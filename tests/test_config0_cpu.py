"""BASELINE configs[0] — "64x64 SynthesisNetwork forward, 1 latent x 1 frame, CPU (torch_utils.ops custom CUDA disabled) — plumbing":
  (1) the UNMODIFIED reference SynthesisNetwork gives the same image on its own ops and, in a fresh interpreter, on the drop-in ops
      installed by stylegan_v_b200.install.install_ops() (INTEGRATION.md route 1);
  (2) the native SynthesisNetwork, loaded with the reference's state dict, reproduces that image on CPU.
(1) and (2) run the reference tree itself and are skipped where it is absent; (2) is also checked against the reference's stored image
(tests/golden/config0_64.npz, oracle/make_goldens.py::gen_config0) everywhere."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT, load_golden, rel_err
from oracle import ref_loader

_SCRIPT = r'''
import sys, numpy as np, torch
sys.path.insert(0, {root!r})
use_dropin = {dropin}
if use_dropin:
    from stylegan_v_b200.install import install_ops
    install_ops()
from oracle import ref_loader, synthesis_ref as sr
ref_loader._install_omegaconf_stub()
for p in ({ref_root!r} + '/src', {ref_root!r}):
    if p not in sys.path: sys.path.insert(0, p)
import importlib
networks = importlib.import_module('training.networks')
ops_mod = sys.modules['src.torch_utils.ops.upfirdn2d'].__name__
cfg = sr.SynthesisConfig(img_resolution=64)
torch.manual_seed(0)
S = networks.SynthesisNetwork(w_dim=cfg.w_dim, img_resolution=64, img_channels=3, channel_base=cfg.channel_base, channel_max=cfg.channel_max,
                              cfg=ref_loader.to_cfg(cfg.reference_generator_cfg())).eval()
g = torch.Generator().manual_seed(1)
ws = torch.randn(1, S.num_ws, cfg.w_dim, generator=g)
t = torch.zeros(1, 1)
mz = torch.randn(1, sr.max_traj_len(cfg, 0.0), cfg.motion_z_dim, generator=g)
with torch.no_grad():
    img = S(ws, t=t, c=torch.zeros(1, 0), motion_z=mz)
out = dict(img=img.numpy(), ws=ws.numpy(), mz=mz.numpy(), ops=np.frombuffer(ops_mod.encode(), dtype=np.uint8))
if not use_dropin:
    out.update({{'p:' + k: v.numpy() for k, v in S.state_dict().items()}})
np.savez({out!r}, **out)
'''


def _run(tmp_path, dropin):
    out = str(tmp_path / f'cfg0_{int(dropin)}.npz')
    code = _SCRIPT.format(root=ROOT, ref_root=ref_loader.REF_ROOT, dropin=dropin, out=out)
    env = dict(os.environ, OMP_NUM_THREADS='4')
    subprocess.run([sys.executable, '-c', code], check=True, env=env, cwd=ROOT, timeout=600)
    return np.load(out)


@pytest.mark.skipif(not ref_loader.available(), reason='reference tree not present')
def test_config0_reference_network_on_dropin_ops_and_native_network(tmp_path):
    ref = _run(tmp_path, False)
    drop = _run(tmp_path, True)
    assert bytes(ref['ops']).decode().startswith('src.torch_utils.ops')            # reference ops in the first interpreter
    assert bytes(drop['ops']).decode().startswith('stylegan_v_b200.ops')           # ours in the second
    img_ref, img_drop = torch.from_numpy(ref['img']), torch.from_numpy(drop['img'])
    assert img_ref.shape == (1, 3, 64, 64) and torch.isfinite(img_ref).all()
    assert rel_err(img_drop, img_ref) < 1e-6                                       # same standard-PyTorch-ops formulation on CPU
    # native network with the reference's parameters
    from oracle import synthesis_ref as sr
    from stylegan_v_b200.synthesis import SynthesisNetwork
    net = SynthesisNetwork.from_config(sr.SynthesisConfig(img_resolution=64)).eval()
    sd = {k[2:]: torch.from_numpy(ref[k]) for k in ref.files if k.startswith('p:')}
    assert set(sd) == set(net.state_dict())
    net.load_state_dict(sd)
    with torch.no_grad():
        img = net(torch.from_numpy(ref['ws']), torch.zeros(1, 1), motion_z=torch.from_numpy(ref['mz']))
    assert rel_err(img, img_ref) < 1e-5


def test_config0_native_network_vs_reference_golden():
    """(2) without the reference tree: the native SynthesisNetwork at 64x64, built from torch seed 0, against the image the reference's
    SynthesisNetwork computed on CPU with the same parameters and inputs."""
    from oracle import synthesis_ref as sr
    from stylegan_v_b200.synthesis import SynthesisNetwork
    g, _ = load_golden('config0_64.npz')
    torch.manual_seed(0)
    net = SynthesisNetwork.from_config(sr.SynthesisConfig(img_resolution=64)).eval()
    assert sum(float(v.double().abs().sum()) for v in net.state_dict().values()) == pytest.approx(float(g['param_sum']), rel=1e-12), \
        'the seeded initialisation of SynthesisNetwork changed: re-mint tests/golden/config0_64.npz (python -m oracle.make_goldens gen_config0)'
    with torch.no_grad():
        img = net(torch.from_numpy(g['ws']), torch.zeros(1, 1), motion_z=torch.from_numpy(g['mz']))
    assert img.shape == (1, 3, 64, 64) and rel_err(img, torch.from_numpy(g['img'])) < 1e-5
