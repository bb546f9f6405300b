"""Reference network pickles (torch_utils.persistence, src/torch_utils/persistence.py:118-126,179-203) load into the native modules without the
reference source tree: a snapshot dict {G, D, G_ema} is pickled by the UNMODIFIED reference in one interpreter and read back by
stylegan_v_b200.checkpoint in a fresh interpreter that has no reference module on its path; the native networks must reproduce the
reference's outputs.  Needs a reference tree to WRITE the pickle (build container or the staged copy); skipped elsewhere."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from oracle import ref_loader

_WRITE = r'''
import sys, pickle, numpy as np, torch
sys.path.insert(0, {root!r})
from oracle import ref_loader, synthesis_ref as sr
ref = ref_loader.load()
import importlib
dnnlib = importlib.import_module('src.dnnlib')
cfg = sr.SynthesisConfig(img_resolution=32, w_dim=64, channel_base=1024, channel_max=32, motion_z_dim=32, motion_v_dim=32, time_enc_dim=16)
def easy(d):
    return dnnlib.EasyDict({{k: easy(v) if isinstance(v, dict) else v for k, v in d.items()}})
gcfg = easy(cfg.reference_generator_cfg())
dcfg = easy(dict(sampling=dict(num_frames_per_video=3, max_num_frames=1024, type='random'), concat_res=16, num_frames_div_factor=2, dummy_c=False))
torch.manual_seed(0)
G = ref.networks.Generator(c_dim=0, w_dim=cfg.w_dim, img_resolution=32, img_channels=3, cfg=gcfg, mapping_kwargs=dnnlib.EasyDict(num_layers=2),
                           synthesis_kwargs=dnnlib.EasyDict(channel_base=cfg.channel_base, channel_max=cfg.channel_max)).eval()
D = ref.networks.Discriminator(c_dim=0, img_resolution=32, img_channels=3, channel_base=1024, channel_max=32, cfg=dcfg,
                               mapping_kwargs=dnnlib.EasyDict(num_layers=2), epilogue_kwargs=dnnlib.EasyDict(mbstd_group_size=2)).eval()
g = torch.Generator().manual_seed(1)
z = torch.randn(2, cfg.w_dim, generator=g); t = torch.tensor([[0.0, 5.0, 9.0], [100.0, 116.5, 131.0]]); c = torch.zeros(2, 0)
mz = torch.randn(2, sr.max_traj_len(cfg, 131.0), cfg.motion_z_dim, generator=g)
with torch.no_grad():
    img = G(z, c, t, motion_z=mz)
    logits = D(img, c, t)['image_logits']
with open({pkl!r}, 'wb') as f:
    pickle.dump(dict(G=G, D=D, G_ema=G, training_set_kwargs=dnnlib.EasyDict(resolution=32), augment_pipe=None), f)
np.savez({npz!r}, z=z.numpy(), t=t.numpy(), mz=mz.numpy(), img=img.numpy(), logits=logits.numpy())
'''

_READ = r'''
import sys, numpy as np, torch
sys.path.insert(0, {root!r})
assert not any('reference' in p or 'pyref' in p for p in sys.path)
from stylegan_v_b200 import checkpoint
snap = checkpoint.load_snapshot({pkl!r})
assert not any(m.startswith(('training.', 'src.training', 'src.torch_utils', 'src.dnnlib')) for m in sys.modules), 'the reference must not be imported'
G, D = snap['G_ema'].eval(), snap['D'].eval()
assert type(G).__module__ == 'stylegan_v_b200.networks' and snap['training_set_kwargs']['resolution'] == 32
d = np.load({npz!r})
with torch.no_grad():
    img = G(torch.from_numpy(d['z']), torch.zeros(2, 0), torch.from_numpy(d['t']), motion_z=torch.from_numpy(d['mz']))
    logits = D(torch.from_numpy(d['img']), torch.zeros(2, 0), torch.from_numpy(d['t']))['image_logits']
e1 = float((img - torch.from_numpy(d['img'])).abs().max() / torch.from_numpy(d['img']).abs().max())
e2 = float((logits - torch.from_numpy(d['logits'])).abs().max() / torch.from_numpy(d['logits']).abs().max())
print('ERR', e1, e2)
assert e1 < 1e-5 and e2 < 1e-5, (e1, e2)
'''


@pytest.mark.skipif(not ref_loader.available(), reason='reference tree not present')
def test_reference_snapshot_loads_into_native_modules(tmp_path):
    pkl, npz = str(tmp_path / 'network-snapshot.pkl'), str(tmp_path / 'out.npz')
    env = dict(os.environ, OMP_NUM_THREADS='4')
    r = subprocess.run([sys.executable, '-c', _WRITE.format(root=ROOT, pkl=pkl, npz=npz)], capture_output=True, text=True, env=env, cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    env.pop('SGV_REFERENCE_ROOT', None)
    r = subprocess.run([sys.executable, '-c', _READ.format(root=ROOT, pkl=pkl, npz=npz)], capture_output=True, text=True, env=env, cwd=str(tmp_path), timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]


def test_unpickler_refuses_arbitrary_globals():
    import pickle
    from stylegan_v_b200 import checkpoint
    evil = pickle.dumps(os.system)
    with pytest.raises(pickle.UnpicklingError):
        checkpoint.load_records(evil)
