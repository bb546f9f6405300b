"""Generator + Discriminator and the training-loss phases on the B200 against the reference's own networks (src/training/networks.py:370-673)
and StyleGAN2Loss (src/training/loss.py:73-173) on the same parameters.

tests/golden/networks_64.npz holds what the reference Generator and Discriminator computed on CPU (its `impl='ref'` ops: BASELINE configs[0]
"custom CUDA disabled") on the parameters of this project's modules built from fixed seeds (oracle/make_goldens.py, `seeded_modules`):
the generated clip, D's logits on it, and the gradients of the softplus(-logits) loss w.r.t. a set of G and D weights (a fixed sample of each).
Here the same modules run on cuda:0 with `conv2d_gradfix.enabled = True` like the reference's training loop (training_loop.py:143): the
native synthesis path, and the discriminator on the drop-in FIR / bias_act / contraction kernels of libsgv_b200, in tf32x3 (fp32-grade) and
in the default TF32 mode.  Images, logits and parameter gradients must match the reference; the launch counter proves the library ran.
tests/golden/loss_phases_32.npz holds the reference loss's Gmain, Dmain and R1 gradients at 32x32 in the same way."""
import json

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from oracle import make_goldens as M
from stylegan_v_b200 import train_step as ts

pytestmark = pytest.mark.gpu


def _rel(a, b):
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def test_generator_and_discriminator_cuda_vs_reference_golden(cuda):
    from stylegan_v_b200 import _lib, precision
    from stylegan_v_b200.ops import conv2d_gradfix
    g = np.load(f'{GOLDEN}/networks_64.npz')
    G, D = M.seeded_modules(M.NET64_G, M.NET64_D)
    assert M.param_sum(G, D) == pytest.approx(float(g['param_sum']), rel=1e-12), \
        'the seeded initialisation of the modules changed: re-mint tests/golden/networks_64.npz (python -m oracle.make_goldens gen_networks_64)'
    G, D = G.to(cuda).train(), D.to(cuda).train()
    z, t, mz = (torch.from_numpy(g[k]).to(cuda) for k in ('z', 't', 'motion_z'))
    c = torch.zeros(len(z), 0, device=cuda)
    want = {k: torch.from_numpy(g[k]).double() for k in g.files if k not in ('z', 't', 'motion_z', 'param_sum', 'meta')}
    w0 = G.mapping.w_avg.clone()

    def run():
        for m in (G, D):
            for p in m.parameters():
                p.grad = None
        img = G(z, c, t, motion_z=mz)
        logits = D(img, c, t)['image_logits']
        torch.nn.functional.softplus(-logits).mean().backward()
        G.mapping.w_avg.copy_(w0)             # a train-mode forward moves the average; keep both evaluations on the same state
        gp, dp = dict(G.named_parameters()), dict(D.named_parameters())
        out = dict(img=img.detach().double().cpu(), logits=logits.detach().double().cpu())
        out.update({'G:' + n: torch.from_numpy(M.sample(gp[n].grad)) for n in M.NET64_G_NAMES})
        out.update({'D:' + n: torch.from_numpy(M.sample(dp[n].grad)) for n in M.NET64_D_NAMES})
        return out

    saved = conv2d_gradfix.enabled, torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    conv2d_gradfix.enabled = True                                   # training_loop.py:143
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    report = {}
    try:
        for mode in ('tf32x3', 'tf32'):
            n0 = _lib.launch_count()
            with precision.precision(mode):
                got = run()
            torch.cuda.synchronize()
            report[mode] = dict(launches=_lib.launch_count() - n0, **{k: _rel(got[k], want[k]) for k in want})
            report[mode]['cos'] = {k: float(torch.nn.functional.cosine_similarity(got[k].flatten(), want[k].flatten(), dim=0))
                                   for k in want if k[1] == ':'}
    finally:
        conv2d_gradfix.enabled, torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = saved
    x3, x1 = report['tf32x3'], report['tf32']
    assert x3['launches'] > 100 and x1['launches'] > 100, report     # FIR / bias_act / tcgen05 launches of libsgv_b200, not a library fallback
    # fp32-grade mode: image, logits and every sampled gradient agree with the reference's CPU evaluation
    assert x3['img'] < 1e-4 and x3['logits'] < 1e-4, x3
    for k, v in x3.items():
        if k[1:2] == ':':
            assert v < 2e-3, (k, v)
    # default TF32 mode: north_star tolerance on outputs; gradients by direction (leaky-ReLU slope flips, tests/test_synthesis_gpu.py docstring)
    assert x1['img'] < 3e-3 and x1['logits'] < 5e-3, x1
    for k, cs in x1['cos'].items():
        if not k.endswith('bias'):
            assert cs > 0.99, (k, cs)
    print('G + D at 64x64 vs the reference:', report)


def loss_phase_grads(g, dev):
    """Gmain, Dmain (with the motion noise the reference drew) and Dreg (gain 16) of the modules of loss_phases_32.npz on `dev`:
    {phase:name: fixed sample of the gradient} for the weights the golden holds."""
    G, D = M.seeded_modules(M.LOSS32_G, M.LOSS32_D)
    assert M.param_sum(G, D) == pytest.approx(float(g['param_sum']), rel=1e-12), \
        'the seeded initialisation of the modules changed: re-mint tests/golden/loss_phases_32.npz (python -m oracle.make_goldens gen_loss_phases_32)'
    G, D = G.to(dev).train(), D.to(dev).train()
    real = torch.from_numpy(g['real']).to(dev)
    real = real.view(-1, *real.shape[2:])
    real_t, gen_t, z = (torch.from_numpy(g[k]).to(dev) for k in ('real_t', 'gen_t', 'z'))
    c = torch.zeros(len(z), 0, device=dev)
    r1_gamma = json.loads(bytes(g['meta']).decode())['r1_gamma']
    w0 = G.mapping.w_avg.clone()
    out = {}
    for phase in ('Gmain', 'Dmain', 'Dreg'):
        module = G if phase == 'Gmain' else D
        G.requires_grad_(module is G)
        D.requires_grad_(module is D)
        for p in module.parameters():
            p.grad = None
        if phase == 'Gmain':
            ts.generator_main_loss(G, D, z, c, gen_t, motion_z=torch.from_numpy(g['motion_z:Gmain']).to(dev)).backward()
        elif phase == 'Dmain':
            a, b = ts.discriminator_main_loss(G, D, real, c, real_t, z, c, gen_t, motion_z=torch.from_numpy(g['motion_z:Dmain']).to(dev))
            (a + b).backward()
        else:
            ts.discriminator_r1_loss(D, real, c, real_t, r1_gamma).mul(16).backward()
        G.mapping.w_avg.copy_(w0)
        P = dict(module.named_parameters())
        for k in g.files:
            if k.startswith(phase + ':') and not k.startswith('motion_z'):
                out[k] = torch.from_numpy(M.sample(P[k.split(':', 1)[1]].grad))
    return out


def test_loss_phases_cuda_vs_reference_golden(cuda):
    """SURVEY §2 row 11: the training loss follows the reference's `StyleGAN2Loss`.  Its Gmain, Dmain and R1 phases (the last differentiates
    the discriminator twice) on cuda:0 in the fp32-grade mode must reproduce the reference's CPU gradients for every weight of the network."""
    from stylegan_v_b200 import _lib, precision
    from stylegan_v_b200.ops import conv2d_gradfix
    g = np.load(f'{GOLDEN}/loss_phases_32.npz')
    saved = conv2d_gradfix.enabled, torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    conv2d_gradfix.enabled = True
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        n0 = _lib.launch_count()
        with precision.precision('tf32x3'):
            got = loss_phase_grads(g, cuda)
        torch.cuda.synchronize()
        launches = _lib.launch_count() - n0
    finally:
        conv2d_gradfix.enabled, torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = saved
    assert launches > 300 and len(got) > 40, (launches, len(got))
    worst = {}
    for k, a in got.items():
        b = torch.from_numpy(g[k]).double()
        w = worst.setdefault(k.split(':')[0], dict(rel=0.0, cos=1.0, n=0))
        rel = _rel(a, b)
        if rel >= w['rel']:
            w['rel'], w['worst'] = rel, k
        w['cos'] = min(w['cos'], float(torch.nn.functional.cosine_similarity(a.flatten(), b.flatten(), dim=0)))
        w['n'] += 1
    for phase, w in worst.items():
        # measured on the B200 with the reference modules on these kernels: worst max-norm error 1.7e-4 (Gmain) / 3.9e-4 (Dmain) / 7.7e-5 (Dreg),
        # cosine 1 - 1e-8; the margin is for leaky-ReLU slope flips of a non-bit-equal forward (tests/test_precision_gpu.py)
        assert w['n'] > 5 and w['cos'] > 0.9999 and w['rel'] < 2e-3, (phase, w)
    print('loss phases vs the reference:', worst)
