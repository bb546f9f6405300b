"""ORACLE (test infrastructure only).  Mints tests/golden/*.npz from the UNMODIFIED reference.

Run in the build container only (needs /root/reference):   python -m oracle.make_goldens

Every vector is produced by the reference's own Python code on CPU — i.e. the `impl='ref'`
branch of its ops (upfirdn2d.py:162-164, bias_act.py:87-89), F.conv2d for the contractions
(conv2d_gradfix.py:51-52) and the reference network classes — with fixed seeds.  The reference's
test-suite has no vectors for this path (SURVEY.md §4), so these files are the parity pin.
"""
import json
import os
import numpy as np
import torch

from . import ref_loader
from . import synthesis_ref as sr

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'tests', 'golden')

UPFIRDN_CASES = [
    # (N, C, H, W, filter, up, down, padding, flip, gain, channels_last)
    dict(shape=[2, 3, 9, 9], f=[1, 3, 3, 1], up=1, down=1, padding=1, flip=False, gain=4),          # G up-layer FIR (2h+1 -> 2h)
    dict(shape=[2, 3, 8, 8], f=[1, 3, 3, 1], up=2, down=1, padding=[2, 1, 2, 1], flip=False, gain=4),  # img upsample2d
    dict(shape=[1, 4, 8, 8], f=[1, 3, 3, 1], up=1, down=2, padding=1, flip=False, gain=1),          # D skip downsample
    dict(shape=[1, 4, 8, 8], f=[1, 3, 3, 1], up=1, down=1, padding=2, flip=False, gain=1),          # D blur before stride-2 conv
    dict(shape=[2, 2, 8, 8], f=[1, 3, 3, 1], up=1, down=1, padding=2, flip=True, gain=4),           # backward of case 0
    dict(shape=[1, 2, 7, 5], f=[[1, 2, 3], [4, 5, 6]], up=[2, 3], down=[3, 2], padding=[1, 2, 0, 3], flip=False, gain=1.5),
    dict(shape=[1, 2, 7, 5], f=[[1, 2, 3], [4, 5, 6]], up=[2, 3], down=[3, 2], padding=[1, 2, 0, 3], flip=True, gain=1.5),
    dict(shape=[1, 3, 10, 12], f=[1, 3, 3, 1], up=1, down=1, padding=[-1, 2, 1, -2], flip=False, gain=1),   # negative padding = crop
    dict(shape=[1, 2, 6, 6], f=None, up=2, down=1, padding=0, flip=False, gain=1),                  # identity filter
    dict(shape=[1, 2, 16, 16], f='sym6', up=2, down=1, padding=[6, 5, 6, 5], flip=False, gain=4),   # separable 12-tap (augment.py path)
    dict(shape=[1, 2, 16, 16], f='sym6', up=1, down=2, padding=[5, 5, 5, 5], flip=True, gain=1),
    dict(shape=[2, 8, 9, 9], f=[1, 3, 3, 1], up=1, down=1, padding=1, flip=False, gain=4, channels_last=True),
    dict(shape=[1, 5, 6, 7], f=[1, 2, 1], up=2, down=2, padding=[1, 1, 1, 1], flip=False, gain=2, channels_last=True),
    dict(shape=[1, 1, 1, 1], f=[1, 3, 3, 1], up=1, down=1, padding=[2, 1, 2, 1], flip=False, gain=1),  # minimal extent
]
SYM6 = [0.015404109327027373, 0.0034907120842174702, -0.11799011114819057, -0.048311742585633, 0.4910559419267466, 0.787641141030194]


def _filter(ref, spec):
    if spec is None:
        return None
    if spec == 'sym6':
        taps = np.asarray(SYM6 + SYM6[::-1])
        return ref.upfirdn2d.setup_filter(taps)      # >= 8 taps -> separable (upfirdn2d.py:100-101)
    return ref.upfirdn2d.setup_filter(spec)


def gen_upfirdn2d(ref):
    out = {}
    meta = []
    for i, c in enumerate(UPFIRDN_CASES):
        g = torch.Generator().manual_seed(100 + i)
        x = torch.randn(c['shape'], generator=g, dtype=torch.float64)
        if c.get('channels_last'):
            x = x.contiguous(memory_format=torch.channels_last)
        f = _filter(ref, c['f'])
        x.requires_grad_(True)
        y = ref.upfirdn2d.upfirdn2d(x, f, up=c['up'], down=c['down'], padding=c['padding'], flip_filter=c['flip'], gain=c['gain'], impl='ref')
        dy = torch.randn(y.shape, generator=g, dtype=torch.float64)
        dx, = torch.autograd.grad(y, x, dy)
        out[f'c{i}_x'] = x.detach().numpy()
        out[f'c{i}_y'] = y.detach().numpy()
        out[f'c{i}_dy'] = dy.numpy()
        out[f'c{i}_dx'] = dx.numpy()
        if f is not None:
            out[f'c{i}_f'] = f.numpy()
        meta.append({k: v for k, v in c.items() if k != 'f'} | {'has_f': f is not None})
    out['meta'] = np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)
    np.savez_compressed(os.path.join(OUT, 'upfirdn2d_cases.npz'), **out)


def gen_bias_act(ref):
    out = {}
    meta = []
    i = 0
    for act in ref.bias_act.activation_funcs.keys():
        for (gain, clamp, alpha, use_b, dim, shape) in [
            (None, None, None, True, 1, [2, 5, 4, 3]),
            (0.7, 0.9, 0.3, True, 1, [2, 5, 4, 3]),
            (2.0, None, None, False, 1, [3, 7]),
            (None, 0.5, None, True, 0, [4, 6]),
        ]:
            g = torch.Generator().manual_seed(200 + i)
            x = (torch.randn(shape, generator=g, dtype=torch.float64) * 2).requires_grad_(True)
            b = torch.randn(shape[dim], generator=g, dtype=torch.float64).requires_grad_(True) if use_b else None
            y = ref.bias_act.bias_act(x, b, dim=dim, act=act, alpha=alpha, gain=gain, clamp=clamp, impl='ref')
            dy = torch.randn(shape, generator=g, dtype=torch.float64).requires_grad_(True)
            ins = [x] + ([b] if use_b else [])
            grads = torch.autograd.grad(y, ins, dy, create_graph=True)
            ddx = torch.randn(shape, generator=g, dtype=torch.float64)
            # second order: d(<dx, ddx>)/d(dy) and /d(x)
            g2 = torch.autograd.grad(grads[0], [dy, x], ddx, allow_unused=True)
            out[f'c{i}_x'] = x.detach().numpy()
            if use_b:
                out[f'c{i}_b'] = b.detach().numpy()
                out[f'c{i}_db'] = grads[1].detach().numpy()
            out[f'c{i}_y'] = y.detach().numpy()
            out[f'c{i}_dy'] = dy.detach().numpy()
            out[f'c{i}_dx'] = grads[0].detach().numpy()
            out[f'c{i}_ddx'] = ddx.numpy()
            out[f'c{i}_g2_dy'] = g2[0].numpy()
            out[f'c{i}_g2_x'] = (g2[1] if g2[1] is not None else torch.zeros(shape, dtype=torch.float64)).numpy()
            meta.append(dict(act=act, gain=gain, clamp=clamp, alpha=alpha, use_b=use_b, dim=dim, shape=shape))
            i += 1
    out['meta'] = np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)
    np.savez_compressed(os.path.join(OUT, 'bias_act_cases.npz'), **out)


MODCONV_CASES = [
    dict(N=2, I=8, O=6, H=6, k=3, up=1, demod=True, fused=False),
    dict(N=2, I=8, O=6, H=6, k=3, up=1, demod=True, fused=True),
    dict(N=2, I=8, O=6, H=5, k=3, up=2, demod=True, fused=False),
    dict(N=2, I=8, O=6, H=5, k=3, up=2, demod=True, fused=True),
    dict(N=3, I=8, O=3, H=6, k=1, up=1, demod=False, fused=False),      # ToRGB
    dict(N=2, I=32, O=32, H=16, k=3, up=1, demod=True, fused=False),     # tensor-core friendly sizes
    dict(N=2, I=32, O=32, H=8, k=3, up=2, demod=True, fused=False),
    dict(N=2, I=64, O=3, H=16, k=1, up=1, demod=False, fused=False),
]


def gen_modconv(ref):
    out = {}
    f = ref.upfirdn2d.setup_filter([1, 3, 3, 1])
    for i, c in enumerate(MODCONV_CASES):
        g = torch.Generator().manual_seed(300 + i)
        x = torch.randn(c['N'], c['I'], c['H'], c['H'], generator=g).requires_grad_(True)
        w = torch.randn(c['O'], c['I'], c['k'], c['k'], generator=g).requires_grad_(True)
        s = (torch.randn(c['N'], c['I'], generator=g) + 1).requires_grad_(True)
        y = ref.networks.modulated_conv2d(x=x, weight=w, styles=s, up=c['up'], padding=c['k'] // 2, resample_filter=f,
                                          demodulate=c['demod'], flip_weight=(c['up'] == 1), fused_modconv=c['fused'])
        dy = torch.randn(y.shape, generator=g)
        dx, dw, ds = torch.autograd.grad(y, [x, w, s], dy)
        for k, v in dict(x=x, w=w, s=s, y=y, dy=dy, dx=dx, dw=dw, ds=ds).items():
            out[f'c{i}_{k}'] = v.detach().numpy()
    out['f'] = f.numpy()
    out['meta'] = np.frombuffer(json.dumps(MODCONV_CASES).encode(), dtype=np.uint8)
    np.savez_compressed(os.path.join(OUT, 'modconv_cases.npz'), **out)


RESAMPLE_CASES = [
    dict(N=1, I=4, O=5, H=8, k=3, up=1, down=1, flip_weight=True),
    dict(N=1, I=4, O=5, H=8, k=3, up=2, down=1, flip_weight=False),
    dict(N=1, I=4, O=5, H=8, k=3, up=1, down=2, flip_weight=True),
    dict(N=1, I=4, O=5, H=8, k=1, up=1, down=2, flip_weight=True),
    dict(N=1, I=4, O=5, H=8, k=1, up=2, down=1, flip_weight=True),
    dict(N=2, I=3, O=8, H=8, k=1, up=1, down=1, flip_weight=True),
]


def gen_conv2d_resample(ref):
    out = {}
    f = ref.upfirdn2d.setup_filter([1, 3, 3, 1])
    for i, c in enumerate(RESAMPLE_CASES):
        g = torch.Generator().manual_seed(400 + i)
        x = torch.randn(c['N'], c['I'], c['H'], c['H'], generator=g).requires_grad_(True)
        w = torch.randn(c['O'], c['I'], c['k'], c['k'], generator=g).requires_grad_(True)
        y = ref.conv2d_resample.conv2d_resample(x=x, w=w, f=f, up=c['up'], down=c['down'], padding=c['k'] // 2, flip_weight=c['flip_weight'])
        dy = torch.randn(y.shape, generator=g)
        dx, dw = torch.autograd.grad(y, [x, w], dy)
        for k, v in dict(x=x, w=w, y=y, dy=dy, dx=dx, dw=dw).items():
            out[f'c{i}_{k}'] = v.detach().numpy()
    out['f'] = f.numpy()
    out['meta'] = np.frombuffer(json.dumps(RESAMPLE_CASES).encode(), dtype=np.uint8)
    np.savez_compressed(os.path.join(OUT, 'conv2d_resample_cases.npz'), **out)


TINY = dict(img_resolution=32, w_dim=64, channel_base=1024, channel_max=32, motion_z_dim=32, motion_v_dim=32, time_enc_dim=16)


def gen_synthesis(ref):
    cfg = sr.SynthesisConfig(**TINY)
    rcfg = ref_loader.to_cfg(cfg.reference_generator_cfg())
    torch.manual_seed(0)
    S = ref.networks.SynthesisNetwork(w_dim=cfg.w_dim, img_resolution=cfg.img_resolution, img_channels=3,
                                      channel_base=cfg.channel_base, channel_max=cfg.channel_max, cfg=rcfg)
    # give biases non-trivial values so they are exercised
    g = torch.Generator().manual_seed(1)
    with torch.no_grad():
        for n, p in S.named_parameters():
            if n.endswith('.bias') and 'affine' not in n:
                p.copy_(torch.randn(p.shape, generator=g) * 0.1)
    B, Fr = 2, 3
    ws = torch.randn(B, S.num_ws, cfg.w_dim, generator=g).requires_grad_(True)
    t = torch.tensor([[0.0, 5.25, 9.0], [100.5, 101.0, 130.75]])
    c = torch.zeros(B, 0)
    L = sr.max_traj_len(cfg, float(t.max()))
    mz = torch.randn(B, L, cfg.motion_z_dim, generator=g)
    out = {}
    S.train()   # => fused_modconv=False (networks.py:232)
    motion_v = S.motion_encoder(c, t, motion_z=mz)['motion_v']
    img = S(ws, t=t, c=c, motion_z=mz)
    dimg = torch.randn(img.shape, generator=g)
    params = dict(S.named_parameters())
    names = sorted(params.keys())
    grads = torch.autograd.grad(img, [ws] + [params[n] for n in names], dimg)
    S.eval()    # => fused_modconv=True for fp32
    with torch.no_grad():
        img_eval = S(ws, t=t, c=c, motion_z=mz)
    for k, v in S.state_dict().items():
        out['p:' + k] = v.detach().numpy()
    out.update(ws=ws.detach().numpy(), t=t.numpy(), motion_z=mz.numpy(), motion_v=motion_v.detach().numpy(),
               img_train=img.detach().numpy(), img_eval=img_eval.numpy(), dimg=dimg.numpy(), d_ws=grads[0].numpy())
    for n, gr in zip(names, grads[1:]):
        out['g:' + n] = gr.numpy()
    out['meta'] = np.frombuffer(json.dumps(TINY).encode(), dtype=np.uint8)
    np.savez_compressed(os.path.join(OUT, 'synthesis_tiny.npz'), **out)


def gen_synthesis_noise(ref):
    """The reference SynthesisNetwork with use_noise = true (networks.py:119-121,130-134), noise_mode='const', non-zero strengths:
    image + gradients incl. d(noise_strength).  Pins the noise-add of the fused layers (a6)."""
    tiny = dict(TINY, img_resolution=16)
    cfg = sr.SynthesisConfig(**tiny, use_noise=True)
    rcfg = ref_loader.to_cfg(cfg.reference_generator_cfg())
    torch.manual_seed(3)
    S = ref.networks.SynthesisNetwork(w_dim=cfg.w_dim, img_resolution=cfg.img_resolution, img_channels=3,
                                      channel_base=cfg.channel_base, channel_max=cfg.channel_max, cfg=rcfg)
    g = torch.Generator().manual_seed(4)
    with torch.no_grad():
        for n, p in S.named_parameters():
            if n.endswith('.bias') and 'affine' not in n:
                p.copy_(torch.randn(p.shape, generator=g) * 0.1)
            if n.endswith('.noise_strength'):
                p.copy_(torch.randn(p.shape, generator=g) * 0.5)
    B, Fr = 2, 2
    ws = torch.randn(B, S.num_ws, cfg.w_dim, generator=g).requires_grad_(True)
    t = torch.tensor([[0.0, 5.25], [100.5, 130.75]])
    c = torch.zeros(B, 0)
    mz = torch.randn(B, sr.max_traj_len(cfg, float(t.max())), cfg.motion_z_dim, generator=g)
    S.train()
    img = S(ws, t=t, c=c, motion_z=mz, noise_mode='const')
    dimg = torch.randn(img.shape, generator=g)
    params = dict(S.named_parameters())
    names = sorted(params.keys())
    grads = torch.autograd.grad(img, [ws] + [params[n] for n in names], dimg)
    out = {}
    for k, v in S.state_dict().items():
        out['p:' + k] = v.detach().numpy()
    out.update(ws=ws.detach().numpy(), t=t.numpy(), motion_z=mz.numpy(), img_train=img.detach().numpy(), dimg=dimg.numpy(), d_ws=grads[0].numpy())
    for n, gr in zip(names, grads[1:]):
        out['g:' + n] = gr.numpy()
    out['meta'] = np.frombuffer(json.dumps(dict(tiny, use_noise=True)).encode(), dtype=np.uint8)
    np.savez_compressed(os.path.join(OUT, 'synthesis_noise_tiny.npz'), **out)


TINY_D = dict(img_resolution=32, channel_base=1024, channel_max=32, num_frames_per_video=3, max_num_frames=1024, concat_res=16,
              num_frames_div_factor=2, mbstd_group_size=2, mapping_layers=2)


def gen_discriminator(ref):
    """Reference Discriminator (networks.py:580-673) on a tiny config: logits, first-order parameter gradients of the Dmain loss terms
    and the R1 double-backward (loss.py:151-160), plus the 2-layer Generator mapping network."""
    d = TINY_D
    dcfg = ref_loader.to_cfg(dict(sampling=dict(num_frames_per_video=d['num_frames_per_video'], max_num_frames=d['max_num_frames'], type='random'),
                                  concat_res=d['concat_res'], num_frames_div_factor=d['num_frames_div_factor'], dummy_c=False))
    torch.manual_seed(3)
    D = ref.networks.Discriminator(c_dim=0, img_resolution=d['img_resolution'], img_channels=3, channel_base=d['channel_base'],
                                   channel_max=d['channel_max'], cfg=dcfg, mapping_kwargs=dict(num_layers=d['mapping_layers']),
                                   epilogue_kwargs=dict(mbstd_group_size=d['mbstd_group_size']))
    g = torch.Generator().manual_seed(4)
    with torch.no_grad():
        for n, p in D.named_parameters():
            if n.endswith('.bias'):
                p.copy_(torch.randn(p.shape, generator=g) * 0.1)
    B, Fr, R = 2, d['num_frames_per_video'], d['img_resolution']
    img = torch.randn(B * Fr, 3, R, R, generator=g).requires_grad_(True)
    t = torch.tensor([[0.0, 5.0, 9.0], [100.0, 101.0, 131.0]])
    c = torch.zeros(B, 0)
    D.train()
    logits = D(img, c, t)['image_logits']
    params = dict(D.named_parameters())
    names = sorted(params.keys())
    loss = torch.nn.functional.softplus(-logits).mean()                                 # loss.py:146 (Dreal term)
    grads = torch.autograd.grad(loss, [params[n] for n in names], retain_graph=True, allow_unused=True)
    # R1: gradient of the logits w.r.t. the images, differentiated again w.r.t. the parameters (loss.py:151-160; gamma = 1)
    with ref.conv2d_gradfix.no_weight_gradients():
        r1_grads, = torch.autograd.grad(logits.sum(), [img], create_graph=True)
    r1_penalty = r1_grads.square().sum([1, 2, 3])
    loss_r1 = (r1_penalty * 0.5).view(-1, Fr).mean(dim=1).mean()
    grads_r1 = torch.autograd.grad(loss_r1, [params[n] for n in names], allow_unused=True)
    out = {}
    for k, v in D.state_dict().items():
        out['p:' + k] = v.detach().numpy()
    out.update(img=img.detach().numpy(), t=t.numpy(), logits=logits.detach().numpy(), r1_grads=r1_grads.detach().numpy(),
               r1_penalty=r1_penalty.detach().numpy())
    for n, a, b in zip(names, grads, grads_r1):
        if a is not None:
            out['g:' + n] = a.numpy()
        if b is not None:
            out['r1:' + n] = b.numpy()
    # Generator mapping network (layers.py:22-104): z -> ws, train mode updates w_avg
    torch.manual_seed(5)
    M = ref.layers.MappingNetwork(z_dim=16, c_dim=0, w_dim=24, num_ws=5, num_layers=2)
    z = torch.randn(4, 16, generator=g)
    for k, v in M.state_dict().items():
        out['m:' + k] = v.detach().numpy().copy()
    M.train()
    ws = M(z, torch.zeros(4, 0))
    out.update(map_z=z.numpy(), map_ws=ws.detach().numpy(), map_w_avg_after=M.w_avg.numpy().copy())
    M.eval()
    out['map_ws_trunc'] = M(z, torch.zeros(4, 0), truncation_psi=0.7, truncation_cutoff=3).detach().numpy()
    out['meta'] = np.frombuffer(json.dumps(TINY_D).encode(), dtype=np.uint8)
    np.savez_compressed(os.path.join(OUT, 'discriminator_tiny.npz'), **out)


def gen_path_length(ref):
    """Path-length regularisation through the reference synthesis network (loss.py:101-119): pl_grads = d(img * noise).sum() / d ws with
    create_graph, penalty gradient w.r.t. parameters — a second-order quantity of the hot path."""
    cfg = sr.SynthesisConfig(**TINY)
    rcfg = ref_loader.to_cfg(cfg.reference_generator_cfg())
    torch.manual_seed(0)
    S = ref.networks.SynthesisNetwork(w_dim=cfg.w_dim, img_resolution=cfg.img_resolution, img_channels=3,
                                      channel_base=cfg.channel_base, channel_max=cfg.channel_max, cfg=rcfg)
    g = torch.Generator().manual_seed(11)
    B = 2
    ws = torch.randn(B, S.num_ws, cfg.w_dim, generator=g).requires_grad_(True)
    t = torch.tensor([[3.0, 20.5, 40.0], [7.25, 8.0, 500.0]])
    c = torch.zeros(B, 0)
    mz = torch.randn(B, sr.max_traj_len(cfg, float(t.max())), cfg.motion_z_dim, generator=g)
    S.train()
    img = S(ws, t=t, c=c, motion_z=mz)
    noise = torch.randn(img.shape, generator=g) / np.sqrt(img.shape[2] * img.shape[3])
    with ref.conv2d_gradfix.no_weight_gradients():
        pl_grads, = torch.autograd.grad([(img * noise).sum()], [ws], create_graph=True)
    pl_lengths = pl_grads.square().sum(2).mean(1).sqrt()
    pl_penalty = (pl_lengths - 0.5).square()
    params = dict(S.named_parameters())
    names = sorted(n for n in params if not n.startswith('motion_encoder'))
    grads = torch.autograd.grad((img[:, 0, 0, 0] * 0 + (pl_penalty * 2.0).repeat_interleave(t.shape[1])).mean(), [params[n] for n in names], allow_unused=True)
    out = {'p:' + k: v.detach().numpy() for k, v in S.state_dict().items()}
    out.update(ws=ws.detach().numpy(), t=t.numpy(), motion_z=mz.numpy(), noise=noise.numpy(), pl_grads=pl_grads.detach().numpy(),
               pl_lengths=pl_lengths.detach().numpy())
    for n, a in zip(names, grads):
        if a is not None:
            out['g:' + n] = a.numpy()
    out['meta'] = np.frombuffer(json.dumps(TINY).encode(), dtype=np.uint8)
    np.savez_compressed(os.path.join(OUT, 'path_length_tiny.npz'), **out)


def gen_mixed_precision(ref):
    """The reference's mixed-precision mode (train.py:173-174: num_fp16_res highest resolutions in fp16, conv_clamp 256) on the tiny
    synthesis network (fp16 in the 16^2 and 32^2 blocks) and the tiny discriminator (fp16 in its 32^2 and 16^2 blocks), CPU."""
    cfg = sr.SynthesisConfig(**TINY)
    rcfg = ref_loader.to_cfg(cfg.reference_generator_cfg())
    torch.manual_seed(0)
    S = ref.networks.SynthesisNetwork(w_dim=cfg.w_dim, img_resolution=cfg.img_resolution, img_channels=3, channel_base=cfg.channel_base,
                                      channel_max=cfg.channel_max, cfg=rcfg, num_fp16_res=2, conv_clamp=256)
    g = torch.Generator().manual_seed(31)
    with torch.no_grad():
        for n, p in S.named_parameters():
            if n.endswith('.bias') and 'affine' not in n:
                p.copy_(torch.randn(p.shape, generator=g) * 0.1)
    B = 2
    ws = torch.randn(B, S.num_ws, cfg.w_dim, generator=g).requires_grad_(True)
    t = torch.tensor([[0.0, 5.25], [100.5, 130.75]])
    c = torch.zeros(B, 0)
    mz = torch.randn(B, sr.max_traj_len(cfg, float(t.max())), cfg.motion_z_dim, generator=g)
    S.train()
    img = S(ws, t=t, c=c, motion_z=mz)
    dimg = torch.randn(img.shape, generator=g)
    keep = ['b32.conv0.weight', 'b16.conv1.bias', 'b8.conv1.weight', 'b32.torgb.weight']
    P = dict(S.named_parameters())
    grads = torch.autograd.grad(img, [ws] + [P[n] for n in keep], dimg)
    S.eval()
    with torch.no_grad():
        img_eval = S(ws, t=t, c=c, motion_z=mz)
        img_eval_b1 = S(ws[:1], t=t[:1], c=c[:1], motion_z=mz[:1])          # batch of one latent: fused_modconv rule of networks.py:232
    out = {'p:' + k: v.detach().numpy().copy() for k, v in S.state_dict().items()}
    out.update(ws=ws.detach().numpy(), t=t.numpy(), motion_z=mz.numpy(), dimg=dimg.numpy(), img_train=img.detach().numpy(),
               img_eval=img_eval.numpy(), img_eval_b1=img_eval_b1.numpy(), d_ws=grads[0].numpy())
    for n, a in zip(keep, grads[1:]):
        out['g:' + n] = a.numpy()
    out['meta'] = np.frombuffer(json.dumps(dict(G=TINY, num_fp16_res=2, conv_clamp=256)).encode(), dtype=np.uint8)
    np.savez_compressed(os.path.join(OUT, 'mixed_precision_g_tiny.npz'), **out)          # G and D in two files: each stays below 1 MB
    # discriminator
    d = TINY_D
    dcfg = ref_loader.to_cfg(dict(sampling=dict(num_frames_per_video=3, max_num_frames=d['max_num_frames'], type='random'),
                                  concat_res=d['concat_res'], num_frames_div_factor=d['num_frames_div_factor'], dummy_c=False))
    torch.manual_seed(3)
    D = ref.networks.Discriminator(c_dim=0, img_resolution=d['img_resolution'], img_channels=3, channel_base=d['channel_base'],
                                   channel_max=d['channel_max'], cfg=dcfg, mapping_kwargs=dict(num_layers=d['mapping_layers']),
                                   epilogue_kwargs=dict(mbstd_group_size=d['mbstd_group_size']), num_fp16_res=2, conv_clamp=256)
    dimg_in = torch.randn(6, 3, 32, 32, generator=g).requires_grad_(True)
    dt = torch.tensor([[0.0, 5.0, 9.0], [100.0, 101.0, 131.0]])
    D.train()
    # the time-difference embedding (1024 rows) is read only at the differences of dt: zero the rows this clip never reads (their
    # gradient is zero), which leaves every output unchanged and keeps the file small
    emb = D.time_encoder.const_embed.weight
    used, = torch.autograd.grad(D(dimg_in, torch.zeros(2, 0), dt)['image_logits'].sum(), [emb])
    with torch.no_grad():
        emb[used.abs().sum(1) == 0] = 0
    logits = D(dimg_in, torch.zeros(2, 0), dt)['image_logits']
    gin, gw = torch.autograd.grad(logits.sum(), [dimg_in, D.b8.conv0.weight])
    out = {'d:' + k: v.detach().numpy().copy() for k, v in D.state_dict().items()}
    out.update(d_img=dimg_in.detach().numpy(), d_t=dt.numpy(), d_logits=logits.detach().numpy(), d_gin=gin.numpy(), d_gw_b8_conv0=gw.numpy())
    out['meta'] = np.frombuffer(json.dumps(dict(D=TINY_D, num_fp16_res=2, conv_clamp=256)).encode(), dtype=np.uint8)
    np.savez_compressed(os.path.join(OUT, 'mixed_precision_d_tiny.npz'), **out)


AUG_CASES = [
    # name, constructor kwargs (train.py:271-279 'bgc' = blit + geom + color, all multipliers 1), p, input shape
    dict(name='bgc', kw=dict(xflip=1, rotate90=1, xint=1, scale=1, rotate=1, aniso=1, xfrac=1, brightness=1, contrast=1, lumaflip=1, hue=1, saturation=1), p=0.8, shape=[4, 3, 32, 32]),
    dict(name='bgc_clip', kw=dict(xflip=1, rotate90=1, xint=1, scale=1, rotate=1, aniso=1, xfrac=1, brightness=1, contrast=1, lumaflip=1, hue=1, saturation=1), p=1.0, shape=[3, 9, 24, 40]),
    dict(name='blit', kw=dict(xflip=1, rotate90=1, xint=1), p=1.0, shape=[5, 3, 16, 16]),
    dict(name='color_gray', kw=dict(brightness=1, contrast=1, lumaflip=1), p=1.0, shape=[3, 1, 16, 16]),
    dict(name='filter_noise_cutout', kw=dict(imgfilter=1, noise=1, cutout=1), p=1.0, shape=[3, 3, 32, 32]),
    dict(name='bgc_debug', kw=dict(xflip=1, rotate90=1, xint=1, scale=1, rotate=1, aniso=1, xfrac=1, brightness=1, contrast=1, lumaflip=1, hue=1, saturation=1,
                                   imgfilter=1, noise=1, cutout=1), p=1.0, shape=[2, 3, 32, 32], debug_percentile=0.7),
]


def gen_augment(ref):
    """Reference AugmentPipe (augment.py:117-436) outputs for fixed generator seeds: the whole random-number stream is part of the contract."""
    out = {}
    g = torch.Generator().manual_seed(41)
    for case in AUG_CASES:
        pipe = ref.augment.AugmentPipe(**case['kw'])
        pipe.p.copy_(torch.as_tensor(case['p']))
        x = torch.randn(case['shape'], generator=g).requires_grad_(True)
        torch.manual_seed(1234)
        y = pipe(x, debug_percentile=case.get('debug_percentile'))
        dy = torch.randn(y.shape, generator=g)
        dx, = torch.autograd.grad(y, [x], dy)
        out[case['name'] + ':x'] = x.detach().numpy()
        out[case['name'] + ':y'] = y.detach().numpy()
        out[case['name'] + ':dy'] = dy.numpy()
        out[case['name'] + ':dx'] = dx.numpy()
        if case['name'] == 'bgc':
            for k, v in pipe.state_dict().items():
                out['buf:' + k] = v.numpy().copy()
    out['meta'] = np.frombuffer(json.dumps(AUG_CASES).encode(), dtype=np.uint8)
    np.savez_compressed(os.path.join(OUT, 'augment_cases.npz'), **out)


def gen_loss_phases(ref):
    """The reference's StyleGAN2Loss.accumulate_gradients (loss.py:73-173) on tiny reference G and D, one call per phase with fixed RNG
    state: per-parameter gradient sums and norms (+ a few full tensors) for Gmain, Dmain and Dreg (R1)."""
    cfg = sr.SynthesisConfig(**TINY)
    gcfg = ref_loader.to_cfg(cfg.reference_generator_cfg())
    d = TINY_D
    dcfg = ref_loader.to_cfg(dict(sampling=dict(num_frames_per_video=3, max_num_frames=d['max_num_frames'], type='random'),
                                  concat_res=d['concat_res'], num_frames_div_factor=d['num_frames_div_factor'], dummy_c=False))
    torch.manual_seed(21)
    G = ref.networks.Generator(c_dim=0, w_dim=cfg.w_dim, img_resolution=cfg.img_resolution, img_channels=3, cfg=gcfg,
                               mapping_kwargs=dict(num_layers=2),
                               synthesis_kwargs=dict(channel_base=cfg.channel_base, channel_max=cfg.channel_max))
    D = ref.networks.Discriminator(c_dim=0, img_resolution=d['img_resolution'], img_channels=3, channel_base=d['channel_base'],
                                   channel_max=d['channel_max'], cfg=dcfg, mapping_kwargs=dict(num_layers=d['mapping_layers']),
                                   epilogue_kwargs=dict(mbstd_group_size=d['mbstd_group_size']))
    loss = ref.loss.StyleGAN2Loss(cfg=None, device=torch.device('cpu'), G_mapping=G.mapping, G_synthesis=G.synthesis, D=D,
                                  style_mixing_prob=0.0, r1_gamma=0.5, pl_weight=0.0)
    g = torch.Generator().manual_seed(22)
    B, Fr, R = 2, 3, cfg.img_resolution
    real = torch.randn(B, Fr, 3, R, R, generator=g).clamp(-1, 1)
    real_t = torch.tensor([[0.0, 4.0, 20.0], [30.0, 31.0, 33.0]])
    gen_t = torch.tensor([[2.0, 10.0, 11.0], [500.0, 516.0, 530.0]])
    z = torch.randn(B, cfg.w_dim, generator=g)
    c = torch.zeros(B, 0)
    out = {'g:' + k: v.detach().numpy().copy() for k, v in G.state_dict().items()}     # copies: w_avg is updated in place below
    out.update({'d:' + k: v.detach().numpy().copy() for k, v in D.state_dict().items()})
    out.update(real=real.numpy(), real_t=real_t.numpy(), gen_t=gen_t.numpy(), z=z.numpy())
    G.train(); D.train()
    for phase, module, gain in [('Gmain', G, 1), ('Dmain', D, 1), ('Dreg', D, 16)]:
        G.requires_grad_(module is G); D.requires_grad_(module is D)
        for p in module.parameters():
            p.grad = None
        torch.manual_seed(100)                                   # motion noise z ~ randn inside G.synthesis (motion.py:83)
        loss.accumulate_gradients(phase=phase, real_img=real, real_c=c, real_t=real_t, gen_z=z, gen_c=c, gen_t=gen_t, sync=True, gain=gain)
        stats = {}
        for n, p in module.named_parameters():
            if p.grad is not None:
                stats[n] = [float(p.grad.double().sum()), float(p.grad.double().norm())]
        out['stats:' + phase] = np.frombuffer(json.dumps(stats).encode(), dtype=np.uint8)
        keep = ['synthesis.b16.conv0.weight', 'mapping.fc1.weight', 'synthesis.b32.torgb.bias'] if module is G else ['b32.conv1.weight', 'b4.out.weight', 'b16.skip.weight']
        for n in keep:
            out[f'grad:{phase}:{n}'] = dict(module.named_parameters())[n].grad.numpy().copy()
    out['w_avg_after'] = G.mapping.w_avg.numpy().copy()
    # the same Dmain phase with the ADA pipe in front of D, video-consistent (loss.py:58-70): generator stream = motion noise, then the
    # pipe's draws for the generated clip, then for the real clip
    loss.cfg = ref_loader.to_cfg(dict(model=dict(loss_kwargs=dict(video_consistent_aug=True)), sampling=dict(num_frames_per_video=3)))
    loss.augment_pipe = ref.augment.AugmentPipe(**AUG_CASES[0]['kw'])
    loss.augment_pipe.p.copy_(torch.as_tensor(0.6))
    G.requires_grad_(False); D.requires_grad_(True)
    for p in D.parameters():
        p.grad = None
    torch.manual_seed(100)
    loss.accumulate_gradients(phase='Dmain', real_img=real, real_c=c, real_t=real_t, gen_z=z, gen_c=c, gen_t=gen_t, sync=True, gain=1)
    stats = {n: [float(p.grad.double().sum()), float(p.grad.double().norm())] for n, p in D.named_parameters() if p.grad is not None}
    out['stats:Dmain_aug'] = np.frombuffer(json.dumps(stats).encode(), dtype=np.uint8)
    out['grad:Dmain_aug:b32.conv1.weight'] = D.b32.conv1.weight.grad.numpy().copy()
    out['meta'] = np.frombuffer(json.dumps(dict(G=TINY, D=TINY_D, r1_gamma=0.5, aug=AUG_CASES[0]['kw'], aug_p=0.6)).encode(), dtype=np.uint8)
    np.savez_compressed(os.path.join(OUT, 'loss_phases_tiny.npz'), **out)


NET64_G = dict(img_resolution=64, w_dim=64, channel_base=4096, channel_max=64, motion_z_dim=32, motion_v_dim=32, time_enc_dim=32)
NET64_D = dict(img_resolution=64, channel_base=4096, channel_max=64, num_frames_per_video=3, max_num_frames=1024, concat_res=16,
               num_frames_div_factor=2, mbstd_group_size=2, mapping_layers=2)
NET64_G_NAMES = ['synthesis.b64.conv1.weight', 'synthesis.b32.conv0.weight', 'synthesis.b8.conv1.weight', 'synthesis.b64.torgb.weight',
                 'synthesis.b16.conv1.bias', 'mapping.fc1.weight', 'synthesis.motion_encoder.conv.0.weight']
NET64_D_NAMES = ['b64.conv0.weight', 'b64.conv1.weight', 'b32.skip.weight', 'b16.conv0.weight', 'b4.conv.weight', 'b4.out.weight', 'b64.fromrgb.weight']
LOSS32_G = dict(img_resolution=32, w_dim=64, channel_base=2048, channel_max=64, motion_z_dim=32, motion_v_dim=32, time_enc_dim=32)
LOSS32_D = dict(NET64_D, img_resolution=32, channel_base=2048)
SAMPLE = 4096


def seeded_modules(gk, dk):
    """The project's own Generator / Discriminator for the configs gk / dk, initialised from torch seed 0, every bias (but the affines')
    drawn from seed 1 in name order.  Goldens minted on these parameters do not have to store them."""
    from stylegan_v_b200.networks import Generator, Discriminator
    cfg = sr.SynthesisConfig(**gk)
    torch.manual_seed(0)
    G = Generator.from_reference_cfg(cfg.reference_generator_cfg(), img_resolution=cfg.img_resolution, channel_base=cfg.channel_base,
                                     channel_max=cfg.channel_max, mapping_layers=2)
    D = Discriminator.from_reference_cfg(d_cfg(dk), img_resolution=dk['img_resolution'], channel_base=dk['channel_base'],
                                         channel_max=dk['channel_max'], mbstd_group_size=dk['mbstd_group_size'], mapping_layers=dk['mapping_layers'])
    g = torch.Generator().manual_seed(1)
    with torch.no_grad():
        for m in (G, D):
            for n, p in sorted(m.named_parameters()):
                if n.endswith('.bias') and 'affine' not in n:
                    p.copy_(torch.randn(p.shape, generator=g) * 0.1)
    return G, D


def d_cfg(dk):
    return dict(sampling=dict(num_frames_per_video=dk['num_frames_per_video'], max_num_frames=dk['max_num_frames'], type='random'),
                concat_res=dk['concat_res'], num_frames_div_factor=dk['num_frames_div_factor'], dummy_c=False)


def param_sum(G, D):
    """sum |p| over both state dicts in float64: tells a changed initialisation of the project's modules from a changed kernel."""
    return float(sum(v.double().abs().sum() for m in (G, D) for v in m.state_dict().values()))


def sample(a, dtype=np.float64):
    """A fixed sample of SAMPLE elements of a (all of it when smaller)."""
    a = a.detach().double().cpu().contiguous().reshape(-1).numpy().astype(dtype)
    if a.size <= SAMPLE:
        return a
    return a[np.sort(np.random.default_rng(a.size).choice(a.size, SAMPLE, replace=False))]


def reference_gd(ref, gk, dk, Gp, Dp):
    """The reference Generator / Discriminator for gk / dk carrying the parameters of the project's modules Gp / Dp."""
    cfg = sr.SynthesisConfig(**gk)
    G = ref.networks.Generator(c_dim=0, w_dim=cfg.w_dim, img_resolution=cfg.img_resolution, img_channels=3, cfg=ref_loader.to_cfg(cfg.reference_generator_cfg()),
                               mapping_kwargs=dict(num_layers=2), synthesis_kwargs=dict(channel_base=cfg.channel_base, channel_max=cfg.channel_max)).train()
    D = ref.networks.Discriminator(c_dim=0, img_resolution=dk['img_resolution'], img_channels=3, channel_base=dk['channel_base'], channel_max=dk['channel_max'],
                                   cfg=ref_loader.to_cfg(d_cfg(dk)), mapping_kwargs=dict(num_layers=dk['mapping_layers']),
                                   epilogue_kwargs=dict(mbstd_group_size=dk['mbstd_group_size'])).train()
    load_parameters(G, Gp)
    load_parameters(D, Dp)
    return G, D


def load_parameters(ref_module, module):
    """Copies the parameters of the project's module into the reference module; the reference keeps its own buffers (FIR filters,
    frequencies, ...), so that those are compared too."""
    missing, unexpected = ref_module.load_state_dict(dict(module.named_parameters()), strict=False)
    buffers = dict(ref_module.named_buffers())
    assert not unexpected and all(k in buffers for k in missing), (unexpected, [k for k in missing if k not in buffers])


def gen_networks_64(ref):
    """The reference Generator + Discriminator (networks.py:370-673) at 64x64, channel_max 64, on CPU (its impl='ref' ops), on the
    parameters of the project's own modules (`seeded_modules`): image, logits of D on the generated clip, and the gradients of the
    softplus(-logits) loss w.r.t. a set of G and D weights.  tests/test_zz_reference_on_dropin_gpu.py runs the same modules on cuda:0."""
    cfg = sr.SynthesisConfig(**NET64_G)
    Gp, Dp = seeded_modules(NET64_G, NET64_D)
    G, D = reference_gd(ref, NET64_G, NET64_D, Gp, Dp)
    g = torch.Generator().manual_seed(2)
    B = 2
    z = torch.randn(B, cfg.w_dim, generator=g)
    t = torch.tensor([[0.0, 5.0, 9.0], [100.0, 116.5, 131.0]])
    c = torch.zeros(B, 0)
    mz = torch.randn(B, sr.max_traj_len(cfg, float(t.max())), cfg.motion_z_dim, generator=g)
    img = G(z, c, t, motion_z=mz)
    logits = D(img, c, t)['image_logits']
    torch.nn.functional.softplus(-logits).mean().backward()
    gp, dp = dict(G.named_parameters()), dict(D.named_parameters())
    out = dict(z=z.numpy(), t=t.numpy(), motion_z=mz.numpy(), img=img.detach().numpy(), logits=logits.detach().numpy(),
               param_sum=np.float64(param_sum(Gp, Dp)))
    out.update({'G:' + n: sample(gp[n].grad) for n in NET64_G_NAMES})
    out.update({'D:' + n: sample(dp[n].grad) for n in NET64_D_NAMES})
    out['meta'] = np.frombuffer(json.dumps(dict(G=NET64_G, D=NET64_D, sample=SAMPLE)).encode(), dtype=np.uint8)
    np.savez_compressed(os.path.join(OUT, 'networks_64.npz'), **out)


def gen_loss_phases_32(ref):
    """The reference's StyleGAN2Loss.accumulate_gradients (loss.py:73-173) for Gmain, Dmain and Dreg (R1, gain 16) at 32x32, channel_max 64,
    on the parameters of the project's own modules (`seeded_modules`), CPU: a fixed float32 sample of every weight gradient of at least 64
    elements.  The motion noise the reference draws inside G (motion.py:83) comes from one CPU generator reseeded per phase and is stored,
    so that a CUDA evaluation can be fed the same draws."""
    Gp, Dp = seeded_modules(LOSS32_G, LOSS32_D)
    G, D = reference_gd(ref, LOSS32_G, LOSS32_D, Gp, Dp)
    loss = ref.loss.StyleGAN2Loss(cfg=None, device=torch.device('cpu'), G_mapping=G.mapping, G_synthesis=G.synthesis, D=D,
                                  style_mixing_prob=0.0, r1_gamma=0.5, pl_weight=0.0)
    g = torch.Generator().manual_seed(2)
    B, Fr, R = 2, 3, LOSS32_G['img_resolution']
    real = torch.randn(B, Fr, 3, R, R, generator=g).clamp(-1, 1)
    real_t = torch.tensor([[0.0, 4.0, 20.0], [30.0, 31.0, 33.0]])
    gen_t = torch.tensor([[2.0, 10.0, 11.0], [500.0, 516.0, 530.0]])
    z = torch.randn(B, LOSS32_G['w_dim'], generator=g)
    c = torch.zeros(B, 0)
    out = dict(real=real.numpy(), real_t=real_t.numpy(), gen_t=gen_t.numpy(), z=z.numpy(), param_sum=np.float64(param_sum(Gp, Dp)))
    randn, draws, gen = torch.randn, [], torch.Generator()

    def recorded_randn(*size, **kw):
        kw.pop('generator', None)
        x = randn(*size, generator=gen, **kw)
        draws.append(x)
        return x
    w0 = G.mapping.w_avg.clone()
    torch.randn = recorded_randn
    try:
        for phase, module, gain in [('Gmain', G, 1), ('Dmain', D, 1), ('Dreg', D, 16)]:
            G.requires_grad_(module is G); D.requires_grad_(module is D)
            for p in module.parameters():
                p.grad = None
            gen.manual_seed(100)
            draws.clear()
            loss.accumulate_gradients(phase=phase, real_img=real, real_c=c, real_t=real_t, gen_z=z, gen_c=c, gen_t=gen_t, sync=True, gain=gain)
            G.mapping.w_avg.copy_(w0)
            assert len(draws) == (0 if phase == 'Dreg' else 1), (phase, len(draws))
            if draws:
                out[f'motion_z:{phase}'] = draws[0].numpy()
            for n, p in module.named_parameters():
                if p.grad is not None and p.grad.numel() >= 64 and not n.endswith('bias'):
                    out[f'{phase}:{n}'] = sample(p.grad, np.float32)
    finally:
        torch.randn = randn
    out['meta'] = np.frombuffer(json.dumps(dict(G=LOSS32_G, D=LOSS32_D, r1_gamma=0.5, sample=SAMPLE)).encode(), dtype=np.uint8)
    np.savez_compressed(os.path.join(OUT, 'loss_phases_32.npz'), **out)


SIGNATURES = {'upfirdn2d': ['setup_filter', 'upfirdn2d', 'filter2d', 'upsample2d', 'downsample2d', '_parse_padding', '_get_filter_size'],
              'bias_act': ['bias_act'], 'conv2d_resample': ['conv2d_resample'], 'conv2d_gradfix': ['conv2d', 'conv_transpose2d', 'no_weight_gradients'],
              'fma': ['fma']}


def gen_signatures(ref):
    """The call signatures of the reference's torch_utils.ops functions that the drop-in ops must keep (tests/test_ops_cpu.py).  Functions
    the reference wraps in misc.profiled_function show `(*args, **kwargs)` and are left out."""
    import inspect
    sigs = {}
    for mod, names in SIGNATURES.items():
        for n in names:
            s = str(inspect.signature(getattr(getattr(ref, mod), n)))
            if s != '(*args, **kwargs)':
                sigs[f'{mod}.{n}'] = s
    out = dict(signatures=np.frombuffer(json.dumps(sigs).encode(), dtype=np.uint8), meta=np.frombuffer(b'{}', dtype=np.uint8))
    np.savez_compressed(os.path.join(OUT, 'reference_signatures.npz'), **out)


def gen_config0(ref):
    """BASELINE configs[0]: the reference SynthesisNetwork at 64x64 (default widths), 1 latent x 1 frame, eval mode, on CPU with its own
    ops, on the parameters of the project's SynthesisNetwork built from torch seed 0 (tests/test_config0_cpu.py rebuilds them)."""
    from stylegan_v_b200.synthesis import SynthesisNetwork
    cfg = sr.SynthesisConfig(img_resolution=64)
    torch.manual_seed(0)
    net = SynthesisNetwork.from_config(cfg)
    S = ref.networks.SynthesisNetwork(w_dim=cfg.w_dim, img_resolution=64, img_channels=3, channel_base=cfg.channel_base, channel_max=cfg.channel_max,
                                      cfg=ref_loader.to_cfg(cfg.reference_generator_cfg())).eval()
    load_parameters(S, net)
    g = torch.Generator().manual_seed(1)
    ws = torch.randn(1, S.num_ws, cfg.w_dim, generator=g)
    mz = torch.randn(1, sr.max_traj_len(cfg, 0.0), cfg.motion_z_dim, generator=g)
    with torch.no_grad():
        img = S(ws, t=torch.zeros(1, 1), c=torch.zeros(1, 0), motion_z=mz)
    out = dict(img=img.numpy(), ws=ws.numpy(), mz=mz.numpy(), param_sum=np.float64(sum(float(v.double().abs().sum()) for v in net.state_dict().values())),
               meta=np.frombuffer(json.dumps(dict(img_resolution=64)).encode(), dtype=np.uint8))
    np.savez_compressed(os.path.join(OUT, 'config0_64.npz'), **out)


def main(only=None):
    os.makedirs(OUT, exist_ok=True)
    ref = ref_loader.load()
    torch.set_num_threads(4)
    if only:            # python -m oracle.make_goldens gen_synthesis_noise ...  (re-mint selected files only)
        for name in only:
            globals()[name](ref)
        return
    gen_upfirdn2d(ref)
    gen_bias_act(ref)
    gen_modconv(ref)
    gen_conv2d_resample(ref)
    gen_synthesis(ref)
    gen_synthesis_noise(ref)
    gen_discriminator(ref)
    gen_path_length(ref)
    gen_loss_phases(ref)
    gen_mixed_precision(ref)
    gen_augment(ref)
    gen_networks_64(ref)
    gen_loss_phases_32(ref)
    gen_signatures(ref)
    gen_config0(ref)
    for fn in sorted(os.listdir(OUT)):
        print(fn, os.path.getsize(os.path.join(OUT, fn)))


if __name__ == '__main__':
    import sys
    main(sys.argv[1:])
