"""Native Generator / Discriminator modules (stylegan_v_b200/networks.py, SynthesisNetwork's any-order-differentiable `unfused` mode)
against goldens minted from the UNMODIFIED reference (oracle/make_goldens.py): state-dict compatibility, logits, first-order
gradients, and the two second-order quantities of the training loop — R1 (loss.py:151-160) and path length (loss.py:101-119).
CPU tensors take the standard-PyTorch-ops formulation of the drop-in ops, so this pins structure and arithmetic order; the CUDA
kernels behind the same modules are checked in tests/test_networks_gpu.py."""
import numpy as np
import pytest
import torch

from conftest import load_golden, rel_err
from oracle import synthesis_ref as sr
from stylegan_v_b200.networks import Discriminator, Generator, MappingNetwork
from stylegan_v_b200.ops import conv2d_gradfix
from stylegan_v_b200.synthesis import SynthesisNetwork


def _t(a):
    return torch.from_numpy(np.asarray(a))


def make_discriminator(g, meta):
    D = Discriminator(c_dim=0, img_resolution=meta['img_resolution'], channel_base=meta['channel_base'], channel_max=meta['channel_max'],
                      num_frames_per_video=meta['num_frames_per_video'], max_num_frames=meta['max_num_frames'], concat_res=meta['concat_res'],
                      num_frames_div_factor=meta['num_frames_div_factor'], mbstd_group_size=meta['mbstd_group_size'],
                      mapping_layers=meta['mapping_layers'])
    sd = {k[2:]: _t(g[k]) for k in g.files if k.startswith('p:')}
    assert set(sd) == set(D.state_dict()), set(sd) ^ set(D.state_dict())      # same keys as the reference's state_dict
    D.load_state_dict(sd)
    return D


def cos_sim(a, b):
    a, b = a.detach().double().cpu().reshape(-1), b.detach().double().cpu().reshape(-1)
    return float((a @ b) / (a.norm() * b.norm()).clamp_min(1e-300))


def discriminator_checks(D, g, dev, tol, tol2, weights_only_cos=None):
    """weights_only_cos: on TF32 hardware compare gradient DIRECTIONS of the weight tensors only.  Bias / embedding gradients of this tiny
    network are ill-conditioned sums: the R1 term reaches them only through the minibatch-std layer's sqrt(var + 1e-8) with a group of 2
    (the rest of D is piecewise linear in its input), i.e. through the few elements whose two group members nearly tie."""
    if weights_only_cos is not None:
        return _discriminator_checks_tf32(D, g, dev, tol, tol2, weights_only_cos)
    names = [k[2:] for k in g.files if k.startswith('g:')]
    img = _t(g['img']).to(dev).requires_grad_(True)
    t = _t(g['t']).to(dev)
    D.train()
    logits = D(img, torch.zeros(len(t), 0, device=dev), t)['image_logits']
    assert rel_err(logits, _t(g['logits'])) < tol
    P = dict(D.named_parameters())
    loss = torch.nn.functional.softplus(-logits).mean()
    grads = torch.autograd.grad(loss, [P[n] for n in names], retain_graph=True)
    for n, a in zip(names, grads):
        assert rel_err(a, _t(g['g:' + n])) < tol2, n
    with conv2d_gradfix.no_weight_gradients():
        r1_grads, = torch.autograd.grad(logits.sum(), [img], create_graph=True)
    assert rel_err(r1_grads, _t(g['r1_grads'])) < tol2
    loss_r1 = (r1_grads.square().sum([1, 2, 3]) * 0.5).view(-1, t.shape[1]).mean(dim=1).mean()
    names2 = [k[3:] for k in g.files if k.startswith('r1:')]
    grads2 = torch.autograd.grad(loss_r1, [P[n] for n in names2], allow_unused=True)
    for n, a in zip(names2, grads2):
        assert a is not None, n
        assert rel_err(a, _t(g['r1:' + n])) < tol2, n


def _discriminator_checks_tf32(D, g, dev, tol, tol2, min_cos):
    names = [k[2:] for k in g.files if k.startswith('g:') and k.endswith('.weight') and 'const_embed' not in k]
    img = _t(g['img']).to(dev).requires_grad_(True)
    t = _t(g['t']).to(dev)
    D.train()
    logits = D(img, torch.zeros(len(t), 0, device=dev), t)['image_logits']
    assert rel_err(logits, _t(g['logits'])) < tol
    P = dict(D.named_parameters())
    grads = torch.autograd.grad(torch.nn.functional.softplus(-logits).mean(), [P[n] for n in names], retain_graph=True)
    for n, a in zip(names, grads):
        assert cos_sim(a, _t(g['g:' + n])) > min_cos, (n, cos_sim(a, _t(g['g:' + n])))
    with conv2d_gradfix.no_weight_gradients():
        r1_grads, = torch.autograd.grad(logits.sum(), [img], create_graph=True)
    assert rel_err(r1_grads, _t(g['r1_grads'])) < tol2
    assert cos_sim(r1_grads, _t(g['r1_grads'])) > min_cos
    loss_r1 = (r1_grads.square().sum([1, 2, 3]) * 0.5).view(-1, t.shape[1]).mean(dim=1).mean()
    names2 = [k[3:] for k in g.files if k.startswith('r1:') and k.endswith('.weight') and 'const_embed' not in k]
    grads2 = torch.autograd.grad(loss_r1, [P[n] for n in names2], allow_unused=True)
    for n, a in zip(names2, grads2):
        assert a is not None, n
        assert cos_sim(a, _t(g['r1:' + n])) > min_cos - 0.04, (n, cos_sim(a, _t(g['r1:' + n])))


def test_discriminator_vs_reference_golden():
    g, meta = load_golden('discriminator_tiny.npz')
    D = make_discriminator(g, meta)
    discriminator_checks(D, g, torch.device('cpu'), 1e-5, 1e-4)


def test_mapping_network_vs_reference_golden():
    g, _ = load_golden('discriminator_tiny.npz')
    M = MappingNetwork(z_dim=16, c_dim=0, w_dim=24, num_ws=5, num_layers=2)
    sd = {k[2:]: _t(g[k]) for k in g.files if k.startswith('m:')}
    assert set(sd) == set(M.state_dict())
    M.load_state_dict(sd)
    M.train()
    z = _t(g['map_z'])
    ws = M(z, torch.zeros(4, 0))
    assert rel_err(ws, _t(g['map_ws'])) < 1e-6
    assert rel_err(M.w_avg, _t(g['map_w_avg_after'])) < 1e-6                     # moving average after that one update (layers.py:86-88)
    M.eval()
    assert rel_err(M(z, torch.zeros(4, 0), truncation_psi=0.7, truncation_cutoff=3), _t(g['map_ws_trunc'])) < 1e-6


def make_synthesis(g, meta):
    cfg = sr.SynthesisConfig(**meta)
    net = SynthesisNetwork.from_config(cfg)
    net.load_state_dict({k[2:]: _t(g[k]) for k in g.files if k.startswith('p:')})
    return net, cfg


def test_synthesis_unfused_mode_vs_reference_golden():
    """The layer-by-layer formulation on the drop-in ops reproduces the reference network (train and eval mode) and all gradients."""
    g, meta = load_golden('synthesis_tiny.npz')
    net, _ = make_synthesis(g, meta)
    ws, t, mz = _t(g['ws']).requires_grad_(True), _t(g['t']), _t(g['motion_z'])
    net.train()
    img = net(ws, t, motion_z=mz)
    assert rel_err(img, _t(g['img_train'])) < 1e-5
    names = [k[2:] for k in g.files if k.startswith('g:')]
    P = dict(net.named_parameters())
    grads = torch.autograd.grad(img, [ws] + [P[n] for n in names], _t(g['dimg']))
    assert rel_err(grads[0], _t(g['d_ws'])) < 1e-5
    for n, a in zip(names, grads[1:]):
        assert rel_err(a, _t(g['g:' + n])) < 1e-4, n
    net.eval()
    with torch.no_grad():
        assert rel_err(net(ws, t, motion_z=mz), _t(g['img_eval'])) < 1e-6


def path_length_checks(net, g, dev, tol):
    ws, t, mz = _t(g['ws']).to(dev).requires_grad_(True), _t(g['t']).to(dev), _t(g['motion_z']).to(dev)
    net.train()
    img = net(ws, t, motion_z=mz, unfused=True)
    with conv2d_gradfix.no_weight_gradients():
        pl_grads, = torch.autograd.grad([(img * _t(g['noise']).to(dev)).sum()], [ws], create_graph=True)
    assert rel_err(pl_grads, _t(g['pl_grads'])) < tol
    pl_lengths = pl_grads.square().sum(2).mean(1).sqrt()
    assert rel_err(pl_lengths, _t(g['pl_lengths'])) < tol
    penalty = (pl_lengths - 0.5).square()
    names = [k[2:] for k in g.files if k.startswith('g:')]
    P = dict(net.named_parameters())
    grads = torch.autograd.grad((img[:, 0, 0, 0] * 0 + (penalty * 2.0).repeat_interleave(t.shape[1])).mean(), [P[n] for n in names])
    for n, a in zip(names, grads):
        assert rel_err(a, _t(g['g:' + n])) < 10 * tol, n


def test_path_length_second_order_vs_reference_golden():
    g, meta = load_golden('path_length_tiny.npz')
    net, _ = make_synthesis(g, meta)
    path_length_checks(net, g, torch.device('cpu'), 1e-4)


def test_generator_wraps_mapping_and_synthesis():
    torch.manual_seed(0)
    G = Generator(z_dim=16, w_dim=64, img_resolution=32, channel_base=1024, channel_max=32, motion_z_dim=32, motion_v_dim=32, time_enc_dim=16)
    z, t = torch.randn(2, 16), torch.tensor([[0.0, 3.0], [10.0, 40.5]])
    img = G(z, torch.zeros(2, 0), t)
    assert img.shape == (4, 3, 32, 32) and torch.isfinite(img).all()
    assert {k.split('.')[0] for k in G.state_dict()} == {'synthesis', 'mapping'}


def test_mixed_precision_mode_vs_reference_golden():
    """num_fp16_res / conv_clamp (the reference's default training precision, train.py:173-174): fp16 activations + clamp 256 in the
    high-resolution blocks of G and D, fp16 pre-normalisation of weights and styles (networks.py:50-52), fused_modconv rule of
    networks.py:232 — on the unfused ops, against the reference run the same way on CPU."""
    g, meta = load_golden('mixed_precision_g_tiny.npz')
    cfg = sr.SynthesisConfig(**meta['G'])
    kw = dict(w_dim=cfg.w_dim, img_resolution=cfg.img_resolution, channel_base=cfg.channel_base, channel_max=cfg.channel_max,
              motion_z_dim=cfg.motion_z_dim, motion_v_dim=cfg.motion_v_dim, time_enc_dim=cfg.time_enc_dim)
    net = SynthesisNetwork(num_fp16_res=meta['num_fp16_res'], conv_clamp=meta['conv_clamp'], **kw)
    net.load_state_dict({k[2:]: _t(g[k]) for k in g.files if k.startswith('p:')})
    assert [getattr(net, f'b{r}').use_fp16 for r in net.block_resolutions] == [False, False, True, True]
    ws, t, mz = _t(g['ws']).requires_grad_(True), _t(g['t']), _t(g['motion_z'])
    net.train()
    img = net(ws, t, motion_z=mz)
    assert img.dtype == torch.float32 and rel_err(img, _t(g['img_train'])) < 2e-3           # fp16 activations: half-ulp flips allowed
    names = [k[2:] for k in g.files if k.startswith('g:')]
    P = dict(net.named_parameters())
    grads = torch.autograd.grad(img, [ws] + [P[n] for n in names], _t(g['dimg']))
    assert rel_err(grads[0], _t(g['d_ws'])) < 1e-2
    for n, a in zip(names, grads[1:]):
        assert rel_err(a, _t(g['g:' + n])) < 1e-2, n
    net.eval()
    with torch.no_grad():
        assert rel_err(net(ws, t, motion_z=mz), _t(g['img_eval'])) < 2e-3
        assert rel_err(net(ws[:1], t[:1], motion_z=mz[:1]), _t(g['img_eval_b1'])) < 2e-3
    g, meta = load_golden('mixed_precision_d_tiny.npz')
    md = meta['D']
    D = Discriminator(c_dim=0, img_resolution=md['img_resolution'], channel_base=md['channel_base'], channel_max=md['channel_max'],
                      num_frames_per_video=md['num_frames_per_video'], max_num_frames=md['max_num_frames'], concat_res=md['concat_res'],
                      num_frames_div_factor=md['num_frames_div_factor'], mbstd_group_size=md['mbstd_group_size'], mapping_layers=md['mapping_layers'],
                      num_fp16_res=meta['num_fp16_res'], conv_clamp=meta['conv_clamp'])
    D.load_state_dict({k[2:]: _t(g[k]) for k in g.files if k.startswith('d:')})
    assert [getattr(D, f'b{r}').use_fp16 for r in D.block_resolutions] == [True, True, False]
    x = _t(g['d_img']).requires_grad_(True)
    D.train()
    logits = D(x, torch.zeros(2, 0), _t(g['d_t']))['image_logits']
    assert rel_err(logits, _t(g['d_logits'])) < 2e-3
    gin, gw = torch.autograd.grad(logits.sum(), [x, D.b8.conv0.weight])
    assert rel_err(gin, _t(g['d_gin'])) < 1e-2 and rel_err(gw, _t(g['d_gw_b8_conv0'])) < 1e-2


def test_modules_from_reference_cfg_nodes():
    """Generator / Discriminator built from the reference's own config nodes (stylegan-v.yaml values) have the reference's state-dict keys and shapes."""
    g, meta = load_golden('loss_phases_tiny.npz')
    cfg = sr.SynthesisConfig(**meta['G'])
    G = Generator.from_reference_cfg(cfg.reference_generator_cfg(), img_resolution=cfg.img_resolution, channel_base=cfg.channel_base,
                                     channel_max=cfg.channel_max, mapping_layers=2)
    want = {k[2:]: tuple(g[k].shape) for k in g.files if k.startswith('g:')}
    assert {k: tuple(v.shape) for k, v in G.state_dict().items()} == want
    md = meta['D']
    dcfg = dict(sampling=dict(num_frames_per_video=md['num_frames_per_video'], max_num_frames=md['max_num_frames'], type='random'),
                concat_res=md['concat_res'], num_frames_div_factor=md['num_frames_div_factor'], dummy_c=False)
    D = Discriminator.from_reference_cfg(dcfg, img_resolution=md['img_resolution'], channel_base=md['channel_base'], channel_max=md['channel_max'],
                                         mbstd_group_size=md['mbstd_group_size'], mapping_layers=md['mapping_layers'])
    want = {k[2:]: tuple(g[k].shape) for k in g.files if k.startswith('d:')}
    assert {k: tuple(v.shape) for k, v in D.state_dict().items()} == want
    noisy = Generator.from_reference_cfg(dict(cfg.reference_generator_cfg(), use_noise=True), img_resolution=32, channel_base=1024, channel_max=32)
    assert 'synthesis.b8.conv0.noise_strength' in noisy.state_dict() and tuple(noisy.synthesis.b16.conv1.noise_const.shape) == (16, 16)
    bad = dict(cfg.reference_generator_cfg(), input=dict(type='const'))
    with pytest.raises(NotImplementedError):
        Generator.from_reference_cfg(bad, img_resolution=32)
