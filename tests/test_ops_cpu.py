"""Host-side logic of the drop-in ops package on CPU: API surface, argument parsing, standard-ops path vs the
golden vectors, conv2d_gradfix custom op (gradients of every order, no_weight_gradients)."""
import inspect

import numpy as np
import pytest
import torch

from conftest import load_golden, rel_err
from stylegan_v_b200.ops import upfirdn2d as U, bias_act as B, conv2d_resample as CR, conv2d_gradfix as CG, fma as FMA


def _t(a):
    return torch.from_numpy(np.asarray(a))


def test_public_surface_matches_reference_signatures():
    sig = lambda f: list(inspect.signature(f).parameters)
    assert sig(U.setup_filter) == ['f', 'device', 'normalize', 'flip_filter', 'gain', 'separable']
    assert sig(U.upfirdn2d) == ['x', 'f', 'up', 'down', 'padding', 'flip_filter', 'gain', 'impl']
    assert sig(U.filter2d) == ['x', 'f', 'padding', 'flip_filter', 'gain', 'impl']
    assert sig(U.upsample2d) == ['x', 'f', 'up', 'padding', 'flip_filter', 'gain', 'impl']
    assert sig(U.downsample2d) == ['x', 'f', 'down', 'padding', 'flip_filter', 'gain', 'impl']
    assert sig(B.bias_act) == ['x', 'b', 'dim', 'act', 'alpha', 'gain', 'clamp', 'impl']
    assert sig(CR.conv2d_resample) == ['x', 'w', 'f', 'up', 'down', 'padding', 'groups', 'flip_weight', 'flip_filter']
    assert sig(CG.conv2d) == ['input', 'weight', 'bias', 'stride', 'padding', 'dilation', 'groups']
    assert sig(CG.conv_transpose2d) == ['input', 'weight', 'bias', 'stride', 'padding', 'output_padding', 'groups', 'dilation']
    assert sig(FMA.fma) == ['a', 'b', 'c']
    assert set(B.activation_funcs) == {'linear', 'relu', 'lrelu', 'tanh', 'sigmoid', 'elu', 'selu', 'softplus', 'swish'}
    assert B.activation_funcs['lrelu'].def_gain == pytest.approx(np.sqrt(2)) and B.activation_funcs['lrelu'].cuda_idx == 3
    assert [B.activation_funcs[k].cuda_idx for k in B.activation_funcs] == list(range(1, 10))


def test_signatures_match_reference_golden():
    """The drop-in ops keep the call signatures of the reference's torch_utils.ops functions (stored by oracle/make_goldens.py::gen_signatures;
    the ones the reference wraps in misc.profiled_function are not stored)."""
    import json
    g, _ = load_golden('reference_signatures.npz')
    theirs = json.loads(bytes(g['signatures']).decode())
    mods = dict(upfirdn2d=U, bias_act=B, conv2d_resample=CR, conv2d_gradfix=CG, fma=FMA)
    assert len(theirs) >= 10
    for name, sig in theirs.items():
        mod, fn = name.split('.')
        assert str(inspect.signature(getattr(mods[mod], fn))) == sig, name


def test_setup_filter():
    f = U.setup_filter([1, 3, 3, 1])
    assert f.shape == (4, 4) and f.dtype == torch.float32
    assert torch.allclose(f, torch.outer(torch.tensor([1., 3, 3, 1]), torch.tensor([1., 3, 3, 1])) / 64)
    assert U.setup_filter(None).shape == (1, 1)
    assert U.setup_filter(list(range(1, 9))).ndim == 1           # >= 8 taps -> separable
    assert U.setup_filter([1, 2, 1], gain=4).sum().item() == pytest.approx(4.0)
    assert torch.equal(U.setup_filter([1, 2, 3], normalize=False, flip_filter=True, separable=True), torch.tensor([3., 2, 1]))


def test_upfirdn2d_standard_ops_path_vs_golden():
    g, meta = load_golden('upfirdn2d_cases.npz')
    for i, m in enumerate(meta):
        x = _t(g[f'c{i}_x']).requires_grad_(True)
        f = _t(g[f'c{i}_f']) if m['has_f'] else None
        y = U.upfirdn2d(x, f, up=m['up'], down=m['down'], padding=m['padding'], flip_filter=m['flip'], gain=m['gain'])
        dx, = torch.autograd.grad(y, x, _t(g[f'c{i}_dy']))
        assert rel_err(y, _t(g[f'c{i}_y'])) < 1e-12 and rel_err(dx, _t(g[f'c{i}_dx'])) < 1e-12


def test_bias_act_standard_ops_path_vs_golden():
    g, meta = load_golden('bias_act_cases.npz')
    for i, m in enumerate(meta):
        x = _t(g[f'c{i}_x'])
        b = _t(g[f'c{i}_b']) if m['use_b'] else None
        y = B.bias_act(x, b, dim=m['dim'], act=m['act'], alpha=m['alpha'], gain=m['gain'], clamp=m['clamp'])
        assert rel_err(y, _t(g[f'c{i}_y'])) < 1e-12


def test_conv2d_resample_vs_golden():
    g, meta = load_golden('conv2d_resample_cases.npz')
    f = _t(g['f'])
    for i, m in enumerate(meta):
        x = _t(g[f'c{i}_x']).requires_grad_(True); w = _t(g[f'c{i}_w']).requires_grad_(True)
        y = CR.conv2d_resample(x=x, w=w, f=f, up=m['up'], down=m['down'], padding=m['k'] // 2, flip_weight=m['flip_weight'])
        dx, dw = torch.autograd.grad(y, [x, w], _t(g[f'c{i}_dy']))
        assert rel_err(y, _t(g[f'c{i}_y'])) < 1e-5 and rel_err(dx, _t(g[f'c{i}_dx'])) < 1e-5 and rel_err(dw, _t(g[f'c{i}_dw'])) < 1e-5


@pytest.mark.parametrize('transpose', [False, True])
def test_conv2d_gradfix_custom_op_all_orders(transpose, monkeypatch):
    monkeypatch.setattr(CG, '_use_custom', lambda x: True)      # exercise the custom op on CPU
    torch.manual_seed(0)
    F = torch.nn.functional
    x = torch.randn(2, 4, 7, 7, dtype=torch.float64, requires_grad=True)
    w = torch.randn(*((4, 5, 3, 3) if transpose else (5, 4, 3, 3)), dtype=torch.float64, requires_grad=True)
    kw = dict(stride=2, padding=1)
    mine = (CG.conv_transpose2d if transpose else CG.conv2d)(x, w, **kw)
    ref = (F.conv_transpose2d if transpose else F.conv2d)(x, w, **kw)
    assert torch.allclose(mine, ref)
    gy = torch.randn_like(ref)
    gm = torch.autograd.grad(mine, [x, w], gy, create_graph=True)
    gr = torch.autograd.grad(ref, [x, w], gy, create_graph=True)
    for a, b in zip(gm, gr):
        assert torch.allclose(a, b, atol=1e-10)
    # second order through both gradient nodes
    vx, vw = torch.randn_like(x), torch.randn_like(w)
    sm = (gm[0] * vx).sum() + (gm[1] * vw).sum()
    s_r = (gr[0] * vx).sum() + (gr[1] * vw).sum()
    g2m = torch.autograd.grad(sm, [x, w])
    g2r = torch.autograd.grad(s_r, [x, w])
    for a, b in zip(g2m, g2r):
        assert torch.allclose(a, b, atol=1e-9)


def test_no_weight_gradients(monkeypatch):
    monkeypatch.setattr(CG, '_use_custom', lambda x: True)
    x = torch.randn(1, 2, 5, 5, requires_grad=True)
    w = torch.randn(3, 2, 3, 3, requires_grad=True)
    with CG.no_weight_gradients():
        assert CG.weight_gradients_disabled
        y = CG.conv2d(x, w, padding=1)
        gx, gw = torch.autograd.grad(y.sum(), [x, w], allow_unused=True)
    assert not CG.weight_gradients_disabled
    assert gx is not None and gw is None


def test_fma_broadcast_grads():
    a = torch.randn(2, 3, 4, 4, dtype=torch.float64, requires_grad=True)
    b = torch.randn(2, 3, 1, 1, dtype=torch.float64, requires_grad=True)
    c = torch.randn(2, 1, 4, 4, dtype=torch.float64, requires_grad=True)
    assert torch.autograd.gradcheck(FMA.fma, (a, b, c))
    assert torch.allclose(FMA.fma(a, b, c), a * b + c)
