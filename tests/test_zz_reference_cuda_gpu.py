"""libsgv_b200 against THE REFERENCE'S OWN CUDA PLUGINS on identical inputs (north_star: "outputs match the reference's own JIT-compiled ops").

oracle/build_ref.py compiles the reference's src/torch_utils/ops/{upfirdn2d,bias_act}.{cpp,cu} UNMODIFIED for sm_100a, and
oracle/ref_cuda_golden.py ran those plugins on a B200 on the cases below and stored their outputs in tests/golden/reference_cuda_cases.npz
(inputs are regenerated from per-case seeds; large outputs are kept as a fixed sample).  Both sides expose the same two pybind-style
entry points (`upfirdn2d(x, f, upx, upy, downx, downy, padx0, padx1, pady0, pady1, flip, gain)`, `bias_act(x, b, xref, yref, dy, grad, dim,
act, alpha, gain, clamp)`), so the comparison is plugin against plugin.

Bars: upfirdn2d and the piecewise-linear activations accumulate in the same order with FMAs on both sides — expected bit-identical, asserted
to 1e-6 of the output range (a wrong tap or index would be O(1)); transcendental activations 2e-3 because the reference is built with
--use_fast_math (bias_act.py:45) and ours uses the accurate functions.
The same plugins are timed by bench.py where they have been built ("beat this kernel": `reference_cuda_kernels` in the bench line)."""
import numpy as np
import pytest
import torch

from conftest import GOLDEN, rel_err
from oracle import ref_cuda_golden as R
from stylegan_v_b200 import plugin

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def golden():
    return np.load(f'{GOLDEN}/reference_cuda_cases.npz')


def _check_inputs(golden, key, total):
    assert total == pytest.approx(float(golden[key + ':x_sum']), rel=1e-12, abs=1e-9), f'{key}: the seeded inputs differ from those the golden was minted on'


@pytest.mark.parametrize('case', R.FIR_CASES)
def test_upfirdn2d_vs_reference_cuda_kernel(cuda, golden, case):
    key = R.fir_key(R.FIR_CASES.index(case))
    x, f = R.fir_inputs(case, cuda)
    _check_inputs(golden, key, x.double().sum().item())
    got = plugin.upfirdn2d(*R.fir_args(case, x, f))
    assert list(got.shape) == golden[key + ':shape'].tolist()
    got, want = R.sample(got), golden[key + ':y']
    assert rel_err(torch.from_numpy(got), torch.from_numpy(want)) <= 1e-6
    if not np.array_equal(got, want):
        print(f'note: not bit-identical for {case}: max |diff| = {np.abs(got - want).max():.3e}')


@pytest.mark.parametrize('act', list(R.ACTS))
@pytest.mark.parametrize('cl', [False, True])
def test_bias_act_vs_reference_cuda_kernel(cuda, golden, act, cl):
    key = R.bias_act_key(act, cl)
    x, dy, b = R.bias_act_inputs(act, cl, cuda)
    _check_inputs(golden, key, x.double().sum().item() + dy.double().sum().item() + b.double().sum().item())
    nil = torch.empty([0], device=cuda)
    alpha, gain, clamp, exact = R.bias_act_params(act)
    tol = 1e-6 if exact else 2e-3
    # forward
    want = torch.from_numpy(golden[key + ':y']).to(cuda).contiguous(memory_format=torch.channels_last if cl else torch.contiguous_format)
    got = plugin.bias_act(x, b, nil, nil, nil, 0, 1, R.ACTS[act], alpha, gain, clamp)
    assert rel_err(got, want) <= tol
    # first-order gradient kernel (grad = 1): xref = x, yref = the reference's y, as BiasActCudaGrad passes them (bias_act.py:164-170)
    got1 = plugin.bias_act(dy, b, x, want, nil, 1, 1, R.ACTS[act], alpha, gain, clamp)
    assert rel_err(torch.from_numpy(R.sample(got1)), torch.from_numpy(golden[key + ':g1'])) <= tol
    # second order (grad = 2) for the activations that have one
    if act in R.SECOND_ORDER:
        got2 = plugin.bias_act(dy, b, x, want, dy, 2, 1, R.ACTS[act], alpha, gain, clamp)
        assert rel_err(torch.from_numpy(R.sample(got2)), torch.from_numpy(golden[key + ':g2'])) <= 5e-3
