"""ORACLE (test infrastructure only).  Mints tests/golden/reference_cuda_cases.npz: the outputs of the REFERENCE'S OWN CUDA plugins
(oracle/build_ref.py, compiled unmodified for sm_100a) on the cases of tests/test_zz_reference_cuda_gpu.py.

    python -m oracle.ref_cuda_golden OUT_DIR     # needs a CUDA device and the plugins under oracle/_ref/ (python -m oracle.build_ref)

The inputs are not stored: every case draws them from its own CPU torch.Generator seed (`fir_inputs`, `bias_act_inputs`); the file keeps
a float64 sum of each input so that a test can tell a changed input stream from a changed kernel.  Outputs are stored in full where the
next kernel call consumes them (the forward of bias_act is the `yref` of its gradient kernels) and otherwise as a fixed sample of
SAMPLE elements (`sample`), which keeps the file small."""
import json
import os
import sys

import numpy as np
import torch

FIR_CASES = [
    # shape, filter taps (outer product of 1-D taps), up, down, (px0, px1, py0, py1), flip, gain, channels_last
    ([2, 8, 33, 33], [1, 3, 3, 1], 1, 1, (1, 1, 1, 1), False, 4.0, False),        # G up-layer FIR (2h+1 -> 2h)
    ([2, 8, 33, 33], [1, 3, 3, 1], 1, 1, (1, 1, 1, 1), False, 4.0, True),
    ([2, 3, 16, 16], [1, 3, 3, 1], 2, 1, (2, 1, 2, 1), False, 4.0, False),        # img upsample2d
    ([2, 16, 32, 32], [1, 3, 3, 1], 1, 1, (2, 2, 2, 2), False, 1.0, False),       # D blur before the stride-2 conv
    ([2, 16, 32, 32], [1, 3, 3, 1], 1, 2, (1, 1, 1, 1), False, 1.0, True),        # D skip down-sampling
    ([1, 4, 20, 24], [1, 3, 3, 1], 1, 1, (2, 2, 2, 2), True, 4.0, False),         # backward of the first case (flipped)
    ([1, 3, 12, 14], [1, 2, 3], 2, 3, (1, 2, 0, 3), False, 1.5, False),           # generic kernel path
    ([1, 3, 12, 14], [1, 3, 3, 1], 1, 1, (-1, 2, 1, -2), False, 1.0, False),      # negative padding = crop
    ([4, 64, 65, 65], [1, 3, 3, 1], 1, 1, (1, 1, 1, 1), False, 4.0, True),        # wide channels_last (TMA kernel on our side)
]

ACTS = {'linear': 1, 'relu': 2, 'lrelu': 3, 'tanh': 4, 'sigmoid': 5, 'elu': 6, 'selu': 7, 'softplus': 8, 'swish': 9}      # bias_act.py:23-33
ALPHA = {'lrelu': 0.2}
SECOND_ORDER = ('tanh', 'sigmoid', 'elu', 'selu', 'softplus', 'swish')          # bias_act.py:23-33 has_2nd_grad
SAMPLE = 2048


def fir_inputs(case, dev):
    """(x, f) of a FIR case on `dev`."""
    shape, taps, up, down, pad, flip, gain, cl = case
    g = torch.Generator().manual_seed(sum(shape))
    x = torch.randn(shape, generator=g).to(dev)
    if cl:
        x = x.contiguous(memory_format=torch.channels_last)
    k = torch.tensor(taps, dtype=torch.float32)
    f = torch.outer(k, k)
    return x, (f / f.sum()).to(dev)


def fir_args(case, x, f):
    shape, taps, up, down, pad, flip, gain, cl = case
    return (x, f, up, up, down, down, pad[0], pad[1], pad[2], pad[3], flip, gain)


def bias_act_inputs(act, cl, dev):
    """(x, dy, b) of a bias_act case on `dev`."""
    g = torch.Generator().manual_seed(ACTS[act])
    x = torch.randn(3, 16, 9, 11, generator=g).to(dev)
    dy = torch.randn(3, 16, 9, 11, generator=g).to(dev)
    if cl:
        x, dy = x.contiguous(memory_format=torch.channels_last), dy.contiguous(memory_format=torch.channels_last)
    return x, dy, torch.randn(16, generator=g).to(dev)


def bias_act_params(act):
    """(alpha, gain, clamp, exact).  Clamp only where the mask is decided by stored values: softplus / swish recompute yref inside the
    gradient kernel (bias_act.cu:113-129), and a fast-math exp can move an element across the clamp threshold on one side only."""
    exact = act in ('linear', 'relu', 'lrelu')
    return ALPHA.get(act, 0.0), 1.3, (2.0 if exact else -1.0), exact


def sample(t):
    """A fixed sample of SAMPLE elements of t in logical (NCHW) order as float64 numpy; all of t when it is smaller."""
    a = t.detach().double().cpu().contiguous().reshape(-1).numpy()
    if a.size <= SAMPLE:
        return a
    return a[np.sort(np.random.default_rng(a.size).choice(a.size, SAMPLE, replace=False))]


def fir_key(i):
    return f'fir{i}'


def bias_act_key(act, cl):
    return f'bias_act:{act}:{int(cl)}'


def mint(out_dir):
    from . import build_ref
    dev = torch.device('cuda', 0)
    up, ba = build_ref.load_plugin('upfirdn2d_plugin'), build_ref.load_plugin('bias_act_plugin')
    assert up is not None and ba is not None, 'build the reference plugins first: python -m oracle.build_ref'
    out = {}
    for i, case in enumerate(FIR_CASES):
        x, f = fir_inputs(case, dev)
        y = up.upfirdn2d(*fir_args(case, x, f))
        torch.cuda.synchronize()
        k = fir_key(i)
        out[k + ':x_sum'] = np.float64(x.double().sum().item())
        out[k + ':shape'] = np.asarray(y.shape, dtype=np.int64)
        out[k + ':y'] = sample(y)
    for act in ACTS:
        for cl in (False, True):
            x, dy, b = bias_act_inputs(act, cl, dev)
            alpha, gain, clamp, _ = bias_act_params(act)
            nil = torch.empty([0], device=dev)
            y = ba.bias_act(x, b, nil, nil, nil, 0, 1, ACTS[act], alpha, gain, clamp)
            g1 = ba.bias_act(dy, b, x, y, nil, 1, 1, ACTS[act], alpha, gain, clamp)
            k = bias_act_key(act, cl)
            out[k + ':x_sum'] = np.float64(x.double().sum().item() + dy.double().sum().item() + b.double().sum().item())
            out[k + ':y'] = y.detach().cpu().contiguous().numpy()          # float32, in full: the yref of the gradient kernels
            out[k + ':g1'] = sample(g1)
            if act in SECOND_ORDER:
                out[k + ':g2'] = sample(ba.bias_act(dy, b, x, y, dy, 2, 1, ACTS[act], alpha, gain, clamp))
            torch.cuda.synchronize()
    props = torch.cuda.get_device_properties(dev)
    out['meta'] = np.frombuffer(json.dumps(dict(device=props.name, torch=torch.__version__, cuda=torch.version.cuda)).encode(), dtype=np.uint8)
    os.makedirs(out_dir, exist_ok=True)
    path = os.path.join(out_dir, 'reference_cuda_cases.npz')
    np.savez_compressed(path, **out)
    print(path, os.path.getsize(path))


if __name__ == '__main__':
    mint(sys.argv[1] if len(sys.argv) > 1 else os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'tests', 'golden'))
