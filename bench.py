#!/usr/bin/env python
"""Benchmark of the StyleGAN-V synthesis hot path on B200 (contract: see DESIGN.md §Measurement).

    python bench.py --gpus N --steps K --warmup W            # this repo (sm_100a kernels)
    python bench.py --impl reference --gpus N --steps K ...  # the UNMODIFIED reference network on the host cores (its impl='ref' ops)

Workload (BASELINE.json metric "256x256 synthesis frames/sec (fwd+bwd)"): one step = forward + backward of the
256x256 SynthesisNetwork (fmaps 0.5, fp32 storage, random-init weights) on 32 synthetic frames per GPU
(32 latents x 1 frame, BASELINE configs[1] batch), gradients w.r.t. all parameters and ws; for N > 1 ranks each
rank runs its own 32 frames (weak scaling) and gradients are averaged with one NCCL all-reduce per step.
Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FRAMES_PER_GPU = 32
RES = 256
DTYPES = {'tf32': 'tf32 (fp32 storage, TF32 tensor-core products, fp32 accumulate) — the headline; the fp32-grade tf32x3 mode is measured beside it',
          'tf32x3': 'tf32x3 (fp32 storage, hi/lo-split TF32 products hi*hi + lo*hi + hi*lo, fp32 accumulate: fp32-grade, ~1e-6 of fp32)'}


def load_peaks():
    try:
        pk = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
        return dict(hbm_gbs=float(pk['hbm_gbs']), bf16_tflops=float(pk['bf16_tflops']),
                    bf16_tflops_sustained=float(pk.get('bf16_tflops_sustained', pk['bf16_tflops'])), source='measured')
    except Exception:
        return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source='fallback')


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md clocks line)."""
    Q = 'clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index=0):
        self.index, self.samples, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-lms', '100', '-i', str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=['nvidia-smi unavailable'])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for s in self.samples:
            f = [x.strip() for x in s.split(',')]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[2:6]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        sm.sort()
        return dict(sm_mhz=(sm[len(sm) // 2] if sm else None), sm_max_mhz=mx, reasons=sorted(reasons), samples=len(sm))


def _reference_cpu_network(frames):
    """The UNMODIFIED reference SynthesisNetwork (src/training/networks.py:270-366) on CPU tensors: every op takes its `impl='ref'` branch
    (upfirdn2d.py:162-164, bias_act.py:87-89) and conv2d_gradfix defers to F.conv2d (conv2d_gradfix.py:51-52) — BASELINE's "torch_utils.ops
    with custom CUDA disabled".  Imported from /root/reference, or on the GPU box from the hash-verified copy under oracle/_ref/pyref
    (oracle/stage_ref.py).  Returns (step_fn, kind) or None when no reference tree is available."""
    from oracle import ref_loader, synthesis_ref as sr
    if not ref_loader.available():
        return None
    ref = ref_loader.load()
    cfg = sr.SynthesisConfig(img_resolution=RES)
    torch.manual_seed(0)
    S = ref.networks.SynthesisNetwork(w_dim=cfg.w_dim, img_resolution=RES, img_channels=3, channel_base=cfg.channel_base, channel_max=cfg.channel_max,
                                      cfg=ref_loader.to_cfg(cfg.reference_generator_cfg())).train()      # train mode => fused_modconv=False (networks.py:232)
    g = torch.Generator().manual_seed(1)
    ws = torch.randn(frames, S.num_ws, cfg.w_dim, generator=g).requires_grad_(True)
    t = torch.zeros(frames, 1)
    c = torch.zeros(frames, 0)
    mz = torch.randn(frames, sr.max_traj_len(cfg, 0.0), cfg.motion_z_dim, generator=g)
    dimg = torch.randn(frames, 3, RES, RES, generator=g)
    params = list(S.parameters())
    opt = torch.optim.Adam(params, lr=0.0025, betas=(0.0, 0.99), eps=1e-8)     # train.py:192-193

    def step():
        t0 = time.perf_counter()
        opt.zero_grad(set_to_none=True)
        ws.grad = None
        img = S(ws, t=t, c=c, motion_z=mz)
        (img * dimg).sum().backward()
        t1 = time.perf_counter()
        for p in params:                                                        # training_loop.py:381-386
            if p.grad is not None:
                torch.nan_to_num(p.grad, nan=0, posinf=1e5, neginf=-1e5, out=p.grad)
        opt.step()
        t2 = time.perf_counter()
        # the parameter update happens once per 32-frame step: the sampled frames are charged their share of it
        return (t1 - t0) + (t2 - t1) * frames / FRAMES_PER_GPU
    return step, 'reference'


def _port_cpu_network(frames):
    """Fallback when no reference tree is reachable: the oracle port of the same path (kind = 'port')."""
    from oracle import synthesis_ref as sr, train_ref
    cfg = sr.SynthesisConfig(img_resolution=RES)
    P = {k: v.requires_grad_(True) for k, v in sr.init_params(cfg, seed=0).items()}
    g = torch.Generator().manual_seed(1)
    ws = torch.randn(frames, cfg.num_ws, cfg.w_dim, generator=g).requires_grad_(True)
    t = torch.zeros(frames, 1)
    mz = torch.randn(frames, sr.max_traj_len(cfg, 0.0), cfg.motion_z_dim, generator=g)
    names = list(P.keys())
    opt = torch.optim.Adam([P[n] for n in names], lr=0.0025, betas=(0.0, 0.99), eps=1e-8)

    def step():
        t0 = time.perf_counter()
        img = sr.synthesis_forward(P, cfg, ws, t, motion_z=mz, fused_modconv=False)
        grads = torch.autograd.grad(img, [ws] + [P[n] for n in names], torch.ones_like(img), allow_unused=True)
        t1 = time.perf_counter()
        for n, gr in zip(names, grads[1:]):
            P[n].grad = train_ref.nan_to_num_ref(gr) if gr is not None else None
        opt.step()
        t2 = time.perf_counter()
        return (t1 - t0) + (t2 - t1) * frames / FRAMES_PER_GPU
    return step, 'port'


def cpu_reference_step(frames, threads=None):
    """One forward + backward + parameter update of the reference's CPU path on `frames` frames at 256x256 -> (step() -> seconds, kind, threads).
    threads=None: the faster of 32 / 64 / all host threads on one probe step (oversubscribed intra-op pools are SLOWER on these 128-core hosts)."""
    made = _reference_cpu_network(frames) or _port_cpu_network(frames)
    step, kind = made
    ncpu = os.cpu_count() or 1
    if threads is None:
        best = None
        for th in sorted({min(32, ncpu), min(64, ncpu), ncpu}):
            torch.set_num_threads(th)
            sec = step()
            if best is None or sec < best[0]:
                best = (sec, th)
        threads = best[1]
    torch.set_num_threads(threads)
    return step, kind, threads


DUMP_SAMPLE = 1 << 23          # elements kept of an output larger than this (32 MB): a fixed seeded choice of indices, the same in every run


def dump_outputs(out_dir, **arrays):
    """Writes each array as out_dir/<name>.npy in float32.  An array above DUMP_SAMPLE elements is flattened and sampled at DUMP_SAMPLE
    sorted indices drawn from seed 0, so two runs sample the same elements and the dump of the synthesis step stays below 64 MB."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = a.detach().float().cpu().numpy()
        if a.size > DUMP_SAMPLE:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, DUMP_SAMPLE, replace=False))]
        np.save(os.path.join(out_dir, f'{name}.npy'), a)


def run_reference(args):
    """--impl reference: the reference's own implementation of the path on the host cores — the unmodified reference SynthesisNetwork with
    custom CUDA disabled — on a bounded sample (8 of the 32 frames of a step) with the requested steps / warm-up (shortened only if the
    whole run would exceed ~3 minutes)."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    sample_frames = args.ref_frames
    step, kind, threads = cpu_reference_step(sample_frames)
    t_probe = step()
    budget = 150.0
    warmup = max(1, min(args.warmup, int(budget * 0.2 / max(t_probe, 1e-3))))
    steps = max(1, min(args.steps, int(budget * 0.8 / max(t_probe, 1e-3))))
    for _ in range(warmup):
        step()
    times = [step() for _ in range(steps)]
    sec = sum(times) / len(times)
    fps = sample_frames / sec
    what = 'UNMODIFIED reference SynthesisNetwork on CPU tensors (torch_utils.ops impl=\'ref\', F.conv2d; custom CUDA disabled), training mode (fused_modconv=False)' \
        if kind == 'reference' else 'oracle CPU port of the reference path (no reference tree reachable), fused_modconv=False'
    line = dict(metric='synthesis_fwd_bwd_frames_per_sec_256', value=fps, unit='frames/s', n_gpus=args.gpus, steps=steps, warmup=warmup,
                ms_per_step=sec * 1e3, higher_is_better=True, scaling='weak', vs_baseline=None, dtype='f32', data='synthetic', impl='reference',
                config=dict(workload='256x256 SynthesisNetwork forward+backward + fused nan_to_num/Adam update of all parameters, 32 frames/GPU (32 latents x 1 frame), '
                                     'fmaps 0.5, random-init weights', implementation=what, frames_per_step=sample_frames, frames_per_gpu=FRAMES_PER_GPU,
                            note=f'each step = a bounded sample of {sample_frames} of the 32 frames: forward/backward of the sample + its {sample_frames}/32 share of the '
                                 'once-per-step per-tensor nan_to_num + torch.optim.Adam update; frames/s = sample frames / that time'),
                cpu_baseline=dict(value=fps, unit='frames/s', cores=threads, kind=kind,
                                  sample=f'{sample_frames} frames fwd+bwd per step, mean of {steps} steps after {warmup} warm-up; {threads} torch threads of {os.cpu_count()} host cores'),
                e2e=dict(value=fps, unit='frames/s', h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line))


def run_gd_step(args):
    """BASELINE configs[2]: 256x256 G + D training step, forward + backward, no regularisation phases, 3 frames / clip, 16 clips / GPU,
    synthetic frames; phases Gmain + Dmain (loss.py:84-99,121-147) each followed by the all-reduce and the fused Adam (+ EMA) update.
    frames/s = 48 frames per GPU and step / step time (SURVEY.md §8d config 3).  A secondary line: the headline metric stays `synthesis`."""
    import torch.distributed as dist
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    assert torch.cuda.is_available(), 'bench.py needs a CUDA device: the b200 implementation has no CPU path'
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=dev)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    from stylegan_v_b200 import _lib
    from stylegan_v_b200.networks import Generator, Discriminator
    from stylegan_v_b200 import train_step
    from stylegan_v_b200.train_step import TrainingPhases
    if args.fused_d is not None:
        train_step.FUSED_DISCRIMINATOR = bool(args.fused_d)
    args.warmup = max(args.warmup, 3)
    torch.manual_seed(rank)
    B, Fr = 16, 3
    G = Generator(img_resolution=RES).to(dev).train()
    D = Discriminator(img_resolution=RES, mbstd_group_size=4).to(dev).train()
    tp = TrainingPhases(G, D, lr=0.0025, r1_gamma=0.0, pl_weight=0.0, batch_size=B * world, device_step=not args.no_graph)
    h_real = torch.randn(B * Fr, 3, RES, RES).clamp_(-1, 1).pin_memory()
    h_z = torch.randn(B, G.z_dim).pin_memory()
    base = torch.randint(0, 900, (B, 1)).float()
    h_t = (base + torch.tensor([[0.0, 5.0, 9.0]])).pin_memory()
    s_real, s_z, s_t = h_real.to(dev), h_z.to(dev), h_t.to(dev)
    h_out = torch.zeros(2).pin_memory()

    def compute():
        out = tp.step(s_real, s_t, s_z, s_t)
        return torch.stack([out['Gmain'], out['Dmain']])
    graph, graph_launches, s_loss = None, 0, None
    if not args.no_graph and world == 1:
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(2):
                    compute()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            l0 = _lib.launch_count()
            with torch.cuda.graph(graph):
                s_loss = compute()
            graph_launches = _lib.launch_count() - l0
        except Exception as e:
            if rank == 0:
                sys.stderr.write(f'[bench] CUDA graph capture failed ({type(e).__name__}: {e}); eager launches\n')
            graph = None
            torch.cuda.synchronize()

    split = None
    if not args.no_graph and world > 1:
        # N > 1: the gradient exchange sits between the phases, so each main phase (loss + backward into the flat gradient buffer) is its own
        # graph and the NCCL all-reduce + fused update run between the replays.  All ranks must agree on the mode: a rank whose capture failed
        # would otherwise issue a different sequence of collectives.
        zeros_c = torch.zeros(B, 0, device=dev)
        g_part = lambda: tp.backward_gmain(s_z, zeros_c, s_t)
        d_part = lambda: tp.backward_dmain(s_real, zeros_c, s_t, s_z, zeros_c, s_t)
        ok = torch.ones(1, device=dev)
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(2):
                    g_part(); tp.finish_g(); d_part(); tp.finish_d()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            gG, gD = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
            l0 = _lib.launch_count()
            with torch.cuda.graph(gG):
                s_lg = g_part()
            with torch.cuda.graph(gD, pool=gG.pool()):
                s_ld = d_part()
            graph_launches = _lib.launch_count() - l0
            split = (gG, gD, s_lg, s_ld)
        except Exception as e:
            sys.stderr.write(f'[bench] rank {rank}: per-phase CUDA graph capture failed ({type(e).__name__}: {e}); eager launches\n')
            ok.zero_()
            torch.cuda.synchronize()
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if float(ok.item()) == 0:
            split = None

    def step():
        if graph is not None:
            graph.replay()
            return s_loss
        if split is not None:
            gG, gD, s_lg, s_ld = split
            gG.replay(); tp.finish_g(); gD.replay(); tp.finish_d()
            return torch.stack([s_lg, s_ld])
        return compute()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = _lib.launch_count()
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), _lib.launch_count() - l0
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms_total, launches = timed(step, args.steps, args.warmup)
    if graph is not None:
        launches = graph_launches * args.steps
    elif split is not None:
        launches += graph_launches * args.steps          # the replayed phases + the update launches counted live
    clocks = sampler.stop() if rank == 0 else None

    def e2e_step():
        s_real.copy_(h_real, non_blocking=True); s_z.copy_(h_z, non_blocking=True); s_t.copy_(h_t, non_blocking=True)
        h_out.copy_(step().detach(), non_blocking=True)
    ms_e2e, _ = timed(e2e_step, args.steps, 1)
    if rank == 0:
        frames = B * Fr * world
        ms_step = ms_total / args.steps
        line = dict(metric='gd_training_step_frames_per_sec_256', value=frames / (ms_step * 1e-3), unit='frames/s', n_gpus=world, steps=args.steps,
                    warmup=args.warmup, ms_per_step=ms_step, higher_is_better=True, scaling='weak', vs_baseline=None,
                    dtype='tf32 (fp32 storage, TF32 tensor-core products, fp32 accumulate)', data='synthetic',
                    config=dict(workload='BASELINE configs[2]: 256x256 G+D training step fwd+bwd (Gmain + Dmain, no reg), 3 frames/clip, 16 clips/GPU, '
                                         'all-reduce + fused Adam/EMA update per phase', clips_per_gpu=B, frames_per_clip=Fr, parallelism=f'dp{world}',
                                cuda_graph=(graph is not None) or ('per phase, all-reduce + update between replays' if split is not None else False),
                                fused_discriminator_layers=bool(train_step.FUSED_DISCRIMINATOR),
                                l2='per-step activation working set >> 126 MB L2; no explicit flush',
                                G_params=int(tp.G_state.numel), D_params=int(tp.D_state.numel)),
                    e2e=dict(value=frames / (ms_e2e / args.steps * 1e-3), unit='frames/s',
                             h2d_bytes_per_step=(h_real.numel() + h_z.numel() + h_t.numel()) * 4, d2h_bytes_per_step=8),
                    gpu_launches=launches, clocks=clocks)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def _dist_setup():
    import torch.distributed as dist
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    assert torch.cuda.is_available(), 'bench.py needs a CUDA device: the b200 implementation has no CPU path'
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=dev)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    return dist, rank, local_rank, world, dev


def _timed(dist, world, dev, fn, steps, warmup):
    from stylegan_v_b200 import _lib
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = _lib.launch_count()
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item()), _lib.launch_count() - l0


def run_synthesis_fwd(args):
    """BASELINE configs[1] / configs[4]: SynthesisNetwork forward only (no_grad), 256^2 x 32 frames or 1024^2 x 8 frames (fmaps 1), replicas at N > 1."""
    dist, rank, local_rank, world, dev = _dist_setup()
    from stylegan_v_b200 import _lib
    from stylegan_v_b200.synthesis import SynthesisNetwork
    from oracle import synthesis_ref as sr     # FLOP model only
    args.warmup = max(args.warmup, 3)
    res = args.res
    N = 32 if res <= 256 else 8
    cb = 16384 if res < 512 else 32768
    torch.manual_seed(rank)
    net = SynthesisNetwork(img_resolution=res, channel_base=cb).to(dev).eval().requires_grad_(False)
    h_ws = torch.randn(N, net.num_ws, net.w_dim).pin_memory()
    h_t = torch.zeros(N, 1).pin_memory()
    h_mz = torch.randn(N, net.motion_encoder.traj_len(), net.motion_encoder.z_dim).pin_memory()
    s_ws, s_t, s_mz = h_ws.to(dev), h_t.to(dev), h_mz.to(dev)
    h_out = torch.zeros(1).pin_memory()

    def compute():
        with torch.no_grad():
            return net(s_ws, s_t, motion_z=s_mz).mean()
    graph, graph_launches, s_out = None, 0, None
    if not args.no_graph:
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(2):
                    compute()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            l0 = _lib.launch_count()
            with torch.cuda.graph(graph):
                s_out = compute()
            graph_launches = _lib.launch_count() - l0
        except Exception as e:
            sys.stderr.write(f'[bench] CUDA graph capture failed ({type(e).__name__}: {e}); eager launches\n')
            graph = None
            torch.cuda.synchronize()

    def step():
        if graph is not None:
            graph.replay()
            return s_out
        return compute()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms_total, launches = _timed(dist, world, dev, step, args.steps, args.warmup)
    if graph is not None:
        launches = graph_launches * args.steps
    clocks = sampler.stop() if rank == 0 else None

    def e2e_step():
        s_ws.copy_(h_ws, non_blocking=True); s_t.copy_(h_t, non_blocking=True); s_mz.copy_(h_mz, non_blocking=True)
        h_out.copy_(step().reshape(1), non_blocking=True)
    ms_e2e, _ = _timed(dist, world, dev, e2e_step, args.steps, 1)
    if rank == 0:
        ms_step = ms_total / args.steps
        frames = N * world
        gflop = sr.conv_flops_per_frame(sr.SynthesisConfig(img_resolution=res, channel_base=cb)) / 1e9
        line = dict(metric=f'synthesis_fwd_frames_per_sec_{res}', value=frames / (ms_step * 1e-3), unit='frames/s', n_gpus=world, steps=args.steps, warmup=args.warmup,
                    ms_per_step=ms_step, higher_is_better=True, scaling='weak', vs_baseline=None, dtype='tf32 (fp32 storage, TF32 tensor-core products, fp32 accumulate)',
                    data='synthetic', config=dict(workload=f'{res}x{res} SynthesisNetwork forward, {N} frames/GPU, random-init weights (BASELINE configs[{1 if res <= 256 else 4}])',
                                                  frames_per_gpu=N, parallelism=f'replicas x{world}', cuda_graph=graph is not None, conv_gflop_per_frame_fwd=gflop,
                                                  l2='activations per layer exceed the 126 MB L2 at res >= 64; no explicit flush'),
                    e2e=dict(value=frames / (ms_e2e / args.steps * 1e-3), unit='frames/s', h2d_bytes_per_step=(h_ws.numel() + h_t.numel() + h_mz.numel()) * 4, d2h_bytes_per_step=4),
                    gpu_launches=launches, clocks=clocks, model_tflops_fwd=gflop * N / ms_step)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def run_full_loop(args):
    """BASELINE configs[3]: the full training iteration with lazy regularisation — R1 every 16 iterations, path-length every 4 (training_loop.py:116-117),
    8 clips x 3 frames per GPU (global batch 64 on 8 GPUs), DDP gradient all-reduce + fused Adam/EMA per phase.  A step here = 16 iterations (one complete
    regularisation cycle: 16 Gmain, 4 Greg, 16 Dmain, 1 Dreg), eager launches (the phase mix changes per iteration)."""
    dist, rank, local_rank, world, dev = _dist_setup()
    from stylegan_v_b200.networks import Generator, Discriminator
    from stylegan_v_b200.train_step import TrainingPhases
    torch.manual_seed(rank)
    B, Fr, CYCLE = 8, 3, 16
    G = Generator(img_resolution=RES).to(dev).train()
    D = Discriminator(img_resolution=RES, mbstd_group_size=4).to(dev).train()
    tp = TrainingPhases(G, D, lr=0.0025, r1_gamma=0.2048, pl_weight=2.0, G_reg_interval=4, D_reg_interval=16, batch_size=B * world)
    real = torch.randn(B * Fr, 3, RES, RES, device=dev).clamp_(-1, 1)
    z = torch.randn(B, G.z_dim, device=dev)
    t = (torch.randint(0, 900, (B, 1)).float() + torch.tensor([[0.0, 5.0, 9.0]])).to(dev)

    def cycle():
        for _ in range(CYCLE):
            out = tp.step(real, t, z, t)
        return out
    steps = max(1, min(args.steps, 3))
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms_total, launches = _timed(dist, world, dev, cycle, steps, 1)
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0:
        ms_iter = ms_total / steps / CYCLE
        frames = B * Fr * world
        line = dict(metric='full_training_loop_frames_per_sec_256', value=frames / (ms_iter * 1e-3), unit='frames/s', n_gpus=world, steps=steps * CYCLE, warmup=CYCLE,
                    ms_per_step=ms_iter, higher_is_better=True, scaling='weak', vs_baseline=None, dtype='tf32 (fp32 storage, TF32 tensor-core products, fp32 accumulate)',
                    data='synthetic', config=dict(workload='BASELINE configs[3]: 256x256 full training loop, R1 every 16 + path length every 4, 3 frames/clip, 8 clips/GPU',
                                                  clips_per_gpu=B, frames_per_clip=Fr, parallelism=f'dp{world}', cuda_graph=False, iterations_timed=steps * CYCLE,
                                                  note='ms_per_step = mean iteration time over whole 16-iteration regularisation cycles'),
                    gpu_launches=launches, clocks=clocks)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-graph', action='store_true', help='launch every kernel from Python instead of replaying a CUDA graph of the step')
    ap.add_argument('--no-optimizer', action='store_true', help='time forward + backward only (no fused Adam update at the end of the step)')
    ap.add_argument('--fused-d', type=int, default=None, help='gd_step: 1 / 0 = discriminator conv layers on the fused conv+bias+act nodes or on the drop-in ops')
    ap.add_argument('--res', type=int, default=256, help='synthesis_fwd: 256 (BASELINE configs[1], 32 frames) or 1024 (configs[4], 8 frames, fmaps 1)')
    ap.add_argument('--precision', default='tf32', choices=['tf32', 'tf32x3'], help='arithmetic mode of the headline number (the other mode is measured beside it)')
    ap.add_argument('--no-second-mode', action='store_true', help='skip the measurement of the other arithmetic mode')
    ap.add_argument('--no-overlap', action='store_true', help='N > 1: one gradient all-reduce after the graph replay instead of the early bucket inside the graph')
    ap.add_argument('--ref-frames', type=int, default=8, help='--impl reference: frames per sampled CPU step (of the 32 of a step)')
    ap.add_argument('--workload', default='synthesis', choices=['synthesis', 'gd_step', 'synthesis_fwd', 'full_loop'],
                    help="synthesis = BASELINE metric (256x256 SynthesisNetwork fwd+bwd, configs[1] batch); gd_step = configs[2] (G+D training step, no reg)")
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='synthesis workload, one GPU: after the timed steps run the timed step once more on the starting parameters and the same '
                         'inputs and write what it computes (image, loss, d loss / d ws, d loss / d parameters) as DIR/<name>.npy in float32, '
                         'for comparing two builds output for output')
    args = ap.parse_args()
    if args.dump_outputs is not None and (args.impl != 'b200' or args.workload != 'synthesis'):
        ap.error('--dump-outputs is implemented for the default synthesis workload of the b200 implementation')
    if args.impl == 'reference':
        return run_reference(args)
    if args.workload == 'gd_step':
        return run_gd_step(args)
    if args.workload == 'synthesis_fwd':
        return run_synthesis_fwd(args)
    if args.workload == 'full_loop':
        return run_full_loop(args)
    args.warmup = max(args.warmup, 3)

    import torch.distributed as dist
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    assert torch.cuda.is_available(), 'bench.py needs a CUDA device: the b200 implementation has no CPU path'
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=dev)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False

    from stylegan_v_b200 import _lib, conv as C, plugin, precision
    from stylegan_v_b200.synthesis import SynthesisNetwork
    from stylegan_v_b200.optim import FlatModuleState, FusedAdamEMA
    from stylegan_v_b200.ops import upfirdn2d as U
    from oracle import synthesis_ref as sr     # FLOP model + cpu_baseline only

    torch.manual_seed(0)                       # every rank builds the SAME replica ...
    net = SynthesisNetwork(img_resolution=RES).to(dev).train()
    # parameters / gradients / Adam moments in flat buffers: one all-reduce (N > 1) and one fused nan_to_num + Adam launch per step
    # (training_loop.py:381-386 semantics; lr as train.py:160).  --no-optimizer times forward + backward alone.
    # N > 1: the 3x3 convolution weights (70 % of the gradient bytes) come FIRST in the flat buffer: their weight-gradient kernels are the last
    # tensor-core kernels of the backward pass, but ~0.7 ms of small kernels follow them (demodulation / affine / motion-encoder gradients,
    # profiles/timeline_r2m_serial.txt), so their all-reduce is issued — inside the captured graph — the moment the last of them has been
    # accumulated and runs under that tail; only the rest of the buffer is reduced after the backward pass.  (--no-overlap: one collective.)
    overlap = world > 1 and not args.no_overlap and not args.no_graph
    state = FlatModuleState(list(net.parameters()), early=(lambda p: p.ndim == 4 and p.shape[-1] == 3) if overlap else None)
    state.broadcast(0)                         # ... and rank 0's parameters are broadcast like the reference's "Distribute across GPUs" (training_loop.py:215-232)
    bucket = dict(armed=False)                 # whether the step being built carries its collectives (stylegan_v_b200/optim.py: begin / finish_backward)
    opt = None if args.no_optimizer else FusedAdamEMA(state, lr=0.0025, betas=(0.0, 0.99), eps=1e-8)
    if args.dump_outputs is not None:
        assert world == 1, '--dump-outputs runs on one GPU'
        p0 = state.param.clone()               # the starting parameters: what the dumped step is computed from
    torch.manual_seed(1 + rank)                # per-rank latents (each rank works on its own 32 frames)
    N = FRAMES_PER_GPU
    L = net.motion_encoder.traj_len()
    # host-side (pinned) inputs for the end-to-end measurement
    h_ws = torch.randn(N, net.num_ws, net.w_dim).pin_memory()
    h_t = torch.zeros(N, 1).pin_memory()
    h_mz = torch.randn(N, L, net.motion_encoder.z_dim).pin_memory()
    d_ws, d_t, d_mz = h_ws.to(dev), h_t.to(dev), h_mz.to(dev)
    dimg = torch.randn(N, 3, RES, RES, device=dev)
    h_out = torch.zeros(1).pin_memory()
    last = {}                                  # image, loss and ws (.grad) of the latest step (graph outputs are rewritten by every replay)

    def step_compute(ws, t, mz):
        if opt is None:
            state.zero_grad()                  # with the optimiser, its update kernel re-zeroes the gradient buffer
        ws = ws.requires_grad_(True)
        img = net(ws, t, motion_z=mz)
        loss = (img * dimg).sum()
        if bucket['armed']:
            state.begin_backward()
        loss.backward()
        if bucket['armed']:
            state.finish_backward()            # waits for the conv-weight bucket (stream-level, capturable), reduces the rest: affines, biases, motion encoder
        last.update(img=img, loss=loss, ws=ws)
        return loss

    # The step (about 670 kernel launches: forward + backward of 20 fused layers) is captured ONCE into a CUDA graph and replayed:
    # the GPU then never waits for the Python/ctypes launch path.  The gradient all-reduce (N > 1) is issued after each replay.
    s_ws, s_t, s_mz = d_ws.clone(), d_t.clone(), d_mz.clone()      # static graph inputs

    def build_step(mode):
        """The step in one arithmetic mode of the contractions (stylegan_v_b200.precision): 'tf32' or the fp32-grade 'tf32x3'.  The mode is
        read when the kernels are issued, i.e. at capture time; a replay needs no context."""
        graph, graph_launches, s_loss = None, 0, None
        in_graph_reduce = False
        if not args.no_graph:
            try:
                bucket['armed'] = overlap                   # the collectives are captured with the step
                with precision.precision(mode):
                    side = torch.cuda.Stream()
                    side.wait_stream(torch.cuda.current_stream())
                    with torch.cuda.stream(side):
                        for _ in range(2):
                            step_compute(s_ws.detach(), s_t, s_mz)
                    torch.cuda.current_stream().wait_stream(side)
                    torch.cuda.synchronize()
                    graph = torch.cuda.CUDAGraph()
                    l0 = _lib.launch_count()
                    with torch.cuda.graph(graph):
                        s_loss = step_compute(s_ws.detach(), s_t, s_mz)
                    graph_launches = _lib.launch_count() - l0
                in_graph_reduce = overlap
            except Exception as e:      # capture is an optimisation, not a requirement
                sys.stderr.write(f'[bench] rank {rank}: CUDA graph capture failed ({type(e).__name__}: {e}); falling back\n')
                graph = None
                torch.cuda.synchronize()
            bucket['armed'] = False
            if overlap:
                # every rank must issue the same collectives: if the capture with NCCL inside failed anywhere, all ranks re-capture without it
                ok = torch.tensor([1.0 if graph is not None else 0.0], device=dev)
                dist.all_reduce(ok, op=dist.ReduceOp.MIN)
                if float(ok.item()) == 0.0:
                    in_graph_reduce = False
                    graph = None
                    try:
                        with precision.precision(mode):
                            torch.cuda.synchronize()
                            graph = torch.cuda.CUDAGraph()
                            l0 = _lib.launch_count()
                            with torch.cuda.graph(graph):
                                s_loss = step_compute(s_ws.detach(), s_t, s_mz)
                            graph_launches = _lib.launch_count() - l0
                    except Exception as e:
                        sys.stderr.write(f'[bench] rank {rank}: CUDA graph capture failed again ({type(e).__name__}: {e}); eager launches\n')
                        graph = None
                        torch.cuda.synchronize()
        state.zero_grad()                          # warm-up / capture passes accumulated into the buffer

        def step(ws, t, mz):
            if graph is not None:
                if ws.data_ptr() != s_ws.data_ptr():
                    s_ws.copy_(ws, non_blocking=True); s_t.copy_(t, non_blocking=True); s_mz.copy_(mz, non_blocking=True)
                graph.replay()
                loss = s_loss
            else:
                with precision.precision(mode):
                    loss = step_compute(ws, t, mz)
            if not (in_graph_reduce and graph is not None):
                state.all_reduce()                 # SUM over ranks; the 1/world of the average is applied inside the update kernel
            if opt is not None:
                opt.step(zero_grad=True)
            elif world > 1:
                state.grad.div_(world)
            return loss
        return step, graph, graph_launches, in_graph_reduce

    step, graph, graph_launches, reduce_in_graph = build_step(args.precision)

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = _lib.launch_count()
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), _lib.launch_count() - l0

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    # (1) device-resident inputs
    ms_total, launches = timed(lambda: step(s_ws if graph is not None else d_ws.detach(), s_t if graph is not None else d_t, s_mz if graph is not None else d_mz),
                               args.steps, args.warmup)
    if graph is not None:
        launches = (graph_launches + (1 if opt is not None else 0)) * args.steps      # launches recorded at capture time, replayed once per step (+ the update kernel)

    # (2) end to end: H2D of the step's inputs from pinned memory, D2H of the loss, every step
    def e2e_step():
        ws = h_ws.to(dev, non_blocking=True); t = h_t.to(dev, non_blocking=True); mz = h_mz.to(dev, non_blocking=True)
        loss = step(ws, t, mz)
        h_out.copy_(loss.detach().reshape(1), non_blocking=True)
    ms_e2e, _ = timed(e2e_step, args.steps, 1)
    clocks = sampler.stop() if rank == 0 else None      # sampled across both timed regions (device-resident and end-to-end)
    if args.dump_outputs is not None:
        # Every timed step updates the parameters, and the atomic reductions of the kernels make each gradient exact only up to rounding; over
        # many Adam steps on this unbounded loss those differences grow, so the state the timed steps end in is not the same in every run.  The
        # dump is the timed step (the same graph, or the same eager launches) evaluated once more on the starting parameters and the same
        # inputs: the same in every run up to rounding.  The parameters the timed steps reached are put back afterwards.
        p_now = state.param.clone()
        state.param.copy_(p0)
        state.zero_grad()
        if graph is not None:
            graph.replay()
        else:
            with precision.precision(args.precision):
                step_compute(d_ws.detach(), d_t, d_mz)
        dump_outputs(args.dump_outputs, img=last['img'], loss=last['loss'], ws_grad=last['ws'].grad, param_grad=state.grad)
        state.param.copy_(p_now)
        state.zero_grad()
        del p0, p_now

    # (3) the same step in the other arithmetic mode, beside the headline (the reference trains with allow_tf32 = False, training_loop.py:141-142:
    #     tf32x3 is the fp32-grade counterpart; tf32 is the north_star's TF32 tensor-core arithmetic)
    other_mode = 'tf32x3' if args.precision == 'tf32' else 'tf32'
    other = None
    if not args.no_second_mode:
        step2, graph2, launches2, _ = build_step(other_mode)
        k2 = max(3, args.steps // 2)
        ms2, l2 = timed(lambda: step2(s_ws if graph2 is not None else d_ws.detach(), s_t if graph2 is not None else d_t, s_mz if graph2 is not None else d_mz), k2, 3)
        other = dict(dtype=DTYPES[other_mode], value=N * world / (ms2 / k2 * 1e-3), unit='frames/s', ms_per_step=ms2 / k2, steps=k2, warmup=3,
                     gpu_launches=(launches2 + (1 if opt is not None else 0)) * k2 if graph2 is not None else l2)
        del step2, graph2

    ms_step = ms_total / args.steps
    frames = N * world
    value = frames / (ms_step * 1e-3)
    e2e_value = frames / (ms_e2e / args.steps * 1e-3)
    def leave():
        """End of a rank's work.  When NCCL collectives were captured into the step's CUDA graph, tearing the process group down (here, or from
        interpreter shutdown) blocked for minutes on this stack (round-2 call O: the result line was printed, the ranks never exited) — the
        graphs hold communicator work the destructor waits for.  Those runs drop the graphs and leave through os._exit after flushing."""
        if world == 1:
            return
        torch.cuda.synchronize()
        if reduce_in_graph:
            sys.stdout.flush(); sys.stderr.flush()
            os._exit(0)
        dist.destroy_process_group()
    if rank != 0:
        leave()
        return

    peaks = load_peaks()
    # ---- roofline of the dominant kernel (largest share of the step): the implicit-GEMM conv at its heaviest layer shape,
    #      and the stand-alone upfirdn2d kernel the metric names ----
    def kernel_ms(fn, iters=10):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        evs = []
        for _ in range(iters):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(); b.record(); evs.append((a, b))
        torch.cuda.synchronize()
        ts = sorted(a.elapsed_time(b) for a, b in evs)
        return sum(ts) / len(ts)
    taps, offs = C.conv3x3_taps()
    conv_shapes = [('b32.conv1', 512, 512, 32), ('b64.conv1', 256, 256, 64), ('b128.conv1', 128, 128, 128), ('b256.conv1', 64, 64, 256)]
    per_layer = []
    x3_headline = args.precision == 'tf32x3'
    for name, ci, co, r in conv_shapes:
        x = torch.randn(N, ci, r, r, device=dev).contiguous(memory_format=torch.channels_last)
        wp = C.prep_weights(torch.randn(co, ci, 3, 3, device=dev), taps, x3=x3_headline)
        s = torch.rand(N, ci, device=dev) + 0.5; d = torch.rand(N, co, device=dev) + 0.5; b = torch.zeros(co, device=dev)
        ms = kernel_ms(lambda: C.igemm_conv(x, wp, offs, a_scale=s, o_scale=d, bias=b, act='lrelu', gain=1.4142135))
        var = C.igemm_conv(x, wp, offs, a_scale=s, o_scale=d, bias=b, act='lrelu', gain=1.4142135, query=True)
        fl = 2.0 * N * r * r * ci * co * 9
        per_layer.append(dict(layer=name, ms=ms, tflops=fl / ms / 1e9, flops=fl, variant=var))
        del x, wp
    dom = max(per_layer, key=lambda z: z['ms'])
    # DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum of ONE `ncu --set full` capture of the current kernels): read from the
    # committed summary profiles/ncu_traffic.json (written by scripts/ncu_traffic.py from the .ncu-rep); null when no capture of this build exists.
    # The algorithmic minimum of the conv is x once + y once.
    try:
        ncu_traffic = json.load(open(os.path.join(ROOT, 'profiles', 'ncu_traffic.json')))
    except Exception:
        ncu_traffic = {}
    roofline = dict(bound='tensor', kernel=f"conv_tf32_v3_kernel @ {dom['layer']} (N={N})", achieved=dom['tflops'], peak=peaks['bf16_tflops'],
                    unit='TFLOP/s', frac=dom['tflops'] / peaks['bf16_tflops'], traffic=ncu_traffic.get(dom['layer']),
                    traffic_unit='bytes/launch (ncu --set full, profiles/ncu_traffic.json: ' + str(ncu_traffic.get('source')) + ')',
                    algorithmic_bytes_per_launch=N * 256 * 256 * 64 * 4 * 2 if dom['layer'] == 'b256.conv1' else None,
                    peak_source=peaks['source'] + ' (dense bf16 cuBLAS; the kernel runs kind::tf32, whose measured issue-rate ceiling is 1164 TFLOP/s for N >= 128 and '
                                                  '776 TFLOP/s for N = 64 output channels — profiles/mma_rate_probe_r1.txt)',
                    tf32_issue_rate_ceiling_tflops=776.0 if dom['layer'] == 'b256.conv1' else 1164.0,
                    algorithmic_flops_per_launch=dom['flops'], per_layer=per_layer)
    # the FIR pass of the up layers as the network runs it (channels_last, TMA-fed kernel) and the NCHW kernel the drop-in op uses
    f = U.setup_filter([1, 3, 3, 1], device=dev)
    xf = torch.randn(N, 64, 257, 257, device=dev)
    fir_bytes = (xf.numel() + N * 64 * 256 * 256) * 4
    fir_nchw_ms = kernel_ms(lambda: plugin.upfirdn2d(xf, f, 1, 1, 1, 1, 1, 1, 1, 1, False, 4.0))
    xf = xf.contiguous(memory_format=torch.channels_last)
    fir_ms = kernel_ms(lambda: plugin.upfirdn2d(xf, f, 1, 1, 1, 1, 1, 1, 1, 1, False, 4.0))
    upfirdn = dict(bound='hbm', kernel='fir_nhwc_tma44 [32,257,257,64]->[32,256,256,64] (channels_last, as the synthesis path runs it)', achieved=fir_bytes / fir_ms / 1e6,
                   peak=peaks['hbm_gbs'], unit='GB/s', frac=fir_bytes / fir_ms / 1e6 / peaks['hbm_gbs'], traffic=ncu_traffic.get('fir_nhwc_tma44'), algorithmic_bytes_per_launch=fir_bytes,
                   peak_source=peaks['source'], nchw=dict(kernel='fir_nchw_tiled, same extents in NCHW (odd row pitch: not TMA-addressable)', achieved=fir_bytes / fir_nchw_ms / 1e6,
                                                          frac=fir_bytes / fir_nchw_ms / 1e6 / peaks['hbm_gbs']))
    # "beat this kernel" (BASELINE.md §4): the reference's OWN CUDA plugins, compiled unmodified for sm_100a (oracle/_ref, oracle/build_ref.py), timed
    # on the same extents in the layout the reference runs them in (NCHW) — a reported baseline, never part of the product path
    ref_cuda = None
    try:
        from oracle import build_ref
        rup, rba = build_ref.load_plugin('upfirdn2d_plugin'), build_ref.load_plugin('bias_act_plugin')
        if rup is not None and rba is not None:
            xn = xf.contiguous()
            ref_fir_ms = kernel_ms(lambda: rup.upfirdn2d(xn, f, 1, 1, 1, 1, 1, 1, 1, 1, False, 4.0))
            ref_fir_cl_ms = kernel_ms(lambda: rup.upfirdn2d(xf, f, 1, 1, 1, 1, 1, 1, 1, 1, False, 4.0))
            xb = torch.randn(N, 64, 256, 256, device=dev); bb = torch.randn(64, device=dev); e = torch.empty(0, device=dev)
            ba_bytes = 2 * xb.numel() * 4
            ref_ba_ms = kernel_ms(lambda: rba.bias_act(xb, bb, e, e, e, 0, 1, 3, 0.2, 1.4142135, -1.0))
            our_ba_ms = kernel_ms(lambda: plugin.bias_act(xb, bb, e, e, e, 0, 1, 3, 0.2, 1.4142135, -1.0))
            ref_cuda = dict(note="the reference's own upfirdn2d / bias_act CUDA kernels (unmodified sources, --use_fast_math, sm_100a) on this B200, same extents",
                            upfirdn2d=dict(shape='[32,64,257,257] -> [32,64,256,256] fp32', reference_nchw_gbs=fir_bytes / ref_fir_ms / 1e6,
                                           reference_channels_last_gbs=fir_bytes / ref_fir_cl_ms / 1e6, ours_nchw_gbs=fir_bytes / fir_nchw_ms / 1e6,
                                           ours_channels_last_gbs=fir_bytes / fir_ms / 1e6, speedup_vs_reference_nchw=ref_fir_ms / fir_ms),
                            bias_act=dict(shape='[32,64,256,256] fp32 lrelu', reference_gbs=ba_bytes / ref_ba_ms / 1e6, ours_gbs=ba_bytes / our_ba_ms / 1e6,
                                          speedup=ref_ba_ms / our_ba_ms,
                                          note='in the synthesis path this pass does not exist at all: bias/lrelu/gain run in the conv / FIR epilogue'))
            del xn, xb
    except Exception as ex:      # a baseline that cannot run is reported, not fatal
        ref_cuda = dict(unavailable=f'{type(ex).__name__}: {ex}')
    del xf
    # the parameter update of the step: one streaming pass over the flat state (4 loads + 4 stores of 4 B per parameter incl. gradient zeroing)
    optimizer = None
    if opt is not None:
        opt_ms = kernel_ms(lambda: opt.step(zero_grad=True))
        opt_bytes = opt.algorithmic_bytes(False, True)
        optimizer = dict(bound='hbm', kernel=f'adam_ema_kernel<EMA=0,ZERO=1> over {state.numel} fp32 parameters (flat state)', ms=opt_ms,
                         achieved=opt_bytes / opt_ms / 1e6, peak=peaks['hbm_gbs'], unit='GB/s', frac=opt_bytes / opt_ms / 1e6 / peaks['hbm_gbs'],
                         algorithmic_bytes_per_launch=opt_bytes)

    cfg = sr.SynthesisConfig(img_resolution=RES)
    conv_gflop_fwd = sr.conv_flops_per_frame(cfg) / 1e9
    cpu_baseline = None
    if not args.no_cpu_baseline:
        cframes = 4
        cstep, ckind, threads = cpu_reference_step(cframes)
        cstep()
        ts = sorted(cstep() for _ in range(3))
        cpu_baseline = dict(value=cframes / ts[1], unit='frames/s', cores=threads, kind=ckind,
                            sample=f'{cframes} of the 32 frames fwd+bwd (+ their share of the nan_to_num/Adam update) at 256x256 on the ' +
                                   ("UNMODIFIED reference SynthesisNetwork, torch_utils.ops impl='ref' (custom CUDA disabled)" if ckind == 'reference'
                                    else 'oracle port of the reference CPU path') +
                                   f', fused_modconv=False; median of 3 after warm-up; {threads} torch threads of {os.cpu_count()} host cores')

    line = dict(metric='synthesis_fwd_bwd_frames_per_sec_256', value=value, unit='frames/s', n_gpus=world, steps=args.steps, warmup=args.warmup,
                ms_per_step=ms_step, higher_is_better=True, scaling='weak', vs_baseline=None, dtype=DTYPES[args.precision],
                data='synthetic',
                config=dict(workload='256x256 SynthesisNetwork forward+backward' + (' + fused nan_to_num/Adam update of all parameters' if opt is not None else '') +
                                     ', 32 frames/GPU (32 latents x 1 frame), fmaps 0.5, random-init weights', optimizer_step=opt is not None,
                            frames_per_gpu=N, parallelism=f'dp{world}', cuda_graph=graph is not None,
                            gradient_all_reduce=('none (1 GPU)' if world == 1 else 'conv-weight bucket inside the graph under the backward tail + rest after it' if reduce_in_graph else 'one collective after the graph replay'), l2='activation working set per step (>= 134 MB per layer at res >= 64, ~6 GB total) exceeds the 126 MB L2; no explicit flush',
                            conv_gflop_per_frame_fwd=conv_gflop_fwd),
                e2e=dict(value=e2e_value, unit='frames/s', h2d_bytes_per_step=(h_ws.numel() + h_t.numel() + h_mz.numel()) * 4, d2h_bytes_per_step=4),
                gpu_launches=launches, clocks=clocks, roofline=roofline, upfirdn2d=upfirdn, optimizer=optimizer, cpu_baseline=cpu_baseline,
                model_tflops_fwd_bwd=3 * conv_gflop_fwd * frames / ms_step / world, reference_cuda_kernels=ref_cuda)
    line[other_mode] = other      # the same step in the other arithmetic mode, measured beside the headline
    print(json.dumps(line))
    leave()


if __name__ == '__main__':
    main()
