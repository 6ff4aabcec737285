#!/usr/bin/env python
"""Training benchmark (BASELINE.json configs[2], "C3"): Transformer-XL d_model 512, 16 layers, 8 heads x 64, d_inner 2048,
mem_len 512, genre-style LM training, bptt 512 with warm memory (S = 1024), dropout 0.1, rand_window_mask, bf16 compute /
fp32 master weights, synthetic LakhMIDI-shaped tokens, data-parallel (batch sharded over ranks, NCCL all-reduce of the flat
gradient overlapped with backward).  A "step" = forward + backward + all-reduce + Adam on `batch` sequences per GPU.
`value` = trained tokens/s over all GPUs (weak scaling).  Run through `python bench.py --workload c3 ...`.
"""
import ctypes as C
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC, UNIT = 'trained_tokens_per_sec', 'tokens/s'
V = 324
WORKLOAD = ('C3: Transformer-XL d_model 512, 16 layers, 8 heads x 64, d_inner 2048, mem_len 512, vocab 324; training step '
            '(fwd + bwd + gradient all-reduce + Adam), bptt 512 over a full 512-slot memory (S=1024), dropout 0.1, '
            'rand_window_mask(mask_steps=1), AR/TAR, bf16 compute / fp32 master')


def flops_per_token(d=512, L=16, H=8, Dh=64, di=2048, M=512, T=512, b=32):
    "SURVEY.md 8(d): dense-count FLOPs per input token; returns (forward, forward+backward)."
    HD, S = H * Dh, M + T
    per_layer = 2 * d * 3 * HD + 2 * d * 2 * HD * (M / T) + 3 * 2 * HD * S + 2 * HD * d + 4 * d * di
    fwd = L * per_layer + L * 2 * d * HD * S / (b * T) + 2 * d * V
    mem_kv_dgrad = L * 2 * d * 2 * HD * (M / T)        # memory rows are detached: no input gradient for their K/V GEMM
    return fwd, 3 * fwd - mem_kv_dgrad


def lakh_shaped_tokens(bs, n, gen):
    "(note, duration) pairs with an xxsep/duration separator every 1-4 notes: the token grammar of the genre model"
    out = torch.empty(bs, n + 8, dtype=torch.int64)
    for b in range(bs):
        toks = []
        while len(toks) < n + 8:
            for _ in range(int(torch.randint(1, 5, (1,), generator=gen))):
                toks += [int(torch.randint(12, 140, (1,), generator=gen)), int(torch.randint(140, 301, (1,), generator=gen))]
            toks += [11, int(torch.randint(140, 301, (1,), generator=gen))]
        out[b] = torch.tensor(toks[:n + 8])
    return out[:, :n + 1]


def run_b200(args):
    outputs = {} if args.dump_outputs else None
    line = measure(args, outputs=outputs)
    if line is not None:
        print(json.dumps(line), flush=True)
        if outputs is not None:
            from bench import dump_outputs
            dump_outputs(args.dump_outputs, outputs)


def measure(args, sample_clocks=True, cpu_leg=True, outputs=None):
    "Runs the C3 leg on every rank; returns the JSON record on rank 0 (None elsewhere)."
    from bench import ClockSampler
    from deepmusicgeneration_b200 import _lib, sharding
    from deepmusicgeneration_b200.app_utils import baseline_config
    from deepmusicgeneration_b200.model import get_language_model
    from deepmusicgeneration_b200.training import TXLTrainer

    rank, local_rank, world = sharding.init_distributed()
    if not torch.cuda.is_available():
        raise SystemExit('bench_train.py: no CUDA device - the CUDA path has no CPU fallback')
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    B, T, K, W = args.train_batch, 512, args.steps, max(args.warmup, 3)
    lib = _lib.load()
    cfg = dict(baseline_config(), mask_steps=1)
    model = get_language_model(V, cfg, dtype='bf16', device=local_rank, max_batch=1, max_seq=64, max_rows=64, keep_hidden=False, seed=0)
    tr = TXLTrainer(model, B, T, cfg, drop_mult=1.0, alpha=2., beta=1., seed=7, distributed=world > 1)
    np.random.seed(1234)          # rand_window_mask draws: identical on every rank, like a shared schedule

    n_batches = 4
    gen = torch.Generator().manual_seed(1234 + rank)
    stream_tokens = lakh_shaped_tokens(B, n_batches * T, gen)
    xs = [stream_tokens[:, i * T:(i + 1) * T].contiguous().pin_memory() for i in range(n_batches)]
    ys = [stream_tokens[:, i * T + 1:(i + 1) * T + 1].contiguous().pin_memory() for i in range(n_batches)]
    xd = [x.to(dev) for x in xs]
    yd = [y.to(dev) for y in ys]

    if os.environ.get('DMG_BENCH_PROFILE'):          # short run for ncu launch lists: 2 warm steps + 1 step, no timing
        tr.reset()
        for i in range(3):
            tr.step(xd[i % n_batches], yd[i % n_batches], lr=1e-4)
        torch.cuda.synchronize()
        print('profile run done', tr.losses())
        tr.close()
        return None
    tr.reset()
    for i in range(W):
        tr.step(xd[i % n_batches], yd[i % n_batches], lr=1e-4)
    torch.cuda.synchronize()
    l0 = tr.losses()

    # ---- timed region: K steps, inputs resident in HBM
    sharding.barrier(); torch.cuda.synchronize()
    clocks = ClockSampler(local_rank) if rank == 0 and sample_clocks else None
    launches0 = lib.dmg_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.time()
    ev0.record()
    for i in range(K):
        tr.step(xd[i % n_batches], yd[i % n_batches], lr=1e-4)
    ev1.record()
    torch.cuda.synchronize()
    t1 = time.time()
    sharding.barrier()
    ms = ev0.elapsed_time(ev1)
    launches = int(lib.dmg_launch_count() - launches0)
    clock_info = clocks.stop(t0, t1) if clocks else None
    ms_max = sharding.max_over_ranks(ms, device=dev)
    value = B * T * world * K / (ms_max / 1e3)
    l1 = tr.losses()
    if outputs is not None:
        outputs['train_losses'] = np.array([l1[k] for k in ('loss', 'ce', 'ar', 'tar', 'grad_norm')])
    grad_exchange = tr.describe_exchange()

    # ---- end to end: every step copies its tokens/targets from pinned host memory and reads the loss back
    Ke = min(K, 20)
    sharding.barrier(); torch.cuda.synchronize()
    ev0.record()
    for i in range(Ke):
        x = xs[i % n_batches].to(dev, non_blocking=True)
        y = ys[i % n_batches].to(dev, non_blocking=True)
        tr.step(x, y, lr=1e-4)
        loss = tr.losses()['loss']
    ev1.record()
    torch.cuda.synchronize()
    e2e_ms = sharding.max_over_ranks(ev0.elapsed_time(ev1), device=dev)
    e2e_value = B * T * world * Ke / (e2e_ms / 1e3)

    # ---- per-phase split of one step (device timed), for the roofline of the GEMMs
    def timed(fn, reps=3):
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps): fn()
        b.record(); torch.cuda.synchronize()
        return a.elapsed_time(b) / reps
    t_fwd = timed(lambda: tr.forward(xd[0], yd[0]))
    def fb():
        tr.forward(xd[0], yd[0]); tr.backward()
    t_fb = timed(fb)
    fwd_f, fb_f = flops_per_token(b=B)
    try:
        pk = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
        peak_tf, peak_src = float(pk['bf16_tflops_sustained']), 'measured sustained (MEASURED_PEAKS.json)'
    except Exception:
        peak_tf, peak_src = 1340.8, 'fallback'
    step_ms = ms_max / K
    achieved = fb_f * B * T / (step_ms / 1e3) / 1e12
    roofline = {'bound': 'tensor', 'kernel': 'whole training step (GEMMs + attention contractions)', 'achieved': achieved,
                'peak': peak_tf, 'unit': 'TFLOP/s', 'frac': achieved / peak_tf, 'traffic': None, 'peak_source': peak_src,
                'flops_per_token_fwd_bwd_dense': fb_f, 'forward_ms': t_fwd, 'forward_backward_ms': t_fb,
                'optimizer_and_rest_ms': step_ms - t_fb}
    comm = tr.profile_comm(lambda: tr.step(xd[0], yd[0], lr=1e-4), reps=3) if world > 1 else None
    tr.close()
    del tr, model
    torch.cuda.empty_cache()
    if rank != 0:
        return None
    cpu = None
    if world == 1 and not args.no_cpu_baseline and cpu_leg:
        v, n, threads, dt = cpu_reference(2, 8, budget_s=15.0)                  # a bounded sample: about 15 s of host work
        cpu = {'value': v, 'unit': UNIT, 'cores': threads, 'kind': 'port',
               'sample': f'{n} training step(s) of 2 sequences x 512 tokens over a full memory, fp32 eager-PyTorch oracle, {dt:.1f} s'}
    line = {'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': K, 'warmup': W, 'ms_per_step': step_ms,
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'bf16', 'data': 'synthetic',
            'config': {'workload': WORKLOAD, 'batch_per_gpu': B, 'global_batch': B * world, 'bptt': T,
                       'parallelism': f'dp{world}: batch sharded; ' + grad_exchange,
                       'l2': 'activations per step (>3 GB) exceed the 126 MB L2',
                       'loss_before': l0['loss'], 'loss_after': l1['loss'], 'loss_parts_before': l0, 'loss_parts_after': l1,
                       'comm': comm},
            'roofline': roofline, 'cpu_baseline': cpu,
            'e2e': {'value': e2e_value, 'unit': UNIT, 'h2d_bytes_per_step': 2 * B * T * 8, 'd2h_bytes_per_step': 16, 'steps': Ke},
            'gpu_launches': launches, 'clocks': clock_info}
    return line


def cpu_reference(batch, steps, budget_s):
    "The reference training step (oracle/train.py) on the host cores: eager PyTorch fp32 autograd."
    from oracle import train as otrain
    from oracle import txl
    torch.manual_seed(0)
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    model = txl.get_language_model(V, txl.baseline_config()).train()
    model.reset()
    opt = otrain.AdamTrueWD(otrain.unique_params(model))
    g = torch.Generator().manual_seed(1)
    toks = torch.randint(12, 301, (batch, 512 * (steps + 2) + 1), generator=g)
    otrain.train_step(model, toks[:, :512], toks[:, 1:513], opt, 1e-4)          # fills the memory (and warms up)
    done, t0 = 0, time.time()
    for s in range(1, steps + 1):
        otrain.train_step(model, toks[:, s * 512:(s + 1) * 512], toks[:, s * 512 + 1:(s + 1) * 512 + 1], opt, 1e-4)
        done += 1
        if time.time() - t0 > budget_s:
            break
    dt = time.time() - t0
    return batch * 512 * done / dt, done, threads, dt


def run_reference(args):
    if int(os.environ.get('RANK', '0')) != 0:
        return
    v, n, threads, dt = cpu_reference(2, max(1, min(args.steps, 3)), budget_s=150.0)
    sample = f'{n} training step(s) of 2 sequences x 512 tokens over a full memory, fp32 eager-PyTorch oracle (reference algorithm), {threads} threads'
    line = {'impl': 'reference', 'metric': METRIC, 'value': v, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': n, 'warmup': 1,
            'ms_per_step': 1e3 * dt / n, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
            'data': 'synthetic', 'config': {'workload': WORKLOAD, 'cpu_batch': 2},
            'cpu_baseline': {'value': v, 'unit': UNIT, 'cores': threads, 'kind': 'port', 'sample': sample},
            'e2e': {'value': v, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}, 'gpu_launches': 0}
    print(json.dumps(line), flush=True)
