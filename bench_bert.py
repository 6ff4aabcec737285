#!/usr/bin/env python
"""Remix-encoder benchmark (BASELINE.json configs[3], "C4"): the masked-BERT encoder of deep_music_remix.py (MultiTransformer msk
branch, app_utils.py:60 config: d_model 512, 8 heads x 64, 10 layers, no FFN, no out-projection), seq 1024, bf16 forward,
`--bert-batch` sequences per GPU (default 512, chunked into 32-sequence activation chunks).  A "step" = one forward over the
batch; `value` = forward tokens/s over all GPUs (batch sharded, no collective).  Run through `python bench.py --workload c4 ...`.
"""
import json
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC, UNIT = 'forward_tokens_per_sec', 'tokens/s'
V, T = 324, 1024


def workload_name(cfg, B):
    return (f"C4: remix (masked-BERT) encoder d_model {cfg['d_model']}, {cfg['enc_layers']} layers, {cfg['n_heads']} heads x {cfg['d_head']}, "
            f"seq {T}, {B} sequences/GPU, bf16 forward (wrap-around _line_shift, no mask, no out-projection / FFN)")


def flops_per_token(cfg):
    "SURVEY.md 8(d): q, k, v projections + AC, BD, PV (dense count) per layer, + the tied head for one position per sequence"
    d, HD = cfg['d_model'], cfg['n_heads'] * cfg['d_head']
    return cfg['enc_layers'] * (3 * 2 * d * HD + 3 * 2 * HD * T)


def synthetic(B, gen):
    x = torch.randint(0, V, (B, T), generator=gen)
    pos = torch.cumsum(torch.randint(0, 9, (B, T), generator=gen), 1).clamp_max(32 * 1024 - 1)
    return x, pos


def run_b200(args):
    outputs = {} if args.dump_outputs else None
    line = measure(args, outputs=outputs)
    if line is not None:
        print(json.dumps(line), flush=True)
        if outputs is not None:
            from bench import dump_outputs
            dump_outputs(args.dump_outputs, outputs)


def measure(args, sample_clocks=True, cpu_leg=True, outputs=None):
    "Runs the C4 leg on every rank; returns the JSON record on rank 0 (None elsewhere)."
    from bench import ClockSampler
    from deepmusicgeneration_b200 import _lib, sharding
    from deepmusicgeneration_b200.app_utils import multitask_config
    from deepmusicgeneration_b200.model import get_multitask_model

    rank, local_rank, world = sharding.init_distributed()
    if not torch.cuda.is_available():
        raise SystemExit('bench_bert.py: no CUDA device - the CUDA path has no CPU fallback')
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    B, K, W = args.bert_batch, args.steps, max(args.warmup, 3)
    lib = _lib.load()
    cfg = multitask_config()
    pm = get_multitask_model(V, cfg, pad_idx=1, dtype='bf16', device=local_rank, max_batch=B, max_seq=T, max_rows=getattr(args, 'bert_chunk', 32) * T, seed=0)
    e = pm._e
    gen = torch.Generator().manual_seed(1234 + rank)
    xh, ph = synthetic(B, gen)
    xh, ph = xh.pin_memory(), ph.pin_memory()
    x, pos = xh.to(dev), ph.to(dev)

    for _ in range(W):
        e.forward(x, pos, _lib.LOGITS_NONE)
    torch.cuda.synchronize()

    # ---- timed region: K forwards, inputs resident in HBM
    sharding.barrier(); torch.cuda.synchronize()
    clocks = ClockSampler(local_rank) if rank == 0 and sample_clocks else None
    launches0 = lib.dmg_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.time()
    ev0.record()
    for _ in range(K):
        e.forward(x, pos, _lib.LOGITS_NONE)
    ev1.record()
    torch.cuda.synchronize()
    t1 = time.time()
    sharding.barrier()
    ms = ev0.elapsed_time(ev1)
    launches = int(lib.dmg_launch_count() - launches0)
    clock_info = clocks.stop(t0, t1) if clocks else None
    ms_max = sharding.max_over_ranks(ms, device=dev)
    value = B * T * world * K / (ms_max / 1e3)

    # ---- end to end: ids and positions come from pinned host memory every step, the last position's logits go back
    Ke = min(K, 5)
    out_host = torch.empty(B, V, dtype=torch.float32).pin_memory()
    def e2e_step():
        xd, pd = xh.to(dev, non_blocking=True), ph.to(dev, non_blocking=True)
        logits = e.forward(xd, pd, _lib.LOGITS_LAST)[0]
        out_host.copy_(logits, non_blocking=True)
        torch.cuda.synchronize()
    e2e_step()                                       # untimed: first use of the logits path and of the pinned result buffer
    sharding.barrier(); torch.cuda.synchronize()
    ev0.record()
    for _ in range(Ke):
        e2e_step()
    ev1.record()
    torch.cuda.synchronize()
    e2e_ms = sharding.max_over_ranks(ev0.elapsed_time(ev1), device=dev)
    e2e_value = B * T * world * Ke / (e2e_ms / 1e3)
    if outputs is not None:
        outputs['bert_logits'] = out_host.numpy().copy()

    del e, pm
    torch.cuda.empty_cache()
    if rank != 0:
        return None
    try:
        pk = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
        peak_tf, peak_src = float(pk['bf16_tflops_sustained']), 'measured sustained (MEASURED_PEAKS.json)'
    except Exception:
        peak_tf, peak_src = 1340.8, 'fallback'
    fpt = flops_per_token(cfg)
    achieved = fpt * B * T / (ms_max / K / 1e3) / 1e12
    roofline = {'bound': 'tensor', 'kernel': 'whole forward (attn_bert_tc_kernel 77 %, q/k/v GEMMs 14 %, residual + LayerNorm 9 % of the listed kernel time)', 'achieved': achieved,
                'peak': peak_tf, 'unit': 'TFLOP/s', 'frac': achieved / peak_tf, 'traffic': None, 'peak_source': peak_src,
                'flops_per_token_dense': fpt}
    cpu = None
    if world == 1 and not args.no_cpu_baseline and cpu_leg:
        v, n, threads, dt = cpu_reference(budget_s=15.0)
        cpu = {'value': v, 'unit': UNIT, 'cores': threads, 'kind': 'port',
               'sample': f'{n} forward(s) of 2 sequences x {T} tokens, fp32 eager-PyTorch oracle (oracle/bert.py), {dt:.1f} s'}
    line = {'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': K, 'warmup': W, 'ms_per_step': ms_max / K,
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'bf16', 'data': 'synthetic',
            'config': {'workload': workload_name(cfg, B), 'batch_per_gpu': B, 'global_batch': B * world, 'seq_len': T,
                       'parallelism': f'sequences sharded over {world} GPU(s), no collective',
                       'l2': 'activations per forward (q|k|v of 32-sequence chunks: 100 MB per layer and chunk, 16 chunks) exceed the 126 MB L2'},
            'roofline': roofline, 'cpu_baseline': cpu,
            'e2e': {'value': e2e_value, 'unit': UNIT, 'h2d_bytes_per_step': 2 * B * T * 8, 'd2h_bytes_per_step': B * V * 4, 'steps': Ke},
            'gpu_launches': launches, 'clocks': clock_info}
    return line


def cpu_reference(budget_s, batch=2):
    "The reference encoder (oracle/bert.py restatement of deep_music_remix.py:1851-2104) on the host cores, eager PyTorch fp32."
    from oracle import bert
    torch.manual_seed(0)
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    model = bert.get_multitask_model(V, bert.multitask_config()).eval()
    x, pos = synthetic(batch, torch.Generator().manual_seed(1))
    with torch.no_grad():
        model({'msk': {'x': x, 'pos': pos}})                     # warm-up
        done, t0 = 0, time.time()
        while True:
            model({'msk': {'x': x, 'pos': pos}})
            done += 1
            if time.time() - t0 > budget_s:
                break
        dt = time.time() - t0
    return batch * T * done / dt, done, threads, dt


def run_reference(args):
    if int(os.environ.get('RANK', '0')) != 0:
        return
    from oracle import bert
    v, n, threads, dt = cpu_reference(budget_s=min(60.0, 10.0 * max(1, args.steps)))
    sample = f'{n} forward(s) of 2 sequences x {T} tokens, fp32 eager-PyTorch oracle (reference algorithm), {threads} threads'
    line = {'impl': 'reference', 'metric': METRIC, 'value': v, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': n, 'warmup': 1,
            'ms_per_step': 1e3 * dt / n, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
            'data': 'synthetic', 'config': {'workload': workload_name(bert.multitask_config(), 2), 'cpu_batch': 2},
            'cpu_baseline': {'value': v, 'unit': UNIT, 'cores': threads, 'kind': 'port', 'sample': sample},
            'e2e': {'value': v, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}, 'gpu_launches': 0}
    print(json.dumps(line), flush=True)
