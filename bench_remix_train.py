#!/usr/bin/env python
"""Remix-encoder training benchmark: masked-LM training step of the C4 encoder (d_model 512, 10 layers, 8 heads x 64, vocab 324,
no memory, wrap-around rel-pos attention) at T = 1024 with B sequences per GPU (default 32), dropout 0.1 (drop_mult 1), bf16
compute / fp32 master weights.  Inputs: synthetic LakhMIDI-shaped token streams through mask_tfm (p 0.3, the preloader golden's
mask range), resident on the device.  A "step" = forward + masked cross entropy + backward + Adam.  Prints one JSON line: trained
tokens/s, ms/step, the dense FLOP count and its share of the sustained bf16 rate, with the GPU name and power limit read in the
same run.  --profile writes a torch.profiler kernel table of one step (a separate run: tracing slows the host) to --out.

    python bench_remix_train.py [--batch 32] [--steps 20] [--warmup 5] [--profile --out DIR]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

V, T = 324, 1024
METRIC, UNIT = 'trained_tokens_per_sec', 'tokens/s'


def flops_per_token(d=512, L=10, H=8, Dh=64, T=T):
    """Dense-count FLOPs per token: per layer the q/k/v projections (3 * 2 d HD) and the attention contractions QK^T, the
    position term and PV (3 * 2 HD T), plus the tied head (2 d V); the step (forward + backward) is 3x the forward."""
    HD = H * Dh
    fwd = L * (3 * 2 * d * HD + 3 * 2 * HD * T) + 2 * d * V
    return fwd, 3 * fwd


def gpu_identity(dev):
    "name and power limit of the card, read now (the numbers of this run belong to them)"
    name, limit = torch.cuda.get_device_name(dev), None
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader,nounits', '-i', str(dev.index)],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        limit = float(out.splitlines()[0])
    except Exception:
        pass
    return name, limit


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--batch', type=int, default=32)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--profile', action='store_true', help='one profiled step instead of the timed run')
    ap.add_argument('--out', default=None, help='directory of the profiler table (with --profile)')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_remix_train.py: no CUDA device - the CUDA path has no CPU fallback')
    import bench_train
    from deepmusicgeneration_b200.codec import MusicDataBunch
    from deepmusicgeneration_b200.learner import multitask_model_learner
    from deepmusicgeneration_b200.preloader import mask_tfm
    from oracle.bert import multitask_config

    dev = torch.device('cuda', 0)
    B, K, W = args.batch, args.steps, max(1, args.warmup)
    data = MusicDataBunch.empty('')
    vocab = data.vocab
    cfg = multitask_config()
    learn = multitask_model_learner(data, config=cfg, dtype='bf16', max_batch=1, max_seq=T, seed=0)
    tr = learn.trainer(B, T, drop_mult=1.0, seed=7)
    n_batches = 4
    toks = bench_train.lakh_shaped_tokens(B, n_batches * T, torch.Generator().manual_seed(1234))
    pos = (torch.arange(T, device=dev) // 2).repeat(B, 1)        # one beat step per (note, duration) pair
    batches = []
    for i in range(n_batches):
        x = toks[:, i * T:(i + 1) * T].contiguous().to(dev)
        batches.append(mask_tfm((x, x), (vocab.note_range[0], vocab.dur_range[1]), vocab.mask_idx, vocab.pad_idx, p=0.3, seed=11 + i))

    def step(i):
        x, y = batches[i % n_batches]
        tr.step(x, y, pos, lr=1e-4)

    for i in range(W):
        step(i)
    torch.cuda.synchronize()
    l0 = tr.losses()

    if args.profile:
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            step(0)
            torch.cuda.synchronize()
        table = prof.key_averages().table(sort_by='cuda_time_total', row_limit=40)
        print(table)
        if args.out:
            os.makedirs(args.out, exist_ok=True)
            with open(os.path.join(args.out, 'remix_train_profile.txt'), 'w') as f:
                f.write(table)
        return

    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for i in range(K):
        step(i)
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1)
    l1 = tr.losses()
    step_ms = ms / K
    fwd_f, fb_f = flops_per_token()
    try:
        pk = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
        peak_tf, peak_src = float(pk['bf16_tflops_sustained']), 'measured sustained (MEASURED_PEAKS.json)'
    except Exception:
        peak_tf, peak_src = 1340.8, 'fallback (the sustained dense bf16 rate bench_train.py assumes)'
    achieved = fb_f * B * T / (step_ms / 1e3) / 1e12
    name, limit = gpu_identity(dev)
    line = {'metric': METRIC, 'value': B * T * K / (ms / 1e3), 'unit': UNIT, 'n_gpus': 1, 'steps': K, 'warmup': W, 'ms_per_step': step_ms,
            'higher_is_better': True, 'dtype': 'bf16', 'data': 'synthetic LakhMIDI-shaped tokens + mask_tfm(p=0.3)',
            'config': {'workload': 'remix encoder masked-LM training: d_model 512, 10 layers, 8 heads x 64, vocab 324, T 1024, '
                                   'dropout 0.1, Adam(true_wd), clip 0.5', 'batch_per_gpu': B, 'bptt': T,
                       'ce_before': l0['ce'], 'ce_after': l1['ce'], 'grad_norm': l1['grad_norm']},
            'roofline': {'bound': 'tensor', 'kernel': 'whole training step', 'achieved': achieved, 'peak': peak_tf, 'unit': 'TFLOP/s',
                         'frac': achieved / peak_tf, 'peak_source': peak_src, 'flops_per_token_fwd_bwd_dense': fb_f,
                         'flops_per_token_fwd_dense': fwd_f},
            'gpu': {'name': name, 'power_limit_w': limit}}
    print(json.dumps(line), flush=True)
    tr.close()


if __name__ == '__main__':
    main()
