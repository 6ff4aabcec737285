#!/usr/bin/env python
"""Validation benchmark: held-out loss and accuracy on the device, as fit_one_cycle(valid_batches=...) runs them after every epoch.

Two workloads, each on synthetic LakhMIDI-shaped tokens resident on the device, bf16 compute / fp32 master weights:
- txl:   the C3 Transformer-XL (d_model 512, 16 layers, 8 heads x 64, d_inner 2048, mem_len 512, vocab 324), 32 x 512 tokens per batch
         over a warm 512-slot memory (S = 1024): valid_loss (CrossEntropyFlat) and accuracy.
- remix: the C4 remix encoder (d_model 512, 10 layers, 8 heads x 64), 32 x 1024 tokens per batch through mask_tfm(p 0.3):
         valid_loss (masked CrossEntropyFlat) and mask_acc.
For each, in the same run and on the same batches: the forward-only eval path (TXLTrainer / RemixTrainer.validate: dmg_train_eval_*,
metrics on the device, one host copy per validation) and, for comparison, the training engine's forward in eval mode
(dmg_train_forward(training=0): saves activations, computes dlogits, AR / TAR; one losses() read per batch as a caller must).
Prints one JSON line per workload with validated tokens/s and ms per batch, and the GPU name and power limit read in the same run.
--profile adds a torch.profiler run of one validation per workload (a separate, untimed pass) and reports the metrics kernel's time
next to the whole forward.

    python bench_validate.py [--batches 8] [--reps 3] [--workload txl,remix] [--profile] [--out DIR]
"""
import argparse
import json
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

V = 324


def setup(workload, B, n_batches, dev):
    import bench_train
    from deepmusicgeneration_b200.codec import MusicDataBunch
    toks = bench_train.lakh_shaped_tokens(B, n_batches * (1024 if workload == 'remix' else 512) + 1, torch.Generator().manual_seed(1234))
    vocab = MusicDataBunch.empty('').vocab
    if workload == 'txl':
        from deepmusicgeneration_b200.app_utils import baseline_config
        from deepmusicgeneration_b200.model import get_language_model
        from deepmusicgeneration_b200.training import TXLTrainer
        T = 512
        cfg = dict(baseline_config(), mask_steps=1)
        model = get_language_model(V, cfg, dtype='bf16', device=0, max_batch=1, max_seq=64, max_rows=64, keep_hidden=False, seed=0)
        tr = TXLTrainer(model, B, T, cfg, drop_mult=1.0, seed=7, distributed=False)
        batches = [(toks[:, i * T:(i + 1) * T].to(dev), toks[:, i * T + 1:(i + 1) * T + 1].to(dev), None) for i in range(n_batches)]
        shape = 'C3 Transformer-XL: d_model 512, 16 layers, 8 heads x 64, d_inner 2048, mem_len 512 (warm, S = 1024), vocab 324'
        return tr, batches, T, shape, lambda: tr.validate([(x, y) for x, y, _ in batches], reset=False)
    from deepmusicgeneration_b200.learner import multitask_model_learner
    from deepmusicgeneration_b200.preloader import mask_tfm
    from oracle.bert import multitask_config
    T = 1024
    learn = multitask_model_learner(MusicDataBunch(vocab), config=multitask_config(), dtype='bf16', max_batch=1, max_seq=T, seed=0)
    tr = learn.trainer(B, T, drop_mult=1.0, seed=7)
    pos = (torch.arange(T, device=dev) // 2).repeat(B, 1)
    batches = []
    for i in range(n_batches):
        x = toks[:, i * T:(i + 1) * T].contiguous().to(dev)
        xm, ym = mask_tfm((x, x), (vocab.note_range[0], vocab.dur_range[1]), vocab.mask_idx, vocab.pad_idx, p=0.3, seed=11 + i)
        batches.append((xm, ym, pos))
    shape = 'C4 remix encoder: d_model 512, 10 layers, 8 heads x 64, vocab 324, masked LM (mask_tfm p 0.3)'
    return tr, batches, T, shape, lambda: tr.validate(batches)


def run(workload, args, dev):
    B, n = args.batch, args.batches
    tr, batches, T, shape, validate = setup(workload, B, n, dev)
    if workload == 'txl':        # warm memory: one training-engine pass first so that every timed batch sees a full memory
        tr.reset()
        for x, y, p in batches[:2]:
            tr.step(x, y, p, lr=1e-5, mask_size=(1, 1))
    tr.eval()

    def train_fwd_eval():
        out = []
        for x, y, p in batches:
            tr.forward(x, y, p, mask_size=(1, 1))
            out.append(tr.losses()['ce'])
        return out

    for _ in range(2):           # warm-up of both paths
        r_eval = validate()
        train_fwd_eval()
    torch.cuda.synchronize()
    t_eval, t_fwd = [], []
    for _ in range(args.reps):   # alternate the two paths
        t0 = time.perf_counter(); r_eval = validate(); torch.cuda.synchronize(); t_eval.append(time.perf_counter() - t0)
        t0 = time.perf_counter(); ces = train_fwd_eval(); torch.cuda.synchronize(); t_fwd.append(time.perf_counter() - t0)
    tokens = B * T * n
    best_eval, best_fwd = min(t_eval), min(t_fwd)
    prof = None
    if args.profile:
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as p:
            validate()
            torch.cuda.synchronize()
        rows = p.key_averages()
        tot = sum(r.device_time_total for r in rows)
        met = sum(r.device_time_total for r in rows if 'eval_metrics' in r.key)
        fin = sum(r.device_time_total for r in rows if 'eval_metrics_final' in r.key)
        prof = {'batches': n, 'kernel_us_total': tot, 'metrics_kernels_us': met, 'metrics_final_us': fin,
                'metrics_us_per_batch': met / n, 'metrics_share': met / tot if tot else None,
                'logits_bytes_per_batch': B * T * ((V + 63) // 64 * 64) * 4}
        prof['metrics_gbps'] = prof['logits_bytes_per_batch'] / (met / n * 1e-6) / 1e9 if met else None
        if args.out:
            os.makedirs(args.out, exist_ok=True)
            with open(os.path.join(args.out, f'validate_{workload}_profile.txt'), 'w') as f:
                f.write(rows.table(sort_by='cuda_time_total', row_limit=30))
    tr.train()
    tr.close()
    return {'metric': 'validated_tokens_per_sec', 'workload': workload, 'value': tokens / best_eval, 'unit': 'tokens/s',
            'higher_is_better': True, 'ms_per_batch': best_eval / n * 1e3,
            'train_forward_eval_mode': {'tokens_per_sec': tokens / best_fwd, 'ms_per_batch': best_fwd / n * 1e3,
                                        'mean_ce': sum(ces) / len(ces)},
            'speedup_vs_train_forward': best_fwd / best_eval, 'result': r_eval, 'batches': n, 'reps': args.reps,
            'config': {'model': shape, 'batch': B, 'bptt': T, 'dtype': 'bf16'}, 'profile': prof}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--batch', type=int, default=32)
    ap.add_argument('--batches', type=int, default=8)
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--workload', default='txl,remix')
    ap.add_argument('--profile', action='store_true')
    ap.add_argument('--out', default=None, help='directory of the profiler tables (with --profile)')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_validate.py: no CUDA device - the CUDA path has no CPU fallback')
    from bench_remix_train import gpu_identity
    dev = torch.device('cuda', 0)
    name, limit = gpu_identity(dev)
    for w in args.workload.split(','):
        line = run(w, args, dev)
        line['gpu'] = {'name': name, 'power_limit_w': limit}
        print(json.dumps(line), flush=True)


if __name__ == '__main__':
    main()
