#!/usr/bin/env python
"""Batched-remix benchmark: MultitaskLearner.predict_mask_batch against the one-item predict_mask on the C4 encoder geometry
(d_model 512, 10 layers, 8 heads x 64, vocab 324, seeded random init, bf16).  Items: B seeded synthetic note streams (default 64) of
seeded lengths in [200, 1024], 60 % of their notes masked as predictMaskModel masks them.  Sampling: top_k 20, top_p 0.8, seed 0.

Reports for the batched loop items/s, masked tokens/s, ms per loop step and the encoder tokens/s of one step (sum of the item lengths
per step time; the one-forward C4 rate is the yardstick), and the same items through predict_mask one by one (a stated subset: the
first --seq-items items, default 4).  Prints one JSON line with the GPU name and power limit read in the same run.

    python bench_remix_predict.py [--items 64] [--seq-items 4]
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from bench_remix_train import gpu_identity  # noqa: E402


def make_items(vocab, n, seed):
    "note groups (note, duration) separated by xxsep + duration, lengths in [200, 1024]; 60 % of the notes masked"
    rng = np.random.default_rng(seed)
    items = []
    for _ in range(n):
        L = int(rng.integers(200, 1025))
        data = [vocab.bos_idx, vocab.pad_idx]
        while len(data) < L:
            data += [vocab.note_range[0] + int(rng.integers(40, 90)), vocab.dur_range[0] + int(rng.integers(1, 16))]
            if rng.random() < 0.4:
                data += [vocab.sep_idx, vocab.dur_range[0] + int(rng.integers(1, 8))]
        it = vocab.to_music_item(np.asarray(data[:L], dtype=np.int64))
        _ = it.position
        notes = np.flatnonzero((it.data >= vocab.note_range[0]) & (it.data < vocab.note_range[1]))
        it.data[rng.choice(notes, int(0.6 * len(notes)), replace=False)] = vocab.mask_idx
        items.append(it)
    return items


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--items', type=int, default=64)
    ap.add_argument('--seq-items', type=int, default=4)
    ap.add_argument('--seed', type=int, default=0)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_remix_predict.py needs a CUDA device')
    from oracle import bert as obert
    from deepmusicgeneration_b200.codec import MusicDataBunch
    from deepmusicgeneration_b200.learner import MultitaskLearner
    from deepmusicgeneration_b200.model import get_multitask_model
    dev = torch.device('cuda', 0)
    data = MusicDataBunch.empty('')
    vocab = data.vocab
    cfg = obert.multitask_config()
    B = args.items
    model = get_multitask_model(len(vocab.itos), cfg, pad_idx=vocab.pad_idx, dtype='bf16', device=0, max_batch=B, max_seq=1024,
                                seed=args.seed)
    learn = MultitaskLearner(data, model)
    items = make_items(vocab, B, args.seed)
    n_masks = [int((it.data == vocab.mask_idx).sum()) for it in items]
    kw = dict(temperatures=(1.0, 1.0), top_k=20, top_p=0.8, seed=0)

    learn.predict_mask_batch(items[:2], **kw)            # warm-up: module load, tensor maps, one-time attributes
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = learn.predict_mask_batch(items, **kw)
    torch.cuda.synchronize()
    t_batch = time.perf_counter() - t0
    assert all((o.data != vocab.mask_idx).all() for o in out)
    steps = max(n_masks)
    step_ms = t_batch * 1e3 / steps

    S = min(args.seq_items, B)
    learn.predict_mask(items[0], **kw)                   # warm-up of the one-item path
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for it in items[:S]:
        learn.predict_mask(it, **kw)
    torch.cuda.synchronize()
    t_seq = time.perf_counter() - t0
    seq_masks = sum(n_masks[:S])

    name, limit = gpu_identity(dev)
    line = {'metric': 'remix_items_per_sec', 'value': B / t_batch, 'unit': 'items/s', 'higher_is_better': True, 'dtype': 'bf16',
            'config': {'workload': 'predict_mask_batch, C4 encoder geometry (d_model 512, 10 layers, 8 heads x 64, vocab 324), seeded init',
                       'items': B, 'lengths': [int(min(len(it.data) for it in items)), int(max(len(it.data) for it in items))],
                       'masked_tokens': int(sum(n_masks)), 'loop_steps': steps, 'top_k': 20, 'top_p': 0.8},
            'batched': {'seconds': t_batch, 'items_per_s': B / t_batch, 'masked_tokens_per_s': sum(n_masks) / t_batch,
                        'ms_per_step': step_ms,
                        'encoder_tokens_per_s_per_step': sum(len(it.data) for it in items) / (step_ms / 1e3)},
            'sequential_predict_mask': {'items': S, 'masked_tokens': seq_masks, 'seconds': t_seq, 'ms_per_mask': t_seq * 1e3 / seq_masks,
                                        'items_per_s': S / t_seq, 'masked_tokens_per_s': seq_masks / t_seq},
            'speedup_masked_tokens_per_s': (sum(n_masks) / t_batch) / (seq_masks / t_seq),
            'gpu': {'name': name, 'power_limit_w': limit}}
    print(json.dumps(line), flush=True)


if __name__ == '__main__':
    main()
