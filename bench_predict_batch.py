#!/usr/bin/env python
"""Genre continuation over seeds of their own lengths: the varlen prefill plus the device token loop of MusicLearner.predict_batch on
the C2 model (Transformer-XL d_model 512, 16 layers, 8 heads x 64, d_inner 2048, mem_len 512, vocab 324, seeded random init, bf16,
keep_hidden=False).  Seeds: B seeded synthetic note streams (default 256: note / duration pairs with separators, as the encoder
writes music) of lengths spread over [64, 1024], so that some memories stay short and some are full.  Loop: --steps steps (default
512) with the break rules off (no early stop, min_bars out of reach), so that every stream runs every step; top_k 30, top_p 0.65.

Reports the prefill time, the loop's ms per step and generated tokens/s, and in the same process the same numbers of generate_batch
on B equal 512-token seeds (the C2 geometry of bench.py) and of predict looped over the first --seq-items items (default 4).  Prints
one JSON line with the GPU name and power limit read in the same run.

    python bench_predict_batch.py [--items 256] [--steps 512] [--seq-items 4]
"""
import argparse
import contextlib
import io
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from bench_remix_train import gpu_identity  # noqa: E402

V = 324


def make_seeds(vocab, n, seed, lo=64, hi=1024):
    "note groups (note, duration) separated by xxsep + duration, lengths in [lo, hi]; every seed ends on a duration token"
    rng = np.random.default_rng(seed)
    items = []
    for _ in range(n):
        L = int(rng.integers(lo, hi + 1))
        data = [vocab.bos_idx, vocab.pad_idx]
        while len(data) < L:
            data += [vocab.note_range[0] + int(rng.integers(40, 90)), vocab.dur_range[0] + int(rng.integers(1, 16))]
            if rng.random() < 0.4:
                data += [vocab.sep_idx, vocab.dur_range[0] + int(rng.integers(1, 8))]
        data = data[:L] if vocab.is_duration(data[L - 1]) else data[:L - 1]
        items.append(vocab.to_music_item(np.asarray(data, dtype=np.int64)))
    return items


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--items', type=int, default=256)
    ap.add_argument('--steps', type=int, default=512)
    ap.add_argument('--seq-items', type=int, default=4)
    ap.add_argument('--seed', type=int, default=0)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_predict_batch.py needs a CUDA device')
    from deepmusicgeneration_b200 import _lib
    from deepmusicgeneration_b200.app_utils import baseline_config
    from deepmusicgeneration_b200.codec import MusicDataBunch
    from deepmusicgeneration_b200.learner import MusicLearner, sampler_params
    from deepmusicgeneration_b200.model import get_language_model
    dev = torch.device('cuda', 0)
    data = MusicDataBunch.empty('')
    vocab = data.vocab
    B, K = args.items, args.steps
    cfg = dict(baseline_config(), ctx_len=1024)
    model = get_language_model(V, cfg, dtype='bf16', device=0, max_batch=B, max_seq=1024, max_rows=B * 64, keep_hidden=False, seed=0)
    # the random-init head would sample the unused vocabulary tail (mt* / dummy tokens), after which predict raises the reference's
    # AssertionError; a trained model never does, so their bias is set far down, as the parity tests do
    sd = model.state_dict()
    sd['1.decoder.bias'][308:] = -50.
    model.load_state_dict(sd)
    learn = MusicLearner(data, model)
    no_break = dict(flags=_lib.SAMPLE_MASK_UNUSED, seed=7)   # no early stop, and min_bars below is out of reach

    def run(x, pos, lens):
        "prefill, then K loop steps: (prefill seconds, loop seconds, tokens [K, B])"
        model.reset()
        _, t_pre = timed(lambda: learn._prefill(x, pos, lens))
        last = (np.asarray(lens) - 1) if lens is not None else np.full(x.shape[0], x.shape[1] - 1)
        rows = np.arange(x.shape[0])
        prev, lp = x.cpu().numpy()[rows, last], pos.cpu().numpy()[rows, last]
        params = sampler_params(vocab, K, (1.0, 1.0, 1.0), 10 ** 6, 30, 0.65, None, **no_break)
        toks, t_loop = timed(lambda: learn._run_loop(K, prev, lp, params))
        return t_pre, t_loop, toks

    # ---- seeds of their own lengths (the predict_batch path)
    items = make_seeds(vocab, B, args.seed)
    lens = np.array([len(it.data) for it in items], dtype=np.int32)
    T = int(lens.max())
    x = np.full((B, T), vocab.pad_idx, dtype=np.int64)
    pos = np.zeros((B, T), dtype=np.int64)
    for b, it in enumerate(items):
        x[b, :lens[b]] = it.data
        pos[b, :lens[b]] = it.position
    xv, pv = torch.from_numpy(x).to(dev), torch.from_numpy(pos).to(dev)
    run(xv, pv, lens)                                   # warm-up: module load, tensor maps, graph capture
    v_pre, v_loop, toks = run(xv, pv, lens)
    stopped = int((toks < 0).any(0).sum())             # expected 0: the break rules are off
    mc = model._e.mem_counts(B)

    # ---- C2 geometry: B equal 512-token seeds (generate_batch's path)
    eq = np.stack([np.resize(it.data[2:], 512) for it in items])      # the same grammar, cut / repeated to 512 tokens
    eq[:, -1] = vocab.dur_range[0] + 1
    xe, pe = torch.from_numpy(eq).to(dev), torch.zeros(B, 512, dtype=torch.int64, device=dev)
    run(xe, pe, None)
    e_pre, e_loop, _ = run(xe, pe, None)

    # ---- predict, one item after the other
    S = min(args.seq_items, B)
    kw = dict(n_words=K, temperatures=(1.0, 1.0, 1.0), min_bars=10 ** 6, top_k=30, top_p=0.65, seed=7)
    with contextlib.redirect_stdout(io.StringIO()):     # predict prints its first prev_idx, as the reference does
        learn.predict(items[0], **dict(kw, n_words=8))
        outs, t_seq = timed(lambda: [learn.predict(it, **kw)[0] for it in items[:S]])
    seq_tokens = sum(len(o.data) for o in outs)

    name, limit = gpu_identity(dev)
    line = {'metric': 'predict_batch_generated_tok_per_sec', 'value': B * K / v_loop, 'unit': 'tok/s', 'higher_is_better': True,
            'dtype': 'bf16',
            'config': {'workload': 'varlen prefill + device token loop, C2 model (d_model 512, 16 layers, 8 heads x 64, d_inner 2048, '
                                   'mem_len 512, vocab 324), seeded init with the unused vocabulary tail biased to -50, keep_hidden=False, break rules off',
                       'items': B, 'steps': K, 'lengths': [int(lens.min()), int(lens.max())], 'seed_tokens': int(lens.sum()),
                       'streams_with_short_memory_after_prefill': int(sum(int(n) < 512 for n in lens)), 'top_k': 30, 'top_p': 0.65},
            'varlen': {'prefill_s': v_pre, 'loop_s': v_loop, 'ms_per_step': v_loop * 1e3 / K, 'generated_tok_per_s': B * K / v_loop,
                       'streams_stopped': stopped, 'mem_counts_after_loop': [min(mc), max(mc)]},
            'equal_512_c2_geometry': {'prefill_s': e_pre, 'loop_s': e_loop, 'ms_per_step': e_loop * 1e3 / K,
                                      'generated_tok_per_s': B * K / e_loop},
            'sequential_predict': {'items': S, 'generated_tokens': seq_tokens, 'seconds': t_seq, 'generated_tok_per_s': seq_tokens / t_seq},
            'gpu': {'name': name, 'power_limit_w': limit}}
    print(json.dumps(line), flush=True)


if __name__ == '__main__':
    main()
