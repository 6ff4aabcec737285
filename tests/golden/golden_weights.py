"""Deterministic weights for the golden model fixtures (shared by make_model_golden.py and the tests).

The fixture file stores inputs and outputs only; the weights are re-created here from numpy's legacy ``RandomState`` stream (frozen by
numpy's compatibility policy, NEP 19), one stream per tensor keyed by (seed, crc32(name)) so that a model holding only a subset of the
reference's tensors (the oracle builds encoder + head only) gets the same values; distributions are the ones fastai's
``init_transformer`` leaves behind (SURVEY.md App. A.6).
``weights_checksum`` of the result is stored in the fixture so a drifted stream would be noticed.

To keep the fixture file under 1 MB, the large outputs keep two positions (axis 1) in five: always the first and the last, the rest
a fixed, seeded draw.  ``sample_positions`` does that when the fixture is written; ``kept_positions`` picks the same positions out of
a full output in the tests.
"""
import re
import zlib

import numpy as np
import torch

SAMPLED = re.compile(r'((txl_logits|txl_core|txl_mem_last|bert_logits)\d+|txl_win_logits)$')


def golden_state_dict(reference_state, seed):
    "`reference_state`: a state_dict (names -> tensors) that gives names and shapes; returns a new dict of fp32 tensors."
    out = {}
    alias = {'1.decoder.weight': '0.encoder.weight', 'head.decoder.weight': 'encoder.embed.embed.weight'}
    for name in sorted(reference_state.keys()):
        t = reference_state[name]
        shape = tuple(t.shape)
        if name.endswith('pos_enc.freq'):
            out[name] = t.clone()
            continue
        src = alias.get(name, name)
        if src.startswith('decoder.embed.'):                       # the remix decoder shares the encoder's embedding module
            src = 'encoder.embed.' + src[len('decoder.embed.'):]
        rs = np.random.RandomState((zlib.crc32(src.encode()) ^ (seed * 2654435761)) & 0xffffffff)
        w = rs.standard_normal(shape).astype(np.float32)
        if 'beat_enc' in name or 'bar_enc' in name:
            w[0] = 0                                              # nn.Embedding(padding_idx=0), N(0, 1)
        elif name.endswith('.bias'):
            w *= 0.01                                             # zero after init_transformer; small non-zero values exercise every bias path
        elif '.ln.' in name or '.ff.layers.6.' in name or name.endswith('ln.weight'):
            w = 1.0 + 0.02 * w
        else:
            w *= 0.02
        out[name] = torch.from_numpy(w)
    return out


def weights_checksum(state):
    "Sum of |w| over the tensors of the hot path (the remix decoder, mha2 and ff blocks are not on it and not in every model)."
    skip = lambda k: k.endswith('pos_enc.freq') or k.startswith('decoder.') or '.mha2.' in k or (k.startswith('encoder.') and '.ff.' in k)
    return float(sum(float(v.double().abs().sum()) for k, v in sorted(state.items()) if not skip(k)))


def sample_positions(out, seed=0):
    "In place: every output named by SAMPLED keeps 2 of 5 positions; `<key>_rows` records which, `<key>_shape` the full shape."
    rng = np.random.default_rng(seed)
    for key in sorted(k for k in out if SAMPLED.match(k)):
        a = out[key]
        T = a.shape[1]
        k = -(-2 * T // 5)
        rows = np.arange(T) if k >= T - 1 else np.sort(np.r_[0, T - 1, 1 + rng.choice(T - 2, k - 2, replace=False)])
        out[key], out[key + '_rows'], out[key + '_shape'] = a[:, rows], rows, np.array(a.shape)


def kept_positions(G, key, full):
    "The positions of `full` (an output computed in full) that fixture `G` kept for `key`, after checking the full shape."
    assert tuple(full.shape) == tuple(G[key + '_shape']), (key, full.shape, G[key + '_shape'])
    return full[:, G[key + '_rows']]
