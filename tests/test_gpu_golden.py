"""The CUDA path (through the C ABI) against tests/golden/model_golden.npz - outputs of the REFERENCE'S OWN source
(deep_music_genre.py / deep_music_remix.py executed by tests/golden/make_model_golden.py; fastai names stubbed).  The oracle is not
involved here except to name the weight tensors: fixture == reference source, CUDA == fixture.

Tolerances: fp32 mode 5e-4 absolute on logits; bf16 mode |a-b| <= 2e-2 * max(|b|, sigma) with sigma = std of the fixture logits.
Token streams and kept sets: exact."""
import ast
import ctypes as C
import os
import sys

import numpy as np
import pytest
import torch

from oracle import bert as obert, txl

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden'))
from golden_weights import golden_state_dict, kept_positions      # noqa: E402

pytestmark = pytest.mark.gpu
V = 324


@pytest.fixture(scope='module')
def G(golden_dir):
    return np.load(os.path.join(golden_dir, 'model_golden.npz'), allow_pickle=False)


def _txl_product(cfg, seed, dtype, max_batch, max_seq, tame=False, **kw):
    from deepmusicgeneration_b200.model import get_language_model
    names = txl.get_language_model(V, cfg).state_dict()            # only names and shapes are taken from the oracle model
    sd = golden_state_dict(names, seed)
    if tame:
        sd['1.decoder.bias'] = sd['1.decoder.bias'].clone()
        sd['1.decoder.bias'][308:] = -50.
    pm = get_language_model(V, cfg, dtype=dtype, max_batch=max_batch, max_seq=max_seq, init=False, **kw)
    pm.load_state_dict(sd)
    return pm


def _bert_product(cfg, seed, dtype, max_batch, max_seq):
    from deepmusicgeneration_b200.model import get_multitask_model
    names = obert.get_multitask_model(V, dict(cfg), pad_idx=1).state_dict()
    pm = get_multitask_model(V, dict(cfg), pad_idx=1, dtype=dtype, max_batch=max_batch, max_seq=max_seq, init=False)
    pm.load_state_dict(golden_state_dict(names, seed))
    return pm


def _bf16_ok(a, b):
    sigma = float(b.std())
    return float((np.abs(a - b) / np.maximum(np.abs(b), sigma)).max())


@pytest.mark.parametrize('dtype', ['f32', 'bf16'])
def test_txl_forward_override_against_reference_source(G, dtype):
    cfg = ast.literal_eval(str(G['txl_cfg']))
    pm = _txl_product(cfg, 11, dtype, 3, 64)
    pm.reset()
    worst = 0.
    for s, T in enumerate(G['txl_segments']):
        x, pos = torch.from_numpy(G[f'txl_x{s}']).cuda(), torch.from_numpy(G[f'txl_pos{s}']).cuda()
        logits, raw, outs = pm({'x': x, 'pos': pos})
        logits = kept_positions(G, f'txl_logits{s}', logits.cpu().numpy())
        core = kept_positions(G, f'txl_core{s}', outs[0].cpu().numpy())
        mem = kept_positions(G, f'txl_mem_last{s}', raw[-1].cpu().numpy())
        if dtype == 'f32':
            assert np.abs(logits - G[f'txl_logits{s}']).max() < 5e-4, s
            assert np.abs(core - G[f'txl_core{s}']).max() < 5e-4, s
            assert np.abs(mem - G[f'txl_mem_last{s}']).max() < 5e-4, s
        else:
            worst = max(worst, _bf16_ok(logits, G[f'txl_logits{s}']))
    x, pos = torch.from_numpy(G['txl_win_x']).cuda(), torch.from_numpy(G['txl_win_pos']).cuda()
    lw = pm({'x': x, 'pos': pos}, mask_size=(3, 0))[0].cpu().numpy()           # the training-time window mask over the memory
    lw = kept_positions(G, 'txl_win_logits', lw)
    if dtype == 'f32':
        assert np.abs(lw - G['txl_win_logits']).max() < 5e-4
    else:
        worst = max(worst, _bf16_ok(lw, G['txl_win_logits']))
        print(f'bf16 vs reference-source fixture: max |a-b| / max(|b|, sigma) = {worst:.3e}')
        assert worst <= 2e-2


@pytest.mark.parametrize('tag', ['a', 'b'])
def test_predict_greedy_stream_against_reference_source(G, tag):
    "MusicLearner.predict (fp32, greedy) reproduces the token stream the reference's own predict loop wrote"
    from deepmusicgeneration_b200.codec import MusicDataBunch, MusicItem
    from deepmusicgeneration_b200.learner import MusicLearner
    cfg = ast.literal_eval(str(G[f'predict_{tag}_cfg']))
    pm = _txl_product(cfg, 12, 'f32', 1, 256, tame=True, keep_hidden=False)
    data = MusicDataBunch.empty('')
    item = MusicItem(G[f'predict_{tag}_seed'].copy(), data.vocab)
    assert np.array_equal(item.position, G['predict_seed_positions_full'][:len(item.data)])
    allowed = [str(a) for a in G[f'predict_{tag}_allowed']] or None
    n_words = {'a': 160, 'b': 120}[tag]
    pred, full = MusicLearner(data, pm).predict(item, n_words=n_words, temperatures=(1.3, 1.1, 0.9), min_bars=12, top_k=1, top_p=0.0,
                                                allowed_ins=allowed)
    assert list(pred.data) == list(G[f'predict_{tag}_tokens'])
    assert list(full.data) == list(G[f'predict_{tag}_seed']) + list(G[f'predict_{tag}_tokens'])
    if allowed:
        assert allowed == [str(a) for a in G[f'predict_{tag}_allowed_after']]


@pytest.mark.parametrize('dtype', ['f32', 'bf16'])
def test_bert_encoder_against_reference_source(G, dtype):
    cfg = ast.literal_eval(str(G['bert_cfg']))
    pm = _bert_product(cfg, 13, dtype, 2, 320)
    worst = 0.
    for T in G['bert_lengths']:
        x, pos = torch.from_numpy(G[f'bert_x{T}']).cuda(), torch.from_numpy(G[f'bert_pos{T}']).cuda()
        out = kept_positions(G, f'bert_logits{T}', pm({'msk': {'x': x, 'pos': pos}})['msk'].cpu().numpy())
        if dtype == 'f32':
            assert np.abs(out - G[f'bert_logits{T}']).max() < 5e-4, T
        else:
            worst = max(worst, _bf16_ok(out, G[f'bert_logits{T}']))
    if dtype == 'bf16':
        print(f'bert bf16 vs reference-source fixture: {worst:.3e}')
        assert worst <= 2e-2


def test_predict_mask_against_reference_source(G):
    from deepmusicgeneration_b200.codec import MusicDataBunch, MusicItem
    from deepmusicgeneration_b200.learner import MultitaskLearner
    cfg = ast.literal_eval(str(G['bert_cfg']))
    pm = _bert_product(cfg, 13, 'f32', 1, 256)
    data = MusicDataBunch.empty('')
    item = MusicItem(G['predict_mask_in'].copy(), data.vocab, position=G['predict_mask_pos'].copy())
    out = MultitaskLearner(data, pm).predict_mask(item, temperatures=(1.1, 0.9), top_k=1, top_p=0.0)
    assert list(out.data) == list(G['predict_mask_out'])


# --------------------------------------------------------------------------------------------- device sampler: kept sets
def _p(t): return C.c_void_p(t.data_ptr())


@pytest.fixture(scope='module')
def engine():
    from deepmusicgeneration_b200.model import get_multitask_model
    cfg = dict(d_model=128, n_heads=2, d_head=64, d_inner=256, enc_layers=1, mem_len=512, bias=True)
    return get_multitask_model(V, cfg, dtype='f32', max_batch=1, max_seq=8, seed=0)._e


def _probs(e, predict_loop, logits, prev, rc, last_xxsep, since, temperatures, min_bars, top_k, top_p, allowed_mask=0, flags=0):
    from deepmusicgeneration_b200.codec import MusicVocab
    from deepmusicgeneration_b200.learner import sampler_params, vocab_layout
    vocab = MusicVocab.create()
    vl = vocab_layout(vocab)
    params = sampler_params(vocab, 1000, temperatures, min_bars, top_k, top_p, None, flags=flags, seed=3)
    params.allowed_ins_mask = int(allowed_mask)
    n = logits.shape[0]
    dev = lambda a, dt: torch.as_tensor(np.asarray(a), dtype=dt).cuda()
    lg, pv, rcd, lx, sn = dev(logits, torch.float32), dev(prev, torch.int32), dev(rc, torch.int32), dev(last_xxsep, torch.int32), dev(since, torch.int64)
    out = torch.zeros(n, dtype=torch.int32, device='cuda'); nc = torch.zeros(n, dtype=torch.int32, device='cuda')
    probs = torch.zeros(n, V, dtype=torch.float32, device='cuda')
    rcode = e.lib.dmg_sample_probs(e.h, predict_loop, _p(lg), _p(pv), _p(rcd), _p(lx), _p(sn), n, C.byref(vl), C.byref(params), 0, _p(out),
                                   _p(nc), _p(probs), C.c_void_p(0))
    assert rcode == 0, e.lib.dmg_last_error()
    torch.cuda.synchronize()
    return out.cpu().numpy(), nc.cpu().numpy(), probs.cpu().numpy()


def test_genre_filter_kept_sets_and_allowed_ins(G, engine):
    "filter_invalid_indexes of deep_music_genre.py:1984-2018 on the device: the support of the probabilities == the reference's kept set"
    prevs, allowed = G['filter_prev'], G['filter_allowed']
    flat = np.zeros((1, V), dtype=np.float32)                    # flat logits: nothing but the filter decides the support
    for a, prev in enumerate(prevs):
        for b, last in enumerate((0, 1)):
            # the loop updates last_xxsep from prev before filtering (:1897-1901); the fixture passed it explicitly, so feed a state the update keeps
            if (prev == 11 and last == 0) or (prev == 10 and last == 1):
                continue
            for c, bits in enumerate(allowed):
                ref = G['filter_genre_kept'][a, b, c]
                tok, nc, probs = _probs(engine, 1, flat, [prev], [0], [last], [10 ** 6], (1., 1., 1.), 0, 0, 0.0, allowed_mask=bits)
                temp_class = (140 <= prev < 301) or prev == 11 or (12 <= prev < 140) or prev == 10 or (301 <= prev < 308) or prev == 1
                if not temp_class:
                    assert tok[0] == -2                                       # the reference raises AssertionError (:1920-1925)
                    continue
                assert np.array_equal(probs[0] > 0, ref), (int(prev), last, int(bits))
                assert int(nc[0]) == int(ref.sum())


def test_remix_filter_kept_sets(G, engine):
    from deepmusicgeneration_b200 import _lib as L
    flat = np.zeros((1, V), dtype=np.float32)
    special = [0, 11, 10, 2, 4, 5, 6, 7, 8, 9]                   # predict_mask removes these before the filter (deep_music_remix.py:2595-2596)
    for a, prev in enumerate(G['filter_prev']):
        ref = G['filter_remix_kept'][a].copy()
        ref[special] = False
        tok, nc, probs = _probs(engine, 0, flat, [prev], [0], [0], [0], (1., 1.), 0, 0, 0.0, flags=L.SAMPLE_REMIX_FILTER)
        assert np.array_equal(probs[0] > 0, ref), int(prev)


def test_top_k_top_p_kept_sets_on_device(G, engine):
    "top_k_top_p (deep_music_genre.py:1679-1706): the kept set of the device sampler == the reference's, row by row"
    logits = G['topk_logits']
    n = logits.shape[0]
    # previous token = a note -> only durations survive the grammar filter; the fixture applied the reference function to rows
    # restricted the same way (make_model_golden.py: topk_kept_after_note)
    for c, (k, p) in enumerate(G['topk_cases']):
        tok, nc, probs = _probs(engine, 1, logits, [60 + 12] * n, [0] * n, [0] * n, [10 ** 6] * n, (1., 1., 1.), 0, int(k), float(p))
        for r in range(n):
            assert np.array_equal(probs[r] > 0, G['topk_kept_after_note'][c, r]), (k, p, r)
            assert probs[r, tok[r]] > 0
