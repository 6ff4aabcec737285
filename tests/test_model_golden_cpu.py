"""The oracle against tests/golden/model_golden.npz - outputs of the REFERENCE'S OWN source (deep_music_genre.py /
deep_music_remix.py) executed by tests/golden/make_model_golden.py with the un-vendored fastai names stubbed.  This is what pins the
oracle's masks, forward override, BERT attention twin, sampling filters and generation loops to the reference (SURVEY.md 8c).
CPU only; the CUDA path is checked against the same fixture in tests/test_gpu_golden.py."""
import ast
import os
import sys

import numpy as np
import pytest
import torch

from oracle import bert as obert, codec as ocodec, sampling as osamp, txl

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden'))
from golden_weights import golden_state_dict, kept_positions, weights_checksum      # noqa: E402


@pytest.fixture(scope='module')
def G(golden_dir):
    return np.load(os.path.join(golden_dir, 'model_golden.npz'), allow_pickle=False)


def oracle_txl(cfg, seed):
    m = txl.get_language_model(324, cfg).eval()
    sd = golden_state_dict(m.state_dict(), seed)
    m.load_state_dict(sd, strict=True)
    return m, sd


def test_vocab_is_the_reference_vocab(G):
    from deepmusicgeneration_b200.codec import MusicVocab
    itos = [str(s) for s in G['vocab_itos']]
    assert ocodec.MusicVocab.create().itos == itos
    assert list(MusicVocab.create().itos) == itos


def test_window_masks(G):
    for i, (x_len, m_len, win, k) in enumerate(G['mask_cases']):
        m = txl.window_mask(int(x_len), 'cpu', int(m_len), size=(int(win), int(k)))[0, 0].numpy()
        assert np.array_equal(m, G[f'mask_{i}']), (x_len, m_len, win, k)


def test_rand_window_mask_draws_and_host_mirror(G):
    from deepmusicgeneration_b200.training import rand_window_mask_size
    np.random.seed(4)
    for ref in G['rand_mask_draws']:
        m = txl.rand_window_mask(8, 2, 'cpu', max_size=4, p=0.2, is_eval=False)[0, 0].numpy()
        assert np.array_equal(m, ref)
    np.random.seed(4)
    for ref in G['rand_mask_draws']:                # the product draws (win, k) on the host and applies them by index arithmetic
        size = rand_window_mask_size(max_size=4, p=0.2, is_eval=False)
        assert np.array_equal(txl.window_mask(8, 'cpu', 2, size=size)[0, 0].numpy(), ref)
    assert np.array_equal(txl.rand_window_mask(8, 2, 'cpu', max_size=4, is_eval=True)[0, 0].numpy(), G['rand_mask_eval'])
    assert rand_window_mask_size(max_size=4, is_eval=True) == (1, 1)


def test_top_k_top_p_kept_sets(G):
    logits = torch.from_numpy(G['topk_logits'])
    for c, (k, p) in enumerate(G['topk_cases']):
        for r, row in enumerate(logits):
            kept = torch.isfinite(osamp.top_k_top_p(row, top_k=int(k), top_p=float(p))).numpy()
            assert np.array_equal(kept, G['topk_kept'][c, r]), (k, p, r)
            dur = osamp.filter_invalid_indexes(row.clone(), 72, ocodec.MusicVocab.create())
            assert np.array_equal(torch.isfinite(osamp.top_k_top_p(dur, top_k=int(k), top_p=float(p))).numpy(),
                                  G['topk_kept_after_note'][c, r])


def test_filter_invalid_indexes_kept_sets(G):
    v = ocodec.MusicVocab.create()
    for a, prev in enumerate(G['filter_prev']):
        for b, last in enumerate((False, True)):
            for c, bits in enumerate(G['filter_allowed']):
                allowed = None if bits == 0 else [f'i{i}' for i in range(7) if bits >> i & 1]
                res = osamp.filter_invalid_indexes(torch.zeros(324), int(prev), v, last_xxsep=last, allowed_ins=allowed)
                assert np.array_equal(torch.isfinite(res).numpy(), G['filter_genre_kept'][a, b, c]), (prev, last, allowed)
        res = osamp.filter_invalid_indexes_remix(torch.zeros(324), int(prev), v)
        assert np.array_equal(torch.isfinite(res).numpy(), G['filter_remix_kept'][a]), prev


def test_txl_forward_override_logits_and_mems(G):
    cfg = ast.literal_eval(str(G['txl_cfg']))
    m, sd = oracle_txl(cfg, seed=11)
    assert sorted(sd.keys()) == [str(k) for k in G['txl_state_keys']]          # fastai state-dict key names (SURVEY App. A.8)
    assert abs(weights_checksum(sd) - float(G['txl_weights_checksum'])) < 1e-6 * float(G['txl_weights_checksum'])
    m.reset()
    with torch.no_grad():
        for s, T in enumerate(G['txl_segments']):
            x, pos = torch.from_numpy(G[f'txl_x{s}']), torch.from_numpy(G[f'txl_pos{s}'])
            decoded, raw, outs = m({'x': x, 'pos': pos.clone()})
            assert np.abs(kept_positions(G, f'txl_logits{s}', decoded.numpy()) - G[f'txl_logits{s}']).max() < 2e-5, s
            assert np.abs(kept_positions(G, f'txl_core{s}', outs[0].numpy()) - G[f'txl_core{s}']).max() < 2e-5, s
            assert np.abs(kept_positions(G, f'txl_mem_last{s}', raw[-1].numpy()) - G[f'txl_mem_last{s}']).max() < 2e-5, s
    # the forced (3, 0) training window over the memory
    orig = txl.rand_window_mask
    txl.rand_window_mask = lambda x_len, m_len, device, **kw: txl.window_mask(x_len, device, m_len, size=(3, 0))
    try:
        m.train()
        for mod in m.modules():
            if hasattr(mod, 'p'): mod.p = 0.
        with torch.no_grad():
            lw = m({'x': torch.from_numpy(G['txl_win_x']), 'pos': torch.from_numpy(G['txl_win_pos'])})[0]
    finally:
        txl.rand_window_mask = orig
    assert np.abs(kept_positions(G, 'txl_win_logits', lw.numpy()) - G['txl_win_logits']).max() < 2e-5


@pytest.mark.parametrize('tag', ['a', 'b'])
def test_predict_loop_greedy_stream(G, tag):
    cfg = ast.literal_eval(str(G[f'predict_{tag}_cfg']))
    m, sd = oracle_txl(cfg, seed=12)
    assert abs(weights_checksum(sd) - float(G[f'predict_{tag}_weights_checksum'])) < 1e-6 * float(G[f'predict_{tag}_weights_checksum'])
    with torch.no_grad():
        m[1].decoder.bias[308:] = -50.
    v = ocodec.MusicVocab.create()
    seed = G[f'predict_{tag}_seed']
    pos = ocodec.position_enc(seed.copy(), v)
    assert np.array_equal(pos, G['predict_seed_positions_full'][:len(seed)])
    allowed = [str(a) for a in G[f'predict_{tag}_allowed']] or None
    n_words = {'a': 160, 'b': 120}[tag]
    got = osamp.predict(m, v, seed, pos, n_words=n_words, temperatures=(1.3, 1.1, 0.9), min_bars=12, top_k=1, top_p=0.0,
                        allowed_ins=allowed)
    assert list(got) == list(G[f'predict_{tag}_tokens'])
    if allowed:
        assert allowed == [str(a) for a in G[f'predict_{tag}_allowed_after']]      # rewritten in place like the reference


def test_bert_encoder_logits(G):
    cfg = ast.literal_eval(str(G['bert_cfg']))
    m = obert.get_multitask_model(324, dict(cfg), pad_idx=1).eval()
    own = m.state_dict()
    assert set(own.keys()) <= set(str(k) for k in G['bert_state_keys'])       # the oracle builds encoder + head only; same key names
    sd = golden_state_dict(own, seed=13)
    assert abs(weights_checksum(sd) - float(G['bert_weights_checksum'])) < 1e-6 * float(G['bert_weights_checksum'])
    m.load_state_dict({k: sd[k] for k in own}, strict=True)
    with torch.no_grad():
        for T in G['bert_lengths']:
            x, pos = torch.from_numpy(G[f'bert_x{T}']), torch.from_numpy(G[f'bert_pos{T}'])
            out = m({'msk': {'x': x, 'pos': pos.clone()}})['msk']
            assert np.abs(kept_positions(G, f'bert_logits{T}', out.numpy()) - G[f'bert_logits{T}']).max() < 2e-5, T
    got = osamp.predict_mask(m, ocodec.MusicVocab.create(), G['predict_mask_in'].copy(), G['predict_mask_pos'].copy(),
                             temperatures=(1.1, 0.9), top_k=1, top_p=0.0)
    assert list(got) == list(G['predict_mask_out'])
