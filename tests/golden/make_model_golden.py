"""Generates tests/golden/model_golden.npz by EXECUTING the reference's own model / sampling source.

Run in the build container only (needs /root/reference):  ``python tests/golden/make_model_golden.py``

The reference modules cannot be imported as a whole (fastai / music21 are not installed, np.int is gone), but the definitions on
the hot path are plain torch once the handful of fastai names they use exist.  Executed from the reference checkout:

  deep_music_genre.py   vocab constants + ``MusicVocab`` (:126-196, :812-890), ``position_enc`` (:1489-1527),
                        ``window_mask`` / ``rand_window_mask`` / ``lm_mask`` (:1577-1594),
                        ``MusicTransformerXL`` (the forward override) + ``BeatPositionEncoder`` (:1603-1665),
                        ``top_k_top_p`` (:1679-1706), ``MusicLearner.predict`` (:1853-1972), ``filter_invalid_indexes`` (:1984-2018)
  deep_music_remix.py   ``get_multitask_model`` / ``MultiTransformer`` / ``TransformerEmbedding`` / ``MTLinearDecoder`` / ``MTEncoder`` /
                        ``MTEncoderBlock`` / ``MemMultiHeadRelativeAttentionKV`` (:1851-2104), ``filter_invalid_indexes`` (:2394-2437),
                        ``MultitaskLearner.predict_mask`` (:2563-2613)

Stubbed (un-vendored fastai==1.0.61, restated in oracle/txl.py): the ``TransformerXL`` base class (``__init__`` / ``reset`` /
``_update_mems`` / ``select_hidden`` and its ``DecoderLayer`` stack), ``PositionalEncoding``, ``feed_forward``, ``_line_shift``,
``init_transformer``, ``RNNDropout``, ``LinearDecoder``, ``SequentialRNN``, ``Activation``, ``ifnone``, ``Learner.pred_batch``.
So the fixture pins everything the reference repository itself holds for the path; the fastai layer arithmetic stays pinned by the
parameter-count known answer and the in-repo twin (``MemMultiHeadRelativeAttentionKV._apply_attention``), which IS executed here.
"""
import math
import os
import pickle
import re
import sys
import textwrap
from enum import Enum
from typing import Collection, List, Tuple

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F
from torch import Tensor

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
from golden_weights import golden_state_dict, sample_positions, weights_checksum      # noqa: E402
from oracle import txl                                               # noqa: E402

REF = '/root/reference'
GENRE, REMIX = os.path.join(REF, 'deep_music_genre.py'), os.path.join(REF, 'deep_music_remix.py')


def grab(path, start_pat, end_pat=None, dedent=False):
    src = open(path).read()
    a = re.search(start_pat, src, re.M).start()
    b = len(src) if end_pat is None else re.search(end_pat, src[a + 1:], re.M).start() + a + 1
    code = src[a:b]
    return textwrap.dedent(code) if dedent else code


class Activation(Enum):
    ReLU, Swish, GeLU = 1, 2, 3


def ifnone(a, b):
    return b if a is None else a


class TransformerXLStub(txl.MusicTransformerXL):
    "fastai TransformerXL: its signature (the reference filters kwargs by it, :1606-1609) + the oracle's restated members."
    def __init__(self, vocab_sz, ctx_len, n_layers, n_heads, d_model, d_head, d_inner, resid_p=0., attn_p=0., ff_p=0., embed_p=0.,
                 bias=False, scale=True, act='relu', double_drop=True, attn_cls=None, learned_pos_enc=False, mask=True, mem_len=0):
        txl.MusicTransformerXL.__init__(self, vocab_sz, ctx_len, n_layers, n_heads, d_model, d_head, d_inner, resid_p=resid_p,
                                        attn_p=attn_p, ff_p=ff_p, embed_p=embed_p, bias=bias, scale=scale, act=act,
                                        double_drop=double_drop, mask=mask, mem_len=mem_len, encode_position=False, mask_steps=1)

    forward = None        # must come from the reference's override


BASE = {'np': np, 'torch': torch, 'nn': nn, 'F': F, 'math': math, 'pickle': pickle, 'Enum': Enum, 'Collection': Collection, 'List': List,
        'Tuple': Tuple, 'Tensor': Tensor, 'MusicItem': object, 'ifnone': ifnone, 'Activation': Activation}

# ------------------------------------------------------------------------------------------------ genre namespace
G = dict(BASE, TransformerXL=TransformerXLStub)
exec(grab(GENRE, r'^BPB = 4', r'^#@title\nACCEP_INS'), G)
exec(grab(GENRE, r'^class MusicVocab\(\):', r'^###\*\*dataloader\.py\*\*'), G)
exec(grab(GENRE, r'^def position_enc\(', r'^def beat2index'), G)
exec(grab(GENRE, r'^def window_mask\(', r'^#@title\n#https://github.com/bearpelican/musicautobot/blob/master/musicautobot/music_transformer/model\.py'), G)
exec(grab(GENRE, r'^class MusicTransformerXL\(TransformerXL\):', r'^###\*\*utils\*\*'), G)
exec(grab(GENRE, r'^def top_k_top_p\(', r'^#@title'), G)
exec(grab(GENRE, r'^def filter_invalid_indexes\('), G)
exec(grab(GENRE, r'^    def predict\(self, item:MusicItem', r'^# High level prediction functions', dedent=True), G)
ref_predict = G['predict']

# ------------------------------------------------------------------------------------------------ remix namespace
R = dict(BASE, PositionalEncoding=txl.PositionalEncoding, feed_forward=txl.feed_forward, init_transformer=txl.init_transformer,
         _line_shift=txl._line_shift, RNNDropout=txl.RNNDropout)
exec(grab(REMIX, r'^BPB = 4', r'^#@title\nACCEP_INS'), R)
exec(grab(REMIX, r'^def window_mask\(', r'^def lm_mask'), R)
exec(grab(REMIX, r'^def get_multitask_model\(', r'^###\*\*utils\*\*'), R)
exec(grab(REMIX, r'^def top_k_top_p\(', r'^#@title'), R)
exec(grab(REMIX, r'^def filter_invalid_indexes\(', r'^# # old filter invalid indexes'), R)
exec(grab(REMIX, r'^    def predict_mask\(self, masked_item:MusicItem', r'^    def predict_s2s', dedent=True), R)
ref_predict_mask = R['predict_mask']

out = {}
vocab = G['MusicVocab'].create()
assert len(vocab.itos) == 324
out['vocab_itos'] = np.array(vocab.itos)


# ------------------------------------------------------------------------------------------------ masks
mask_cases = [(1, 0, 1, 1), (1, 5, 1, 1), (6, 0, 1, 1), (6, 4, 1, 1), (7, 3, 2, 0), (12, 0, 3, 0), (12, 5, 4, 0), (9, 2, 1, 0), (16, 16, 5, 0)]
out['mask_cases'] = np.array(mask_cases)
for i, (x_len, m_len, win, k) in enumerate(mask_cases):
    out[f'mask_{i}'] = G['window_mask'](x_len, 'cpu', m_len, size=(win, k))[0, 0].numpy()
np.random.seed(4)
draws = []
for i in range(40):                                  # rand_window_mask: which (win, k) the numpy stream selects for max_size = 4
    m = G['rand_window_mask'](8, 2, 'cpu', max_size=4, p=0.2, is_eval=False)[0, 0].numpy()
    draws.append(m)
out['rand_mask_draws'] = np.stack(draws)
out['rand_mask_eval'] = G['rand_window_mask'](8, 2, 'cpu', max_size=4, is_eval=True)[0, 0].numpy()

# ------------------------------------------------------------------------------------------------ top_k_top_p and the filters
g = torch.Generator().manual_seed(3)
tk_logits = torch.randn(24, 324, generator=g) * 2.0
tk_cases = [(1, 0.0), (20, 0.8), (40, 0.6), (0, 0.9), (5, 0.0), (0, 0.0), (400, 0.3), (30, 0.65)]
out['topk_logits'], out['topk_cases'] = tk_logits.numpy(), np.array(tk_cases, dtype=np.float64)
out['topk_kept'] = np.stack([np.stack([torch.isfinite(G['top_k_top_p'](row, top_k=int(k), top_p=float(p))).numpy() for row in tk_logits])
                             for k, p in tk_cases])
# the same after the reference's grammar filter for a previous NOTE token (durations stay finite - and mt*/dummy*, which the
# reference never filters): what the predict loop feeds top_k_top_p
dur_only = torch.stack([G['filter_invalid_indexes'](row.clone(), vocab.stoi['n60'], vocab) for row in tk_logits])
out['topk_kept_after_note'] = np.stack([np.stack([torch.isfinite(G['top_k_top_p'](row, top_k=int(k), top_p=float(p))).numpy() for row in dur_only])
                                        for k, p in tk_cases])
prevs = ['xxpad', 'd4', 'd160', 'i0', 'i6', 'n60', 'n0', 'xxsep', 'xxni', 'xxbos', 'xxmask', 'xxpop', 'mt3']
out['filter_prev'] = np.array([vocab.stoi[t] for t in prevs])
allowed_sets = [None, ['i0'], ['i1', 'i5'], ['i6', 'i2', 'i3']]
out['filter_allowed'] = np.array([0 if a is None else sum(1 << int(t[1:]) for t in a) for a in allowed_sets])
kept = np.zeros((len(prevs), 2, len(allowed_sets), 324), dtype=bool)
for a, tok in enumerate(prevs):
    for b, last_xxsep in enumerate((False, True)):
        for c, allowed in enumerate(allowed_sets):
            res = torch.zeros(324)
            res = G['filter_invalid_indexes'](res, vocab.stoi[tok], vocab, last_xxsep=last_xxsep, allowed_ins=None if allowed is None else list(allowed))
            kept[a, b, c] = torch.isfinite(res).numpy()
out['filter_genre_kept'] = kept
kept = np.zeros((len(prevs), 324), dtype=bool)
for a, tok in enumerate(prevs):
    kept[a] = torch.isfinite(R['filter_invalid_indexes'](torch.zeros(324), vocab.stoi[tok], vocab)).numpy()
out['filter_remix_kept'] = kept


# ------------------------------------------------------------------------------------------------ Transformer-XL forward (the override)
def build_txl(cfg, seed):
    cfg = dict(cfg)
    tie_weights, output_p, out_bias = map(cfg.pop, ['tie_weights', 'output_p', 'out_bias'])
    enc = G['MusicTransformerXL'](324, **cfg)                               # reference class on the stubbed fastai base
    dec = txl.LinearDecoder(324, cfg['d_model'], output_p, tie_encoder=enc.encoder if tie_weights else None, bias=out_bias)
    model = txl.SequentialRNN(enc, dec)
    sd = golden_state_dict(model.state_dict(), seed)
    missing = model.load_state_dict(sd, strict=True)
    return model.eval(), sd


TXL_CFG = dict(txl.default_config(), n_layers=2, d_model=128, n_heads=2, d_head=64, d_inner=256, mem_len=32, ctx_len=64,
               encode_position=True, mask_steps=4)
out['txl_cfg'] = np.array(repr({k: v for k, v in TXL_CFG.items()}))
model, sd = build_txl(TXL_CFG, seed=11)
out['txl_weights_checksum'] = np.float64(weights_checksum(sd))
out['txl_state_keys'] = np.array(sorted(sd.keys()))
g = torch.Generator().manual_seed(21)
model.reset()
pos_last = torch.zeros(3, 1, dtype=torch.int64)
segs = [40, 1, 1, 7, 1, 33]
out['txl_segments'] = np.array(segs)
with torch.no_grad():
    for s, T in enumerate(segs):
        x = torch.randint(0, 324, (3, T), generator=g)
        pos = pos_last + torch.cumsum(torch.randint(0, 9, (3, T), generator=g), 1)
        pos_last = pos[:, -1:]
        decoded, raw_outputs, outputs = model({'x': x, 'pos': pos.clone()})
        out[f'txl_x{s}'], out[f'txl_pos{s}'], out[f'txl_logits{s}'] = x.numpy(), pos.numpy(), decoded.numpy()
        out[f'txl_core{s}'] = outputs[0].numpy()
        out[f'txl_mem_last{s}'] = raw_outputs[-1].numpy()
# training-mode masks of the override (dropout = 0 so that only the mask differs): forced window (3, 0) over the memory
model.train()
for m in model.modules():
    if isinstance(m, (nn.Dropout, txl.RNNDropout)):
        m.p = 0.
saved = G['rand_window_mask']
G['rand_window_mask'] = lambda x_len, m_len, device, max_size=None, p=0.2, is_eval=False: G['window_mask'](x_len, device, m_len, size=(3, 0))
with torch.no_grad():
    x = torch.randint(0, 324, (3, 20), generator=g)
    pos = pos_last + torch.cumsum(torch.randint(0, 9, (3, 20), generator=g), 1)
    out['txl_win_x'], out['txl_win_pos'] = x.numpy(), pos.numpy()
    out['txl_win_logits'] = model({'x': x, 'pos': pos.clone()})[0].numpy()
G['rand_window_mask'] = saved
model.eval()


# ------------------------------------------------------------------------------------------------ MusicLearner.predict (greedy)
class Item:                                        # the slice of MusicItem (:1152-1278) predict touches
    def __init__(self, data, vocab, ins=None):
        self.data, self.vocab, self.ins = np.asarray(data, dtype=np.int64), vocab, ins
        self.position = G['position_enc'](self.data.copy(), vocab)
    def to_tensor(self): return torch.from_numpy(self.data).long()
    def get_pos_tensor(self): return torch.from_numpy(self.position).long()
    def to_text(self): return self.vocab.textify(self.data)
    def append(self, other): return Item(np.concatenate([self.data, other.data]), self.vocab, self.ins)


G['MusicItem'] = Item
vocab.to_music_item = lambda idxenc, ins=None: Item(idxenc, vocab, ins)


class Data:
    pass


class LearnerStub:
    def __init__(self, model):
        self.model, self.data = model, Data()
        self.data.vocab = vocab
    def pred_batch(self, batch):
        with torch.no_grad():
            return self.model.eval()(batch[0])


seed_text = open(os.path.join(HERE, 'megalovania_seed64.txt')).read().split()
seed_ids = np.array(vocab.numericalize(seed_text), dtype=np.int64)
out['predict_seed_positions_full'] = G['position_enc'](seed_ids.copy(), vocab)
for tag, cfg, n_seed, n_words, allowed in (('a', dict(TXL_CFG, encode_position=True), 120, 160, None),
                                            ('b', dict(TXL_CFG, encode_position=False, mem_len=64), 200, 120, ['Piano', 'Bass'])):
    model, sd = build_txl(cfg, seed=12)
    with torch.no_grad():
        model[1].decoder.bias[308:] = -50.          # mt*/dummy* ids: the reference never filters them, a trained model never emits them
    item = Item(seed_ids[:n_seed], vocab)
    allowed_arg = None if allowed is None else list(allowed)
    pred, full = ref_predict(LearnerStub(model), item, n_words=n_words, temperatures=(1.3, 1.1, 0.9), min_bars=12, top_k=1, top_p=0.0,
                             allowed_ins=allowed_arg)
    out[f'predict_{tag}_seed'], out[f'predict_{tag}_tokens'] = item.data, pred.data
    out[f'predict_{tag}_weights_checksum'] = np.float64(weights_checksum(sd))
    out[f'predict_{tag}_cfg'] = np.array(repr(cfg))
    out[f'predict_{tag}_allowed'] = np.array([] if allowed is None else allowed)
    out[f'predict_{tag}_allowed_after'] = np.array([] if allowed is None else allowed_arg)     # rewritten in place (:1878-1880)
    print(f'predict {tag}: {len(pred.data)} tokens')


# ------------------------------------------------------------------------------------------------ remix encoder + head, predict_mask
BERT_CFG = dict(enc_layers=2, dec_layers=1, d_model=128, n_heads=2, d_head=64, d_inner=256, mem_len=512, resid_p=0.1, attn_p=0.1, ff_p=0.1,
                embed_p=0.1, output_p=0.1, bias=True, scale=True, double_drop=True, tie_weights=True, out_bias=True, mask_steps=1)
out['bert_cfg'] = np.array(repr(BERT_CFG))
bmodel = R['get_multitask_model'](324, dict(BERT_CFG), pad_idx=1)
bsd = golden_state_dict(bmodel.state_dict(), seed=13)
bmodel.load_state_dict(bsd, strict=True)
bmodel.eval()
out['bert_weights_checksum'] = np.float64(weights_checksum(bsd))
out['bert_state_keys'] = np.array(sorted(bsd.keys()))
lens = [1, 2, 31, 70, 130, 257]
out['bert_lengths'] = np.array(lens)
g = torch.Generator().manual_seed(22)
with torch.no_grad():
    for T in lens:
        x = torch.randint(0, 324, (2, T), generator=g)
        pos = torch.cumsum(torch.randint(0, 9, (2, T), generator=g), 1)
        out[f'bert_x{T}'], out[f'bert_pos{T}'] = x.numpy(), pos.numpy()
        out[f'bert_logits{T}'] = bmodel({'msk': {'x': x, 'pos': pos.clone()}})['msk'].numpy()
R['MusicItem'] = Item
item = Item(seed_ids[:150], vocab)
notes = [i for i, t in enumerate(item.data) if vocab.note_range[0] <= t < vocab.note_range[1]]
durs = [i for i, t in enumerate(item.data) if vocab.dur_range[0] <= t < vocab.dur_range[1]]
masked = item.data.copy()
masked[notes[::2]] = vocab.mask_idx
masked[durs[1::3]] = vocab.mask_idx
mitem = Item(masked, vocab)
mitem.position = item.position.copy()               # the app masks after encoding: positions are those of the unmasked item
res = ref_predict_mask(LearnerStub(bmodel), mitem, temperatures=(1.1, 0.9), top_k=1, top_p=0.0)
out['predict_mask_in'], out['predict_mask_pos'], out['predict_mask_out'] = masked, mitem.position, res.data

sample_positions(out)
np.savez_compressed(os.path.join(HERE, 'model_golden.npz'), **out)
print('wrote', len(out), 'arrays,', os.path.getsize(os.path.join(HERE, 'model_golden.npz')) // 1024, 'KiB')
