"""The batched remix: per-sequence lengths in the encoder attention (dmg_forward_varlen, dmg_attn_bert_varlen) and
MultitaskLearner.predict_mask_batch (dmg_predict_mask_batch) against the oracle's one-item predict_mask and the one-item CUDA paths."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

import remix_attention_ref as ref_attn
from oracle import bert as obert, codec as ocodec, sampling as osamp
from test_gpu_train_kernels import row_err

pytestmark = pytest.mark.gpu

V = 324
SMALL_BERT = dict(obert.multitask_config(), enc_layers=2, d_model=128, n_heads=2, d_head=64, d_inner=256)
ITEM_LENS = (23, 64, 100, 127, 128, 200, 311, 517)          # both sides of 128: the flash and the tcgen05 attention classes
VARLEN_LENS = (1, 2, 37, 64, 127, 128, 129, 255, 256, 623, 1024)
# Worst 64-wide row error (row_err) of the varlen attention against the float64 reference; measured on one B200 (1000 W) over both
# kernel classes: see test_varlen_attention_against_float64_reference.  The tolerance is at most 3x that.
ATTN_TOL = 1.5e-2


def _pair(dtype, max_batch, max_seq, seed=0, **kw):
    from deepmusicgeneration_b200.model import get_multitask_model
    torch.manual_seed(seed)
    om = obert.get_multitask_model(V, SMALL_BERT, pad_idx=1).eval()
    pm = get_multitask_model(V, SMALL_BERT, pad_idx=1, dtype=dtype, max_batch=max_batch, max_seq=max_seq, init=False, **kw)
    pm.load_state_dict(om.state_dict())
    return om, pm


def _items(golden_dir, lens=ITEM_LENS, every=2):
    "Cuts of fur_elise of the given lengths, every `every`-th note masked."
    from deepmusicgeneration_b200.codec import MusicDataBunch, MusicItem
    data = MusicDataBunch.empty('')
    full = MusicItem.from_file(os.path.join(golden_dir, 'fur_elise.mid'), data.vocab)
    vocab = data.vocab
    items = []
    for k, L in enumerate(lens):
        off = 7 * k
        it = vocab.to_music_item(full.data[off:off + L].copy())
        _ = it.position                                      # positions of the unmasked cut
        notes = [i for i, t in enumerate(it.data) if vocab.note_range[0] <= t < vocab.note_range[1]]
        it.data[notes[::every]] = vocab.mask_idx
        items.append(it)
    return data, items


def _learner(data, pm):
    from deepmusicgeneration_b200.learner import MultitaskLearner
    return MultitaskLearner(data, pm)


def test_batch_greedy_equals_independent_oracle_predict_masks(golden_dir):
    "fp32, greedy: every item of predict_mask_batch == the oracle's predict_mask run on that item alone"
    om, pm = _pair('f32', 8, 520)
    data, items = _items(golden_dir)
    out = _learner(data, pm).predict_mask_batch(items, temperatures=(1.1, 0.9), top_k=1, top_p=0.0)
    ov = ocodec.MusicVocab.create()
    for it, got in zip(items, out):
        ref = osamp.predict_mask(om, ov, it.data, it.position, temperatures=(1.1, 0.9), top_k=1, top_p=0.0)
        assert list(got.data) == list(ref), len(it.data)
        assert (got.data != data.vocab.mask_idx).all()


def test_batch_sampled_streams_and_chunking(golden_dir):
    "fp32, sampled: item 0 == the one-item predict_mask with the same seed; max_batch 3 / 8 and a reversed item order change nothing"
    _, pm8 = _pair('f32', 8, 520)
    _, pm3 = _pair('f32', 3, 520)
    data, items = _items(golden_dir)
    kw = dict(temperatures=(1.0, 1.0), top_k=20, top_p=0.8, seed=1234)
    a = _learner(data, pm8).predict_mask_batch(items, **kw)
    single = _learner(data, pm8).predict_mask(items[0], **kw)
    assert list(a[0].data) == list(single.data)
    b = _learner(data, pm3).predict_mask_batch(items, **kw)
    for x, y in zip(a, b):
        assert list(x.data) == list(y.data)
    # a reversed list is another assignment of streams: item i of the reversed list draws from stream i.  Reversing it back and
    # giving the reversed list's streams must reproduce that run, whatever the internal grouping
    r = _learner(data, pm8).predict_mask_batch(items[::-1], **kw)
    r3 = _learner(data, pm3).predict_mask_batch(items[::-1], **kw)
    for x, y in zip(r, r3):
        assert list(x.data) == list(y.data)
    assert list(r[0].data) == list(_learner(data, pm8).predict_mask(items[-1], **kw).data)


def _varlen_inputs(B_lens, T_max, seed, pad_random=False):
    g = torch.Generator().manual_seed(seed)
    B = len(B_lens)
    x = torch.randint(12, V, (B, T_max), generator=g)
    pos = torch.cumsum(torch.randint(0, 9, (B, T_max), generator=g), 1)
    for b, L in enumerate(B_lens):
        if not pad_random:
            x[b, L:] = 1
            pos[b, L:] = 0
    return x, pos


@pytest.mark.parametrize('dtype', ['bf16', 'f32'])
@pytest.mark.parametrize('flags', [0, 8, 2])          # default, DMG_KF_BERT_MMA_SYNC, DMG_KF_NO_FLASH
def test_varlen_forward_equals_standalone(dtype, flags):
    if dtype == 'f32' and flags:
        pytest.skip('the selectors choose between bf16 kernels')
    lens = VARLEN_LENS
    T_max = max(lens)
    _, pm = _pair(dtype, len(lens), 1024, kernel_flags=flags)
    e = pm._e
    x, pos = _varlen_inputs(lens, T_max, 5)
    lv, _ = e.forward(x, pos, 1, lens=lens)
    # Bit-identical for every length, as measured on the B200: each sequence gets the attention kernel it gets alone (a one-token
    # sequence: the flash kernel in the batch, the FFMA kernel alone - softmax over one key, out = v either way), and at d_model 128
    # every GEMM kernel the row count can select accumulates its two 64-wide k-blocks in the same order
    for b, L in enumerate(lens):
        ls, _ = e.forward(x[b:b + 1, :L], pos[b:b + 1, :L], 1)
        assert torch.isfinite(lv[b]).all(), L
        assert torch.equal(lv[b, :L], ls[0]), (L, (lv[b, :L] - ls[0]).abs().max().item())
    # random tokens instead of pad_idx in the padding: valid rows bit-identical
    xr, pr = _varlen_inputs(lens, T_max, 5, pad_random=True)
    for b, L in enumerate(lens):
        xr[b, :L], pr[b, :L] = x[b, :L], pos[b, :L]
    lr, _ = e.forward(xr, pr, 1, lens=lens)
    for b, L in enumerate(lens):
        assert torch.equal(lr[b, :L], lv[b, :L]), L
    # other neighbours (same B and T_max): the valid rows of the sequence in row 3 are bit-identical
    lens2 = list(lens[::-1])
    lens2[3] = lens[3]
    x2, p2 = _varlen_inputs(lens2, T_max, 9)
    x2[3], p2[3] = x[3], pos[3]
    l2, _ = e.forward(x2, p2, 1, lens=lens2)
    assert torch.equal(l2[3, :lens[3]], lv[3, :lens[3]])
    if flags == 0 and dtype == 'bf16':
        # a sequence of at least 128 tokens whose neighbours change but which keeps its row: same tcgen05 items, same output
        lens3 = list(lens)
        lens3[0], lens3[1] = 200, 5
        x3, p3 = _varlen_inputs(lens3, T_max, 11)
        x3[9], p3[9] = x[9], pos[9]
        l3, _ = e.forward(x3, p3, 1, lens=lens3)
        assert torch.equal(l3[9, :lens[9]], lv[9, :lens[9]])


def _direct_inputs(scale):
    lens = VARLEN_LENS
    B, T_max, H = len(lens), max(lens), 2
    HD, Dcap = H * 64, max(lens) + 1
    g = torch.Generator().manual_seed(3)
    qkv = (torch.randn(B * T_max, 3 * HD, generator=g) * scale).to(torch.bfloat16).cuda()
    rk = (torch.randn(H, Dcap, 64, generator=g) * scale).to(torch.bfloat16).cuda()
    u = (torch.randn(HD, generator=g) * 0.3).cuda()
    v = (torch.randn(HD, generator=g) * 0.3).cuda()
    return lens, B, T_max, H, HD, Dcap, qkv, rk, u, v


def _direct(lib, qkv, rk, Dcap, u, v, lens, B, T_max, H, mma_sync_only, fill=7.):
    from deepmusicgeneration_b200.model import _ptr
    out = torch.full((B * T_max, H * 64), fill, dtype=torch.bfloat16, device='cuda')
    ln = np.array(lens, dtype=np.int32)
    rc = lib.dmg_attn_bert_varlen(_ptr(qkv), _ptr(rk), Dcap, _ptr(u), _ptr(v), _ptr(out), ln.ctypes.data_as(C.c_void_p), B, T_max, H,
                                  mma_sync_only, C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0, lib.dmg_last_error()
    return out


@pytest.mark.parametrize('mma_sync_only', [0, 1])
def test_varlen_attention_against_float64_reference(mma_sync_only):
    """Every sequence's valid rows of the direct launch against the float64 attention of remix_attention_ref.py at its own length
    (line 3 with L_b).  Inputs x1.5: scores of std ~3, so attention is peaked and a dropped, duplicated or misplaced key moves the
    rows that put their weight on it; NaN in the padding rows of q|k|v."""
    from deepmusicgeneration_b200 import _lib
    lib = _lib.load()
    lens, B, T_max, H, HD, Dcap, qkv, rk, u, v = _direct_inputs(1.5)
    q = qkv.clone()
    for b, L in enumerate(lens):
        q[b * T_max + L:(b + 1) * T_max] = float('nan')
    out = _direct(lib, q, rk, Dcap, u, v, lens, B, T_max, H, mma_sync_only)
    worst = {}
    for b, L in enumerate(lens):
        x = qkv[b * T_max:b * T_max + L].double().view(L, 3, H, 64).permute(1, 2, 0, 3)      # [3, H, L, 64]
        ref, _, _ = ref_attn.remix_attention(x[0][None], x[1][None], x[2][None], rk[:, :L].double().permute(1, 0, 2),
                                             u.double().view(H, 64), v.double().view(H, 64))
        got = out[b * T_max:b * T_max + L].view(L, H, 64)
        worst[L] = row_err(got, ref[0].permute(1, 0, 2))
    print(f'varlen attention (mma_sync_only={mma_sync_only}) worst row error per length:', {L: f'{e:.2e}' for L, e in worst.items()})
    bad = {L: e for L, e in worst.items() if not e <= ATTN_TOL}
    assert not bad, f'over tolerance: {bad}'


@pytest.mark.parametrize('mma_sync_only', [0, 1])
def test_varlen_attention_ignores_padding_rows(mma_sync_only):
    "direct launch on caller-owned q|k|v: NaN or zeros in the padding rows give bit-identical valid rows; padding rows come out zero"
    from deepmusicgeneration_b200 import _lib
    from deepmusicgeneration_b200.model import _ptr
    lib = _lib.load()
    lens, B, T_max, H, HD, Dcap, qkv, rk, u, v = _direct_inputs(0.5)
    ln = np.array(lens, dtype=np.int32)
    valid = torch.zeros(B * T_max, dtype=torch.bool)
    for b, L in enumerate(lens):
        valid[b * T_max:b * T_max + L] = True
    valid = valid.cuda()
    outs = []
    for fill in (0., float('nan')):
        q = qkv.clone()
        q[~valid] = fill
        out = torch.full((B * T_max, HD), 7., dtype=torch.bfloat16, device='cuda')
        rc = lib.dmg_attn_bert_varlen(_ptr(q), _ptr(rk), Dcap, _ptr(u), _ptr(v), _ptr(out), ln.ctypes.data_as(C.c_void_p), B, T_max, H,
                                      mma_sync_only, C.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert rc == 0, lib.dmg_last_error()
        outs.append(out)
    assert torch.isfinite(outs[1][valid].float()).all()
    assert torch.equal(outs[0][valid], outs[1][valid])
    for o in outs:
        assert (o[~valid].float() == 0).all()
    # a sequence alone (B = 1, its own T) through the same entry gives the same rows: same kernel, same arithmetic
    for b in (2, 5, 9):
        L = lens[b]
        q1 = qkv[b * T_max:b * T_max + L].contiguous()
        o1 = torch.empty(L, HD, dtype=torch.bfloat16, device='cuda')
        l1 = np.array([L], dtype=np.int32)
        assert lib.dmg_attn_bert_varlen(_ptr(q1), _ptr(rk), Dcap, _ptr(u), _ptr(v), _ptr(o1), l1.ctypes.data_as(C.c_void_p), 1, L, H,
                                        mma_sync_only, C.c_void_p(torch.cuda.current_stream().cuda_stream)) == 0
        assert torch.equal(o1, outs[0][b * T_max:b * T_max + L]), L


def test_loop_mechanics_graph_zero_masks_and_validation(golden_dir):
    from deepmusicgeneration_b200 import _lib
    from deepmusicgeneration_b200.learner import sampler_params, vocab_layout
    from deepmusicgeneration_b200.model import _ptr, _stream_ptr
    data, items = _items(golden_dir, lens=(40, 150, 90, 300))
    untouched = data.vocab.to_music_item(items[1].data.copy())
    untouched.data[untouched.data == data.vocab.mask_idx] = data.vocab.note_range[0] + 60
    items = items + [untouched]
    kw = dict(temperatures=(1.0, 1.0), top_k=20, top_p=0.8, seed=77)
    _, pm = _pair('bf16', 8, 512)
    _, png = _pair('bf16', 8, 512, kernel_flags=_lib.KF_NO_GRAPH)
    a = _learner(data, pm).predict_mask_batch(items, **kw)
    b = _learner(data, png).predict_mask_batch(items, **kw)
    for x, y in zip(a, b):
        assert list(x.data) == list(y.data)
        assert (x.data != data.vocab.mask_idx).all()
    assert list(a[-1].data) == list(untouched.data)
    for it, got in zip(items, a):                              # only the masks change
        keep = it.data != data.vocab.mask_idx
        assert (got.data[keep] == it.data[keep]).all()
    # validation: rejected before anything launches
    e = pm._e
    vl = vocab_layout(data.vocab)
    params = sampler_params(data.vocab, 1, (1., 1.), 0, 1, 0., None, flags=_lib.SAMPLE_REMIX_FILTER, seed=0)
    x = torch.full((2, 64), 5, dtype=torch.int64, device='cuda')
    pos = torch.zeros_like(x)

    def call(lens, mpos, n, B=2, T=64, n_max=3, streams=(0, 1)):
        ln, mp, nm, sm = (np.ascontiguousarray(np.asarray(a_, dtype=np.int32)) for a_ in (lens, mpos, n, streams))
        return e.lib.dmg_predict_mask_batch(e.h, _ptr(x), _ptr(pos), ln.ctypes.data_as(C.c_void_p), mp.ctypes.data_as(C.c_void_p),
                                            nm.ctypes.data_as(C.c_void_p), sm.ctypes.data_as(C.c_void_p), B, T, n_max, C.byref(vl),
                                            C.byref(params), _stream_ptr())
    before = e.lib.dmg_launch_count()
    assert call((64, 65), [[0, 1, 2], [0, 1, 2]], (3, 3)) != 0             # length past T_max
    assert call((64, 0), [[0, 1, 2], [0, 1, 2]], (3, 3)) != 0              # empty item
    assert call((64, 10), [[0, 2, 1], [0, 1, 2]], (3, 3)) != 0             # not ascending
    assert call((64, 10), [[0, 1, 2], [0, 1, 10]], (3, 3)) != 0            # position past the item's end
    assert call((64, 10), [[0, 1, 2], [0, 1, 2]], (3, 4)) != 0             # more masks than n_max
    assert call((64, 10), [[0, 1, 2], [0, 1, 2]], (3, 3), T=1024) != 0     # T_max > max_seq
    assert call([64] * 9, [[0, 1, 2]] * 9, [3] * 9, B=9, streams=range(9)) != 0   # B > max_batch
    assert e.lib.dmg_launch_count() == before
    from deepmusicgeneration_b200.codec import MusicItem
    too_long = data.vocab.to_music_item(np.full(600, data.vocab.mask_idx, dtype=np.int64))
    with pytest.raises(ValueError, match='max_seq'):
        _learner(data, pm).predict_mask_batch([too_long])


def test_bf16_batch_follows_single_item_path(golden_dir):
    """bf16, greedy: every item agrees with the one-item bf16 predict_mask up to the first mask where the two paths pick different
    tokens, and there the one-item run's logits of the two picks lie within what the two head computations can differ by.  The
    encoder rows are the same (test_varlen_forward_equals_standalone); the head row is the mask step's dot product in one path and the
    head GEMM's tile accumulation in the other - both bf16 x bf16 products summed in fp32, so a logit differs by at most
    d * 2^-24 * sum_k |h_k E_vk| between them"""
    _, pm = _pair('bf16', 8, 520)
    data, items = _items(golden_dir)
    vocab = data.vocab
    kw = dict(temperatures=(1.0, 1.0), top_k=1, top_p=0.0)
    learn = _learner(data, pm)
    out = learn.predict_mask_batch(items, **kw)
    for it, got in zip(items, out):
        single = learn.predict_mask(it, **kw)
        masks = np.flatnonzero(it.data == vocab.mask_idx)
        diff = [p for p in masks if got.data[p] != single.data[p]]
        if not diff:
            continue
        p = diff[0]
        state = single.data.copy()
        state[masks[masks >= p]] = vocab.mask_idx
        logits, core = pm._e.forward(torch.from_numpy(state)[None], torch.from_numpy(np.asarray(it.position))[None], 1, want_core=True)
        row = logits[0, p]
        ta, tb = int(single.data[p]), int(got.data[p])
        h = core[0, p].bfloat16().double()
        emb = pm.state_dict()['encoder.embed.embed.weight'].bfloat16().double().cuda()
        d = h.numel()
        bound = max((h * emb[t]).abs().sum().item() for t in (ta, tb)) * d * 2.0 ** -24
        gap = (row[ta] - row[tb]).abs().item()
        print(f'L={len(it.data)}: first different pick at mask {p}, top-two gap {gap:.3g}, bound {2 * bound:.3g}')
        assert gap <= 2 * bound, (len(it.data), p, gap, bound)
