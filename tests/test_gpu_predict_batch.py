"""GPU tests of genre continuation over many seeds of their own lengths: the per-stream Transformer-XL memory, the varlen prefill
(dmg_forward_varlen for the Transformer-XL), MusicLearner.predict_batch / generate_batch(lens=...), and the per-stream forms of the
attention unit-test entries (dmg_attn_decode_streams, dmg_attn_segment_streams).

fp32 results are compared token for token: every row of a GEMM of the FFMA kernel is computed on its own, and for the rows of a seed
the key tiles that the padding of a shorter seed adds to the general attention kernel are fully masked (they add exact zeros), so a
stream does not depend on its companions or on the padded length.  bf16 logits are held to the suite's gate: max rel <= 2e-2 with
rel = |a - b| / max(|b|, 1.0)."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

import decode_ref
import segment_ref
from oracle import codec as ocodec, sampling as osamp, txl
from deepmusicgeneration_b200 import _lib
from deepmusicgeneration_b200._lib import DmgError, check
from test_gpu_decode_kernels import Ring, TOL as DECODE_TOL, bits, same_bits
from test_gpu_segment_attention import Seg, TOL as SEG_TOL
from test_gpu_train_kernels import _st, row_err

pytestmark = pytest.mark.gpu

V = 324
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
SMALL_M128 = dict(txl.default_config(), n_layers=2, d_model=128, n_heads=2, d_head=64, d_inner=256, mem_len=128,
                  encode_position=False)
SEED_LENS = (5, 40, 127, 128, 129, 200, 300, 77)


def _pair(cfg, dtype, max_batch, max_seq, seed=0, keep_hidden=False, **kw):
    "oracle model and CUDA model on the same random-init weights (the unused vocabulary tail tamed, as in the parity tests)"
    from deepmusicgeneration_b200.model import get_language_model
    torch.manual_seed(seed)
    om = txl.get_language_model(V, cfg).eval()
    with torch.no_grad():
        om[1].decoder.bias[308:] = -50.
    pm = get_language_model(V, cfg, dtype=dtype, max_batch=max_batch, max_seq=max_seq, keep_hidden=keep_hidden, init=False, **kw)
    pm.load_state_dict(om.state_dict())
    return om, pm


def _rel(a, b):
    return ((a - b).abs() / b.abs().clamp_min(1.0)).max().item()


def _items(lens=SEED_LENS):
    """seeds of the given lengths (moved up to the next token with a temperature class, so that predict can start from it), cut from
    the Megalovania and uploadedMidi goldens, alternating"""
    from deepmusicgeneration_b200.codec import MusicDataBunch, MusicItem
    data = MusicDataBunch.empty('')
    vocab = data.vocab
    full = [MusicItem.from_file(os.path.join(GOLDEN, f), vocab).data for f in ('Undertale_-_Megalovania.mid', 'uploadedMidi.mid')]
    items = []
    for n, L in enumerate(lens):
        src = full[n % 2]
        while not (vocab.is_duration(src[L - 1]) or vocab.is_note(src[L - 1]) or vocab.is_ins(src[L - 1]) or src[L - 1] == vocab.pad_idx):
            L += 1
        d = src[:L].copy()
        d[0] = vocab.stoi['xxpop']
        items.append(MusicItem(d, vocab))
    return data, items


def _learner(data, pm):
    from deepmusicgeneration_b200.learner import MusicLearner
    return MusicLearner(data, pm)


# ---------------------------------------------------------------------------------------------------------------------------
# fp32: predict_batch token for token against the oracle's predict on each item alone
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('encode_position', [False, True])
def test_predict_batch_greedy_f32_equals_oracle_per_item(encode_position):
    cfg = dict(SMALL_M128, encode_position=encode_position)
    om, pm = _pair(cfg, 'f32', 8, 320)
    data, items = _items()
    ends = {('dur' if data.vocab.is_duration(it.data[-1]) else 'note' if data.vocab.is_note(it.data[-1]) else 'other') for it in items}
    assert len(ends) >= 2, 'the seeds are meant to end on different token classes'
    ov = ocodec.MusicVocab.create()
    kw = dict(n_words=90, temperatures=(1.3, 1.1, 0.9), min_bars=2, top_k=1, top_p=0.0)
    out = _learner(data, pm).predict_batch(items, **kw)
    stopped_early = 0
    for i, (it, (pred, full)) in enumerate(zip(items, out)):
        ref = osamp.predict(om, ov, it.data, it.position, **kw)
        assert list(pred.data) == ref, (i, len(it.data), len(pred.data), len(ref))
        assert list(full.data) == list(it.data) + ref
        stopped_early += len(ref) < kw['n_words']
    print(f'encode_position={encode_position}: {stopped_early} of {len(items)} streams stopped before n_words')


def test_predict_batch_allowed_ins_f32_equals_oracle():
    om, pm = _pair(SMALL_M128, 'f32', 4, 320)
    data, items = _items((40, 129, 300, 5))
    ov = ocodec.MusicVocab.create()
    kw = dict(n_words=60, temperatures=(1.2, 1.0, 1.0), min_bars=2, top_k=1, top_p=0.0)
    allowed = ['Piano', 'Guitar']
    mine = list(allowed)
    out = _learner(data, pm).predict_batch(items, allowed_ins=mine, **kw)
    assert mine == ['i' + str(ocodec.ACCEP_INS[a]) for a in allowed]          # rewritten in place once, as predict does
    for i, it in enumerate(items):
        ref = osamp.predict(om, ov, it.data, it.position, allowed_ins=list(allowed), **kw)
        assert list(out[i][0].data) == ref, i


# ---------------------------------------------------------------------------------------------------------------------------
# fp32: a stream does not depend on its companions; item 0 makes predict's draws
# ---------------------------------------------------------------------------------------------------------------------------
def test_predict_batch_item0_equals_predict_and_streams_are_isolated_f32():
    om, pm = _pair(SMALL_M128, 'f32', 8, 320)
    data, items = _items()
    learn = _learner(data, pm)
    kw = dict(n_words=80, temperatures=(1.0, 1.0, 1.0), min_bars=2, top_k=20, top_p=0.8)
    for s in (5, 11):
        alone = learn.predict(items[0], seed=s, **kw)[0]
        batch = learn.predict_batch(items, seed=s, **kw)
        assert list(batch[0][0].data) == list(alone.data), s
        # item 2 at the same index (same Philox stream) with other companions and another padded length
        others = [items[5], items[7], items[2], items[3]]
        again = learn.predict_batch(others, seed=s, **kw)
        assert list(again[2][0].data) == list(batch[2][0].data), s
        # and the same again with the longest seed in the batch (the padded length grows)
        longer = [items[1], items[6], items[2]]
        assert list(learn.predict_batch(longer, seed=s, **kw)[2][0].data) == list(batch[2][0].data), s


# ---------------------------------------------------------------------------------------------------------------------------
# bf16: logits of every stream after a varlen prefill and one-token steps, against the oracle run per stream
# ---------------------------------------------------------------------------------------------------------------------------
def _oracle_per_stream(om, x, lens, steps):
    "the oracle (fp32 on the GPU, TF32 off) run on each stream alone: [len(steps) + 1, B, V] last-position logits"
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    omg = om.cuda()
    out = []
    with torch.no_grad():
        for b in range(x.shape[0]):
            omg.reset()
            rows = [omg(x[b:b + 1, :lens[b]].cuda())[0][0, -1].cpu()]
            for xs in steps:
                rows.append(omg(xs[b:b + 1].cuda())[0][0, -1].cpu())
            out.append(torch.stack(rows))
    om.cpu()
    return torch.stack(out, 1)


def _varlen_run(pm, x, lens, steps):
    "prefill (LOGITS_LAST) then the one-token steps: [len(steps) + 1, B, V]"
    e = pm._e
    pm.reset()
    rows = [e.forward(x.cuda(), None, _lib.LOGITS_LAST, lens=lens)[0].cpu()]
    assert e.mem_counts(len(lens)) == [min(int(n), e.cfg.mem_len) for n in lens]
    for xs in steps:
        rows.append(pm[0].forward(xs.cuda(), logits_mode=_lib.LOGITS_ALL)[0][:, -1].cpu())
    return torch.stack(rows)


@pytest.mark.parametrize('M,B', [(512, 64), (192, 6)])
def test_varlen_prefill_and_decode_bf16_against_oracle(M, B):
    """M = 512: the third-generation decode kernel, with >= 64 streams the two-half dual-role pipeline, checked also against the
    KF_NO_DUAL_DECODE (bit for bit: the pipeline reorders launches, not arithmetic), KF_NO_FUSED_DECODE and KF_NO_DECODE_KERNEL
    engines on the same batch.  M = 192: the second-generation kernel.  Seeds below, at and above M."""
    cfg = dict(txl.baseline_config(), n_layers=2, mem_len=M, ctx_len=M + 200)
    T = M + 150
    om, pm = _pair(cfg, 'bf16', B, T)
    g = torch.Generator().manual_seed(M + B)
    lens = torch.randint(1, T + 1, (B,), generator=g).numpy().astype(np.int32)
    lens[:4] = [1, M, M + 1, T][:4]
    x = torch.randint(0, V, (B, T), generator=g)
    steps = [torch.randint(0, V, (B, 1), generator=g) for _ in range(10)]
    ref = _oracle_per_stream(om, x, lens, steps)
    got = _varlen_run(pm, x, lens, steps)
    worst = max(_rel(got[s], ref[s]) for s in range(len(steps) + 1))
    print(f'M={M}, B={B}: varlen prefill + 10 steps, max rel {worst:.3e} (lengths {sorted(lens.tolist())[:6]}...)')
    assert worst <= 2e-2
    if M == 512:
        from deepmusicgeneration_b200 import _lib as L
        for flags in (L.KF_NO_DUAL_DECODE, L.KF_NO_FUSED_DECODE, L.KF_NO_DECODE_KERNEL | L.KF_NO_FUSED_DECODE):
            _, pk = _pair(cfg, 'bf16', B, T, kernel_flags=flags)
            other = _varlen_run(pk, x, lens, steps)
            if flags == L.KF_NO_DUAL_DECODE:
                assert torch.equal(other, got), 'dual-role pipeline vs whole-batch launches'
            else:
                assert max(_rel(other[s], ref[s]) for s in range(len(steps) + 1)) <= 2e-2, flags
                assert max(_rel(other[s], got[s]) for s in range(len(steps) + 1)) <= 3e-2, flags


def test_generate_batch_lens_graph_replay_equals_eager():
    from deepmusicgeneration_b200 import _lib as L
    _, pm = _pair(SMALL_M128, 'bf16', 6, 256)
    _, pe = _pair(SMALL_M128, 'bf16', 6, 256, kernel_flags=L.KF_NO_GRAPH)
    data, items = _items((5, 40, 127, 128, 129, 200))
    lens = np.array([len(it.data) for it in items], dtype=np.int32)
    x = torch.full((6, int(lens.max())), data.vocab.pad_idx, dtype=torch.int64)
    for b, it in enumerate(items):
        x[b, :lens[b]] = torch.from_numpy(it.data)
    kw = dict(n_words=150, top_k=1, top_p=0.0, min_bars=10 ** 6, lens=lens)
    a = _learner(data, pm).generate_batch(x, **kw).cpu()
    b = _learner(data, pe).generate_batch(x, **kw).cpu()
    assert torch.equal(a, b)
    assert pm._e.mem_counts(6) == [128] * 6                  # every ring is full after 150 steps


# ---------------------------------------------------------------------------------------------------------------------------
# kernel level: the per-stream entries
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('kernel,M', [(0, 512), (1, 192), (0, 128)])
def test_attn_decode_streams_against_float64_reference(kernel, M):
    "one launch over streams at pos_total 0 < p < M, = M and > M (wrapped), each against ring_attention with its own pos_total"
    pts = [1, 37, M - 1, M, M + 1, 2 * M + 37, 10 ** 6 + 3]
    B, b0, Bcap = len(pts), 2, len(pts) + 3
    x = Ring(B, 8, M, 0, Bcap=Bcap, b0=b0, seed=M + kernel)
    g = torch.Generator(device='cuda').manual_seed(M)
    x.kring = (torch.randn(Bcap, 8, M, 64, device='cuda', generator=g) * 0.8).bfloat16()
    x.vring = (torch.randn(Bcap, 8, M, 64, device='cuda', generator=g) * 0.8).bfloat16()
    state = torch.full((Bcap, 2), -7, device='cuda', dtype=torch.int32)       # rows outside [b0, b0 + B) are not read
    state[b0:b0 + B] = torch.tensor([[p, min(p, M)] for p in pts], dtype=torch.int32)
    kr, vr = x.kring.clone(), x.vring.clone()
    out = torch.full((B, 8 * 64), float('nan'), device='cuda', dtype=torch.bfloat16)
    torch.cuda.synchronize()
    check(_lib.load().dmg_attn_decode_streams(C.byref(x.args(out, state, kernel, kr, vr, over={'state': None, 'pos_total': -1})),
                                              state.data_ptr(), _st()), 'dmg_attn_decode_streams')
    HD = 8 * 64
    q, k, v = (x.qkv[:, i * HD:(i + 1) * HD].view(B, 8, 64) for i in range(3))
    for b, p in enumerate(pts):
        s = slice(b0 + b, b0 + b + 1)
        ref, rk, rv = decode_ref.ring_attention(q[b:b + 1], k[b:b + 1], v[b:b + 1], x.kring[s], x.vring[s], x.rd, x.u.view(8, 64),
                                                x.v.view(8, 64), p, M)
        err = row_err(out[b:b + 1], ref.reshape(1, HD))
        assert err <= DECODE_TOL['attn'], (p, err)
        assert same_bits(kr[s], rk) and same_bits(vr[s], rv), f'append of stream {b0 + b} (pos_total {p})'
    for s in list(range(b0)) + list(range(b0 + B, Bcap)):
        assert same_bits(kr[s], x.kring[s]) and same_bits(vr[s], x.vring[s]), f'stream {s} outside the launch moved'


@pytest.mark.parametrize('dtype', [_lib.F32, _lib.BF16])
def test_attn_segment_streams_general_kernel_over_unequal_memories(dtype):
    pts = [0, 5, 99, 100, 137, 10 ** 6 + 3]
    B, b0, M, T = len(pts), 1, 100, 33
    x = Seg(_lib.ARCH_TXL, dtype, B, T, 2, M, 10 ** 6 + 3, kernel=0, ran=_lib.SEG_GENERAL, Bcap=B + 2, b0=b0, seed=dtype)
    state = torch.zeros(B + 2, 2, device='cuda', dtype=torch.int32)
    state[b0:b0 + B] = torch.tensor([[p, min(p, M)] for p in pts], dtype=torch.int32)
    kr, vr = x.kring.clone(), x.vring.clone()
    out = torch.full((B * T, 2 * 64), float('nan'), device='cuda', dtype=x.rd.dtype)
    a = x.args(out, kr, vr, {'pos_total': -1})
    torch.cuda.synchronize()
    check(_lib.load().dmg_attn_segment_streams(C.byref(a), state.data_ptr(), _st()), 'dmg_attn_segment_streams')
    assert a.kernel_ran == _lib.SEG_GENERAL
    HD = 2 * 64
    q, k, v = (x.qkv[:, i * HD:(i + 1) * HD].view(B, T, 2, 64).permute(0, 2, 1, 3).double() for i in range(3))
    for b, p in enumerate(pts):
        s = slice(b0 + b, b0 + b + 1)
        ref, rk, rv = segment_ref.segment_attention(q[b:b + 1], k[b:b + 1], v[b:b + 1], x.kring[s], x.vring[s], x.rd, x.u.view(2, 64).double(),
                                                    x.v.view(2, 64).double(), p, M)
        err = row_err(out[b * T:(b + 1) * T], ref.permute(0, 2, 1, 3).reshape(T, HD))
        assert err <= SEG_TOL['general_f32' if dtype == _lib.F32 else 'general_bf16'], (p, err)
        assert same_bits(kr[s], rk) and same_bits(vr[s], rv), f'append of stream {b0 + b} (pos_total {p})'
    # equal memories in bf16 route as dmg_forward does (flash without memory); a bad state row is refused before any launch
    if dtype == _lib.BF16:
        zero = torch.zeros_like(state)
        q16 = x.qkv.bfloat16()                                 # the flash kernel reads q|k|v as bf16
        a = x.args(out, kr, vr, {'qkv': q16.data_ptr()})
        check(_lib.load().dmg_attn_segment_streams(C.byref(a), zero.data_ptr(), _st()), 'dmg_attn_segment_streams')
        assert a.kernel_ran == _lib.SEG_FLASH
        bad = state.clone()
        bad[b0 + 2, 1] = 3
        lib = _lib.load()
        torch.cuda.synchronize()
        n = lib.dmg_launch_count()
        with pytest.raises(DmgError, match=r'not \{pos_total, min'):
            check(lib.dmg_attn_segment_streams(C.byref(x.args(out, kr, vr)), bad.data_ptr(), _st()), 'dmg_attn_segment_streams')
        assert lib.dmg_launch_count() == n


# ---------------------------------------------------------------------------------------------------------------------------
# state handling
# ---------------------------------------------------------------------------------------------------------------------------
def test_select_hidden_after_varlen_prefill_carries_memories_and_counts():
    om, pm = _pair(SMALL_M128, 'f32', 5, 320, keep_hidden=True)
    e = pm._e
    g = torch.Generator().manual_seed(8)
    lens = np.array([30, 200, 128, 7], dtype=np.int32)
    x = torch.randint(0, V, (4, 200), generator=g)
    pm.reset()
    e.forward(x.cuda(), None, _lib.LOGITS_LAST, lens=lens)
    pm[0]._bs = 4
    assert e.mem_counts(5) == [30, 128, 128, 7, 0]
    with pytest.raises(ValueError, match='mem_counts'):
        e.mem_count()
    with pytest.raises(ValueError, match=r'per-stream counts \[30, 128, 128, 7\]'):
        pm[0].hidden
    idx = [1, 3, 0, 3, 2]
    pm[0].select_hidden(idx)
    assert e.mem_counts(5) == [128, 7, 30, 7, 128]
    x2 = torch.randint(0, V, (5, 3), generator=g)
    got = pm(x2.cuda())[0].cpu()                              # a multi-token segment over unequal memories: the general kernel
    for j, i in enumerate(idx):
        om.reset()
        with torch.no_grad():
            om(x[i:i + 1, :lens[i]])
            want = om(x2[j:j + 1])[0]
        assert (got[j:j + 1] - want).abs().max() < 5e-4, j
    # streams 1 and 3 now hold the same count: hidden of a batch whose counts agree works again
    pm[0].select_hidden([1, 3])
    assert e.mem_count() == 10
    hid = pm[0].hidden
    assert len(hid) == 3 and tuple(hid[0].shape) == (2, 10, 128)


def test_varlen_refusals_fire_before_any_launch():
    from deepmusicgeneration_b200.codec import MusicItem
    _, pm = _pair(SMALL_M128, 'f32', 3, 64)
    data, items = _items((5, 40))
    learn = _learner(data, pm)
    e = pm._e
    lib = _lib.load()
    x = torch.randint(0, V, (2, 20), device='cuda')
    torch.cuda.synchronize()
    n = lib.dmg_launch_count()
    with pytest.raises(ValueError, match='max_batch=3'):
        learn.predict_batch(items * 2)
    with pytest.raises(ValueError, match='item 1 is empty'):
        learn.predict_batch([items[0], MusicItem(np.zeros(0, dtype=np.int64), data.vocab)])
    with pytest.raises(ValueError, match=r'item 1 has \d+ tokens.*max_seq=64.*music_model_learner\(\.\.\., max_seq='):
        learn.predict_batch([items[0], _items((100,))[1][0]])
    with pytest.raises(DmgError, match='outside'):
        e.forward(x, None, _lib.LOGITS_LAST, lens=[3, 21])
    assert lib.dmg_launch_count() == n
    pm.reset()
    e.forward(x, None, _lib.LOGITS_LAST, lens=[3, 20])
    torch.cuda.synchronize()
    n = lib.dmg_launch_count()
    with pytest.raises(DmgError, match='empty memory'):
        e.forward(x, None, _lib.LOGITS_LAST, lens=[3, 20])
    assert lib.dmg_launch_count() == n
    assert learn.predict_batch([]) == []
