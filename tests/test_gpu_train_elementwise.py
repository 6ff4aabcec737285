"""GPU unit tests of the training step's elementwise kernels (train_kernels.cu) through their C-ABI test entries, each against
the float64 references of tests/train_elementwise_ref.py: dropout masks, dropout + residual + LayerNorm forward / backward at
every width the kernels are instantiated for, cross-entropy, embedding forward / backward, the head's RNN dropout and
backward, the AR / TAR sums, bias column sums, the gradient wire format and the fused Adam (through the trainer, so that its
real chunk table runs).  Where the kernel's arithmetic is a fixed sequence (masks, bf16 casts, counts, untouched elements) the
comparison is exact; elsewhere it is bounded by the worst error measured on a B200, which every test prints."""
import ctypes as C

import numpy as np
import pytest
import torch

import train_elementwise_ref as ref
from deepmusicgeneration_b200 import _lib
from deepmusicgeneration_b200._lib import DmgError, check
from oracle import txl

pytestmark = pytest.mark.gpu

V = 324
WIDTHS = [128, 256, 384, 512, 768, 1024]


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _st():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _lib_():
    return _lib.load()


def maxrel(a, b):
    "max |a - b| over max |b|: one wrong element anywhere is the result"
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def host(t):
    return t.detach().float().cpu().double().numpy() if t.dtype == torch.bfloat16 else t.detach().cpu().double().numpy()


def mask_t(m, shape=None):
    "a float64 numpy mask as the fp32 device tensor the kernels multiply by (the scale is a float32)"
    t = torch.tensor(m, dtype=torch.float32, device='cuda')
    return t.view(*shape) if shape is not None else t


# ---------------------------------------------------------------------------------------------- dropout masks
def test_embed_dropout_mask_is_the_hash():
    "an all-ones table: x32 is exactly the mask of element row*d + c"
    lib = _lib_()
    rows, d, p, seed = 777, 384, 0.1, 0x1234567
    emb = torch.ones(V, d, device='cuda')
    ids = torch.randint(0, V, (rows,), device='cuda')
    x32 = torch.full((rows, d), 5.0, device='cuda')
    xa = torch.zeros(rows, d, device='cuda', dtype=torch.bfloat16)
    check(lib.dmg_train_embed(_p(ids), None, _p(emb), None, None, _p(x32), _p(xa), rows, d, V, p, seed, _st()), 'embed')
    torch.cuda.synchronize()
    want = ref.row_mask(seed, p, rows, d)
    assert np.array_equal(host(x32), want.astype(np.float32).astype(np.float64))
    assert abs((want == 0).mean() - p) < 0.01
    assert torch.equal(xa, x32.bfloat16())


def test_ln_forward_and_backward_draw_the_same_mask():
    "x = 0, add = 1: the forward's z is the mask on add; the backward's dadd is zero exactly where that mask drops"
    lib = _lib_()
    rows, d, p, seed = 300, 256, 0.25, 4242
    x32 = torch.zeros(rows, d, device='cuda')
    add = torch.ones(rows, d, device='cuda', dtype=torch.bfloat16)
    w, b = torch.ones(d, device='cuda'), torch.zeros(d, device='cuda')
    xa = torch.empty(rows, d, device='cuda', dtype=torch.bfloat16)
    zs = torch.empty(rows, d, device='cuda', dtype=torch.bfloat16)
    st = torch.empty(rows, 2, device='cuda')
    check(lib.dmg_train_ln_fwd(_p(x32), _p(add), _p(w), _p(b), _p(xa), _p(zs), _p(st), rows, d, p, seed, _st()), 'ln fwd')
    dy = torch.randn(rows, d, device='cuda')
    dadd = torch.empty(rows, d, device='cuda', dtype=torch.bfloat16)
    dw, db = torch.zeros(d, device='cuda'), torch.zeros(d, device='cuda')
    check(lib.dmg_train_ln_bwd(_p(dy), None, _p(zs), _p(st), _p(w), _p(dadd), _p(dw), _p(db), None, rows, d, p, seed, _st()), 'ln bwd')
    torch.cuda.synchronize()
    want = ref.row_mask(seed, p, rows, d)
    assert np.array_equal(host(zs), torch.tensor(want, dtype=torch.float32).bfloat16().double().numpy())
    assert (dy != 0).all()
    assert np.array_equal(host(dadd) == 0, want == 0)


def test_head_dropout_mask_is_per_stream_and_constant_over_t():
    lib = _lib_()
    B, T, d, p, seed = 3, 130, 256, 0.1, 99
    x = torch.ones(B, T, d, device='cuda', dtype=torch.bfloat16)
    y = torch.zeros_like(x)
    check(lib.dmg_train_rnn_dropout(_p(x), _p(y), B, T, d, p, seed, _st()), 'rnn dropout')
    dx = torch.full((B, T, d), 7.0, device='cuda')
    check(lib.dmg_train_head_bwd(_p(x), _p(torch.zeros(B, T, d, device='cuda')), _p(dx), B, T, d, p, seed, 0.0, _st()), 'head bwd')
    torch.cuda.synchronize()
    m = np.broadcast_to(ref.stream_mask(seed, p, B, d), (B, T, d))
    assert np.array_equal(host(y), torch.tensor(m, dtype=torch.float32).bfloat16().double().numpy())
    assert np.array_equal(host(dx), m.astype(np.float32).astype(np.float64))
    assert (y.float() == y.float()[:, :1]).all()


# ---------------------------------------------------------------------------------------------- dropout + residual + LayerNorm
# Worst over every case on one B200 (1000 W), max |err| / max |ref| per tensor.  Logic tier (float64 on the kernel's own zsave /
# stats): y 2.2e-7, stats 6.2e-7, dz 1.5e-7, dw 5.9e-7, db 5.2e-7, dsum 5.6e-7.  Design tier (float64 on the true z, so the cost
# of saving z in bf16): dz 6.6e-4, dw 6.7e-3.  Each tolerance is at most 3x that.
LN_TOL = {'y': 6e-7, 'stats': 1.8e-6, 'dz': 4.4e-7, 'dw': 1.7e-6, 'db': 1.5e-6, 'dsum': 1.6e-6, 'design_dz': 1.9e-3, 'design_dw': 2e-2}


def _run_ln(d, rows, use_dbr, use_dsum, p, offset_sigma=0.0, seed=0):
    lib = _lib_()
    g = torch.Generator(device='cuda').manual_seed(rows * 7 + d + int(p * 10) + 2 * use_dbr + use_dsum)
    dseed = 0xABCDEF + rows
    x = torch.randn(rows, d, device='cuda', generator=g)
    if offset_sigma:
        x += offset_sigma * torch.sign(torch.randn(rows, 1, device='cuda', generator=g))
    add = (torch.randn(rows, d, device='cuda', generator=g) * 0.5).bfloat16()
    w = 1 + 0.2 * torch.randn(d, device='cuda', generator=g)
    b = 0.1 * torch.randn(d, device='cuda', generator=g)
    x32 = x.clone()
    xa = torch.empty(rows, d, device='cuda', dtype=torch.bfloat16)
    zs = torch.empty(rows, d, device='cuda', dtype=torch.bfloat16)
    st = torch.full((rows, 2), float('nan'), device='cuda')
    check(lib.dmg_train_ln_fwd(_p(x32), _p(add), _p(w), _p(b), _p(xa), _p(zs), _p(st), rows, d, p, dseed, _st()), 'ln fwd')
    mask = ref.row_mask(dseed, p, rows, d) if p > 0 else None
    mk = mask_t(mask) if mask is not None else None
    # forward: bf16 copies are the RNE casts of what the kernel computed
    assert torch.equal(xa, x32.bfloat16())
    if p == 0:
        assert torch.equal(zs, (x + add.float()).bfloat16())              # one fp32 add, then the cast
    y_ref, z_ref, mean_ref, rstd_ref = ref.ln_fwd(host(x), host(add), host(w), host(b), mask)
    # with dropout, nvcc may contract x + add * keep into one FMA: zsave is then within one bf16 step of the true z, plus the
    # fp32 rounding of the product where x and the product cancel
    branch = np.abs(host(add) * (mask if mask is not None else 1.0))
    assert (np.abs(host(zs) - z_ref) <= 2.0 ** -7 * np.abs(z_ref) + 2.0 ** -22 * (np.abs(host(x)) + branch)).all()
    errs = {'y': maxrel(host(x32), y_ref),
            'stats': max(maxrel(host(st[:, 0]), mean_ref), maxrel(host(st[:, 1]), rstd_ref))}
    # backward
    dy0 = torch.randn(rows, d, device='cuda', generator=g)
    dbr = (torch.randn(rows, d, device='cuda', generator=g) * 0.5).bfloat16() if use_dbr else None
    dy = dy0.clone()
    dadd = torch.empty(rows, d, device='cuda', dtype=torch.bfloat16)
    fills = [torch.randn(d, device='cuda', generator=g) + 3.0 for _ in range(3)]      # dw / db / dsum are added into these
    dw, db, ds = (f.clone() for f in fills)
    check(lib.dmg_train_ln_bwd(_p(dy), _p(dbr), _p(zs), _p(st), _p(w), _p(dadd), _p(dw), _p(db), _p(ds) if use_dsum else None, rows, d,
                               p, dseed, _st()), 'ln bwd')
    torch.cuda.synchronize()
    gy = host(dy0) + (host(dbr) if use_dbr else 0.0)
    # logic tier: the formula on the kernel's own saved z and statistics
    r = ref.ln_bwd(gy, host(zs), host(w), host(st[:, 0]), host(st[:, 1]), mask)
    errs.update(dz=maxrel(host(dy), r['dz']), dw=maxrel(host(dw) - host(fills[0]), r['dw']),
                db=maxrel(host(db) - host(fills[1]), r['db']))
    assert torch.equal(dadd, (dy * mk if mk is not None else dy).bfloat16())           # dy now holds dz; dadd = bf16(mask * dz)
    if use_dsum:
        errs['dsum'] = maxrel(host(ds) - host(fills[2]), r['dsum'])
    else:
        assert torch.equal(ds, fills[2])
    # design tier: the true z (fp32 inputs in float64) instead of the bf16 copy the backward reads
    rd = ref.ln_bwd(gy, z_ref, host(w), mask=mask)
    errs.update(design_dz=maxrel(host(dy), rd['dz']), design_dw=maxrel(host(dw) - host(fills[0]), rd['dw']))
    return errs


@pytest.mark.parametrize('rows', [1, 7, 8, 1237, 5000])        # 5000 > 296 blocks x 8 warps: warps of the backward walk several rows
@pytest.mark.parametrize('d', WIDTHS)
def test_ln_forward_backward_matches_float64(d, rows):
    for use_dbr, use_dsum, p in ((True, True, 0.1), (False, False, 0.0)):
        errs = _run_ln(d, rows, use_dbr, use_dsum, p)
        print(f'd {d} rows {rows} dbr {use_dbr} dsum {use_dsum} p {p}:', {k: f'{v:.2e}' for k, v in errs.items()}, flush=True)
        for k, v in errs.items():
            assert v < LN_TOL[k], (k, v, d, rows, use_dbr, use_dsum, p)


@pytest.mark.parametrize('use_dbr,use_dsum,p', [(True, False, 0.0), (False, True, 0.1)])
def test_ln_row_offset_of_four_sigma(use_dbr, use_dsum, p):
    "rows whose mean sits 4 standard deviations from zero: the variance must not cancel, the bf16 z costs more in the design tier"
    errs = _run_ln(512, 1237, use_dbr, use_dsum, p, offset_sigma=4.0)
    print('offset 4 sigma:', {k: f'{v:.2e}' for k, v in errs.items()}, flush=True)
    for k, v in errs.items():
        assert v < LN_TOL[k], (k, v)


# ---------------------------------------------------------------------------------------------- cross-entropy
# Worst on one B200 (1000 W): loss sum 6.9e-7 relative, dlogits 3.1e-3 of max |dlogits| (a bf16 output).  Tolerances <= 3x.
CE_TOL = {'loss': 2e-6, 'dlogits': 9e-3}


def _ce_inputs(rows, Vp, seed):
    g = torch.Generator(device='cuda').manual_seed(seed)
    logits = torch.full((rows, Vp), 1e30, device='cuda')                 # padding columns must never be read
    logits[:, :V] = torch.randn(rows, V, device='cuda', generator=g) * 3
    big = torch.arange(rows, device='cuda') % 5 == 0                    # rows of magnitude 80
    logits[big, :V] = (torch.rand(int(big.sum()), V, device='cuda', generator=g) * 2 - 1) * 80
    t = torch.randint(0, V, (rows,), device='cuda', generator=g)
    t[3::17] = -5; t[4::17] = V; t[5::17] = 400                         # out of range: clamped
    return logits, t


def test_cross_entropy_matches_float64():
    lib = _lib_()
    rows, Vp = 1237, 384
    logits, t = _ce_inputs(rows, Vp, 1)
    dl = torch.full((rows, Vp), 7.0, device='cuda', dtype=torch.bfloat16)
    acc = torch.zeros(1, device='cuda')
    check(lib.dmg_train_ce(_p(logits), Vp, _p(t), -1, _p(dl), _p(acc), None, rows, V, _st()), 'ce')
    torch.cuda.synchronize()
    lg = host(logits)
    loss, dref, _ = ref.cross_entropy(lg, host(t).astype(np.int64), V)
    errs = {'loss': abs(acc.item() - loss) / abs(loss), 'dlogits': maxrel(host(dl), dref)}
    print('ce:', errs, flush=True)
    assert (dl[:, V:] == 0).all()
    assert errs['loss'] < CE_TOL['loss'] and errs['dlogits'] < CE_TOL['dlogits']


@pytest.mark.parametrize('rows', [203, 1237])
def test_cross_entropy_masked_matches_float64(rows):
    lib = _lib_()
    Vp, ignore = 384, 1
    logits, t = _ce_inputs(rows, Vp, rows)
    t[torch.arange(rows, device='cuda') % 3 == 1] = ignore
    dl = torch.full((rows, Vp), 7.0, device='cuda', dtype=torch.bfloat16)
    acc, cnt = torch.zeros(1, device='cuda'), torch.full((1,), -1.0, device='cuda')
    check(lib.dmg_train_ce(_p(logits), Vp, _p(t), ignore, _p(dl), _p(acc), _p(cnt), rows, V, _st()), 'ce masked')
    torch.cuda.synchronize()
    loss, dref, count = ref.cross_entropy(host(logits), host(t).astype(np.int64), V, ignore)
    assert cnt.item() == count
    ign = (t == ignore).cpu()
    assert (dl[ign.cuda()] == 0).all()                                   # every ldl column of an ignored row
    assert (dl[:, V:] == 0).all()
    errs = {'loss': abs(acc.item() - loss) / abs(loss), 'dlogits': maxrel(host(dl), dref)}
    print('ce masked:', errs, flush=True)
    assert errs['loss'] < CE_TOL['loss'] and errs['dlogits'] < CE_TOL['dlogits']
    # nothing to predict: count 0, no loss, zero gradient, and the mean is NaN as in torch
    t.fill_(ignore)
    acc.zero_(); dl.fill_(7.0)
    check(lib.dmg_train_ce(_p(logits), Vp, _p(t), ignore, _p(dl), _p(acc), _p(cnt), rows, V, _st()), 'ce masked')
    torch.cuda.synchronize()
    assert cnt.item() == 0 and acc.item() == 0 and (dl == 0).all()
    assert np.isnan(np.float32(acc.item()) / np.float32(cnt.item()))


# ---------------------------------------------------------------------------------------------- embedding
# Worst on one B200 (1000 W): 3.1e-7 of max |ref| (fp32 atomics in no fixed order).  Tolerance <= 3x.
EMB_TOL = 9e-7


def _embed_inputs(rows, d, seed):
    g = torch.Generator(device='cuda').manual_seed(seed)
    emb, beat, bar = (torch.randn(n, d, device='cuda', generator=g) for n in (V, 32, 1024))
    ids = torch.randint(0, 24, (rows,), device='cuda', generator=g)      # many duplicates: the atomics collide
    ids[::11] = 5                                                        # pad_idx
    ids[1::13] = -3; ids[2::13] = V + 7                                  # clamped
    pos = torch.randint(0, 40000, (rows,), device='cuda', generator=g)
    pos[::7] = torch.randint(0, 32, (len(pos[::7]),), device='cuda', generator=g)          # bar 0
    pos[1::9] = 32 * torch.randint(0, 2000, (len(pos[1::9]),), device='cuda', generator=g)   # beat 0
    pos[2::5] += 32768                                                   # bar wraps
    pos[3::6] = -torch.randint(1, 70000, (len(pos[3::6]),), device='cuda', generator=g)      # negative: floor semantics
    return emb, beat, bar, ids, pos


@pytest.mark.parametrize('p', [0.0, 0.1])
def test_embedding_forward_matches_reference(p):
    lib = _lib_()
    rows, d, seed = 1000, 256, 31337
    emb, beat, bar, ids, pos = _embed_inputs(rows, d, 5)
    x32 = torch.full((rows, d), 9.0, device='cuda')
    xa = torch.empty(rows, d, device='cuda', dtype=torch.bfloat16)
    check(lib.dmg_train_embed(_p(ids), _p(pos), _p(emb), _p(beat), _p(bar), _p(x32), _p(xa), rows, d, V, p, seed, _st()), 'embed')
    torch.cuda.synchronize()
    bt, br = (torch.tensor(a, device='cuda') for a in ref.beat_bar(host(pos).astype(np.int64)))
    want = emb[ids.clamp(0, V - 1)] + (beat[bt] + bar[br])              # the kernel's order of the fp32 adds
    if p > 0:
        want = want * mask_t(ref.row_mask(seed, p, rows, d))
    assert torch.equal(x32, want)
    assert torch.equal(xa, want.bfloat16())
    np.testing.assert_allclose(host(x32), ref.embed_fwd(host(ids).astype(np.int64), host(pos).astype(np.int64), host(emb), host(beat),
                                                        host(bar), ref.row_mask(seed, p, rows, d) if p > 0 else None), rtol=1e-6,
                               atol=1e-6)


@pytest.mark.parametrize('with_pos,with_dbr,p', [(True, True, 0.1), (True, False, 0.0), (False, True, 0.0)])
def test_embedding_backward_matches_float64(with_pos, with_dbr, p):
    lib = _lib_()
    rows, d, seed, pad = 1000, 256, 2024, 5
    _, _, _, ids, pos = _embed_inputs(rows, d, 6)
    g = torch.Generator(device='cuda').manual_seed(7)
    dx = torch.randn(rows, d, device='cuda', generator=g)
    dbr = (torch.randn(rows, d, device='cuda', generator=g) * 0.5).bfloat16() if with_dbr else None
    demb, dbeat, dbar = torch.zeros(V, d, device='cuda'), torch.zeros(32, d, device='cuda'), torch.zeros(1024, d, device='cuda')
    check(lib.dmg_train_embed_bwd(_p(ids), _p(pos) if with_pos else None, _p(dx), _p(dbr), _p(demb), _p(dbeat), _p(dbar), rows, d, V,
                                  pad, p, seed, _st()), 'embed bwd')
    torch.cuda.synchronize()
    gsum = host(dx) + (host(dbr) if with_dbr else 0.0)
    mask = ref.row_mask(seed, p, rows, d) if p > 0 else None
    re, rb, rr = ref.embed_bwd(host(ids).astype(np.int64), host(pos).astype(np.int64) if with_pos else None, gsum, V, pad, mask)
    assert (demb[pad] == 0).all()
    errs = {'demb': maxrel(host(demb), re)}
    if with_pos:
        assert (dbeat[0] == 0).all() and (dbar[0] == 0).all()
        errs.update(dbeat=maxrel(host(dbeat), rb), dbar=maxrel(host(dbar), rr))
    else:
        assert (dbeat == 0).all() and (dbar == 0).all()
    print('embedding backward:', errs, flush=True)
    for k, v in errs.items():
        assert v < EMB_TOL, (k, v)


def test_negative_positions_match_the_oracle_in_the_f32_model():
    "the inference embedding: positions of both signs through the f32 forward against BeatPositionEncoder's floor semantics"
    from deepmusicgeneration_b200.model import get_language_model
    cfg = dict(txl.default_config(), n_layers=1, d_model=128, n_heads=2, d_head=64, d_inner=256, mem_len=32, encode_position=True)
    torch.manual_seed(0)
    om = txl.get_language_model(V, cfg).eval()
    pm = get_language_model(V, cfg, dtype='f32', max_batch=2, max_seq=64, keep_hidden=False, init=False)
    pm.load_state_dict(om.state_dict())
    g = torch.Generator().manual_seed(3)
    x = torch.randint(0, V, (2, 40), generator=g)
    pos = torch.cumsum(torch.randint(0, 40, (2, 40), generator=g), 1) - 700      # starts far below zero, crosses it
    pos[1, 5] = -32768 * 2 - 40
    om.reset(); pm.reset()
    with torch.no_grad():
        ol = om({'x': x, 'pos': pos.clone()})[0]
    pl = pm({'x': x.cuda(), 'pos': pos.cuda()})[0]
    assert (pl.cpu() - ol).abs().max() < 5e-4


# ---------------------------------------------------------------------------------------------- head, AR / TAR, column sums
# Worst on one B200 (1000 W): head backward 4.2e-8, sumsq 3.2e-8 (both flavours), tar 3.2e-7, colsum 5.2e-8.  Tolerances <= 3x.
HEAD_TOL = {'head_bwd': 1.2e-7, 'sumsq': 9e-8, 'tar': 9e-7, 'colsum': 1.5e-7}


def test_rnn_dropout_and_head_backward_match_float64():
    lib = _lib_()
    B, T, d, p, seed, ar = 4, 192, 384, 0.1, 555, 2.0 / (4 * 192 * 384)
    g = torch.Generator(device='cuda').manual_seed(8)
    x = torch.randn(B, T, d, device='cuda', generator=g).bfloat16()
    y = torch.empty_like(x)
    check(lib.dmg_train_rnn_dropout(_p(x), _p(y), B, T, d, p, seed, _st()), 'rnn dropout')
    m = ref.stream_mask(seed, p, B, d)
    mk = mask_t(m)
    torch.cuda.synchronize()
    assert torch.equal(y, (x.float() * mk).bfloat16())
    dxd = torch.randn(B, T, d, device='cuda', generator=g).bfloat16()
    core = torch.randn(B, T, d, device='cuda', generator=g)
    dx = torch.empty(B, T, d, device='cuda')
    check(lib.dmg_train_head_bwd(_p(dxd), _p(core), _p(dx), B, T, d, p, seed, ar * 1e4, _st()), 'head bwd')
    torch.cuda.synchronize()
    e = maxrel(host(dx), ref.head_bwd(host(dxd), host(core), m, np.float32(ar * 1e4)))
    print('head backward:', e, flush=True)
    assert e < HEAD_TOL['head_bwd']


@pytest.mark.parametrize('n', [1, 4099, 1_500_003])        # 1.5 M > one pass of the 592-block grid; none a multiple of 4
def test_sumsq_both_flavours(n):
    lib = _lib_()
    x = torch.randn(n, device='cuda', generator=torch.Generator(device='cuda').manual_seed(n))
    want = float((host(x) ** 2).sum())
    acc = torch.full((1,), 2.0, device='cuda')
    check(lib.dmg_train_sumsq(_p(x), n, 0, None, 0, _p(acc), _st()), 'sumsq')
    part = torch.full((592,), float('nan'), device='cuda')
    out1, out2 = torch.full((1,), 5.0, device='cuda'), torch.full((1,), 5.0, device='cuda')
    check(lib.dmg_train_sumsq(_p(x), n, 1, _p(part), 592, _p(out1), _st()), 'sumsq det')
    check(lib.dmg_train_sumsq(_p(x), n, 1, _p(part), 592, _p(out2), _st()), 'sumsq det')
    torch.cuda.synchronize()
    e_atomic, e_det = abs(acc.item() - 2.0 - want) / want, abs(out1.item() - want) / want
    print('sumsq', n, e_atomic, e_det, flush=True)
    assert e_atomic < HEAD_TOL['sumsq'] + 2.0 ** -22 * (2.0 + want) / want      # + the rounding of 2 + sum
    assert e_det < HEAD_TOL['sumsq']
    assert torch.equal(out1, out2)                                       # a fixed order: the same bits every time


def test_tar_over_the_right_aligned_memory():
    lib = _lib_()
    B, M, d, cnt = 3, 256, 384, 192                                      # the valid rows are the last cnt of each stream
    mem = torch.randn(B, M, d, device='cuda').bfloat16()
    acc = torch.full((1,), 3.0, device='cuda')
    h = mem[:, M - cnt:]
    check(lib.dmg_train_tar(C.c_void_p(mem.data_ptr() + (M - cnt) * d * 2), M * d, B, cnt, d, _p(acc), _st()), 'tar')
    torch.cuda.synchronize()
    want = ref.tar(host(h))
    e = abs(acc.item() - 3.0 - want) / want
    print('tar', e, flush=True)
    assert e < HEAD_TOL['tar']
    # one row per stream: nothing to difference, nothing launched, the accumulator untouched
    acc.fill_(3.0)
    torch.cuda.synchronize()
    n0 = lib.dmg_launch_count()
    check(lib.dmg_train_tar(_p(mem), M * d, B, 1, d, _p(acc), _st()), 'tar n=1')
    torch.cuda.synchronize()
    assert lib.dmg_launch_count() == n0 and acc.item() == 3.0


@pytest.mark.parametrize('rows,n,ld', [(1000, 324, 384), (777, 325, 330), (3, 1536, 1536)])
def test_colsum_matches_float64(rows, n, ld):
    lib = _lib_()
    x = torch.randn(rows, ld, device='cuda', generator=torch.Generator(device='cuda').manual_seed(rows)).bfloat16()
    x[:, n:] = float('nan')                                              # columns past n must not be read
    dst = torch.full((n + 8,), 1.5, device='cuda')
    check(lib.dmg_train_colsum(_p(x), ld, rows, n, _p(dst), _st()), 'colsum')
    torch.cuda.synchronize()
    want = host(x)[:, :n].sum(0)
    e = maxrel(host(dst[:n]) - 1.5, want)
    print('colsum', rows, n, ld, e, flush=True)
    assert e < HEAD_TOL['colsum']
    assert (dst[n:] == 1.5).all()


# ---------------------------------------------------------------------------------------------- gradient wire format
def _small_trainer(d_model=128, bs=1, bptt=64, **kw):
    from deepmusicgeneration_b200.model import get_language_model
    from deepmusicgeneration_b200.training import TXLTrainer
    cfg = dict(txl.default_config(), n_layers=2, d_model=d_model, n_heads=d_model // 64, d_head=64, d_inner=2 * d_model, mem_len=64,
               encode_position=False, mask_steps=1)
    cfg.update(kw)
    torch.manual_seed(0)
    om = txl.get_language_model(V, cfg, drop_mult=0.)
    pm = get_language_model(V, cfg, dtype='bf16', device=0, max_batch=bs, max_seq=max(bptt, 64), keep_hidden=False, init=False)
    pm.load_state_dict(om.state_dict())
    return cfg, pm, TXLTrainer(pm, bs, bptt, cfg, drop_mult=0., seed=1, distributed=False)


def test_grad_wire_format_round_trip_odd_spans():
    cfg, pm, tr = _small_trainer()
    lib, h = tr.lib, tr.e.h
    G = tr.grad
    G.copy_(torch.randn(G.numel(), device='cuda') * 3)
    # rounding ties, a denormal, large values
    G[:8] = torch.tensor([1.0 + 2 ** -8, 1.0 + 3 * 2 ** -8, -1.0 - 2 ** -8, 1e-40, 3e38, 0.0, -0.0, 65504.0], device='cuda')
    sentinel = torch.tensor(-123.0, dtype=torch.bfloat16)
    for off, cnt in ((0, 8), (1, 1), (3, 3), (7, 5), (5, 4 * 1000 + 3), (4, 4 * 257 + 3), (1001, 4 * 40000 + 3)):
        for shift in (0, 1):                                             # a wire pointer one element off: the scalar paths
            before = G.clone()
            wire = torch.full((cnt + 2,), float(sentinel), device='cuda', dtype=torch.bfloat16)
            w = C.c_void_p(wire.data_ptr() + 2 * shift)
            check(lib.dmg_train_grad_pack(h, off, cnt, w, _st()), 'pack')
            torch.cuda.synchronize()
            got = wire[shift:shift + cnt]
            assert torch.equal(got, G[off:off + cnt].bfloat16()), (off, cnt, shift)
            assert (wire[:shift] == sentinel).all() and (wire[shift + cnt:] == sentinel).all()
            got.mul_(2)                                                  # what an all-reduce of two equal ranks returns
            check(lib.dmg_train_grad_unpack(h, off, cnt, w, _st()), 'unpack')
            torch.cuda.synchronize()
            assert torch.equal(G[off:off + cnt], got.float()), (off, cnt, shift)
            assert torch.equal(G[:off], before[:off]) and torch.equal(G[off + cnt:], before[off + cnt:])
            G.copy_(before)
    tr.close()


# ---------------------------------------------------------------------------------------------- Adam through the trainer
# Worst on one B200 (1000 W): parameter change 2.6e-5 of lr beyond two ulps of p, exp_avg 2.7e-7, exp_avg_sq 1.4e-6 relative,
# grad_norm 9.2e-8.  Tolerances <= 3x.
ADAM_TOL = {'dp': 7.8e-5, 'm1': 8e-7, 'm2': 4e-6, 'gn': 2.7e-7}


def _names_and_shapes(tr):
    return {n: s for n, s in tr.e.weight_names().items() if n != '1.decoder.weight'}


@pytest.mark.parametrize('step,clip,grad_scale', [
    (1, 0.5, 1.0),          # first step, clip active
    (1, 0.0, 0.5),          # no clipping, averaged over two ranks
    (1000, 1e6, 0.5),       # resumed, clip inactive
    (1000, 0.5, 1.0),       # resumed, clip active
])
def test_adam_step_matches_float64(step, clip, grad_scale):
    cfg, pm, tr = _small_trainer()
    lib, h = tr.lib, tr.e.h
    assert lib.dmg_train_grad_buffer(h) == tr.grad.data_ptr()
    shapes = _names_and_shapes(tr)
    assert sum(int(np.prod(s)) for s in shapes.values()) == tr.grad.numel()      # no padding in the flat buffer
    assert int(np.prod(shapes['0.encoder.weight'])) == 41472                     # three Adam chunks: 16384 + 16384 + 8704
    rng = np.random.default_rng(step + int(clip * 10))
    lr, betas, eps, wd = 3e-3, (0.9, 0.99), 1e-8, 0.01
    # the flat gradient, written through the buffer dmg_train_grad_buffer names.  Its layout is found by writing the element
    # index into it and reading every parameter back by name.
    tr.grad.copy_(torch.arange(tr.grad.numel(), dtype=torch.float32, device='cuda'))
    torch.cuda.synchronize()
    offs = {}
    for n, g in tr.grads().items():
        offs[n] = int(g.view(-1)[0])
        assert torch.equal(g.view(-1), torch.arange(offs[n], offs[n] + g.numel(), dtype=torch.float32)), n
    flat = rng.normal(size=tr.grad.numel()) * 0.05
    o = offs['0.encoder.weight']
    flat[o + 16000:o + 17000] = 0                                       # exact zeros across the first chunk boundary
    o = offs['1.decoder.bias']
    flat[o:o + V] = 0                                                   # a whole tensor without gradient
    tr.grad.copy_(torch.tensor(flat, dtype=torch.float32, device='cuda'))
    torch.cuda.synchronize()
    grads = tr.grads()
    w0 = {n: v.clone() for n, v in pm.state_dict().items() if n in shapes}
    m1 = {n: rng.normal(size=s).astype(np.float32) * 0.01 if step > 1 else np.zeros(s, np.float32) for n, s in shapes.items()}
    m2 = {n: (rng.random(size=s).astype(np.float32) * 1e-3) if step > 1 else np.zeros(s, np.float32) for n, s in shapes.items()}
    for n in shapes:
        for which, arr in ((1, m1[n]), (2, m2[n])):
            a = np.ascontiguousarray(arr)
            check(lib.dmg_train_opt_state(h, n.encode(), which, 1, a.ctypes.data_as(C.c_void_p), a.size), 'opt_state')
    lib.dmg_train_opt_steps(h, step - 1)
    check(lib.dmg_train_optimizer_step(h, lr, betas[0], betas[1], eps, wd, clip, grad_scale, _st()), 'optimizer step')
    torch.cuda.synchronize()
    assert lib.dmg_train_opt_steps(h, -1) == step
    names = list(shapes)
    P, M1, M2 = ref.adam([host(w0[n]) for n in names], [grads[n].double().numpy() for n in names], [m1[n] for n in names],
                         [m2[n] for n in names], step, lr, betas, eps, wd, clip, grad_scale)
    w1 = pm.state_dict()
    errs = {'dp': 0.0, 'm1': 0.0, 'm2': 0.0}
    for i, n in enumerate(names):
        got_m1, got_m2 = np.empty(shapes[n], np.float32), np.empty(shapes[n], np.float32)
        check(lib.dmg_train_opt_state(h, n.encode(), 1, 0, got_m1.ctypes.data_as(C.c_void_p), got_m1.size), 'opt_state')
        check(lib.dmg_train_opt_state(h, n.encode(), 2, 0, got_m2.ctypes.data_as(C.c_void_p), got_m2.size), 'opt_state')
        p0 = host(w0[n])
        dp = host(w1[n]) - p0
        ulp = np.spacing(np.abs(p0).astype(np.float32)).astype(np.float64)
        errs['dp'] = max(errs['dp'], float(((np.abs(dp - (P[i] - p0)) - 2 * ulp).clip(0) / lr).max()))
        errs['m1'] = max(errs['m1'], maxrel(got_m1, M1[i]))
        errs['m2'] = max(errs['m2'], maxrel(got_m2, M2[i]))
    gn_ref = float(np.sqrt(sum((grads[n].double().numpy() ** 2).sum() for n in names)))
    errs['gn'] = abs(tr.losses()['grad_norm'] - gn_ref) / gn_ref
    print(f'adam step {step} clip {clip} grad_scale {grad_scale}:', {k: f'{v:.2e}' for k, v in errs.items()}, flush=True)
    for k, v in errs.items():
        assert v < ADAM_TOL[k], (k, v)
    tr.close()


def test_adam_refreshes_every_bf16_weight_copy():
    """After a few optimizer steps, a trainer built afresh from the stepped fp32 weights (which casts every bf16 copy itself)
    validates to the same bits: the validation metrics are summed in a fixed order, so one stale bf16 chunk anywhere shows."""
    cfg, pm, tr = _small_trainer(bs=2)
    g = torch.Generator().manual_seed(11)
    batches = [(torch.randint(0, V, (2, 64), generator=g), torch.randint(0, V, (2, 64), generator=g)) for _ in range(3)]
    for x, y in batches:
        tr.step(x, y, lr=1e-2, clip=0.0)
    got = tr.validate(batches[:2])
    _, pm2, tr2 = _small_trainer(bs=2)
    pm2.load_state_dict(pm.state_dict())
    want = tr2.validate(batches[:2])
    print('validate after 3 steps:', got, 'fresh trainer:', want, flush=True)
    assert got == want
    tr.close(); tr2.close()


def test_train_create_rejects_unsupported_d_model():
    with pytest.raises(DmgError, match='128, 256, 384, 512, 768 or 1024'):
        _small_trainer(d_model=640)


def test_entries_reject_bad_arguments_before_launching():
    lib = _lib_()
    f = torch.zeros(4096, device='cuda')
    b16 = torch.zeros(4096, device='cuda', dtype=torch.bfloat16)
    ids = torch.zeros(8, device='cuda', dtype=torch.int64)
    st = _st()
    cases = [
        ('dmg_train_embed: null', lambda: lib.dmg_train_embed(None, None, _p(f), None, None, _p(f), _p(b16), 8, 128, V, 0., 0, st)),
        ('beat / bar', lambda: lib.dmg_train_embed(_p(ids), _p(ids), _p(f), None, None, _p(f), _p(b16), 8, 128, V, 0., 0, st)),
        ('rows -1', lambda: lib.dmg_train_embed(_p(ids), None, _p(f), None, None, _p(f), _p(b16), -1, 128, V, 0., 0, st)),
        ('dmg_train_embed_bwd: rows -2', lambda: lib.dmg_train_embed_bwd(_p(ids), None, _p(f), None, _p(f), None, None, -2, 128, V, -1,
                                                                        0., 0, st)),
        ('dmg_train_ln_fwd: d=640 unsupported', lambda: lib.dmg_train_ln_fwd(_p(f), _p(b16), _p(f), _p(f), _p(b16), None, None, 4, 640,
                                                                              0., 0, st)),
        ('dmg_train_ln_fwd: rows -1', lambda: lib.dmg_train_ln_fwd(_p(f), _p(b16), _p(f), _p(f), _p(b16), None, None, -1, 128, 0., 0,
                                                                    st)),
        ('dmg_train_ln_bwd: null', lambda: lib.dmg_train_ln_bwd(_p(f), None, _p(b16), None, _p(f), _p(b16), _p(f), _p(f), None, 4, 128,
                                                                 0., 0, st)),
        ('dmg_train_ln_bwd: d=96 unsupported', lambda: lib.dmg_train_ln_bwd(_p(f), None, _p(b16), _p(f), _p(f), _p(b16), _p(f), _p(f),
                                                                             None, 4, 96, 0., 0, st)),
        ('ldl 300', lambda: lib.dmg_train_ce(_p(f), 300, _p(ids), -1, _p(b16), _p(f), None, 8, V, st)),
        ('needs the count', lambda: lib.dmg_train_ce(_p(f), 384, _p(ids), 0, _p(b16), _p(f), None, 8, V, st)),
        ('dmg_train_ce: rows -1', lambda: lib.dmg_train_ce(_p(f), 384, _p(ids), -1, _p(b16), _p(f), None, -1, V, st)),
        ('dmg_train_rnn_dropout: B 1, T 2, d 130', lambda: lib.dmg_train_rnn_dropout(_p(b16), _p(b16), 1, 2, 130, 0.1, 0, st)),
        ('dmg_train_rnn_dropout: dropout probability', lambda: lib.dmg_train_rnn_dropout(_p(b16), _p(b16), 1, 2, 128, 1.5, 0, st)),
        ('dmg_train_head_bwd: null', lambda: lib.dmg_train_head_bwd(_p(b16), None, _p(f), 1, 2, 128, 0., 0, 0., st)),
        ('dmg_train_sumsq: n -1', lambda: lib.dmg_train_sumsq(_p(f), -1, 0, None, 0, _p(f), st)),
        ('16-byte aligned', lambda: lib.dmg_train_sumsq(C.c_void_p(f.data_ptr() + 4), 16, 0, None, 0, _p(f), st)),
        ('needs part', lambda: lib.dmg_train_sumsq(_p(f), 16, 1, None, 0, _p(f), st)),
        ('dmg_train_tar: B 1, n 4, d 3', lambda: lib.dmg_train_tar(_p(b16), 12, 1, 4, 3, _p(f), st)),
        ('dmg_train_tar: null', lambda: lib.dmg_train_tar(_p(b16), 512, 1, 4, 128, None, st)),
        ('dmg_train_colsum: rows 4, n 10, ld 8', lambda: lib.dmg_train_colsum(_p(b16), 8, 4, 10, _p(f), st)),
        ('dmg_train_colsum: null', lambda: lib.dmg_train_colsum(None, 16, 4, 10, _p(f), st)),
    ]
    torch.cuda.synchronize()
    n0 = lib.dmg_launch_count()
    for what, call in cases:
        assert call() != 0, what
        assert what in lib.dmg_last_error().decode(), (what, lib.dmg_last_error())
    assert lib.dmg_launch_count() == n0
