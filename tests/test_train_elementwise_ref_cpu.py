"""CPU anchor of tests/train_elementwise_ref.py: the LayerNorm backward equals float64 autograd, the embedding backward equals
autograd through nn.Embedding(padding_idx) and the oracle's BeatPositionEncoder, the cross-entropy equals torch's, the Adam
reference equals oracle.train.AdamTrueWD step by step, and the dropout hash keeps 1 - p of the elements with pairs sharing one
32-bit hash.  A wrong formula in the reference fails here, before any kernel is compared with it."""
import numpy as np
import pytest
import torch

import train_elementwise_ref as ref
from oracle import txl
from oracle.train import AdamTrueWD


@pytest.mark.parametrize('p', [0.0, 0.1, 0.3])
def test_ln_forward_backward_equals_autograd(p):
    rng = np.random.default_rng(1)
    rows, d = 9, 32
    x, add, gy = rng.normal(size=(rows, d)), rng.normal(size=(rows, d)), rng.normal(size=(rows, d))
    w, b = 1 + 0.3 * rng.normal(size=d), 0.2 * rng.normal(size=d)
    mask = ref.row_mask(77, p, rows, d)
    tx, ta, tw, tb = (torch.tensor(a, requires_grad=True) for a in (x, add, w, b))
    z = tx + ta * torch.tensor(mask)
    y = torch.nn.functional.layer_norm(z, (d,), tw, tb, eps=ref.LN_EPS)
    y.backward(torch.tensor(gy))
    yr, zr, mean, rstd = ref.ln_fwd(x, add, w, b, mask)
    np.testing.assert_allclose(yr, y.detach().numpy(), rtol=1e-12, atol=1e-12)
    g = ref.ln_bwd(gy, zr, w, mean, rstd, mask)
    np.testing.assert_allclose(g['dz'], tx.grad.numpy(), rtol=1e-10, atol=1e-12)       # z = x + ...: dz is x's gradient
    np.testing.assert_allclose(g['dadd'], ta.grad.numpy(), rtol=1e-10, atol=1e-12)
    np.testing.assert_allclose(g['dw'], tw.grad.numpy(), rtol=1e-10, atol=1e-12)
    np.testing.assert_allclose(g['db'], tb.grad.numpy(), rtol=1e-10, atol=1e-12)
    np.testing.assert_allclose(g['dsum'], ta.grad.numpy().sum(0), rtol=1e-10, atol=1e-12)


def test_embedding_equals_oracle_position_encoder_and_autograd():
    "positions of both signs, beat 0 / bar 0 rows, bar wrap past 32768, duplicate ids and the pad id"
    rng = np.random.default_rng(2)
    V, d, pad = 11, 8, 3
    ids = np.array([0, 3, 5, 5, 10, 3, 7, 5, 12, -2])
    pos = np.array([0, 31, 32, 33, -1, -40, 32768 + 65, -32768 * 3 - 7, 64, 5])
    emb, beat, bar = rng.normal(size=(V, d)), rng.normal(size=(32, d)), rng.normal(size=(1024, d))
    enc = txl.BeatPositionEncoder(d).double()
    with torch.no_grad():
        enc.beat_enc.weight.copy_(torch.tensor(beat)); enc.bar_enc.weight.copy_(torch.tensor(bar))
    x = ref.embed_fwd(ids, pos, emb, beat, bar)
    tpos = torch.tensor(pos)
    np.testing.assert_allclose(x - emb[np.clip(ids, 0, V - 1)], enc(tpos).detach().numpy(), rtol=0, atol=1e-14)
    bt, br = ref.beat_bar([-40])
    assert (int(bt[0]), int(br[0])) == (24, 1022)
    # backward: autograd through nn.Embedding(padding_idx) (ids clamped as the kernels do) and the encoder's padding rows
    g = rng.normal(size=(len(ids), d))
    mask = ref.row_mask(9, 0.25, len(ids), d)
    e = torch.nn.Embedding(V, d, padding_idx=pad).double()
    out = e(torch.tensor(np.clip(ids, 0, V - 1))) + enc(tpos)
    (out * torch.tensor(mask)).backward(torch.tensor(g))
    demb, dbeat, dbar = ref.embed_bwd(ids, pos, g, V, pad, mask)
    np.testing.assert_allclose(demb, e.weight.grad.numpy(), rtol=1e-12, atol=1e-14)
    np.testing.assert_allclose(dbeat, enc.beat_enc.weight.grad.numpy(), rtol=1e-12, atol=1e-14)
    np.testing.assert_allclose(dbar, enc.bar_enc.weight.grad.numpy(), rtol=1e-12, atol=1e-14)
    assert not demb[pad].any() and not dbeat[0].any() and not dbar[0].any()


@pytest.mark.parametrize('ignore', [-1, 4])
def test_cross_entropy_equals_torch(ignore):
    rng = np.random.default_rng(3)
    rows, V, ldl = 13, 10, 16
    logits = rng.normal(size=(rows, ldl)) * 3
    t = rng.integers(0, V, rows)
    t[[1, 5, 6]] = ignore if ignore >= 0 else 2
    loss, dl, count = ref.cross_entropy(logits, t, V, ignore)
    x = torch.tensor(logits[:, :V], requires_grad=True)
    tl = torch.nn.functional.cross_entropy(x, torch.tensor(t), ignore_index=ignore if ignore >= 0 else -100)
    tl.backward()
    assert count == (rows if ignore < 0 else int((t != ignore).sum())) and (ignore < 0 or count <= rows - 3)
    np.testing.assert_allclose(loss / count, tl.item(), rtol=1e-12)
    np.testing.assert_allclose(dl[:, :V], x.grad.numpy(), rtol=1e-10, atol=1e-14)
    assert not dl[:, V:].any()


def test_adam_reference_equals_adam_true_wd_over_steps():
    "several steps, several tensors, clipping active on some steps, grad_scale folded into the gradient"
    rng = np.random.default_rng(4)
    shapes = [(5, 3), (7,), (2, 2, 2)]
    ps = [rng.normal(size=s) for s in shapes]
    tp = [torch.tensor(p.copy()) for p in ps]
    opt = AdamTrueWD(tp, betas=(0.9, 0.99), eps=1e-8)
    m1 = [np.zeros(s) for s in shapes]
    m2 = [np.zeros(s) for s in shapes]
    for step in range(1, 6):
        gs = [rng.normal(size=s) * (3.0 if step % 2 else 0.05) for s in shapes]
        for t, g in zip(tp, gs):
            t.grad = torch.tensor(g * 0.5)
        opt.step(1e-2, wd=0.1, clip=0.5)
        ps, m1, m2 = ref.adam(ps, gs, m1, m2, step, 1e-2, (0.9, 0.99), 1e-8, 0.1, 0.5, grad_scale=0.5)
        for a, t, m, tm, v, tv in zip(ps, tp, m1, opt.m, m2, opt.v):
            np.testing.assert_allclose(a, t.numpy(), rtol=1e-12, atol=1e-15)
            np.testing.assert_allclose(m, tm.numpy(), rtol=1e-12, atol=1e-15)
            np.testing.assert_allclose(v, tv.numpy(), rtol=1e-12, atol=1e-15)


def test_adam_reference_eps_outside_sqrt_and_bias_correction():
    "one element by hand: step 3, no clip"
    p, g, m, v = 0.5, 0.2, 0.1, 0.03
    lr, b1, b2, eps, wd = 1e-2, 0.9, 0.99, 1e-3, 0.1
    (pn,), (mn,), (vn,) = ref.adam([np.array([p])], [np.array([g])], [np.array([m])], [np.array([v])], 3, lr, (b1, b2), eps, wd, 0)
    m_ = b1 * m + (1 - b1) * g
    v_ = b2 * v + (1 - b2) * g * g
    want = p * (1 - lr * wd) - lr * (m_ / (1 - b1 ** 3)) / (np.sqrt(v_ / (1 - b2 ** 3)) + eps)
    np.testing.assert_allclose([pn[0], mn[0], vn[0]], [want, m_, v_], rtol=1e-14)


def test_dropout_hash_keep_rate_and_pairs():
    n = 1 << 20
    for p in (0.1, 0.25, 0.5):
        keep = ref.drop_keep(1234, np.arange(n, dtype=np.uint32), ref.drop_thresh16(p))
        assert abs(keep.mean() - (1 - p)) < 3e-3
    assert ref.drop_thresh16(0.1) == 6554 and ref.drop_thresh16(0.0) == 0 and ref.drop_thresh16(1.0) == 65535
    assert ref.drop_scale(0.1) == np.float32(1.0) / (np.float32(1.0) - np.float32(6554) / np.float32(65536))
    # elements 2k and 2k+1 read the low and high half of one hash
    seed, k = 987654321, np.arange(1000, dtype=np.uint32)
    h = ref.drop_pair_bits(seed, k)
    t = 30000
    assert np.array_equal(ref.drop_keep(seed, 2 * k, t), (h & 0xFFFF) >= t)
    assert np.array_equal(ref.drop_keep(seed, 2 * k + 1, t), (h >> 16) >= t)
    # the numpy uint32 arithmetic wraps exactly like the kernels' 32-bit integers (checked against Python integers)
    def mix32_int(x):
        x ^= x >> 16; x = (x * 0x7feb352d) & 0xFFFFFFFF; x ^= x >> 15; x = (x * 0x846ca68b) & 0xFFFFFFFF; x ^= x >> 16
        return x
    xs = np.random.default_rng(6).integers(0, 1 << 32, 500, dtype=np.uint64).astype(np.uint32)
    assert [int(v) for v in ref.mix32(xs)] == [mix32_int(int(v)) for v in xs]
    m = ref.row_mask(5, 0.5, 4, 8)
    assert set(np.unique(m)) <= {0.0, 2.0}
    s = ref.stream_mask(5, 0.5, 3, 8)
    assert s.shape == (3, 1, 8) and np.array_equal(s.reshape(-1), ref.dropout_mask(5, 0.5, 24))
