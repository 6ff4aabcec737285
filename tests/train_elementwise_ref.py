"""Float64 references of the training step's elementwise kernels (train_kernels.cu), no CUDA: the counter-based dropout hash,
embedding forward / backward, dropout + residual + LayerNorm forward / backward, cross-entropy, the RNN (per-stream) dropout
and head backward, TAR and the fused Adam.  tests/test_train_elementwise_ref_cpu.py anchors them to autograd and to
oracle.train.AdamTrueWD; tests/test_gpu_train_elementwise.py compares the kernels with them."""
import numpy as np
import torch

from oracle.train import AdamTrueWD

LN_EPS = 1e-5


# ---------------------------------------------------------------------------------------------- dropout hash (train_kernels.cuh)
def mix32(x):
    x = np.asarray(x, dtype=np.uint32).copy()
    x ^= x >> np.uint32(16)
    x *= np.uint32(0x7feb352d)
    x ^= x >> np.uint32(15)
    x *= np.uint32(0x846ca68b)
    x ^= x >> np.uint32(16)
    return x


def drop_pair_bits(seed, pair_idx):
    "one 32-bit hash per pair of neighbouring elements: the low half for the even element, the high half for the odd one"
    return mix32(np.asarray(pair_idx, dtype=np.uint32) ^ np.uint32(seed))


def drop_keep(seed, idx, thresh16):
    idx = np.asarray(idx, dtype=np.uint32)
    h = drop_pair_bits(seed, idx >> np.uint32(1))
    return ((h >> ((idx & np.uint32(1)) * np.uint32(16))) & np.uint32(0xFFFF)) >= thresh16


def drop_thresh16(p):
    "round(p * 65536) clamped to [0, 65535], in float32 as the host computes it"
    t = int(np.float32(p) * np.float32(65536.0) + np.float32(0.5))
    return min(max(t, 0), 65535)


def drop_scale(p):
    "1 / the exact keep probability, a float32"
    return float(np.float32(1.0) / (np.float32(1.0) - np.float32(drop_thresh16(p)) / np.float32(65536.0)))


def dropout_mask(seed, p, n):
    "keep ? scale : 0 for element indices 0 .. n-1 (float64); all ones for p = 0"
    if p <= 0:
        return np.ones(n)
    return np.where(drop_keep(seed, np.arange(n, dtype=np.uint32), drop_thresh16(p)), drop_scale(p), 0.0)


def row_mask(seed, p, rows, d):
    "the mask of the embedding and LayerNorm sites: element row*d + c"
    return dropout_mask(seed, p, rows * d).reshape(rows, d)


def stream_mask(seed, p, B, d):
    "the RNN (output) dropout: one mask per stream and feature, element b*d + c, shared over t -> [B, 1, d]"
    return dropout_mask(seed, p, B * d).reshape(B, 1, d)


# ---------------------------------------------------------------------------------------------- embedding
def beat_bar(pos):
    "Python floor semantics, as oracle.txl.BeatPositionEncoder: beat = pos mod 32, bar = floor(pos / 32) mod 1024"
    pos = np.asarray(pos, dtype=np.int64)
    return pos % 32, (pos // 32) % 1024


def embed_fwd(ids, pos, emb, beat, bar, mask=None):
    "x [rows, d] = (emb[clamp(id)] (+ beat[pos mod 32] + bar[floor(pos/32) mod 1024])) * mask"
    emb = np.asarray(emb, dtype=np.float64)
    ids = np.clip(np.asarray(ids, dtype=np.int64), 0, emb.shape[0] - 1)
    x = emb[ids]
    if pos is not None:
        bt, br = beat_bar(pos)
        x = x + np.asarray(beat, dtype=np.float64)[bt] + np.asarray(bar, dtype=np.float64)[br]
    return x * mask if mask is not None else x


def embed_bwd(ids, pos, g, vocab, pad_idx=-1, mask=None):
    """nn.Embedding(padding_idx=pad_idx) and the two position tables with padding_idx 0: (demb, dbeat, dbar) of the row
    gradients g [rows, d] (dx + dbr, before the dropout mask)."""
    g = np.asarray(g, dtype=np.float64)
    if mask is not None:
        g = g * mask
    d = g.shape[1]
    ids = np.clip(np.asarray(ids, dtype=np.int64), 0, vocab - 1)
    demb = np.zeros((vocab, d))
    keep = ids != pad_idx
    np.add.at(demb, ids[keep], g[keep])
    if pos is None:
        return demb, None, None
    bt, br = beat_bar(pos)
    dbeat, dbar = np.zeros((32, d)), np.zeros((1024, d))
    np.add.at(dbeat, bt[bt != 0], g[bt != 0])
    np.add.at(dbar, br[br != 0], g[br != 0])
    return demb, dbeat, dbar


# ---------------------------------------------------------------------------------------------- dropout + residual + LayerNorm
def ln_fwd(x, add, w, b, mask=None):
    "z = x + add * mask; y = LayerNorm(z) * w + b.  Returns (y, z, mean, rstd), float64"
    z = np.asarray(x, dtype=np.float64) + np.asarray(add, dtype=np.float64) * (mask if mask is not None else 1.0)
    mean = z.mean(1)
    rstd = 1.0 / np.sqrt(((z - mean[:, None]) ** 2).mean(1) + LN_EPS)
    y = (z - mean[:, None]) * rstd[:, None] * np.asarray(w, dtype=np.float64) + np.asarray(b, dtype=np.float64)
    return y, z, mean, rstd


def ln_bwd(gy, z, w, mean=None, rstd=None, mask=None):
    """Backward of y = LayerNorm(z) * w + b for the output gradient gy [rows, d].  mean / rstd default to z's own; pass the
    saved statistics (and the saved z) to evaluate the formula on what a kernel saved.  Returns a dict:
    dz (gradient wrt z), dadd = dz * mask (wrt the dropped branch), dw, db, dsum = column sums of dadd."""
    gy, z, w = (np.asarray(a, dtype=np.float64) for a in (gy, z, w))
    if mean is None:
        mean = z.mean(1)
        rstd = 1.0 / np.sqrt(((z - mean[:, None]) ** 2).mean(1) + LN_EPS)
    mean, rstd = np.asarray(mean, dtype=np.float64)[:, None], np.asarray(rstd, dtype=np.float64)[:, None]
    xh = (z - mean) * rstd
    g = gy * w
    dz = rstd * (g - g.mean(1, keepdims=True) - xh * (g * xh).mean(1, keepdims=True))
    dadd = dz * mask if mask is not None else dz
    return {'dz': dz, 'dadd': dadd, 'dw': (gy * xh).sum(0), 'db': gy.sum(0), 'dsum': dadd.sum(0)}


# ---------------------------------------------------------------------------------------------- cross-entropy
def cross_entropy(logits, targets, V, ignore=-1):
    """CrossEntropyFlat over the first V columns of logits [rows, ldl]; targets clamped to [0, V).  ignore < 0: every row
    counts and dlogits = (softmax - onehot) / rows; otherwise rows with target == ignore get no loss and zero dlogits, the
    others / count.  Returns (loss sum, dlogits [rows, ldl] with zero padding columns, count)."""
    logits = np.asarray(logits, dtype=np.float64)
    rows, ldl = logits.shape
    t = np.asarray(targets, dtype=np.int64)
    kept = np.ones(rows, dtype=bool) if ignore < 0 else t != ignore
    tc = np.clip(t, 0, V - 1)
    x = logits[:, :V]
    mx = x.max(1, keepdims=True)
    lse = mx[:, 0] + np.log(np.exp(x - mx).sum(1))
    loss = lse - x[np.arange(rows), tc]
    count = int(kept.sum())
    scale = 1.0 / rows if ignore < 0 else (1.0 / count if count else 0.0)
    d = np.exp(x - lse[:, None])
    d[np.arange(rows), tc] -= 1.0
    dl = np.zeros((rows, ldl))
    dl[:, :V] = d * scale
    dl[~kept] = 0.0
    return float(loss[kept].sum()), dl, count


# ---------------------------------------------------------------------------------------------- head
def rnn_dropout(x, mask):
    "x [B, T, d] * mask [B, 1, d]"
    return np.asarray(x, dtype=np.float64) * mask


def head_bwd(dxd, core, mask, ar_coef):
    "dx [B, T, d] = dxd * mask[b] + ar_coef * core (the activation regulariser's gradient)"
    return np.asarray(dxd, dtype=np.float64) * mask + ar_coef * np.asarray(core, dtype=np.float64)


def tar(h):
    "temporal activation regulariser value: sum over b, t >= 1 of ||h[b, t] - h[b, t-1]||^2 for h [B, n, d]"
    h = np.asarray(h, dtype=np.float64)
    return float(((h[:, 1:] - h[:, :-1]) ** 2).sum())


# ---------------------------------------------------------------------------------------------- Adam
def adam(params, grads, exp_avg, exp_avg_sq, step, lr, betas, eps, wd, clip, grad_scale=1.0):
    """One fused-Adam step in float64 through oracle.train.AdamTrueWD: gradients times grad_scale, clipped to global norm `clip`
    (<= 0: none) with coefficient clip / (||g * grad_scale|| + 1e-6), true_wd decay p *= 1 - lr*wd, then Adam with bias correction
    at step `step` (1 = the first) and eps outside the sqrt.  Lists of arrays in, (params, exp_avg, exp_avg_sq) lists out."""
    ps = [torch.tensor(np.asarray(p, dtype=np.float64)) for p in params]
    for p, g in zip(ps, grads):
        p.grad = torch.tensor(np.asarray(g, dtype=np.float64)) * grad_scale
    opt = AdamTrueWD(ps, betas=betas, eps=eps)
    opt.m = [torch.tensor(np.asarray(m, dtype=np.float64)) for m in exp_avg]
    opt.v = [torch.tensor(np.asarray(v, dtype=np.float64)) for v in exp_avg_sq]
    opt.t = step - 1
    opt.step(lr, wd=wd, clip=clip if clip > 0 else None)
    return [p.numpy() for p in ps], [m.numpy() for m in opt.m], [v.numpy() for v in opt.v]
