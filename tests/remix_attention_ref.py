"""Plain float64 restatement of the remix (masked-BERT) encoder's attention (oracle.bert.MemMultiHeadRelativeAttentionKV.
_apply_attention with mem_len 0 and r_mask=False, DESIGN.md section 9), and the map of dS into the (query row, distance)
coordinates of the kernels' ds_dist.  No CUDA: the CPU test anchors it to the oracle, the GPU test compares the kernels with it."""
import math

import torch

from oracle.txl import _line_shift


def remix_attention(q, k, v, rk, u, vb, drop_mask=None):
    """q, k, v [B, H, T, D]; rk [T, H, D] with row = distance; u, vb [H, D]; drop_mask [B, H, T, T] (already scaled) or None.
    Returns out [B, H, T, D], lse [B, H, T] of the scaled scores, and the raw scores AC + BD [B, H, T, T] (before the 1/sqrt(D)),
    whose gradient is the dS the kernels write."""
    ac, bd = score_terms(q + u[:, None], q + vb[:, None], k, rk)
    raw = ac + bd
    s = raw / math.sqrt(q.shape[-1])
    p = torch.softmax(s, dim=-1)
    if drop_mask is not None:
        p = p * drop_mask
    return p @ v, torch.logsumexp(s, dim=-1), raw


def score_terms(qu, qv, k, rk):
    "content term AC = (q + u) K^T and position term BD = _line_shift((q + v) Rk.flip(0)^T) of the raw scores, [B, H, T, T]"
    return qu @ k.transpose(-1, -2), _line_shift(qv @ rk.flip(0).permute(1, 2, 0), mask=False)   # r[-T:] runs over positions T-1 .. 0


def ds_to_dist(ds):
    """dS [B, H, T, T] (gradient of the raw scores) -> ds_dist [B, T, H, T]: row r holds dS[r, r - x] at distances x <= r (line 1)
    and dS[r - 1, T + r - x] at x > r (line 3 of the row above); row 0 is zero past distance 0."""
    B, H, T, _ = ds.shape
    r = torch.arange(T, device=ds.device)[:, None]
    x = torch.arange(T, device=ds.device)[None, :]
    line1 = x <= r
    rows = torch.where(line1, r, r - 1).clamp_min(0).expand(T, T)
    cols = torch.where(line1, r - x, T + r - x).clamp(0, T - 1)
    dist = ds[:, :, rows, cols]
    dist = torch.where(line1 | (r >= 1), dist, torch.zeros((), dtype=ds.dtype, device=ds.device))
    return dist.permute(0, 2, 1, 3)


def position_grads(ds_dist, rk, qv):
    """What the trainer's GEMMs make of ds_dist [B, T, H, T]: the position part of dq [B, T, H, D] = ds_dist . Rk per head,
    dv [H, D] = its column sum, dRk [T, H, D] = ds_dist^T (q + v) with qv [B, T, H, D]."""
    dq_pos = torch.einsum('bthx,xhd->bthd', ds_dist, rk)
    return dq_pos, dq_pos.sum((0, 1)), torch.einsum('bthx,bthd->xhd', ds_dist, qv)
