"""Float64 reference of the attention of a Transformer-XL segment of T tokens over a K/V ring (the kernels behind dmg_attn_segment:
attention.cu, attention_flash.cu, attention_train_tc.cu with the ring, and the ring append of elementwise.cu).  No CUDA:
tests/test_segment_ref_cpu.py anchors it to the oracle, tests/test_gpu_segment_attention.py compares the kernels with it.  The BERT
encoder's segment attention is remix_attention_ref.remix_attention."""
import math

import torch

from oracle import txl


def memory_slots(pos_total, M):
    "ring slot of memory token j (oldest first) after pos_total appended tokens: (pos_total - mem_count + j) mod M"
    mc = min(pos_total, M)
    return [(pos_total - mc + j) % M for j in range(mc)]


def append_slots(pos_total, M, T):
    "(segment token t, ring slot) of the append: the last min(T, M) tokens, token t in slot (pos_total + t) mod M"
    return [(t, (pos_total + t) % M) for t in range(max(0, T - M), T)] if M else []


def segment_attention(q, k, v, kring, vring, rd, u, vb, pos_total, M, win=1, k_mask=1):
    """The relative-position attention of a segment over the memory in a ring, in float64.

    q, k, v [B, H, T, 64] of the segment; kring, vring [B, H, M, 64]; rd [H, Dcap, 64] (rel-pos keys by distance, Dcap >= mem_count + T);
    u, vb [H, 64].  The memory is mem_count = min(pos_total, M) tokens (memory_slots); key j of the context (memory, then the segment) is
    at distance mem_count + i - j from query i.  score = ((q + u) . k + (q + v) . rd[dist]) / 8, masked by
    txl.window_mask(T, m_len=mem_count, size=(win, k_mask)).  Returns (out [B, H, T, 64] float64, kring, vring after the append of
    append_slots, converted to the rings' dtype; every other slot as given)."""
    B, H, T, _ = q.shape
    mc = min(pos_total, M)
    f = lambda t: t.double()
    q, k, v, rd, u, vb = map(f, (q, k, v, rd, u, vb))
    slots = memory_slots(pos_total, M)
    K = torch.cat([f(kring[:, :, slots]), k], dim=2)            # [B, H, mc + T, 64]
    V = torch.cat([f(vring[:, :, slots]), v], dim=2)
    i = torch.arange(T, device=q.device)[:, None]
    j = torch.arange(mc + T, device=q.device)[None, :]
    dist = mc + i - j                                           # [T, mc + T]
    masked = txl.window_mask(T, q.device, m_len=mc, size=(win, k_mask))[0, 0]
    assert not (~masked & (dist < 0)).any(), 'a visible key after the query: the kernels do not implement this mask'
    bd = torch.einsum('bhid,hxd->bhix', q + vb[:, None], rd)   # (q + v) . rd[x] for every distance x of the cache
    bd = bd.gather(3, dist.clamp_min(0).expand(B, H, T, mc + T))
    s = torch.einsum('bhid,bhjd->bhij', q + u[:, None], K) + bd
    s = (s / 8).masked_fill(masked, -math.inf)
    out = torch.softmax(s, dim=-1) @ V
    kr, vr = kring.clone(), vring.clone()
    for t, slot in append_slots(pos_total, M, T):
        kr[:, :, slot] = k[:, :, t].to(kr.dtype)
        vr[:, :, slot] = v[:, :, t].to(vr.dtype)
    return out, kr, vr
