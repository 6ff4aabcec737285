"""Float64 references of the one-token decode kernels (no CUDA): the decode attention over a K/V ring (attention_decode2.cuh,
attention_decode3.cuh) and the fused layer step (decode_layer.cu).  tests/test_decode_ref_cpu.py anchors both to the oracle;
tests/test_gpu_decode_kernels.py compares the kernels with them."""
import math

import torch


def gelu_tanh(x):
    return 0.5 * x * (1 + torch.tanh(math.sqrt(2 / math.pi) * (x + 0.044715 * x ** 3)))


def slot_distance(pos_total, M, device=None):
    """Distance of the key in every ring slot [M] after pos_total appended tokens: slot p holds the token appended
    ((pos_total % M) - p - 1) mod M + 1 steps ago, so the slot the new token is written to (pos_total % M) holds the oldest, M."""
    p = torch.arange(M, device=device)
    return (pos_total % M - p - 1) % M + 1


def ring_attention(q, k_new, v_new, kring, vring, rd, u, v, pos_total, M):
    """One-token relative-position attention over a ring, in float64.

    q, k_new, v_new [B, H, 64]; kring, vring [B, H, M, 64]; rd [H, Dcap, 64] (rel-pos keys by distance, Dcap >= M + 1); u, v [H, 64].
    Slot p holds the key at distance slot_distance(pos_total, M)[p]; it is part of the memory iff that distance is at most
    mem_count = min(pos_total, M).  The new token sits at distance 0.  score = ((q + u) . k + (q + v) . rd[dist]) / 8, exact softmax
    over the memory and the new token.  Returns (out [B, H, 64] float64, kring, vring after the append: slot pos_total % M holds k_new /
    v_new converted to the rings' dtype, everything else as given)."""
    f = lambda t: t.double()
    q, k_new, v_new, K, V, rd, u, v = map(f, (q, k_new, v_new, kring, vring, rd, u, v))
    mc = min(pos_total, M)
    dist = slot_distance(pos_total, M, device=q.device)
    valid = dist <= mc
    qu, qv = q + u[None], q + v[None]
    s_mem = torch.einsum('bhd,bhmd->bhm', qu, K) + torch.einsum('bhd,hmd->bhm', qv, rd[:, dist])
    s_mem = torch.where(valid, s_mem / 8, torch.full_like(s_mem, -math.inf))
    s_new = ((qu * k_new).sum(-1) + (qv * rd[None, :, 0]).sum(-1)) / 8
    p = torch.softmax(torch.cat([s_mem, s_new[..., None]], dim=-1), dim=-1)
    p_mem = torch.where(valid, p[..., :M], torch.zeros_like(p[..., :M]))      # masked slots contribute nothing, whatever they hold
    out = torch.einsum('bhm,bhmd->bhd', p_mem, V) + p[..., M:] * v_new
    head = pos_total % M
    kr, vr = kring.clone(), vring.clone()
    kr[:, :, head] = k_new.to(kr.dtype)
    vr[:, :, head] = v_new.to(vr.dtype)
    return out, kr, vr


def _ln(x, w, b):
    mu = x.mean(-1, keepdim=True)
    var = ((x - mu) ** 2).mean(-1, keepdim=True)
    return (x - mu) / torch.sqrt(var + 1e-5) * w + b


def layer_step(x, attn, wo, bo, ln1w, ln1b, w1, b1, w2, b2, ln2w, ln2b, wqkv, bqkv, mode, operand_rounding=False):
    """The fused one-token layer step, in float64.  x [B, d]; attn [B, HD]; weights in nn.Linear layout; biases may be None.

    mode bit 0 (layer body): x1 = LN1(x + attn Wo^T + bo), x = LN2(x1 + gelu_tanh(x1 W1^T + b1) W2^T + b2); bit 1: q|k|v =
    x Wqkv^T + bqkv (of the x the body left, or of the given x without the body).  LayerNorm eps 1e-5.  Returns (x, qkv, xa):
    xa is the bf16-valued copy of the body's output (None without the body), qkv None without bit 1.

    operand_rounding=True applies the rounding points of decode_layer.cu (every other value stays float64, as the kernel's are fp32):
      * the attention rows are bf16 (the TMA-loaded B operand of the out-projection);
      * the LN1 output feeds FFN-up as bf16 (the slices every CTA writes into its XA), while LN2 adds the fp32 LN1 output (X1);
      * the GeLU output is bf16 (HS, the B operand of the split-K FFN-down);
      * the LN2 output feeds the next q|k|v as bf16 (the rows broadcast into XA) and is stored to xa_out as bf16;
      * in mode 2 the given x rows feed q|k|v as bf16 (dl_store_xa of the embedded rows).
    The weights are bf16 in the kernel; pass bf16-valued weights to compare with it."""
    r = (lambda t: t.to(torch.bfloat16).double()) if operand_rounding else (lambda t: t)
    lin = lambda a, w, b: a @ w.double().t() + (b.double() if b is not None else 0)
    x = x.double()
    qkv = xa = None
    if mode & 1:
        x1 = _ln(x + lin(r(attn.double()), wo, bo), ln1w.double(), ln1b.double())
        h = r(gelu_tanh(lin(r(x1), w1, b1)))
        x = _ln(x1 + lin(h, w2, None) + (b2.double() if b2 is not None else 0), ln2w.double(), ln2b.double())
        xa = x.to(torch.bfloat16).double()
    if mode & 2:
        qkv = lin(r(x), wqkv, bqkv)
    return x, qkv, xa
