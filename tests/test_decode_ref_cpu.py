"""CPU anchor of tests/decode_ref.py: the ring attention and the fused layer step of the reference equal the oracle's
MultiHeadRelativeAttention / DecoderLayer / next layer's q|k|v Linear in float64 (operand rounding off).  A wrong distance map,
mask or append slot in the reference fails here, before any kernel is compared with it."""
import pytest
import torch

import decode_ref
from oracle import txl

D, H, DH, DI = 128, 2, 64, 256


def _mhra(seed):
    torch.manual_seed(seed)
    m = txl.MultiHeadRelativeAttention(H, D, DH, bias=True).double().eval()
    for p in m.parameters():          # O(1) weights: every term of the score and of the output matters
        torch.nn.init.normal_(p, std=0.3)
    return m


def test_slot_distance_covers_one_to_m():
    for pos_total in (0, 1, 7, 8, 9, 29):
        d = decode_ref.slot_distance(pos_total, 8)
        assert sorted(d.tolist()) == list(range(1, 9))
        assert d[pos_total % 8] == 8                 # the slot about to be overwritten holds the oldest key
        assert d[(pos_total - 1) % 8] == 1           # the previous token


@pytest.mark.parametrize('M,pos_total', [
    (8, 0),      # no memory: only the new token
    (8, 1),      # one token
    (8, 5),      # part of the ring, head inside it
    (8, 8),      # exactly full, head back at slot 0
    (8, 13),     # wrapped, head at 5
    (8, 16),     # wrapped, head at 0
    (12, 40),    # wrapped more than once, head at 4
])
def test_ring_attention_equals_oracle(M, pos_total):
    B = 3
    mhra = _mhra(M + pos_total)
    g = torch.Generator().manual_seed(pos_total)
    mc = min(pos_total, M)
    x = torch.randn(B, 1, D, generator=g, dtype=torch.float64)
    mem = torch.randn(B, mc, D, generator=g, dtype=torch.float64) if mc else torch.empty(0, dtype=torch.float64)
    u = torch.randn(H, 1, DH, generator=g, dtype=torch.float64)
    v = torch.randn(H, 1, DH, generator=g, dtype=torch.float64)
    pe = txl.PositionalEncoding(D).double()
    with torch.no_grad():
        want = mhra._apply_attention(x, r=pe(torch.arange(mc, -1, -1, dtype=torch.float64)), u=u, v=v, mask=None, mem=mem)
        heads = lambda t: t.view(B, -1, H, DH).permute(0, 2, 1, 3)           # [B, H, T, DH]
        q, k_new, v_new = (heads(t)[:, :, 0] for t in mhra.attention(x).chunk(3, dim=-1))
        Dcap = M + 3
        rd = mhra.r_attn(pe(torch.arange(Dcap, dtype=torch.float64))).view(Dcap, H, DH).permute(1, 0, 2)
        kring = torch.randn(B, H, M, DH, generator=g, dtype=torch.float64) * 1e4        # garbage in the slots outside the memory
        vring = torch.randn(B, H, M, DH, generator=g, dtype=torch.float64) * 1e4
        if mc:
            _, km, vm = (heads(t) for t in mhra.attention(mem).chunk(3, dim=-1))
            for j in range(mc):                     # memory token j (oldest first) lives in slot (pos_total - mc + j) mod M
                kring[:, :, (pos_total - mc + j) % M] = km[:, :, j]
                vring[:, :, (pos_total - mc + j) % M] = vm[:, :, j]
        got, kr, vr = decode_ref.ring_attention(q, k_new, v_new, kring, vring, rd, u[:, 0], v[:, 0], pos_total, M)
    assert torch.allclose(got.reshape(B, 1, H * DH), want, rtol=1e-10, atol=1e-10)
    head = pos_total % M
    assert torch.equal(kr[:, :, head], k_new) and torch.equal(vr[:, :, head], v_new)
    others = [p for p in range(M) if p != head]
    assert torch.equal(kr[:, :, others], kring[:, :, others]) and torch.equal(vr[:, :, others], vring[:, :, others])


@pytest.mark.parametrize('mode', [1, 2, 3])
def test_layer_step_equals_oracle(mode):
    torch.manual_seed(5)
    layer = txl.DecoderLayer(H, D, DH, DI, bias=True, act='gelu').double().eval()
    nxt = txl.DecoderLayer(H, D, DH, DI, bias=True, act='gelu').double().eval()
    for p in list(layer.parameters()) + list(nxt.parameters()):
        torch.nn.init.normal_(p, std=0.2)
    B = 4
    x = torch.randn(B, D, dtype=torch.float64)
    attn = torch.randn(B, H * DH, dtype=torch.float64)
    a, f = layer.mhra, layer.ff.layers
    with torch.no_grad():
        want_x = layer.ff(a.ln(x + a.out(attn))) if mode & 1 else x
        want_qkv = nxt.mhra.attention(want_x)
        got_x, got_qkv, xa = decode_ref.layer_step(x, attn, a.out.weight, a.out.bias, a.ln.weight, a.ln.bias, f[0].weight, f[0].bias,
                                                   f[3].weight, f[3].bias, f[6].weight, f[6].bias, nxt.mhra.attention.weight,
                                                   nxt.mhra.attention.bias, mode)
    assert torch.allclose(got_x, want_x, rtol=1e-10, atol=1e-10)
    if mode & 2:
        assert torch.allclose(got_qkv, want_qkv, rtol=1e-10, atol=1e-10)
    else:
        assert got_qkv is None
    if mode & 1:
        assert torch.equal(xa, got_x.to(torch.bfloat16).double())
