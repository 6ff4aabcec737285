"""CPU anchor of tests/segment_ref.py: the segment attention over a ring equals the oracle's MultiHeadRelativeAttention._apply_attention
(memory as hidden states, the window mask of window_mask) in float64, and the append leaves exactly the last min(T, M) tokens of the
segment in their slots.  A wrong slot map, distance, mask or append slot in the reference fails here, before any kernel is compared
with it."""
import pytest
import torch

import decode_ref
import segment_ref
from oracle import txl

D, H, DH = 128, 2, 64
GARBAGE = 1e4


def _mhra(seed):
    torch.manual_seed(seed)
    m = txl.MultiHeadRelativeAttention(H, D, DH, bias=True).double().eval()
    for p in m.parameters():          # O(1) weights: every term of the score and of the output matters
        torch.nn.init.normal_(p, std=0.3)
    return m


def _pos(M):
    return {'empty': 0, 'partial': M // 2 + 1, 'full': M, 'wrapped': M + 3, 'wrapped2': 2 * M + 5}


def _masks(T):
    return {'1,1': (1, 1), '1,0': (1, 0), '3,0': (3, 0), 'T+5,0': (T + 5, 0)}


CASES = [(M, pname, tname, mname) for M in (8, 12) for pname in _pos(M) for tname in ('T<M', 'T=M', 'T>M')
         for mname in _masks(0)]


@pytest.mark.parametrize('M,pname,tname,mname', CASES, ids=[f'M{M}-{p}-{t}-mask{m}' for M, p, t, m in CASES])
def test_segment_attention_equals_oracle(M, pname, tname, mname, monkeypatch):
    pos_total = _pos(M)[pname]
    T = {'T<M': M // 2 - 1, 'T=M': M, 'T>M': M + 5}[tname]
    win, k = _masks(T)[mname]
    B = 2
    mhra = _mhra(M * 1000 + pos_total * 10 + T)
    g = torch.Generator().manual_seed(pos_total + 7 * T)
    mc = min(pos_total, M)
    x = torch.randn(B, T, D, generator=g, dtype=torch.float64)
    mem = torch.randn(B, mc, D, generator=g, dtype=torch.float64) if mc else torch.empty(0, dtype=torch.float64)
    u = torch.randn(H, 1, DH, generator=g, dtype=torch.float64)
    v = torch.randn(H, 1, DH, generator=g, dtype=torch.float64)
    pe = txl.PositionalEncoding(D).double()
    mask = txl.window_mask(T, 'cpu', m_len=mc, size=(win, k))
    r = pe(torch.arange(mc + T - 1, -1, -1, dtype=torch.float64))
    with torch.no_grad(), monkeypatch.context() as mp:
        # the oracle masks in fp32 (attn_score.float().masked_fill(...).type_as(...)); lift that rounding so float64 is float64 throughout
        mp.setattr(torch.Tensor, 'float', lambda t: t)
        want = mhra._apply_attention(x, r=r, u=u, v=v, mask=mask, mem=mem)
    with torch.no_grad():
        heads = lambda t: t.view(B, -1, H, DH).permute(0, 2, 1, 3)           # [B, H, T, DH]
        q, k_seg, v_seg = (heads(t) for t in mhra.attention(x).chunk(3, dim=-1))
        Dcap = M + T + 1
        rd = mhra.r_attn(pe(torch.arange(Dcap, dtype=torch.float64))).view(Dcap, H, DH).permute(1, 0, 2)
        kring = torch.randn(B, H, M, DH, generator=g, dtype=torch.float64) * GARBAGE      # garbage in the slots outside the memory
        vring = torch.randn(B, H, M, DH, generator=g, dtype=torch.float64) * GARBAGE
        slots = segment_ref.memory_slots(pos_total, M)
        # the slot map agrees with the decode kernels': memory token j is mem_count - j tokens before the next one
        assert [decode_ref.slot_distance(pos_total, M)[s].item() for s in slots] == [mc - j for j in range(mc)]
        if mc:
            _, km, vm = (heads(t) for t in mhra.attention(mem).chunk(3, dim=-1))
            kring[:, :, slots], vring[:, :, slots] = km, vm
        got, kr, vr = segment_ref.segment_attention(q, k_seg, v_seg, kring, vring, rd, u[:, 0], v[:, 0], pos_total, M, win, k)
    assert torch.allclose(got.permute(0, 2, 1, 3).reshape(B, T, H * DH), want, rtol=1e-10, atol=1e-10)
    # the append, slot by slot: slot (pos_total + t) mod M holds segment token t for the last min(T, M) tokens, the rest is as given
    written = {}
    for t in range(T):
        written[(pos_total + t) % M] = t                  # a later token overwrites an earlier one in the same slot
    assert len(written) == min(T, M)
    for slot in range(M):
        if slot in written:
            t = written[slot]
            assert t >= T - M
            assert torch.equal(kr[:, :, slot], k_seg[:, :, t]) and torch.equal(vr[:, :, slot], v_seg[:, :, t]), f'slot {slot}'
        else:
            assert torch.equal(kr[:, :, slot], kring[:, :, slot]) and torch.equal(vr[:, :, slot], vring[:, :, slot]), f'slot {slot}'
    assert sorted(s for _, s in segment_ref.append_slots(pos_total, M, T)) == sorted(written)


def test_append_converts_to_the_ring_dtype():
    B, M, T = 1, 8, 3
    k = torch.randn(B, H, T, DH, dtype=torch.float64)
    kring = torch.zeros(B, H, M, DH, dtype=torch.bfloat16)
    _, kr, vr = segment_ref.segment_attention(k, k, k, kring, kring.clone(), torch.zeros(H, M + T + 1, DH), torch.zeros(H, DH),
                                              torch.zeros(H, DH), 6, M)
    assert kr.dtype == torch.bfloat16
    for t in range(T):
        assert torch.equal(kr[:, :, (6 + t) % M], k[:, :, t].to(torch.bfloat16))


def test_reference_refuses_a_mask_that_shows_later_keys():
    "(3, 1) lets query 31 see key 32 (31 // 3 == 32 // 3): no kernel implements that, and dmg_forward refuses it"
    T = 33
    q = torch.randn(1, 1, T, DH, dtype=torch.float64)
    with pytest.raises(AssertionError, match='visible key after the query'):
        segment_ref.segment_attention(q, q, q, torch.zeros(1, 1, 8, DH), torch.zeros(1, 1, 8, DH), torch.zeros(1, T + 9, DH),
                                      torch.zeros(1, DH), torch.zeros(1, DH), 0, 8, 3, 1)
