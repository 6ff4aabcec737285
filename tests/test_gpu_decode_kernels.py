"""GPU unit tests of the one-token decode kernels on their own, through dmg_attn_decode / dmg_decode_layer_step / dmg_decode_dual,
against the float64 references of decode_ref.py (which tests/test_decode_ref_cpu.py anchors to the oracle).

The model-level parity tests see these kernels only through the logits of a small random-init model, where the attention is
nearly uniform and the residual stream hides every GEMM term.  Here every comparison is per row (row_err: a 64-wide (stream, head)
row of the attention output and of q|k|v, a 512-wide row of the residual stream), the weights are scaled so that each GEMM term is
as large as the residual, every output starts as NaN, and the ring append, the masked ring slots, the rel-pos rows past M, the
padding rows of a 32-row cluster and the partial-sum scratch are probed directly."""
import ctypes as C
import math

import pytest
import torch

import decode_ref
from deepmusicgeneration_b200 import _lib
from deepmusicgeneration_b200._lib import DmgError, check
from test_gpu_train_kernels import _st, row_err

pytestmark = pytest.mark.gpu

D, DI = 512, 2048                   # the geometry of the fused layer kernel
GARBAGE = 1e4                       # finite values in the ring slots outside the memory

# Worst row errors measured on one NVIDIA B200 (1000 W power limit) over the cases below; each tolerance is at most 3x its value.
#   attention output, inputs x0.8:          kernel 0 4.2e-3, kernel 1 4.3e-3
#   attention output, q x3 / x4:            kernel 0 1.5e-2, kernel 1 1.7e-2  (bf16 q + u / q + v operands against exact scores)
#   layer step (1/sqrt(fan_in) weights):    x32 6.9e-4, q|k|v 2.2e-3, xa_out 1.3e-3
#   layer step (0.02 weights):              x32 7.3e-5, q|k|v 8.8e-4, xa_out 7.3e-4
TOL = {'attn': 1.2e-2, 'attn_peaked': 5e-2, 'x32': 2e-3, 'qkv': 6e-3, 'xa': 3.5e-3}
TOL_SMALL_W = {'x32': 2e-4, 'qkv': 2.5e-3, 'xa': 2e-3}


def bits(t):
    "a bit-level view (NaN == NaN) for bit-identity checks"
    return t.contiguous().view(torch.int16 if t.element_size() == 2 else torch.int32)


def same_bits(a, b):
    return torch.equal(bits(a), bits(b))


# ---------------------------------------------------------------------------------------------------------------------------
# decode attention
# ---------------------------------------------------------------------------------------------------------------------------
class Ring:
    "inputs of one decode-attention call: q|k|v of B streams, the K/V rings of Bcap streams (ours at [b0, b0 + B)), Rd, u, v"
    def __init__(self, B, H, M, pos_total, scale=0.8, q_scale=1.0, Bcap=None, b0=0, seed=0):
        g = torch.Generator(device='cuda').manual_seed(seed)
        self.B, self.H, self.M, self.pos_total, self.b0 = B, H, M, pos_total, b0
        self.Bcap = Bcap or B + b0
        self.Dcap = M + 65                       # rows past M inside the cache: the kernels must never use them
        HD = H * 64
        rn = lambda *s: torch.randn(*s, device='cuda', generator=g)
        self.qkv = rn(B, 3 * HD) * scale
        self.qkv[:, :HD] *= q_scale
        self.kring = (rn(self.Bcap, H, M, 64) * scale).bfloat16()
        self.vring = (rn(self.Bcap, H, M, 64) * scale).bfloat16()
        self.rd = (rn(H, self.Dcap, 64) * scale).bfloat16()
        self.u, self.v = rn(HD) * 0.3, rn(HD) * 0.3
        self.masked = decode_ref.slot_distance(pos_total, M, device='cuda') > min(pos_total, M)   # slots outside the memory
        self.junk = (rn(self.Bcap, H, M, 64).sign() * GARBAGE * (0.5 + torch.rand(self.Bcap, H, M, 64, device='cuda', generator=g)))
        self.fill(masked=GARBAGE, rd_tail=float('nan'))

    def fill(self, masked, rd_tail):
        "what the masked slots (GARBAGE: large random finite values, or 0) and the Rd rows past M (NaN or 0) hold"
        for ring in (self.kring, self.vring):
            ring[:, :, self.masked] = (self.junk[:, :, self.masked] if masked == GARBAGE else torch.zeros_like(self.junk[:, :, self.masked])).bfloat16()
        self.rd[:, self.M + 1:] = rd_tail
        return self

    def args(self, out, state, kernel, kring=None, vring=None, over={}):
        a = _lib.DecodeAttnArgs()
        a.qkv, a.kring, a.vring, a.rd, a.u, a.v, a.out, a.state = (
            t.data_ptr() for t in (self.qkv, kring if kring is not None else self.kring, vring if vring is not None else self.vring,
                                   self.rd, self.u, self.v, out, state))
        a.pos_total, a.B, a.H, a.Dh, a.M, a.Dcap, a.Bcap, a.b0, a.kernel = (
            self.pos_total, self.B, self.H, 64, self.M, self.Dcap, self.Bcap, self.b0, kernel)
        for k, v in over.items():
            setattr(a, k, v)
        return a

    def run(self, kernel):
        "one call on copies of the rings; returns (out, kring after, vring after)"
        kr, vr = self.kring.clone(), self.vring.clone()
        out = torch.full((self.B, self.H * 64), float('nan'), device='cuda', dtype=torch.bfloat16)
        state = torch.zeros(2, device='cuda', dtype=torch.int32)
        torch.cuda.synchronize()                 # the ring must not be written by the kernel launched just before
        check(_lib.load().dmg_attn_decode(C.byref(self.args(out, state, kernel, kr, vr)), _st()), 'dmg_attn_decode')
        assert state.tolist() == [self.pos_total, min(self.pos_total, self.M)]
        return out, kr, vr

    def reference(self):
        B, H, HD, s = self.B, self.H, self.H * 64, slice(self.b0, self.b0 + self.B)
        q, k, v = (self.qkv[:, i * HD:(i + 1) * HD].view(B, H, 64) for i in range(3))
        out, kr, vr = decode_ref.ring_attention(q, k, v, self.kring[s], self.vring[s], self.rd, self.u.view(H, 64), self.v.view(H, 64),
                                                self.pos_total, self.M)
        kring, vring = self.kring.clone(), self.vring.clone()
        kring[s], vring[s] = kr, vr
        return out, kring, vring


def n_sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def straddling_ctas(B, H, M):
    "CTAs of the third kernel whose (stream, head) items span two heads (the prologue reloads Rd for the second one)"
    per = 16 * n_sms() // H                      # streams per launch (D3_CAP items per CTA)
    n = 0
    for c0 in range(0, B, per):
        b = min(per, B - c0)
        ni, grid = b * H, min(b * H, n_sms())
        for cta in range(grid):
            lo, hi = ni * cta // grid, ni * (cta + 1) // grid
            n += hi > lo and lo // b != (hi - 1) // b
    return n


POS = lambda M: [0, 1, M - 1, M, M + 1, 2 * M + 37, 10 ** 6 + 3]
KERNEL_M = [(0, 128), (0, 256), (0, 384), (0, 512), (1, 64), (1, 192), (1, 512), (1, 1024)]

ATTN_CASES = (   # kernel, B, H, M, pos_total, q scale, Bcap, b0
    [(k, 5, 8, M, pt, 1.0, None, 0) for k, M in KERNEL_M for pt in POS(M)]            # one item per CTA, every ring position class
    + [(k, 1, 1, M, pt, 1.0, None, 0) for k, M in KERNEL_M for pt in (M + 1, 2 * M + 37)]
    + [(k, 40, 8, M, pt, 1.0, None, 0) for k, M in [(0, 128), (0, 384), (0, 512), (1, 64), (1, 192), (1, 512)]
       for pt in (M - 1, 2 * M + 37)]
    + [(0, 300, 8, 128, pt, 1.0, None, 0) for pt in (129, 10 ** 6 + 3)]                # the third kernel's two stream chunks
    + [(k, 64, 8, M, 2 * M + 37, 1.0, 80, 7) for k, M in [(0, 256), (1, 192)]]        # streams [7, 71) of an 80-stream ring
    + [(1, 8, 16, 1024, pt, 1.0, None, 0) for pt in (1000, 10 ** 6 + 3)]                # the C5 geometry
    + [(k, B, 8, M, 2 * M + 37, qs, None, 0) for k, M in KERNEL_M for B, qs in ((5, 3.0), (40, 4.0))]   # peaked softmax
)


def _attn_id(c):
    k, B, H, M, pt, qs, Bcap, b0 = c
    return f'k{k}-B{B}-H{H}-M{M}-pos{pt}' + (f'-q{qs:g}' if qs != 1 else '') + (f'-b0{b0}' if b0 else '')


@pytest.mark.parametrize('kernel,B,H,M,pos_total,q_scale,Bcap,b0', ATTN_CASES, ids=[_attn_id(c) for c in ATTN_CASES])
def test_attention_against_float64_reference(kernel, B, H, M, pos_total, q_scale, Bcap, b0):
    if B == 40:
        assert straddling_ctas(B, H, M) >= 1, 'B=40 is meant to give CTAs whose items straddle a head boundary'
    x = Ring(B, H, M, pos_total, q_scale=q_scale, Bcap=Bcap, b0=b0, seed=kernel * 7919 + B * 131 + M + pos_total % 9973)
    ref_out, ref_k, ref_v = x.reference()
    out, kr, vr = x.run(kernel)
    assert not torch.isnan(out).any(), 'output elements left unwritten (or NaN from the masked slots / Rd rows past M)'
    err = row_err(out, ref_out)
    tol = TOL['attn_peaked' if q_scale > 1 else 'attn']
    print(f'attention {_attn_id((kernel, B, H, M, pos_total, q_scale, Bcap, b0))}: row error {err:.2e}', flush=True)
    assert err <= tol, f'worst (stream, head) row error {err:.2e} > {tol:.1e}'
    # the append: exactly slot pos_total % M of the covered streams, as bf16(k_new) / bf16(v_new); nothing else moves
    for name, got, want in (('K', kr, ref_k), ('V', vr, ref_v)):
        if not same_bits(got, want):
            diff = (bits(got) != bits(want)).any(-1).nonzero().tolist()
            pytest.fail(f'{name} ring after the call differs at (stream, head, slot) {diff[:8]} (append slot {pos_total % M}, '
                        f'streams [{b0}, {b0 + B}))')
    # masked slots: large finite garbage there and zeros there give the same bits; so do NaN and zeros in the Rd rows past M
    x.fill(masked=0.0, rd_tail=float('nan'))
    out_zero_slots = x.run(kernel)[0]
    assert same_bits(out, out_zero_slots), 'the slots outside the memory reach the output'
    x.fill(masked=0.0, rd_tail=0.0)
    out_zero_rd = x.run(kernel)[0]
    assert same_bits(out_zero_slots, out_zero_rd), 'the rel-pos rows past M reach the output'
    assert same_bits(out_zero_rd, x.run(kernel)[0]), 'two runs from the same ring differ'


def test_attention_rejects_bad_arguments_before_launching():
    lib = _lib.load()
    x = Ring(4, 2, 128, 200)
    out = torch.zeros(4, 128, device='cuda', dtype=torch.bfloat16)
    state = torch.zeros(2, device='cuda', dtype=torch.int32)
    call = lambda over={}: check(lib.dmg_attn_decode(C.byref(x.args(out, state, 0, over=over)), _st()), 'dmg_attn_decode')
    torch.cuda.synchronize()
    launches = lib.dmg_launch_count()
    bad = [({'Dh': 32}, 'head size'), ({'M': 96}, 'mem_len'), ({'M': 100, 'kernel': 1}, 'mem_len'), ({'M': 4096, 'Dcap': 4097}, 'mem_len'),
           ({'Dcap': 128}, 'rel-pos cache'), ({'b0': 1}, 'outside the ring'), ({'B': 5}, 'outside the ring'),
           ({'pos_total': -1}, 'pos_total'), ({'kernel': 2}, 'kernel'), ({'qkv': None}, 'null'), ({'state': None}, 'null'),
           ({'rd': None}, 'null')]
    for over, msg in bad:
        with pytest.raises(DmgError, match=msg):
            call(over)
    assert lib.dmg_launch_count() == launches
    call()                                       # the same arguments without the fault do run
    assert lib.dmg_launch_count() > launches


# ---------------------------------------------------------------------------------------------------------------------------
# fused layer step
# ---------------------------------------------------------------------------------------------------------------------------
class Layer:
    "weights of one layer body + the next layer's q|k|v projection, bf16 as the kernel reads them"
    def __init__(self, w_scale=None, seed=0):
        g = torch.Generator(device='cuda').manual_seed(seed)
        rn = lambda *s: torch.randn(*s, device='cuda', generator=g)
        w = lambda n, k: (rn(n, k) * (w_scale or 1 / math.sqrt(k))).bfloat16()     # 1/sqrt(fan_in): each GEMM term ~ the residual
        self.wo, self.w1, self.w2, self.wqkv = w(D, D), w(DI, D), w(D, DI), w(3 * D, D)
        self.bo, self.b1, self.b2, self.bqkv = rn(D) * 0.1, rn(DI) * 0.1, rn(D) * 0.1, rn(3 * D) * 0.1
        self.ln1w, self.ln1b, self.ln2w, self.ln2b = 1 + 0.1 * rn(D), 0.1 * rn(D), 1 + 0.1 * rn(D), 0.1 * rn(D)


class Rows:
    "the row buffers of one step: residual stream, attention rows, q|k|v, xa_out, the partial-sum scratch"
    def __init__(self, n_rows, attn_rows, seed):
        g = torch.Generator(device='cuda').manual_seed(seed)
        self.x32 = torch.randn(n_rows, D, device='cuda', generator=g)
        self.attn = torch.randn(attn_rows, D, device='cuda', generator=g).bfloat16()
        self.qkv = torch.full((n_rows, 3 * D), float('nan'), device='cuda')
        self.xa = torch.full((n_rows, D), float('nan'), device='cuda', dtype=torch.bfloat16)
        self.pp = torch.full((8, n_rows * D), float('nan'), device='cuda')

    def clone(self):
        r = Rows.__new__(Rows)
        r.__dict__.update({k: v.clone() for k, v in self.__dict__.items()})
        return r


def layer_args(L, R, row_base, B, mode, xa_out=True, over={}):
    a = _lib.DecodeLayerArgs()
    for name, t in (('x32', R.x32), ('attn', R.attn), ('qkv', R.qkv), ('pp', R.pp), ('xa_out', R.xa if xa_out else None)):
        setattr(a, name, t.data_ptr() if t is not None else None)
    for name in ('wo', 'w1', 'w2', 'wqkv', 'bo', 'ln1w', 'ln1b', 'b1', 'b2', 'ln2w', 'ln2b', 'bqkv'):
        setattr(a, name, getattr(L, name).data_ptr())
    a.pp_stride, a.attn_rows, a.row_base, a.B, a.mode = R.pp.shape[1], R.attn.shape[0], row_base, B, mode
    a.d_model, a.n_heads, a.d_head, a.d_inner = D, 8, 64, DI
    for k, v in over.items():
        setattr(a, k, v)
    return a


def run_layer(L, R, row_base, B, mode, xa_out):
    torch.cuda.synchronize()
    check(_lib.load().dmg_decode_layer_step(C.byref(layer_args(L, R, row_base, B, mode, xa_out)), _st()), 'dmg_decode_layer_step')


def rows_padded(row_base, B):
    return row_base + (B - row_base + 31) // 32 * 32


LAYER_CASES = ([(B, 0, mode, None) for B in (1, 5, 32, 40, 256) for mode in (1, 2, 3)]
               + [(40, 32, mode, None) for mode in (1, 2, 3)] + [(256, 128, mode, None) for mode in (1, 2, 3)]
               + [(40, 0, 3, 0.02), (40, 0, 1, 0.02)])


@pytest.mark.parametrize('B,row_base,mode,w_scale', LAYER_CASES,
                         ids=[f'B{B}-rb{rb}-mode{m}' + (f'-w{w}' if w else '') for B, rb, m, w in LAYER_CASES])
def test_layer_step_against_float64_reference(B, row_base, mode, w_scale):
    L = Layer(w_scale, seed=B + mode)
    n_rows = rows_padded(row_base, B) + 8
    R0 = Rows(n_rows, rows_padded(row_base, B) + 32, seed=3 * B + row_base)
    R0.attn[B:] = float('nan')                   # rows of the last cluster past B (and beyond): read, never used
    xa_out = mode == 1
    R = R0.clone()
    run_layer(L, R, row_base, B, mode, xa_out)
    s = slice(row_base, B)
    x_ref, qkv_ref, xa_ref = decode_ref.layer_step(R0.x32[s], R0.attn[s], L.wo, L.bo, L.ln1w, L.ln1b, L.w1, L.b1, L.w2, L.b2, L.ln2w,
                                                   L.ln2b, L.wqkv, L.bqkv, mode, operand_rounding=True)
    errs = {}
    if mode & 1:
        errs['x32'] = row_err(R.x32[s], x_ref, D)
        if xa_out:
            assert not torch.isnan(R.xa[s]).any()
            errs['xa'] = row_err(R.xa[s], xa_ref, D)
    if mode & 2:
        assert not torch.isnan(R.qkv[s]).any(), 'q|k|v elements left unwritten'
        errs['qkv'] = row_err(R.qkv[s], qkv_ref)
    print(f'layer step B={B} row_base={row_base} mode={mode} w={w_scale or "1/sqrt(fan_in)"}:',
          {n: f'{e:.2e}' for n, e in errs.items()}, flush=True)
    tol = TOL_SMALL_W if w_scale else TOL
    bad = {n: e for n, e in errs.items() if not e <= tol[n]}
    assert not bad, f'worst row error over tolerance: {bad}'
    # rows outside [row_base, B) of every output, and every output the mode does not write, are untouched
    outside = lambda t: torch.cat([t[:row_base], t[B:]])
    assert same_bits(outside(R.x32), outside(R0.x32)), 'x32 rows outside [row_base, B) written'
    assert same_bits(outside(R.qkv), outside(R0.qkv)), 'q|k|v rows outside [row_base, B) written'
    assert same_bits(outside(R.xa), outside(R0.xa)), 'xa_out rows outside [row_base, B) written'
    if not mode & 1:
        assert same_bits(R.x32, R0.x32) and same_bits(R.xa, R0.xa), 'mode 2 wrote the residual stream'
    if not mode & 2:
        assert same_bits(R.qkv, R0.qkv), 'mode 1 wrote q|k|v'
    # the partial-sum scratch and the attention rows past B: NaN there and zeros there give the same bits; two runs agree
    R1 = R0.clone()
    R1.pp.zero_()
    R1.attn[B:] = 0
    run_layer(L, R1, row_base, B, mode, xa_out)
    for name in ('x32', 'qkv', 'xa'):
        assert same_bits(getattr(R, name), getattr(R1, name)), f'{name}: the NaN in the scratch or in attention rows past B leaked in'
    R2 = R0.clone()
    R2.pp.zero_()
    R2.attn[B:] = 0
    run_layer(L, R2, row_base, B, mode, xa_out)
    for name in ('x32', 'qkv', 'xa', 'pp'):
        assert same_bits(getattr(R1, name), getattr(R2, name)), f'{name}: two runs differ'


def test_layer_step_rejects_bad_arguments_before_launching():
    lib = _lib.load()
    L, R = Layer(seed=1), Rows(72, 96, seed=1)
    call = lambda over={}: check(lib.dmg_decode_layer_step(C.byref(layer_args(L, R, 32, 40, 3, over=over)), _st()),
                                 'dmg_decode_layer_step')
    torch.cuda.synchronize()
    launches = lib.dmg_launch_count()
    bad = [({'d_model': 256}, 'geometry'), ({'d_inner': 1024}, 'geometry'), ({'n_heads': 4}, 'geometry'), ({'d_head': 32}, 'geometry'),
           ({'pp_stride': 63 * D}, 'pp_stride'), ({'row_base': 40}, 'empty'), ({'attn_rows': 39}, 'attn_rows'), ({'mode': 0}, 'mode'),
           ({'mode': 4}, 'mode'), ({'w2': None}, 'null'), ({'qkv': None}, 'null'), ({'pp': None}, 'null')]
    for over, msg in bad:
        with pytest.raises(DmgError, match=msg):
            call(over)
    assert lib.dmg_launch_count() == launches
    call({'pp_stride': 64 * D})                       # rows [32, 40) are one cluster [32, 64): 64 rows of scratch are enough
    assert lib.dmg_launch_count() > launches


# ---------------------------------------------------------------------------------------------------------------------------
# dual-role launch
# ---------------------------------------------------------------------------------------------------------------------------
DUAL_CASES = [(64, 128), (64, 512), (256, 128), (256, 512), (300, 128)]


@pytest.mark.parametrize('B,M', DUAL_CASES, ids=[f'B{B}-M{M}' for B, M in DUAL_CASES])
@pytest.mark.parametrize('order', ['A(Y)+F(X)', 'A(X)+F(Y)'])
def test_dual_launch_equals_each_role_alone(B, M, order):
    """The fused step over one half of the streams and the attention over the other half in one launch: every buffer bit-identical to
    dmg_decode_layer_step over the fused rows followed by dmg_attn_decode(kernel 0) over the attention rows, so neither role touches
    the other's rows and the attention role's CTA split changes no bit."""
    lib = _lib.load()
    hx = ((B + 31) // 32 + 1) // 2 * 32          # the step's split: the first half is whole 32-row clusters
    (f0, f1), (a0, a1) = ((0, hx), (hx, B)) if order == 'A(Y)+F(X)' else ((hx, B), (0, hx))
    L = Layer(seed=B)
    H = 8
    n_rows = (B + 31) // 32 * 32
    R0 = Rows(n_rows, n_rows, seed=B + M)
    R0.qkv.normal_(0, 0.8)                       # the attention role's input rows
    R0.qkv[f0:f1] = float('nan')                 # each role's output rows start as NaN: both must write all of them
    R0.attn[a0:a1] = float('nan')
    R0.pp.zero_()
    ring = Ring(B, H, M, 2 * M + 37, seed=B * M)
    k0, v0 = ring.kring.clone(), ring.vring.clone()

    def attn_args(R, kr, vr, out_state):
        sub = Ring.__new__(Ring)
        sub.__dict__.update(ring.__dict__)
        sub.qkv, sub.B, sub.b0 = R.qkv[a0:a1], a1 - a0, a0
        out = R.attn[a0:a1]
        return sub.args(out, out_state, 0, kr, vr)

    # each role alone
    Ra, ka, va, sa = R0.clone(), k0.clone(), v0.clone(), torch.zeros(2, device='cuda', dtype=torch.int32)
    torch.cuda.synchronize()
    check(lib.dmg_decode_layer_step(C.byref(layer_args(L, Ra, f0, f1, 3, xa_out=False)), _st()), 'dmg_decode_layer_step')
    check(lib.dmg_attn_decode(C.byref(attn_args(Ra, ka, va, sa)), _st()), 'dmg_attn_decode')
    # one dual-role launch
    Rd, kd, vd, sd = R0.clone(), k0.clone(), v0.clone(), torch.zeros(2, device='cuda', dtype=torch.int32)
    torch.cuda.synchronize()
    check(lib.dmg_decode_dual(C.byref(layer_args(L, Rd, f0, f1, 3, xa_out=False)), C.byref(attn_args(Rd, kd, vd, sd)), 0, _st()),
          'dmg_decode_dual')
    assert not torch.isnan(Rd.attn[a0:a1]).any() and not torch.isnan(Rd.qkv[f0:f1]).any()
    for name, got, want in (('x32', Rd.x32, Ra.x32), ('q|k|v', Rd.qkv, Ra.qkv), ('attention output', Rd.attn, Ra.attn),
                            ('K ring', kd, ka), ('V ring', vd, va), ('scratch', Rd.pp, Ra.pp)):
        if not same_bits(got, want):
            rows = (bits(got) != bits(want)).reshape(got.shape[0], -1).any(-1).nonzero().flatten().tolist()
            pytest.fail(f'{order} B={B} M={M}: {name} differs from the roles launched alone at rows {rows[:8]} '
                        f'(fused rows [{f0}, {f1}), attention rows [{a0}, {a1}))')
    # and neither role wrote into the other's rows
    assert same_bits(Rd.x32[a0:a1], R0.x32[a0:a1]) and same_bits(Rd.qkv[a0:a1], R0.qkv[a0:a1])
    assert same_bits(Rd.attn[f0:f1], R0.attn[f0:f1])
    other = torch.ones(B, dtype=torch.bool, device='cuda')
    other[a0:a1] = False
    assert same_bits(kd[other], k0[other]) and same_bits(vd[other], v0[other])


def test_dual_rejects_bad_arguments_before_launching():
    lib = _lib.load()
    L, R = Layer(seed=2), Rows(64, 64, seed=2)
    ring = Ring(32, 8, 128, 300, seed=2)
    out, state = torch.zeros(32, D, device='cuda', dtype=torch.bfloat16), torch.zeros(2, device='cuda', dtype=torch.int32)
    call = lambda clusters=0, f_over={}, a_over={}: check(lib.dmg_decode_dual(
        C.byref(layer_args(L, R, 0, 32, 3, over=f_over)), C.byref(ring.args(out, state, 0, over=a_over)), clusters, _st()), 'dmg_decode_dual')
    torch.cuda.synchronize()
    launches = lib.dmg_launch_count()
    bad = [({'a_over': {'kernel': 1}}, 'third-generation'), ({'a_over': {'M': 192, 'Dcap': 193}}, 'third-generation'),
           ({'clusters': 1}, 'do not fit'), ({'clusters': -1}, 'attn_clusters'), ({'f_over': {'d_inner': 1024}}, 'geometry'),
           ({'a_over': {'Dcap': 100}}, 'rel-pos cache'), ({'f_over': {'pp_stride': 16 * D}}, 'pp_stride')]
    for kw, msg in bad:
        with pytest.raises(DmgError, match=msg):
            call(**kw)
    assert lib.dmg_launch_count() == launches
    call(clusters=2)                             # 32 x 8 items fit two clusters of 8 CTAs x 16 items
    assert lib.dmg_launch_count() > launches
