"""GPU unit tests of the attention of a multi-token segment on its own, through dmg_attn_segment: the general FFMA kernel (fp32 and
bf16), the flash kernel (Transformer-XL prefill, short BERT sequences), the tcgen05 kernel over the warm K/V rings and the BERT tcgen05
kernel, with the ring append that follows them, against the float64 references of segment_ref.py (anchored to the oracle by
tests/test_segment_ref_cpu.py) and remix_attention_ref.py.

The model-level parity tests see these kernels only through the logits of a small random-init model, where the attention is nearly
uniform and the residual stream hides most of the attention term.  Here every comparison is per 64-wide (stream, head) row of the
output, every output starts as NaN, and the ring slots outside the memory, the rel-pos rows past the last live distance, the ring
streams outside [b0, b0 + B) and the append are probed directly."""
import ctypes as C

import pytest
import torch

import remix_attention_ref
import segment_ref
from deepmusicgeneration_b200 import _lib
from deepmusicgeneration_b200._lib import DmgError, check
from test_gpu_decode_kernels import bits, same_bits
from test_gpu_train_kernels import _st, row_err

pytestmark = pytest.mark.gpu

GARBAGE = 1e4                       # finite values in the ring slots outside the memory and in the rel-pos rows past the last distance
GENERAL, FLASH, TC_RING, BERT_TC = _lib.SEG_GENERAL, _lib.SEG_FLASH, _lib.SEG_TC_RING, _lib.SEG_BERT_TC
KNAME = {GENERAL: 'general', FLASH: 'flash', TC_RING: 'tc_ring', BERT_TC: 'bert_tc'}

# Worst row errors measured on one NVIDIA B200 (1000 W power limit) over the cases below; each tolerance is at most 3x its value.
#   inputs x0.8:    general fp32 7.2e-7, general bf16 2.3e-3, flash 5.4e-3 (TXL) / 4.4e-3 (BERT), tcgen05 ring 5.5e-3, BERT tcgen05 5.7e-3
#   q x3 (peaked):  general fp32 1.1e-6, general bf16 2.2e-3, flash 9.2e-3, tcgen05 ring 1.0e-2, BERT tcgen05 1.05e-2
# The fp32 general kernel keeps a tolerance of its own: one bf16 rounding anywhere in its path would cost ~1e-3.  The bf16 kernels'
# errors are those of bf16 operands and a bf16 output against exact scores.  No row with a near-zero true output was seen to inflate
# row_err (its denominator carries 0.1 x the median row norm).
TOL = {'general_f32': 2e-6, 'general_bf16': 6e-3, 'flash': 1.5e-2, 'tc_ring': 1.5e-2, 'bert_tc': 1.5e-2}
TOL_PEAKED = {'general_f32': 3e-6, 'general_bf16': 6e-3, 'flash': 2.5e-2, 'tc_ring': 3e-2, 'bert_tc': 3e-2}


class Seg:
    """Inputs of one dmg_attn_segment call: q|k|v of B streams x T tokens, the K/V rings of Bcap streams (ours at [b0, b0 + B)), Rd with
    the fewest rows the entry allows (M + T + 1), u, v.  kernel: the one asked for (0 = the model's choice); ran: the one expected."""
    def __init__(self, arch, dtype, B, T, H, M, pos_total, win=1, k=1, kernel=0, ran=GENERAL, q_scale=1.0, Bcap=None, b0=0,
                 append=1, seed=0):
        g = torch.Generator(device='cuda').manual_seed(seed)
        self.arch, self.dtype, self.B, self.T, self.H, self.M, self.pos_total = arch, dtype, B, T, H, M, pos_total
        self.win, self.k, self.kernel, self.ran, self.b0, self.append = win, k, kernel, ran, b0, append
        self.Bcap = Bcap or B + b0
        self.Dcap = M + T + 1
        self.mc = min(pos_total, M)
        HD = H * 64
        rn = lambda *s: torch.randn(*s, device='cuda', generator=g)
        el = torch.float32 if dtype == _lib.F32 else torch.bfloat16
        qkv = rn(B * T, 3 * HD) * 0.8
        qkv[:, :HD] *= q_scale
        self.qkv = qkv if ran == GENERAL else qkv.bfloat16()          # as the q|k|v GEMM writes it for each kernel
        Mr = max(M, 1)
        self.kring = (rn(self.Bcap, H, Mr, 64) * 0.8).to(el)
        self.vring = (rn(self.Bcap, H, Mr, 64) * 0.8).to(el)
        self.rd = (rn(H, self.Dcap, 64) * 0.8).to(el)
        self.u, self.v = rn(HD) * 0.3, rn(HD) * 0.3
        self.masked = torch.ones(Mr, dtype=torch.bool, device='cuda')  # ring slots outside the memory
        self.masked[segment_ref.memory_slots(pos_total, M)] = False
        self.live = self.mc + T if arch == _lib.ARCH_TXL else T         # rel-pos rows [0, live) can be used
        self.junk_ring = rn(self.Bcap, H, Mr, 64).sign() * GARBAGE * (0.5 + torch.rand(self.Bcap, H, Mr, 64, device='cuda', generator=g))
        self.junk_rd = rn(H, self.Dcap, 64).sign() * GARBAGE
        self.fill(GARBAGE, GARBAGE)

    def fill(self, masked, rd_tail):
        "what the ring slots outside the memory and the Rd rows past the last live distance hold: GARBAGE (large finite values) or 0"
        for ring in (self.kring, self.vring):
            ring[:, :, self.masked] = (self.junk_ring[:, :, self.masked] * (masked == GARBAGE)).to(ring.dtype)
        self.rd[:, self.live:] = (self.junk_rd[:, self.live:] * (rd_tail == GARBAGE)).to(self.rd.dtype)
        return self

    def args(self, out, kring, vring, over={}):
        a = _lib.SegmentAttnArgs()
        a.qkv, a.kring, a.vring, a.rd, a.u, a.v, a.out = (t.data_ptr() for t in (self.qkv, kring, vring, self.rd, self.u, self.v, out))
        a.pos_total = self.pos_total
        a.arch, a.dtype, a.B, a.T, a.H, a.M, a.Dcap, a.Bcap, a.b0 = (self.arch, self.dtype, self.B, self.T, self.H, self.M, self.Dcap,
                                                                     self.Bcap, self.b0)
        a.win, a.k, a.append, a.kernel, a.kernel_ran = self.win, self.k, self.append, self.kernel, -1
        for name, val in over.items():
            setattr(a, name, val)
        return a

    def run(self, over={}):
        "one call on copies of the rings; returns (out, kring after, vring after, the kernel that ran)"
        kr, vr = self.kring.clone(), self.vring.clone()
        out = torch.full((self.B * self.T, self.H * 64), float('nan'), device='cuda', dtype=self.rd.dtype)
        a = self.args(out, kr, vr, over)
        torch.cuda.synchronize()
        check(_lib.load().dmg_attn_segment(C.byref(a), _st()), 'dmg_attn_segment')
        return out, kr, vr, a.kernel_ran

    def reference(self):
        "(out [B*T, H*64] float64, kring, vring after the call)"
        B, T, H, HD, s = self.B, self.T, self.H, self.H * 64, slice(self.b0, self.b0 + self.B)
        q, k, v = (self.qkv[:, i * HD:(i + 1) * HD].view(B, T, H, 64).permute(0, 2, 1, 3).double() for i in range(3))
        u, vb = self.u.view(H, 64).double(), self.v.view(H, 64).double()
        kring, vring = self.kring.clone(), self.vring.clone()
        if self.arch == _lib.ARCH_BERT:
            out = remix_attention_ref.remix_attention(q, k, v, self.rd[:, :T].permute(1, 0, 2).double(), u, vb)[0]
        else:
            out, kr, vr = segment_ref.segment_attention(q, k, v, self.kring[s, :, :max(self.M, 1)], self.vring[s, :, :max(self.M, 1)],
                                                        self.rd, u, vb, self.pos_total, self.M, self.win, self.k)
            if self.append and self.M:
                kring[s], vring[s] = kr, vr
        return out.permute(0, 2, 1, 3).reshape(B * T, HD), kring, vring


def tol_key(x):
    return KNAME[x.ran] + ('_f32' if x.dtype == _lib.F32 else '_bf16' if x.ran == GENERAL else '')


# ---------------------------------------------------------------------------------------------------------------------------
# cases: Seg keyword arguments (ids from _id)
# ---------------------------------------------------------------------------------------------------------------------------
TXL, BERT, F32, BF16 = _lib.ARCH_TXL, _lib.ARCH_BERT, _lib.F32, _lib.BF16
POS = lambda M: [0, 37, M - 1, M, M + 1, 2 * M + 37, 10 ** 6 + 3]
T_GEN = lambda M: [1, 2, 31, 32, 33, 100, M + 7]
MASKS = lambda T: [(1, 1), (1, 0), (3, 0), (T + 5, 0)]


def _general_cases():
    out = []
    for dtype in (F32, BF16):
        for mi, M in enumerate((32, 100, 256)):
            for pi, pt in enumerate(POS(M)):
                T = T_GEN(M)[(pi + 2 * mi) % 7]
                win, k = MASKS(T)[(pi + mi) % 4]
                H = (1, 2, 8)[(pi + mi) % 3]
                out.append(dict(arch=TXL, dtype=dtype, B=2, T=T, H=H, M=M, pos_total=pt, win=win, k=k,
                                kernel=0 if dtype == F32 else GENERAL, ran=GENERAL))
    # peaked softmax, and streams [3, 5) of a 7-stream ring
    for dtype in (F32, BF16):
        kern = 0 if dtype == F32 else GENERAL
        out.append(dict(arch=TXL, dtype=dtype, B=2, T=33, H=2, M=100, pos_total=237, kernel=kern, ran=GENERAL, q_scale=3.0))
        out.append(dict(arch=TXL, dtype=dtype, B=2, T=40, H=2, M=32, pos_total=101, win=3, k=0, kernel=kern, ran=GENERAL, Bcap=7, b0=3))
    return out


def _flash_cases():
    out = [dict(arch=TXL, dtype=BF16, B=2, T=T, H=8, M=256, pos_total=0, ran=FLASH) for T in (2, 63, 64, 65, 200, 512)]
    out.append(dict(arch=TXL, dtype=BF16, B=2, T=65, H=8, M=256, pos_total=0, ran=FLASH, q_scale=3.0))
    out.append(dict(arch=TXL, dtype=BF16, B=2, T=200, H=8, M=128, pos_total=0, ran=FLASH, Bcap=6, b0=4))   # prefill of streams [4, 6)
    out += [dict(arch=BERT, dtype=BF16, B=3, T=T, H=8, M=0, pos_total=0, ran=FLASH, append=0) for T in (2, 63, 65, 127)]
    out += [dict(arch=BERT, dtype=BF16, B=3, T=T, H=8, M=0, pos_total=0, kernel=FLASH, ran=FLASH, append=0) for T in (128, 384)]
    return out


def _tc_ring_cases():
    out = []
    for mi, M in enumerate((128, 256, 512, 1024)):
        for pi, pt in enumerate((128, M, M + 128, 2 * M + 256, 7813 * 128)):
            T = (128, 256, M + 128)[(pi + mi) % 3]
            win, k = ((1, 1), (3, 0), (200, 0))[(pi + 2 * mi) % 3]
            H = 16 if M == 1024 else (1, 8)[(pi + mi) % 2]             # M 1024, 16 heads: the C5 geometry
            out.append(dict(arch=TXL, dtype=BF16, B=2, T=T, H=H, M=M, pos_total=pt, win=win, k=k, ran=TC_RING))
    out.append(dict(arch=TXL, dtype=BF16, B=2, T=256, H=8, M=512, pos_total=1280, ran=TC_RING, q_scale=3.0))
    out.append(dict(arch=TXL, dtype=BF16, B=2, T=128, H=8, M=256, pos_total=640, win=3, k=0, ran=TC_RING, Bcap=5, b0=2))
    return out


def _bert_tc_cases():
    out = [dict(arch=BERT, dtype=BF16, B=2, T=T, H=8, M=0, pos_total=0, ran=BERT_TC, append=0) for T in (128, 129, 200, 384)]
    out.append(dict(arch=BERT, dtype=BF16, B=8, T=384, H=8, M=0, pos_total=0, ran=BERT_TC, append=0))    # 192 items > 148 SMs
    out.append(dict(arch=BERT, dtype=BF16, B=2, T=200, H=8, M=0, pos_total=0, ran=BERT_TC, append=0, q_scale=3.0))
    return out


CASES = _general_cases() + _flash_cases() + _tc_ring_cases() + _bert_tc_cases()


def _id(c):
    arch = 'bert' if c['arch'] == BERT else 'txl'
    s = f"{KNAME[c['ran']]}-{arch}-{'f32' if c['dtype'] == F32 else 'bf16'}-B{c['B']}-T{c['T']}-H{c['H']}"
    if c['arch'] == TXL:
        s += f"-M{c['M']}-pos{c['pos_total']}-w{c.get('win', 1)}k{c.get('k', 1)}"
    if c.get('kernel'):
        s += '-forced'
    if c.get('q_scale', 1) != 1:
        s += f"-q{c['q_scale']:g}"
    if c.get('b0'):
        s += f"-b0{c['b0']}of{c['Bcap']}"
    return s


def _seed(c):
    return (c['T'] * 131 + c['M'] * 7 + c['pos_total'] % 9973 + c['H'] * 3 + c['dtype'] + 17 * c.get('b0', 0)) % (2 ** 31)


@pytest.mark.parametrize('case', CASES, ids=[_id(c) for c in CASES])
def test_segment_attention_against_float64_reference(case):
    x = Seg(**case, seed=_seed(case))
    ref_out, ref_k, ref_v = x.reference()
    out, kr, vr, ran = x.run()
    assert ran == x.ran, f'kernel {KNAME.get(ran, ran)} ran, expected {KNAME[x.ran]}'
    assert not torch.isnan(out).any(), 'output elements left unwritten'
    err = row_err(out, ref_out)
    tol = (TOL_PEAKED if case.get('q_scale', 1) != 1 else TOL)[tol_key(x)]
    print(f'segment attention {_id(case)}: row error {err:.2e}', flush=True)
    assert err <= tol, f'worst (stream, head) row error {err:.2e} > {tol:.1e}'
    # the append: the last min(T, M) tokens of streams [b0, b0 + B) in slots (pos_total + t) mod M, converted to the ring dtype;
    # nothing else moves (without append, or without memory, nothing at all)
    for name, got, want in (('K', kr, ref_k), ('V', vr, ref_v)):
        if not same_bits(got, want):
            diff = (bits(got) != bits(want)).any(-1).nonzero().tolist()
            pytest.fail(f'{name} ring after the call differs at (stream, head, slot) {diff[:8]} (streams [{x.b0}, {x.b0 + x.B}), '
                        f'append slots {[s for _, s in segment_ref.append_slots(x.pos_total, x.M, x.T)][:8]})')
    # ring slots outside the memory and Rd rows past the last live distance: garbage there and zeros there give the same bits
    x.fill(0.0, GARBAGE)
    out_zero_slots = x.run()[0]
    assert same_bits(out, out_zero_slots), 'the ring slots outside the memory reach the output'
    x.fill(0.0, 0.0)
    out_zero_rd = x.run()[0]
    assert same_bits(out_zero_slots, out_zero_rd), 'the rel-pos rows past the last live distance reach the output'
    assert same_bits(out_zero_rd, x.run()[0]), 'two runs differ'


# ---------------------------------------------------------------------------------------------------------------------------
# routing, argument checks, dmg_forward's mask check
# ---------------------------------------------------------------------------------------------------------------------------
ROUTES = [   # id, Seg keyword arguments (kernel 0), the kernel dmg_forward runs
    ('f32', dict(arch=TXL, dtype=F32, B=1, T=128, H=2, M=128, pos_total=256), GENERAL),
    ('f32-bert', dict(arch=BERT, dtype=F32, B=1, T=200, H=2, M=0, pos_total=0, append=0), GENERAL),
    ('bf16-txl-prefill', dict(arch=TXL, dtype=BF16, B=1, T=64, H=2, M=128, pos_total=0), FLASH),
    ('bf16-txl-prefill-mask3,0', dict(arch=TXL, dtype=BF16, B=1, T=64, H=2, M=128, pos_total=0, win=3, k=0), GENERAL),
    ('bf16-txl-warm-aligned', dict(arch=TXL, dtype=BF16, B=1, T=128, H=2, M=256, pos_total=384), TC_RING),
    ('bf16-txl-warm-pos-unaligned', dict(arch=TXL, dtype=BF16, B=1, T=128, H=2, M=256, pos_total=300), GENERAL),
    ('bf16-txl-warm-T-unaligned', dict(arch=TXL, dtype=BF16, B=1, T=100, H=2, M=256, pos_total=384), GENERAL),
    ('bf16-txl-warm-M-unaligned', dict(arch=TXL, dtype=BF16, B=1, T=128, H=2, M=192, pos_total=384), GENERAL),
    ('bf16-bert-128', dict(arch=BERT, dtype=BF16, B=1, T=128, H=2, M=0, pos_total=0, append=0), BERT_TC),
    ('bf16-bert-100', dict(arch=BERT, dtype=BF16, B=1, T=100, H=2, M=0, pos_total=0, append=0), FLASH),
    ('bf16-bert-1', dict(arch=BERT, dtype=BF16, B=1, T=1, H=2, M=0, pos_total=0, append=0), GENERAL),
]


@pytest.mark.parametrize('kw,want', [(kw, want) for _, kw, want in ROUTES], ids=[r[0] for r in ROUTES])
def test_routing_picks_the_model_kernel(kw, want):
    x = Seg(**kw, ran=want)
    out, _, _, ran = x.run()
    assert ran == want, f'kernel {KNAME.get(ran, ran)} ran, dmg_forward runs {KNAME[want]} for this shape'
    assert not torch.isnan(out).any()


def test_one_token_bf16_segment_is_left_to_the_decode_entry():
    x = Seg(TXL, BF16, 2, 1, 2, 128, 300)
    with pytest.raises(DmgError, match='dmg_attn_decode'):
        x.run()
    assert x.run({'kernel': GENERAL})[3] == GENERAL        # forced, the general kernel serves it


def test_rejects_bad_arguments_before_launching():
    lib = _lib.load()
    x = Seg(TXL, BF16, 2, 128, 2, 256, 384, ran=TC_RING, Bcap=3, b0=1)
    bad = [({'qkv': None}, 'null'), ({'kring': None}, 'null'), ({'rd': None}, 'null'), ({'u': None}, 'null'), ({'out': None}, 'null'),
           ({'b0': 2}, 'outside the ring'), ({'Bcap': 2}, 'outside the ring'), ({'b0': -1}, 'outside the ring'),
           ({'Dcap': 256 + 128}, 'rel-pos cache'),
           ({'win': 3, 'k': 1}, r'window mask \(3,1\)'), ({'k': 2}, r'window mask \(1,2\)'), ({'k': -1}, r'window mask \(1,-1\)'),
           ({'win': 0, 'k': 0}, r'window mask \(0,0\)'),
           ({'kernel': FLASH}, 'does not support'), ({'kernel': BERT_TC}, 'does not support'),
           ({'kernel': TC_RING, 'pos_total': 300}, 'does not support'), ({'kernel': TC_RING, 'dtype': F32}, 'does not support'),
           ({'arch': 2}, 'arch'), ({'dtype': 2}, 'dtype'), ({'kernel': 5}, 'kernel'), ({'kernel': -1}, 'kernel'),
           ({'pos_total': -1}, 'pos_total'), ({'append': 2}, 'append'), ({'arch': BERT}, 'no memory'), ({'H': 0}, 'H 0')]
    out = torch.zeros(2 * 128, 128, device='cuda', dtype=torch.bfloat16)
    torch.cuda.synchronize()
    launches = lib.dmg_launch_count()
    for over, msg in bad:
        kr, vr = x.kring.clone(), x.vring.clone()
        a = x.args(out, kr, vr, over)
        with pytest.raises(DmgError, match=msg):
            check(lib.dmg_attn_segment(C.byref(a), _st()), 'dmg_attn_segment')
    assert lib.dmg_launch_count() == launches
    assert x.run()[3] == TC_RING                   # the same arguments without the fault do run
    assert lib.dmg_launch_count() > launches


def test_forward_refuses_masks_the_kernels_do_not_implement():
    from oracle import txl
    from deepmusicgeneration_b200.model import get_language_model
    cfg = dict(txl.default_config(), n_layers=1, d_model=128, n_heads=2, d_head=64, d_inner=256, mem_len=64, encode_position=False)
    pm = get_language_model(324, cfg, dtype='bf16', device=0, max_batch=2, max_seq=64, keep_hidden=False)
    lib = _lib.load()
    x = torch.randint(0, 324, (2, 40), device='cuda')
    pm.reset()
    for mask in ((3, 1), (1, 2), (1, -1)):
        torch.cuda.synchronize()
        launches = lib.dmg_launch_count()
        with pytest.raises(DmgError, match=r'window mask \(%d,%d\) unsupported' % mask):
            pm[0].forward(x, logits_mode=_lib.LOGITS_ALL, mask_size=mask)
        assert lib.dmg_launch_count() == launches
        assert pm[0]._e.mem_count() == 0
    for mask in ((1, 1), (5, 0)):
        logits = pm[0].forward(x, logits_mode=_lib.LOGITS_ALL, mask_size=mask)[0]
        assert torch.isfinite(logits).all()
