"""GPU unit tests of the remix (masked-BERT) encoder's training attention kernels (attention_bert_train.cu and the dK/dV kernel it
shares with attention_train.cu) through dmg_attn_bert_train_fwd / _bwd, against the float64 reference of remix_attention_ref.py
(which tests/test_remix_train_cpu.py anchors to the oracle).

Errors are taken per row: for every 64-wide head row (a query row for out and dq, a key row for dk and dv, a distance row for
dRk) ||x - ref|| / (||ref|| + 0.1 median row norm), and the worst row is asserted on.  A norm over the whole tensor would let
one wrong query row, one wrong distance column of ds_dist or a stale row 0 through: at T 1024 one row in 2048 moves it ~2 %."""
import pytest
import torch

import remix_attention_ref as ref_attn
from deepmusicgeneration_b200 import _lib
from deepmusicgeneration_b200._lib import DmgError, check
from test_gpu_train_kernels import _p, _st, attn_mask_from_device, row_err

pytestmark = pytest.mark.gpu

RK_BEFORE, RK_AFTER = 64, 128      # Rk rows the line-1 / line-3 windows may read below distance 0 and past distance T-1
SEED = 77

CASES = [   # B, T, H, attention dropout p, input scale
    (1, 64, 1, 0.0, 0.8),      # one tile: both rel-pos windows partly in the padding
    (3, 64, 2, 0.1, 0.8),      # the last tile's next-row q is row 0 of the next sequence
    (2, 128, 2, 0.0, 0.8),     # diagonal and off-diagonal tiles
    (2, 128, 2, 0.5, 0.8),     # forward / backward dropout agreement made prominent
    (1, 192, 1, 0.1, 0.8),     # odd tile count
    (2, 320, 2, 0.0, 3.0),     # peaked softmax: the running max changes across key tiles (l / O rescaling)
    (1, 1024, 8, 0.1, 0.8),    # one sequence of the C4 geometry
]

# Row errors, LSE absolute, ds_dist relative to |ref| + row RMS.  The worst value over the x0.8 cases on one B200 (1000 W) was
# out 5.6e-3, lse 1.4e-3, dq_content 5.7e-3, dq 5.6e-3, dk 5.8e-3, dv 6.0e-3, du 2.9e-3, dv-bias 3.6e-3, dRk 5.3e-3, ds_dist 8.6e-3;
# each tolerance is at most 3x that.
TOL = {'out': 1.5e-2, 'lse': 4e-3, 'dq': 1.5e-2, 'dq_content': 1.5e-2, 'dk': 1.5e-2, 'dv': 1.5e-2, 'du': 8e-3, 'dvb': 1e-2, 'drk': 1.5e-2,
       'ds_dist': 2e-2}


class Inputs:
    "q|k|v with its extra row, the Rk table inside its padding, u, v and dO - bf16 values the reference reads exactly"
    def __init__(self, B, T, H, scale, seed):
        g = torch.Generator(device='cuda').manual_seed(seed)
        HD = H * 64
        self.B, self.T, self.H = B, T, H
        self.qkv = (torch.randn(B * T + 1, 3 * HD, device='cuda', generator=g) * scale).bfloat16()
        self.rk_buf = (torch.randn(RK_BEFORE + T + RK_AFTER, HD, device='cuda', generator=g) * scale).bfloat16()
        self.u = torch.randn(HD, device='cuda', generator=g) * 0.3
        self.v = torch.randn(HD, device='cuda', generator=g) * 0.3
        self.dout = (torch.randn(B * T, HD, device='cuda', generator=g) * 0.5).bfloat16()

    @property
    def rk(self):
        return self.rk_buf[RK_BEFORE:RK_BEFORE + self.T]

    def padded(self, fill):
        "a copy whose q|k|v row past the last sequence and Rk padding rows hold `fill`"
        x = Inputs.__new__(Inputs)
        x.__dict__.update(self.__dict__)
        x.qkv, x.rk_buf = self.qkv.clone(), self.rk_buf.clone()
        x.qkv[-1] = fill
        x.rk_buf[:RK_BEFORE] = fill
        x.rk_buf[RK_BEFORE + self.T:] = fill
        return x


def run_kernels(x, p, du0, prefill=float('nan')):
    "forward then backward through the C ABI; every output starts as `prefill`, du starts as du0 (it is accumulated into)"
    lib = _lib.load()
    B, T, H, HD = x.B, x.T, x.H, x.H * 64
    full = lambda shape, dt: torch.full(shape, prefill, device='cuda', dtype=dt)
    out, lse = full((B * T, HD), torch.bfloat16), full((B, H, T), torch.float32)
    check(lib.dmg_attn_bert_train_fwd(_p(x.qkv), 3 * HD, _p(x.rk), _p(x.u), _p(x.v), _p(out), _p(lse), B, T, H, p, SEED, _st()),
          'dmg_attn_bert_train_fwd')
    delta, dqkv, ds_dist = full((B, H, T), torch.float32), full((B * T, 3 * HD), torch.bfloat16), full((B * T, H * T), torch.bfloat16)
    du = du0.clone()
    p_buf = torch.empty(B * H, T, T, device='cuda', dtype=torch.bfloat16)
    ds_buf = torch.empty_like(p_buf)
    check(lib.dmg_attn_bert_train_bwd(_p(x.qkv), 3 * HD, _p(x.rk), _p(x.u), _p(x.v), _p(out), _p(lse), _p(x.dout), B, T, H, p, SEED,
                                      _p(delta), _p(dqkv), _p(ds_dist), _p(du), _p(p_buf), _p(ds_buf), _st()), 'dmg_attn_bert_train_bwd')
    torch.cuda.synchronize()
    return {'out': out, 'lse': lse, 'dqkv_x': dqkv, 'ds_dist': ds_dist, 'du': du}


def make_inputs(B, T, H, p, scale):
    return Inputs(B, T, H, scale, seed=B * 1000 + T + H + int(p * 10))


@pytest.mark.parametrize('B,T,H,p,scale', CASES)
def test_forward_backward_against_float64_reference(B, T, H, p, scale):
    x = make_inputs(B, T, H, p, scale)
    HD = H * 64
    # float64 reference from the exact bf16 inputs, on the GPU
    qkv = x.qkv[:B * T].double().view(B, T, 3, H, 64)
    q, k, v = (qkv[:, :, i].permute(0, 2, 1, 3) for i in range(3))           # [B, H, T, 64]
    rk, u, vb = x.rk.double().view(T, H, 64), x.u.double().view(H, 64), x.v.double().view(H, 64)
    mask = attn_mask_from_device(B, H, T, T, 0, 0, p, SEED).double() if p > 0 else None
    leaves = [t.clone().requires_grad_(True) for t in (q, k, v, rk, u, vb)]
    ref_out, ref_lse, raw = ref_attn.remix_attention(*leaves, drop_mask=mask)
    raw.retain_grad()
    ref_out.backward(x.dout.double().view(B, T, H, 64).permute(0, 2, 1, 3))
    gq, gk, gv, grk, gu, gvb = [t.grad for t in leaves]
    bthd = lambda t: t.permute(0, 2, 1, 3)                                    # [B, H, T, 64] -> [B, T, H, 64]

    du0 = torch.randn(HD, device='cuda', generator=torch.Generator(device='cuda').manual_seed(5)) * gu.norm().item() / 8
    got = run_kernels(x.padded(float('nan')), p, du0)
    for name in ('out', 'lse', 'dqkv_x', 'ds_dist'):           # every element written, no padding value leaked in
        assert not torch.isnan(got[name]).any(), f'{name} has unwritten or NaN elements'
    dsd = got['ds_dist'].double().view(B, T, H, T)
    assert (dsd[:, 0, :, 1:] == 0).all(), 'row 0 of a sequence has no line-3 predecessor: distances 1 .. T-1 must be zero'

    errs = {
        'out': row_err(got['out'], bthd(ref_out)),
        'lse': (got['lse'].double() - ref_lse).abs().max().item(),
    }
    if scale > 1:
        check_peaked_forward(x, q, k, v, rk, mask, ref_out, ref_lse, errs)
        return
    d = got['dqkv_x'].double().view(B, T, 3, H, 64)
    dq_pos, dvb, drk = ref_attn.position_grads(dsd, rk, bthd(q + vb[:, None]))
    ref_dist = ref_attn.ds_to_dist(raw.grad)
    rms = ref_dist.pow(2).mean(-1, keepdim=True).sqrt()
    errs.update({
        'dq_content': row_err(d[:, :, 0], bthd(raw.grad @ k)),
        'dq': row_err(d[:, :, 0] + dq_pos, bthd(gq)),
        'dk': row_err(d[:, :, 1], bthd(gk)),
        'dv': row_err(d[:, :, 2], bthd(gv)),
        'du': row_err(got['du'].double() - du0.double(), gu),
        'dvb': row_err(dvb, gvb),
        'drk': row_err(drk, grk),
        'ds_dist': ((dsd - ref_dist).abs() / (ref_dist.abs() + rms)).max().item(),
    })
    print(f'errors B={B} T={T} H={H} p={p} x{scale}:', {n: f'{e:.2e}' for n, e in errs.items()}, flush=True)
    bad = {n: e for n, e in errs.items() if not e <= TOL[n]}
    assert not bad, f'over tolerance: {bad}'


def check_peaked_forward(x, q, k, v, rk, mask, ref_out, ref_lse, errs):
    """Inputs x3: raw scores reach ~500, and the kernels' mma operands (q + u) and (q + v) are bf16 (rounding 2^-9 relative):
    that alone moves a score by up to ~0.1 and the LSE by ~0.07, ten times the fp16 rel-pos strip (2^-11 of |BD|, <= 0.016).
    The tolerance of out and LSE is TOL plus twice that floor, measured here: the float64 forward recomputed from the operands
    as the kernels round them (bf16 q + bias, fp16 BD).  This case exists for the running maximum changing across key tiles.
    Its backward is not compared: in near-one-hot rows dS = P (dP - delta) cancels far below the bf16 resolution of the
    output O that delta = dO . O is formed from, so the float64 reference and any bf16 backward part by more than the signal
    (the gradients of the other cases, which cover every backward index path, are compared)."""
    H = x.H
    rnd = lambda bias: (q.float() + bias.view(H, 1, 64)).bfloat16().double()     # q_frags: fp32 add, round to bf16
    ac, bd = ref_attn.score_terms(rnd(x.u), rnd(x.v), k, rk)
    s = (ac + bd.half().double()) / 8
    pr = torch.softmax(s, dim=-1)
    out_r = (pr * mask if mask is not None else pr) @ v
    floor = {'out': row_err(out_r, ref_out), 'lse': (torch.logsumexp(s, dim=-1) - ref_lse).abs().max().item()}
    print('errors x3 forward:', {n: f'{e:.2e}' for n, e in errs.items()}, 'operand-rounding floor:',
          {n: f'{e:.2e}' for n, e in floor.items()}, flush=True)
    bad = {n: e for n, e in errs.items() if not e <= TOL[n] + 2 * floor[n]}
    assert not bad, f'over tolerance: {bad}'


@pytest.mark.parametrize('B,T,H,p,scale', CASES)
def test_padding_rows_never_reach_the_outputs(B, T, H, p, scale):
    """The rel-pos windows read Rk 64 rows below distance 0 and up to 128 past T-1, and the next-row q of the last tile reads one
    q|k|v row past the last sequence; the line selection must discard everything computed from those rows: NaN there and
    zero there give bit-identical results."""
    x = make_inputs(B, T, H, p, scale)
    du0 = torch.zeros(H * 64, device='cuda')
    a = run_kernels(x.padded(float('nan')), p, du0)
    b = run_kernels(x.padded(0.0), p, du0)
    for name in ('out', 'lse', 'dqkv_x', 'ds_dist'):
        assert not torch.isnan(a[name]).any() and torch.equal(a[name], b[name]), name
    assert torch.isfinite(a['du']).all()
    assert (a['du'] - b['du']).abs().max() <= 1e-5 * b['du'].abs().max()      # atomics: summation order only


@pytest.mark.parametrize('B,T,H,p,scale', CASES)
def test_bitwise_deterministic(B, T, H, p, scale):
    "out, lse, dqkv_x and ds_dist are written without atomics: two runs agree bit for bit; du (atomics) to rounding"
    x = make_inputs(B, T, H, p, scale).padded(0.0)
    du0 = torch.zeros(H * 64, device='cuda')
    a, b = run_kernels(x, p, du0), run_kernels(x, p, du0)
    for name in ('out', 'lse', 'dqkv_x', 'ds_dist'):
        assert torch.equal(a[name], b[name]), name
    assert (a['du'] - b['du']).abs().max() <= 1e-5 * b['du'].abs().max()


def test_entry_points_reject_bad_arguments_before_launching():
    lib = _lib.load()
    B, T, H = 1, 128, 1
    HD = H * 64
    x = make_inputs(B, T, H, 0.0, 0.8).padded(0.0)
    out = torch.zeros(B * T, HD, device='cuda', dtype=torch.bfloat16)
    lse, delta = torch.zeros(B, H, T, device='cuda'), torch.zeros(B, H, T, device='cuda')
    dqkv = torch.zeros(B * T, 3 * HD, device='cuda', dtype=torch.bfloat16)
    ds_dist = torch.zeros(B * T, H * T, device='cuda', dtype=torch.bfloat16)
    du = torch.zeros(HD, device='cuda')
    bufs = [torch.zeros(B * H, T, T, device='cuda', dtype=torch.bfloat16) for _ in range(2)]

    def bwd(T_, ds_dist_, p_buf_):
        check(lib.dmg_attn_bert_train_bwd(_p(x.qkv), 3 * HD, _p(x.rk), _p(x.u), _p(x.v), _p(out), _p(lse), _p(x.dout), B, T_, H, 0.0,
                                          SEED, _p(delta), _p(dqkv), _p(ds_dist_), _p(du), _p(p_buf_), _p(bufs[1]), _st()), 'bwd')

    check(lib.dmg_attn_bert_train_fwd(_p(x.qkv), 3 * HD, _p(x.rk), _p(x.u), _p(x.v), _p(out), _p(lse), B, T, H, 0.0, SEED, _st()), 'fwd')
    torch.cuda.synchronize()
    launches = lib.dmg_launch_count()
    with pytest.raises(DmgError, match='multiple of 64'):
        check(lib.dmg_attn_bert_train_fwd(_p(x.qkv), 3 * HD, _p(x.rk), _p(x.u), _p(x.v), _p(out), _p(lse), B, 96, H, 0.0, SEED, _st()),
              'fwd')
    with pytest.raises(DmgError, match='multiple of 64'):
        bwd(96, ds_dist, bufs[0])
    with pytest.raises(DmgError, match='ds_dist'):
        bwd(T, None, bufs[0])
    with pytest.raises(DmgError, match='p_buf'):
        bwd(T, ds_dist, None)
    assert lib.dmg_launch_count() == launches
    bwd(T, ds_dist, bufs[0])                                   # the same arguments with the constraint met do run
    assert lib.dmg_launch_count() > launches
