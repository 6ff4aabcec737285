"""GPU unit tests of the training kernels through the C ABI: the persistent tcgen05 GEMM (all operand majors and fused
epilogues) and the flash attention forward/backward with the rel-pos term, each against a plain PyTorch fp32 restatement
of the oracle's arithmetic (oracle/txl.py MultiHeadRelativeAttention._apply_attention, _line_shift, window_mask)."""
import ctypes as C
import math

import pytest
import torch

from deepmusicgeneration_b200 import _lib
from deepmusicgeneration_b200._lib import DmgError, check
from oracle import txl

pytestmark = pytest.mark.gpu


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _st():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def gelu_tanh(x):
    return 0.5 * x * (1 + torch.tanh(math.sqrt(2 / math.pi) * (x + 0.044715 * x ** 3)))


def gemm_train(a, a_mn, b, b_mn, M, N, K, splitk=1, bias=None, gelu=0, aux=None, aux_mode=0, out_mode=0, out=None, want_pre=False,
               drop_p=0., seed=0):
    lib = _lib.load()
    dev = a.device
    if out is None:
        out = torch.zeros(M, N, device=dev, dtype=torch.bfloat16 if out_mode == 1 else torch.float32)
    pre = torch.zeros(M, N, device=dev, dtype=torch.bfloat16) if want_pre else None
    check(lib.dmg_gemm_train(_p(a), a_mn, a.stride(0), _p(b), b_mn, b.stride(0), M, N, K, splitk, _p(bias), gelu, _p(aux),
                             aux.stride(0) if aux is not None else 0, aux_mode, _p(out), out.stride(0), out_mode, _p(pre),
                             pre.stride(0) if pre is not None else 0, drop_p, seed, _st()), 'dmg_gemm_train')
    torch.cuda.synchronize()
    return (out, pre) if want_pre else out


def rel_err(a, b):
    return ((a.float() - b.float()).norm() / b.float().norm().clamp_min(1e-12)).item()


def row_err(a, b, width=64):
    """Worst row of `width` elements (one head row of a query, key or distance): ||a - b|| / (||b|| + 0.1 median row norm of b).
    One wrong row out of thousands barely moves the norm of the whole tensor; here it is the result."""
    a, b = a.double().reshape(-1, width), b.double().reshape(-1, width)
    d, n = (a - b).norm(dim=1), b.norm(dim=1)
    return (d / (n + 0.1 * n.median()).clamp_min(1e-30)).max().item()


@pytest.mark.parametrize('a_mn,b_mn', [(0, 0), (0, 1), (1, 0), (1, 1)])
@pytest.mark.parametrize('M,N,K', [(256, 512, 512), (1000, 324, 320), (384, 64, 1024), (2048, 1536, 192)])
def test_gemm_train_operand_majors(a_mn, b_mn, M, N, K):
    torch.manual_seed(M + N + K + 2 * a_mn + b_mn)
    dev = 'cuda'
    Kp, Mp, Np = (K + 7) // 8 * 8, (M + 7) // 8 * 8, (N + 7) // 8 * 8
    A = torch.randn(M, K, device=dev)
    B = torch.randn(N, K, device=dev)
    a_store = torch.zeros(K, Mp, device=dev, dtype=torch.bfloat16) if a_mn else torch.zeros(M, Kp, device=dev, dtype=torch.bfloat16)
    b_store = torch.zeros(K, Np, device=dev, dtype=torch.bfloat16) if b_mn else torch.zeros(N, Kp, device=dev, dtype=torch.bfloat16)
    if a_mn: a_store[:, :M] = A.t()
    else: a_store[:, :K] = A
    if b_mn: b_store[:, :N] = B.t()
    else: b_store[:, :K] = B
    ref = A.bfloat16().float() @ B.bfloat16().float().t()
    out = gemm_train(a_store, a_mn, b_store, b_mn, M, N, K)
    assert rel_err(out, ref) < 2e-3, (a_mn, b_mn, M, N, K)


def test_gemm_train_splitk_atomic_accumulates():
    torch.manual_seed(1)
    M, N, K = 512, 256, 4096
    A = torch.randn(K, M, device='cuda').bfloat16()      # dY^T X weight-gradient shape: both operands MN-major
    B = torch.randn(K, N, device='cuda').bfloat16()
    base = torch.randn(M, N, device='cuda')
    out = base.clone()
    gemm_train(A, 1, B, 1, M, N, K, splitk=6, out_mode=2, out=out)
    ref = base + A.float().t() @ B.float()
    assert rel_err(out, ref) < 2e-3


def test_gemm_train_residual_and_dropout_epilogues():
    "residual adds (bf16 / fp32 aux, in place) and the fused dropout on the fp32 output path"
    torch.manual_seed(2)
    M, N, K = 640, 768, 256
    A = torch.randn(M, K, device='cuda').bfloat16()
    W = (torch.randn(N, K, device='cuda') * 0.1).bfloat16()
    bias = torch.randn(N, device='cuda')
    acc = A.float() @ W.float().t() + bias
    # residual adds
    aux = torch.randn(M, N, device='cuda').bfloat16()
    res32 = torch.randn(M, N, device='cuda')
    out = gemm_train(A, 0, W, 0, M, N, K, aux=res32, aux_mode=3, out_mode=0)
    assert rel_err(out, acc - bias + res32) < 2e-3
    out = gemm_train(A, 0, W, 0, M, N, K, aux=aux, aux_mode=2, out_mode=0)
    assert rel_err(out, acc - bias + aux.float()) < 2e-3
    # in-place residual accumulate (the backward pass adds input gradients into the running fp32 gradient)
    run = res32.clone()
    gemm_train(A, 0, W, 0, M, N, K, aux=run, aux_mode=3, out_mode=0, out=run)
    assert rel_err(run, acc - bias + res32) < 2e-3
    # fused dropout: kept entries scaled, dropped entries zero, keep rate right
    out = gemm_train(A, 0, W, 0, M, N, K, out_mode=0, drop_p=0.25, seed=1234)
    plain = acc - bias
    kept = out != 0
    assert abs(kept.float().mean().item() - 0.75) < 0.01
    assert rel_err(out[kept], plain[kept] / 0.75) < 2e-3


def test_gemm_train_gradient_saving_gelu_epilogue():
    "act = 2: out = dropout(gelu(acc + bias)), second output = gelu'(acc + bias) * the same dropout factor; aux_mode 4 multiplies by it"
    torch.manual_seed(6)
    M, N, K = 1024, 2048, 512
    A = (torch.randn(M, K, device='cuda') * 0.5).bfloat16()
    W = (torch.randn(N, K, device='cuda') * 0.1).bfloat16()
    bias = torch.randn(N, device='cuda') * 0.3
    x = (A.float() @ W.float().t() + bias).requires_grad_(True)
    gelu_tanh(x).sum().backward()
    out, gfac = gemm_train(A, 0, W, 0, M, N, K, bias=bias, gelu=2, out_mode=1, want_pre=True)
    assert rel_err(out, gelu_tanh(x.detach())) < 5e-3 and rel_err(gfac, x.grad) < 5e-3
    out, gfac = gemm_train(A, 0, W, 0, M, N, K, bias=bias, gelu=2, out_mode=1, want_pre=True, drop_p=0.25, seed=11)
    plain = gemm_train(A, 0, W, 0, M, N, K, bias=bias, gelu=1, out_mode=1, drop_p=0.25, seed=11)
    kept = plain != 0
    assert torch.equal(out != 0, kept) and rel_err(out, plain) < 2e-3  # same mask as the act = 1 epilogue (the GeLU is factored differently)
    assert (gfac[~kept] == 0).all()
    assert rel_err(gfac[kept], (x.grad / 0.75)[kept]) < 5e-3
    dy = (torch.randn(M, K, device='cuda') * 0.5).bfloat16()          # dh = (dY W2) * factor with W2 [K, N] MN-major
    W2 = (torch.randn(K, N, device='cuda') * 0.1).bfloat16()
    dh = gemm_train(dy, 0, W2, 1, M, N, K, aux=gfac, aux_mode=4, out_mode=1)
    assert rel_err(dh, (dy.float() @ W2.float()) * gfac.float()) < 5e-3


def test_gemm_train_persistent_loop_wraps_around():
    "more tiles than CTA pairs: the persistent loop, both TMEM stages, the TMA-store strips and the aux-box prefetch wrap around"
    torch.manual_seed(4)
    M, N, K = 8192, 2048, 192
    A = (torch.randn(M, K, device='cuda') * 0.5).bfloat16()
    W = (torch.randn(N, K, device='cuda') * 0.1).bfloat16()
    bias = torch.randn(N, device='cuda')
    acc = A.float() @ W.float().t()
    x = (acc + bias).requires_grad_(True)
    gelu_tanh(x).sum().backward()
    out, gfac = gemm_train(A, 0, W, 0, M, N, K, bias=bias, gelu=2, out_mode=1, want_pre=True)
    assert rel_err(gfac, x.grad) < 5e-3 and rel_err(out, gelu_tanh(x.detach())) < 5e-3
    out = gemm_train(A, 0, W, 0, M, N, K, aux=gfac, aux_mode=4, out_mode=1)
    assert torch.isfinite(out.float()).all()
    assert rel_err(out, acc * gfac.float()) < 5e-3
    aux = torch.randn(M, N, device='cuda').bfloat16()
    out = gemm_train(A, 0, W, 0, M, N, K, aux=aux, aux_mode=2, out_mode=1)
    assert rel_err(out, acc + aux.float()) < 5e-3
    out = gemm_train(A, 0, W, 0, M, N, K, out_mode=0)
    assert rel_err(out, acc) < 2e-3
    Wm = W.t().contiguous()                                   # [K, N]: MN-major B
    out = gemm_train(A, 0, Wm, 1, M, N, K, out_mode=1)
    assert rel_err(out, acc) < 5e-3


def test_gemm_train_rejects_unsupported_epilogues():
    "aux_mode 1, and a second output with any GeLU but the gradient-saving one, are refused before anything is launched"
    torch.manual_seed(7)
    lib = _lib.load()
    M, N, K = 256, 256, 128
    A = torch.randn(M, K, device='cuda').bfloat16()
    W = torch.randn(N, K, device='cuda').bfloat16()
    aux = torch.randn(M, N, device='cuda').bfloat16()
    out = torch.full((M, N), 5.0, device='cuda', dtype=torch.bfloat16)
    torch.cuda.synchronize()
    launches = lib.dmg_launch_count()
    with pytest.raises(DmgError, match='aux_mode 1'):
        gemm_train(A, 0, W, 0, M, N, K, aux=aux, aux_mode=1, out_mode=1, out=out)
    with pytest.raises(DmgError, match='second output'):
        gemm_train(A, 0, W, 0, M, N, K, gelu=1, out_mode=1, out=out, want_pre=True)
    assert lib.dmg_launch_count() == launches
    assert (out == 5.0).all()


def test_gemm_train_grouped_heads():
    "the dRk contraction: one launch, group h reads A columns [h*S,(h+1)*S) and B columns [h*64,(h+1)*64)"
    torch.manual_seed(3)
    lib = _lib.load()
    H, S, rows = 4, 192, 1024
    A = (torch.randn(rows, H * S, device='cuda') * 0.5).bfloat16()
    B = (torch.randn(rows, H * 64, device='cuda') * 0.5).bfloat16()
    out = torch.zeros(S, H * 64, device='cuda')
    # exported test entry has no group arguments: run the per-head launches and the library's grouped path must agree with
    # the einsum (the grouped path itself is exercised by the training-step tests through dWr)
    for h in range(H):
        o = out[:, h * 64:]
        check(lib.dmg_gemm_train(_p(A[:, h * S:]), 1, A.stride(0), _p(B[:, h * 64:]), 1, B.stride(0), S, 64, rows, 3, None, 0, None,
                                 0, 0, _p(o), out.stride(0), 2, None, 0, 0., 0, _st()), 'gemm')
    torch.cuda.synchronize()
    ref = torch.einsum('rhs,rhd->shd', A.float().view(rows, H, S), B.float().view(rows, H, 64)).reshape(S, H * 64)
    assert rel_err(out, ref) < 2e-3


# ---------------------------------------------------------------------------------------------- attention
def ref_attention(q, k, v, rk, u, vb, win, kk, mem_count, drop_mask=None):
    """q [B,T,H,D]; k, v [B,Sc,H,D] (Sc = mem_count + T compact context); rk [Sc,H,D] by distance; fp32.
    Mirrors oracle.txl.MultiHeadRelativeAttention._apply_attention."""
    B, T, H, D = q.shape
    Sc = k.shape[1]
    wq, wk, wv = q.permute(0, 2, 1, 3), k.permute(0, 2, 3, 1), v.permute(0, 2, 1, 3)
    wkr = rk.flip(0).permute(1, 2, 0)                      # oracle's r runs over positions Sc-1 .. 0
    AC = torch.matmul(wq + u.view(1, H, 1, D), wk)
    BD = txl._line_shift(torch.matmul(wq + vb.view(1, H, 1, D), wkr))
    score = (AC + BD) * (1 / math.sqrt(D))
    mask = txl.window_mask(T, q.device, m_len=mem_count, size=(win, kk))
    score = score.masked_fill(mask, -float('inf'))
    p = torch.softmax(score, dim=-1)
    lse = torch.logsumexp(score, dim=-1)
    ref_attention.last_probs = p.detach()                  # undropped probabilities [B, H, T, Sc] (saved-P format test)
    if drop_mask is not None:
        p = p * drop_mask
    o = torch.matmul(p, wv)
    return o.permute(0, 2, 1, 3).reshape(B, T, H * D), lse


def make_attn_inputs(B, T, H, M, seed):
    g = torch.Generator(device='cuda').manual_seed(seed)
    HD = H * 64
    qkv_x = (torch.randn(B * T, 3 * HD, device='cuda', generator=g) * 0.8).bfloat16()
    kv_m = (torch.randn(B * max(M, 1), 2 * HD, device='cuda', generator=g) * 0.8).bfloat16()
    rk = (torch.randn(M + T, HD, device='cuda', generator=g) * 0.8).bfloat16()
    u = torch.randn(HD, device='cuda', generator=g) * 0.3
    v = torch.randn(HD, device='cuda', generator=g) * 0.3
    return qkv_x, kv_m, rk, u, v


def split_ref_inputs(qkv_x, kv_m, rk, B, T, H, M, mem_count):
    HD = H * 64
    x = qkv_x.float().view(B, T, 3, H, 64)
    q, kx, vx = x[:, :, 0], x[:, :, 1], x[:, :, 2]
    if mem_count > 0:
        mm = kv_m.float().view(B, M, 2, H, 64)[:, M - mem_count:]
        k = torch.cat([mm[:, :, 0], kx], 1)
        v = torch.cat([mm[:, :, 1], vx], 1)
    else:
        k, v = kx, vx
    r = rk.float()[:mem_count + T].view(mem_count + T, H, 64)
    return q, k, v, r


def attn_mask_from_device(B, H, T, S, M, mem_count, p, seed):
    "the attention-dropout mask as the kernels index it: element ((b*H+h)*T+i)*S + j, j in full-context coordinates"
    lib = _lib.load()
    n = B * H * T * S
    out = torch.empty(n, device='cuda')
    # reuse the model-free export through a GEMM-free path: the hash is exposed by dmg_gemm_train's dropout, so derive it
    # from a ones matrix: out = dropout(ones)  (row = (b,h,i), col = j)
    ones_a = torch.ones(B * H * T, 64, device='cuda', dtype=torch.bfloat16)
    ones_b = torch.zeros(S, 64, device='cuda', dtype=torch.bfloat16)
    ones_b[:, 0] = 1
    o = gemm_train(ones_a, 0, ones_b, 0, B * H * T, S, 64, out_mode=0, drop_p=p, seed=seed)
    return o.view(B, H, T, S)[..., M - mem_count:]


# Worst row error (row_err) over every case on one B200 (1000 W): out 4.4e-3, dq 4.4e-2, dk 7.6e-3, dv 5.9e-3, dk_mem 6.6e-3,
# dv_mem 5.5e-3, du 2.9e-3, dv-bias 3.5e-3, dRk 6.8e-3; each tolerance is at most 3x that.  dq is 6.7e-3 or less except with
# no memory (M = 0): there the first query rows see one or a few keys, their true dq is ~0 (dS = P (dP - dO . O) cancels), and
# what the kernels give is the bf16 rounding of the O that delta is formed from.
ROW_TOL = {'out': 1.2e-2, 'dq': 8e-2, 'dk': 2e-2, 'dv': 1.5e-2, 'dk_mem': 2e-2, 'dv_mem': 1.5e-2, 'du': 8e-3, 'dvb': 1e-2, 'drk': 2e-2}


@pytest.mark.parametrize('B,T,H,M,mem_count,win,kk,p', [
    (2, 64, 2, 0, 0, 1, 1, 0.0),
    (2, 128, 2, 128, 128, 1, 1, 0.0),
    (1, 192, 1, 128, 64, 1, 0, 0.0),
    (2, 128, 2, 64, 64, 3, 0, 0.0),
    (2, 128, 2, 128, 128, 1, 1, 0.1),
    # shapes served by the tcgen05 forward (attention_train_tc.cu: T, M, mem_count multiples of 128)
    (1, 384, 2, 0, 0, 1, 1, 0.0),          # no memory: the diagonal tile's lower Rk block lies at negative distances
    (1, 256, 2, 256, 128, 1, 1, 0.1),      # partly filled memory
    (2, 256, 1, 128, 128, 3, 0, 0.0),      # window mask (3, 0)
    (1, 512, 2, 512, 512, 1, 1, 0.1),      # C3 geometry
])
@pytest.mark.parametrize('save_p', [False, True])
def test_attention_train_forward_backward(B, T, H, M, mem_count, win, kk, p, save_p):
    if save_p and not (T % 128 == 0 and M % 128 == 0 and mem_count % 128 == 0):
        pytest.skip('p_save needs the tcgen05 forward')
    lib = _lib.load()
    HD, S = H * 64, M + T
    seed = 99
    qkv_x, kv_m, rk, u, v = make_attn_inputs(B, T, H, M, seed=B * 1000 + T + M)
    out = torch.zeros(B * T, HD, device='cuda', dtype=torch.bfloat16)
    lse = torch.zeros(B, H, T, device='cuda')
    # shapes the tcgen05 forward serves also save the undropped probabilities for the backward (p_save / m_save)
    saved = T % 128 == 0 and M % 128 == 0 and mem_count % 128 == 0 and save_p
    p_save = torch.full((B * H, T, S), float('nan'), device='cuda', dtype=torch.bfloat16) if saved else None
    m_save = torch.full((B * H, T, S // 64), float('nan'), device='cuda') if saved else None
    check(lib.dmg_attn_train_fwd(_p(qkv_x), 3 * HD, _p(kv_m), 2 * HD, _p(rk), _p(u), _p(v), _p(out), _p(lse), B, T, H, M, mem_count,
                                 win, kk, p, seed, _p(p_save), _p(m_save), _st()), 'fwd')
    torch.cuda.synchronize()
    drop = attn_mask_from_device(B, H, T, S, M, mem_count, p, seed) if p > 0 else None
    q, k, vv, r = split_ref_inputs(qkv_x, kv_m, rk, B, T, H, M, mem_count)
    leaves = [t.clone().requires_grad_(True) for t in (q, k, vv, r, u.view(H, 64), v.view(H, 64))]
    ref, ref_lse = ref_attention(*leaves, win, kk, mem_count, drop)
    assert rel_err(lse, ref_lse) < 2e-3
    assert rel_err(out.view(B, T, HD), ref) < 1e-2
    errs = {'out': row_err(out, ref)}
    if saved:
        # the saved format: P = p_save * exp(m_save * scale - lse) wherever the forward visited a tile (bf16 rounding only);
        # tiles above the diagonal are never written (still NaN) and hold no probability mass
        fac = torch.exp(m_save.view(B, H, T, S // 64) * 0.125 - lse.view(B, H, T, 1))
        rebuilt = p_save.float().view(B, H, T, S // 64, 64) * fac.unsqueeze(-1)
        rebuilt = torch.nan_to_num(rebuilt, nan=0.0).view(B, H, T, S)[..., M - mem_count:]
        assert rel_err(rebuilt, ref_attention.last_probs) < 1e-2

    dout = (torch.randn(B * T, HD, device='cuda') * 0.5).bfloat16()
    ref.backward(dout.float().view(B, T, HD))
    gq, gk, gv, gr, gu, gvb = [t.grad for t in leaves]
    delta = torch.zeros(B, H, T, device='cuda')
    dqkv_x = torch.zeros_like(qkv_x)
    dkv_m = torch.full_like(kv_m, 7.0)
    ds_dist = torch.full((B * T, H * S), 3.0, device='cuda', dtype=torch.bfloat16)
    du = torch.zeros(HD, device='cuda'); dv = torch.zeros(HD, device='cuda')
    check(lib.dmg_attn_train_bwd(_p(qkv_x), 3 * HD, _p(kv_m), 2 * HD, _p(rk), _p(u), _p(v), _p(out), _p(lse), _p(dout), B, T, H, M,
                                 mem_count, win, kk, p, seed, _p(delta), _p(dqkv_x), _p(dkv_m), _p(ds_dist), _p(du), _p(dv), _p(p_save),
                                 _p(m_save), _st()),
          'bwd')
    torch.cuda.synchronize()
    d = dqkv_x.float().view(B, T, 3, H, 64)
    tol = 2e-2
    assert rel_err(d[:, :, 0], gq) < tol
    assert rel_err(d[:, :, 1], gk[:, mem_count:]) < tol
    assert rel_err(d[:, :, 2], gv[:, mem_count:]) < tol
    if M > 0:
        dm = dkv_m.float().view(B, M, 2, H, 64)
        if mem_count > 0:
            assert rel_err(dm[:, M - mem_count:, 0], gk[:, :mem_count]) < tol
            assert rel_err(dm[:, M - mem_count:, 1], gv[:, :mem_count]) < tol
        if mem_count < M:
            assert dm[:, :M - mem_count].abs().max().item() == 0.0
    assert rel_err(du.view(H, 64), gu) < tol
    assert rel_err(dv.view(H, 64), gvb) < tol
    errs.update(dq=row_err(d[:, :, 0], gq), dk=row_err(d[:, :, 1], gk[:, mem_count:]), dv=row_err(d[:, :, 2], gv[:, mem_count:]),
                du=row_err(du, gu), dvb=row_err(dv, gvb))
    if mem_count > 0:
        errs.update(dk_mem=row_err(dm[:, M - mem_count:, 0], gk[:, :mem_count]), dv_mem=row_err(dm[:, M - mem_count:, 1], gv[:, :mem_count]))
    # dRk from the (row, distance) dS tensor, the way train.cu contracts it
    qv = (qkv_x.float().view(B * T, 3, H, 64)[:, 0] + v.view(1, H, 64)).bfloat16().float()       # [rows, H, 64]
    dsd = ds_dist.float().view(B * T, H, S)
    drk = torch.einsum('rhs,rhd->shd', dsd, qv)
    assert rel_err(drk[:mem_count + T], gr) < tol
    errs['drk'] = row_err(drk[:mem_count + T], gr)
    print('row errors', {n: f'{e:.2e}' for n, e in errs.items()}, flush=True)
    for n, e in errs.items():
        assert e < ROW_TOL[n], (n, e)
    if mem_count < M:
        assert drk[mem_count + T:].abs().max().item() == 0.0
