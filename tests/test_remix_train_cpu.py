"""CPU checks of the remix (masked-BERT) encoder's training step: the wrap-around attention backward identity the CUDA kernels
use, the oracle's masked cross entropy and padding row, and the training-config ABI (no GPU needed)."""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

import remix_attention_ref
from deepmusicgeneration_b200 import _lib
from oracle import bert
from oracle import bert_train
from oracle.txl import _line_shift


@pytest.mark.parametrize('T', [1, 2, 5, 8, 13])
def test_line_shift_lines_and_ds_dist_identity(T):
    """_line_shift(mask=False) of (q + v) Rk^T is the three lines of attention_bert_train.cu, and its gradient is dS put into
    (q-row, distance) coordinates (line 1 of row r, line 3 of row r - 1) times Rk / (q + v) - float64 against autograd."""
    g = torch.Generator().manual_seed(T)
    Dh = 4
    qv = torch.randn(T, Dh, dtype=torch.float64, generator=g, requires_grad=True)   # q + v rows
    Rk = torch.randn(T, Dh, dtype=torch.float64, generator=g, requires_grad=True)   # Rk[x] = r_attn(pe(position x))
    BD = _line_shift((qv @ Rk.flip(0).t())[None, None], mask=False)[0, 0]           # r[-T:] rows are positions T-1 .. 0
    q, R = qv.detach(), Rk.detach()
    for i in range(T):
        for j in range(T):
            if j <= i: want = q[i] @ R[i - j]
            elif j == i + 1: want = torch.zeros((), dtype=torch.float64)
            else: want = q[i + 1] @ R[T + 1 + i - j]
            assert abs(BD[i, j].item() - want.item()) < 1e-9, (i, j)
    dS = torch.randn(T, T, dtype=torch.float64, generator=g)
    (BD * dS).sum().backward()
    dist = torch.zeros(T, T, dtype=torch.float64)
    for r in range(T):
        for x in range(T):
            if x <= r: dist[r, x] = dS[r, r - x]
            elif r >= 1: dist[r, x] = dS[r - 1, T + r - x]
    assert torch.allclose(qv.grad, dist @ R)
    assert torch.allclose(Rk.grad, dist.t() @ q)


@pytest.mark.parametrize('T', [1, 2, 5, 8, 13])
@pytest.mark.parametrize('dropout', [False, True])
def test_float64_attention_reference_matches_the_oracle(T, dropout):
    """remix_attention_ref (the reference of tests/test_gpu_remix_attention.py) against the oracle's _apply_attention fed q, k, v
    and Rk directly (identity projections): same output, same gradients, and the gradients rebuilt from dS the way the kernels
    and the trainer's GEMMs split them (content part of dq from dS K, position part and dRk from ds_dist)."""
    B, H, D = 2, 2, 64
    g = torch.Generator().manual_seed(100 + T)
    q, k, v = (torch.randn(B, H, T, D, dtype=torch.float64, generator=g) for _ in range(3))
    rk = torch.randn(T, H, D, dtype=torch.float64, generator=g)
    u, vb = (0.3 * torch.randn(H, D, dtype=torch.float64, generator=g) for _ in range(2))
    mask = (torch.rand(B, H, T, T, generator=g) > 0.3).double() / 0.7 if dropout else None
    dout = torch.randn(B, H, T, D, dtype=torch.float64, generator=g)

    att = bert.MemMultiHeadRelativeAttentionKV(H, H * D, D, mem_len=0, r_mask=False).double()
    with torch.no_grad():
        for lin in (att.q_wgt, att.k_wgt, att.v_wgt, att.r_attn):
            lin.weight.copy_(torch.eye(H * D, dtype=torch.float64))
            lin.bias.zero_()
    att.drop_att = bert_train.FixedMask()
    att.drop_att.mask = mask
    leaves = [t.clone().requires_grad_(True) for t in (q, k, v, rk, u, vb)]
    lq, lk, lv, lrk, lu, lvb = leaves
    flat = lambda t: t.permute(0, 2, 1, 3).reshape(B, T, H * D)
    want = att._apply_attention(flat(lq), flat(lk), flat(lv), r=lrk.flip(0).reshape(T, H * D), g_u=lu[:, None], g_v=lvb[:, None])
    want.backward(flat(dout))
    want_grads = [t.grad for t in leaves]

    leaves = [t.clone().requires_grad_(True) for t in (q, k, v, rk, u, vb)]
    out, lse, raw = remix_attention_ref.remix_attention(*leaves, drop_mask=mask)
    raw.retain_grad()
    assert torch.allclose(flat(out), want, rtol=1e-12, atol=1e-12)
    assert torch.allclose(lse, torch.logsumexp(raw / 8, -1))
    out.backward(dout)
    for got, ref in zip([t.grad for t in leaves], want_grads):
        assert torch.allclose(got, ref, rtol=1e-10, atol=1e-12)

    dS = raw.grad
    dist = remix_attention_ref.ds_to_dist(dS)
    assert (dist[:, 0, :, 1:] == 0).all()
    qv = (q + vb[:, None]).permute(0, 2, 1, 3)
    dq_pos, dvb, drk = remix_attention_ref.position_grads(dist, rk, qv)
    dq_content = dS @ k
    gq, gk, gv, grk, gu, gvb = want_grads
    assert torch.allclose(dq_content + dq_pos.permute(0, 2, 1, 3), gq, rtol=1e-10, atol=1e-12)
    assert torch.allclose(dq_content.sum((0, 2)), gu, rtol=1e-10, atol=1e-12)
    assert torch.allclose(dvb, gvb, rtol=1e-10, atol=1e-12)
    assert torch.allclose(drk, grk, rtol=1e-10, atol=1e-12)
    assert torch.allclose(dS.transpose(-1, -2) @ (q + u[:, None]), gk, rtol=1e-10, atol=1e-12)


def small_model(pad_idx, V=40):
    cfg = dict(bert.multitask_config(), d_model=32, n_heads=2, d_head=16, d_inner=64, enc_layers=2)
    torch.manual_seed(0)
    return bert.get_multitask_model(V, cfg, drop_mult=0., pad_idx=pad_idx), V


def test_masked_ce_is_cross_entropy_with_ignore_index():
    g = torch.Generator().manual_seed(1)
    logits = torch.randn(3, 7, 11, generator=g)
    y = torch.randint(0, 11, (3, 7), generator=g)
    y[torch.rand(3, 7, generator=g) < 0.6] = 4
    ref = F.cross_entropy(logits.reshape(-1, 11), y.reshape(-1), ignore_index=4)
    assert torch.allclose(bert_train.masked_ce(logits, y, 4), ref)
    none = torch.full((3, 7), 4)
    assert torch.isnan(bert_train.masked_ce(logits, none, 4)) and torch.isnan(F.cross_entropy(logits.reshape(-1, 11), none.reshape(-1), ignore_index=4))


def test_pad_lookups_leave_only_the_head_gradient_on_the_pad_row():
    pad = 1
    model, V = small_model(pad)
    model.train()
    g = torch.Generator().manual_seed(2)
    x = torch.randint(2, V, (2, 9), generator=g)
    x[:, ::3] = pad                                   # pad tokens in the input
    pos = torch.cumsum(torch.randint(0, 5, (2, 9), generator=g), 1)
    y = torch.full_like(x, pad)
    y[:, 1::2] = torch.randint(2, V, (2, 9), generator=g)[:, 1::2]
    seen = {}
    model.head.decoder.register_forward_pre_hook(lambda mod, inp: seen.__setitem__('h', inp[0]))
    logits = model({'msk': {'x': x, 'pos': pos}})['msk']
    logits.retain_grad()
    bert_train.masked_ce(logits, y, pad).backward()
    head_only = torch.einsum('btv,btd->vd', logits.grad, seen['h'])[pad]
    emb = model.encoder.embed.embed.weight
    assert emb is model.head.decoder.weight
    assert torch.allclose(emb.grad[pad], head_only, atol=1e-7)
    other = x[0, 1].item()                            # a looked-up non-pad token also gets the embedding's gradient
    assert not torch.allclose(emb.grad[other], torch.einsum('btv,btd->vd', logits.grad, seen['h'])[other], atol=1e-7)


def test_oracle_train_step_moves_the_model_and_reports_the_masked_ce():
    from oracle.train import AdamTrueWD
    pad = 1
    model, V = small_model(pad)
    model.train()
    sites = bert_train.install_dropout_masks(model)
    assert {k: len(v) for k, v in sites.items()} == {'embed': 1, 'attn': 2, 'res1': 2, 'out': 1}
    opt = AdamTrueWD(bert_train.unique_params(model))
    g = torch.Generator().manual_seed(3)
    x = torch.randint(2, V, (2, 8), generator=g)
    pos = torch.arange(8).repeat(2, 1)
    y = torch.full_like(x, pad)
    y[:, 2] = 5
    w0 = model.encoder.layers[0].mha1.q_wgt.weight.detach().clone()
    out = bert_train.train_step(model, x, pos, y, opt, 1e-3, pad)
    ref = F.cross_entropy(model({'msk': {'x': x, 'pos': pos}})['msk'].reshape(-1, V), y.reshape(-1), ignore_index=pad)
    assert out['grad_norm'] > 0 and out['ce'] > 0 and abs(out['ce'] - ref.item()) < 1.0
    assert not torch.equal(w0, model.encoder.layers[0].mha1.q_wgt.weight)


def test_train_config_carries_pad_idx_at_offset_48():
    assert C.sizeof(_lib.TrainConfig) == 64
    assert _lib.TrainConfig.pad_idx.offset == 48 and _lib.TrainConfig.seed.offset == 40 and _lib.TrainConfig.alpha.offset == 28
    assert _lib.TrainConfig.reserved.offset == 52
