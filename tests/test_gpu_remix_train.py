"""GPU parity of the remix (masked-BERT) encoder's training step (dmg_train_* on a DMG_ARCH_BERT model, RemixTrainer,
MultitaskLearner.fit_one_cycle) against the oracle's restatement of the fastai step (oracle/bert_train.py on oracle/bert.py):
masked cross entropy, every parameter gradient, the gradient norm and the Adam update, with and without dropout (the oracle is fed
the very masks the kernels draw), pad tokens in x."""
import os
import socket

import numpy as np
import pytest
import torch

from deepmusicgeneration_b200.model import get_multitask_model
from deepmusicgeneration_b200.training import RemixTrainer
from oracle import bert as obert
from oracle import bert_train as obt
from oracle import train as otrain

pytestmark = pytest.mark.gpu

V, PAD, MASK = 324, 1, 3


def small_config(**kw):
    c = dict(obert.multitask_config(), enc_layers=2, d_model=128, n_heads=2, d_head=64, d_inner=256)
    c.update(kw)
    return c


def build_pair(cfg, bs, bptt, drop_mult, seed=0):
    torch.manual_seed(seed)
    om = obert.get_multitask_model(V, cfg, drop_mult=drop_mult, pad_idx=PAD)
    pm = get_multitask_model(V, cfg, pad_idx=PAD, dtype='bf16', max_batch=bs, max_seq=bptt, init=False)
    pm.load_state_dict(om.state_dict())
    tr = RemixTrainer(pm, bs, bptt, cfg, pad_idx=PAD, drop_mult=drop_mult, seed=1234, distributed=False)
    return om, pm, tr


def rel(a, b):
    return ((a.float() - b.float()).norm() / b.float().norm().clamp_min(1e-20)).item()


def compare_grads(got, om, tol, world=1):
    """Relative error of every gradient, except the k_wgt biases: softmax is invariant to a per-row shift of the scores, so their
    gradient is zero up to rounding on both sides - it must be small next to the q_wgt bias gradient of the same layer instead."""
    ref = {n: p.grad for n, p in om.state_dict(keep_vars=True).items() if getattr(p, 'grad', None) is not None}
    worst = (0., None)
    for name, g in got.items():
        r = ref.get(name)
        assert r is not None, f'oracle has no gradient for {name}'
        if name.endswith('k_wgt.bias'):
            scale = ref[name.replace('k_wgt', 'q_wgt')].norm()
            e = ((g / world - r).norm() / scale).item()
        else:
            e = rel(g / world, r.reshape(g.shape))
        if e > worst[0]:
            worst = (e, name)
    assert worst[0] < tol, f'worst gradient mismatch {worst}'
    print('worst gradient rel err', worst, flush=True)
    return len(got)


def install_masks(tr, sites, cfg, bs, bptt, step):
    d, H = cfg['d_model'], cfg['n_heads']
    sites['embed'][0].mask = tr.dropout_mask(0, 0, (bs, bptt, d), step).cpu()
    sites['out'][0].mask = tr.dropout_mask(5, 0, (bs, 1, d), step).cpu()
    for l in range(cfg['enc_layers']):
        sites['attn'][l].mask = tr.dropout_mask(1, l, (bs, H, bptt, bptt), step).cpu()
        sites['res1'][l].mask = tr.dropout_mask(2, l, (bs, bptt, d), step).cpu()


def masked_batch(g, bs, bptt, p=0.3):
    "tokens with pad tokens in x; y = the original token at ~p of the positions (x there = mask), pad elsewhere"
    x = torch.randint(4, V, (bs, bptt), generator=g)
    x[torch.rand(bs, bptt, generator=g) < 0.1] = PAD
    sel = torch.rand(bs, bptt, generator=g) < p
    y = torch.where(sel, x, torch.full_like(x, PAD))
    x = torch.where(sel, torch.full_like(x, MASK), x)
    pos = torch.cumsum(torch.randint(0, 9, (bs, bptt), generator=g), 1)
    return x, y, pos


@pytest.mark.parametrize('bptt', [64, 128, 192])
@pytest.mark.parametrize('drop_mult', [0., 1.])
def test_remix_training_step_matches_oracle(drop_mult, bptt):
    cfg = small_config()
    bs, steps, lr = 3, 3, 1e-3
    om, pm, tr = build_pair(cfg, bs, bptt, drop_mult)
    om.train()
    sites = obt.install_dropout_masks(om)
    opt = otrain.AdamTrueWD(otrain.unique_params(om), eps=1e-3)
    sd0 = {k: v.clone() for k, v in om.state_dict().items()}
    g = torch.Generator().manual_seed(5)
    for s in range(steps):
        x, y, pos = masked_batch(g, bs, bptt)
        if drop_mult > 0:
            install_masks(tr, sites, cfg, bs, bptt, s)
        ref = obt.train_step(om, x, pos, y, opt, lr, PAD, wd=0.01, clip=0.5)
        tr.forward(x, y, pos)
        tr.backward()
        got = tr.losses()
        assert got['ar'] == 0. and got['tar'] == 0.
        assert abs(got['ce'] - ref['ce']) < 2e-2 * max(1., abs(ref['ce'])), (s, got, ref)
        n = compare_grads(tr.grads(), om, tol=2e-2)
        assert n == 6 + 10 * cfg['enc_layers']
        tr.optimizer_step(lr, betas=(0.9, 0.99), eps=1e-3, wd=0.01, clip=0.5)
        got = tr.losses()
        assert abs(got['grad_norm'] - ref['grad_norm']) < 3e-2 * ref['grad_norm'], (s, got, ref)
    sd_ref, sd_got = om.state_dict(), pm.state_dict()
    for name, w in sd_got.items():
        if name.endswith('k_wgt.bias'):          # zero gradient (see compare_grads): Adam moves it by rounding noise only
            continue
        d_got, d_ref = w - sd0[name].reshape(w.shape), (sd_ref[name] - sd0[name]).reshape(w.shape)
        assert rel(d_got, d_ref) < 0.1, (name, rel(d_got, d_ref))
    tr.close()


def test_remix_geometry_gradients_and_20_step_loss_curve():
    """The C4 encoder (d_model 512, 8 heads x 64, 10 layers) at T 1024, 2 sequences of LakhMIDI-shaped tokens through mask_tfm, dropout
    off: one step's gradients against the oracle, then 20 steps of the recipe (Adam(0.9, 0.99), true_wd 0.01, clip 0.5) on two
    repeating batches - every step's masked CE follows the oracle and the loss falls."""
    import bench_train
    from deepmusicgeneration_b200.preloader import mask_tfm
    cfg = obert.multitask_config()
    bs, bptt, steps, lr = 2, 1024, 20, 5e-4
    om, pm, tr = build_pair(cfg, bs, bptt, 0.)
    om.train()
    opt = otrain.AdamTrueWD(otrain.unique_params(om))
    toks = bench_train.lakh_shaped_tokens(bs, 2 * bptt, torch.Generator().manual_seed(3))
    batches = []
    for i in range(2):
        x = toks[:, i * bptt:(i + 1) * bptt].contiguous().cuda()
        pos = (torch.arange(bptt) // 2).repeat(bs, 1)
        xm, ym = mask_tfm((x, x), (12, 300), MASK, PAD, p=0.3, seed=7 + i)
        batches.append((xm.cpu(), ym.cpu(), pos))
    curve = []
    for s in range(steps):
        x, y, pos = batches[s % 2]
        ref = obt.train_step(om, x, pos, y, opt, lr, PAD, wd=0.01, clip=0.5)
        tr.forward(x, y, pos)
        tr.backward()
        if s == 0:
            compare_grads(tr.grads(), om, tol=3e-2)
        tr.optimizer_step(lr, betas=(0.9, 0.99), eps=1e-8, wd=0.01, clip=0.5)
        curve.append((ref['ce'], tr.losses()['ce']))
    print('loss curve (oracle ce, cuda ce):', [(round(a, 3), round(b, 3)) for a, b in curve])
    for s, (rce, gce) in enumerate(curve):
        assert abs(gce - rce) < 3e-2 * rce + 2e-2, (s, curve[s])
    assert curve[-1][1] < curve[0][1] - 1.0
    tr.close()


def _corpus_preloader(vocab, bs, bptt):
    from deepmusicgeneration_b200.preloader import MusicPreloader
    from oracle import preloader as opl
    rng = np.random.default_rng(0)
    pattern = rng.integers(vocab.note_range[0], vocab.dur_range[1], 48)
    items = [opl.Item(np.tile(pattern, 8)[:int(n)], np.arange(int(n))) for n in rng.integers(160, 380, 12)]
    return MusicPreloader(items, vocab, bs=bs, bptt=bptt, shuffle=True, transpose_range=None, encode_position=True, y_offset=0)


def test_fit_one_cycle_over_the_preloader_then_inference_follows(golden_dir):
    "multitask_model_learner(...).fit_one_cycle(epochs, lr, MusicPreloader(y_offset=0)): the loss falls; inference sees the weights"
    from deepmusicgeneration_b200.codec import MusicDataBunch, MusicItem
    from deepmusicgeneration_b200.learner import multitask_model_learner
    cfg = small_config()
    data = MusicDataBunch.empty('')
    learn = multitask_model_learner(data, config=cfg, dtype='bf16', max_batch=4, max_seq=512, seed=0)
    pl = _corpus_preloader(data.vocab, 4, 64)
    ces = []
    last = learn.fit_one_cycle(8, 3e-3, pl, callback=lambda i, tr: ces.append(tr.losses()['ce']))
    first3, last3 = np.mean(ces[:3]), np.mean(ces[-3:])
    print('masked CE first / last batches', first3, last3, last)
    assert last3 < 0.7 * first3, (first3, last3)
    # the inference forward on the trained weights equals the oracle's forward on the trained state_dict
    torch.manual_seed(0)
    om = obert.get_multitask_model(len(data.vocab.itos), cfg, pad_idx=data.vocab.pad_idx).eval()
    om.load_state_dict(learn.model.state_dict(), strict=False)
    g = torch.Generator().manual_seed(4)
    x = torch.randint(0, len(data.vocab.itos), (2, 128), generator=g)
    pos = torch.cumsum(torch.randint(0, 5, (2, 128), generator=g), 1)
    with torch.no_grad():
        ol = om({'msk': {'x': x, 'pos': pos.clone()}})['msk']
    pl_logits = learn.model({'msk': {'x': x.cuda(), 'pos': pos.cuda()}})['msk'].cpu()
    assert rel(pl_logits, ol) < 2e-2
    item = MusicItem.from_file(os.path.join(golden_dir, 'uploadedMidi.mid'), data.vocab).trim_to_beat(8)
    notes = [i for i, t in enumerate(item.data) if data.vocab.note_range[0] <= t < data.vocab.note_range[1]]
    item.data[notes[::2]] = data.vocab.mask_idx
    out = learn.predict_mask(item, top_k=1, top_p=0.0)
    assert len(out.data) == len(item.data) and data.vocab.mask_idx not in list(out.data)


def test_checkpoint_round_trip_resumes_adam(tmp_path):
    "save(with_opt) -> multitask_model_learner(pretrained_path=...) -> fit_one_cycle starts from the saved Adam moments and step count"
    from deepmusicgeneration_b200.codec import MusicDataBunch
    from deepmusicgeneration_b200.learner import multitask_model_learner
    from deepmusicgeneration_b200.training import one_cycle_lr
    cfg = small_config()
    data = MusicDataBunch.empty('')
    learn = multitask_model_learner(data, config=cfg, dtype='bf16', max_batch=4, max_seq=64, seed=3)
    g = torch.Generator().manual_seed(8)
    batches = []
    for _ in range(3):
        x, y, pos = masked_batch(g, 4, 64)
        batches.append(({'x': x, 'pos': pos}, y))
    path = str(tmp_path / 'remix.pth')
    assert torch.load(learn.save(path), weights_only=False)['opt'] is None       # no trainer yet
    learn.fit_one_cycle(1, 3e-3, batches)
    learn.save(path, config=dict(cfg))
    state = torch.load(path, map_location='cpu', weights_only=False)
    assert state['opt'] is not None and len(state['opt']['state']) == len(state['opt']['param_names']) == 6 + 10 * cfg['enc_layers']
    assert state['opt']['step_count'] == 3
    learn2 = multitask_model_learner(data, config=None, pretrained_path=path, dtype='bf16', max_batch=4, max_seq=64)
    for k, v in learn.model.state_dict().items():
        assert torch.equal(v, learn2.model.state_dict()[k]), k
    seen = []
    learn2.fit_one_cycle(1, 3e-3, batches[:1], callback=lambda i, tr: seen.append(tr.step_count))
    assert seen == [4]
    # the same step on the original learner's live trainer moves the weights identically
    lr, mom = one_cycle_lr(0, 1, 3e-3)
    tr1 = learn.trainer(4, 64)
    tr1.step(batches[0][0]['x'], batches[0][1], batches[0][0]['pos'], lr=lr, betas=(mom, 0.99))
    sd1, sd2 = learn.model.state_dict(), learn2.model.state_dict()
    for k in sd1:
        assert (sd1[k] - sd2[k]).abs().max() < 1e-6, k


def test_error_paths_name_the_constraint():
    from deepmusicgeneration_b200._lib import DmgError
    cfg = small_config()
    torch.manual_seed(0)
    pm = get_multitask_model(V, cfg, pad_idx=PAD, dtype='bf16', max_batch=2, max_seq=128)
    with pytest.raises(DmgError, match='multiple of 64'):
        RemixTrainer(pm, 2, 96, cfg, pad_idx=PAD, distributed=False)
    tr = RemixTrainer(pm, 2, 64, cfg, pad_idx=PAD, distributed=False)
    x, y, pos = masked_batch(torch.Generator().manual_seed(1), 2, 64)
    with pytest.raises(ValueError, match=r'\(1, 1\)'):
        tr.forward(x, y, pos, mask_size=(2, 0))
    with pytest.raises(ValueError, match='pos'):
        tr.forward(x, y, None)
    # the library refuses a window mask for the encoder too
    from deepmusicgeneration_b200.model import _ptr, _stream_ptr
    xd, yd, pd = x.cuda(), y.cuda(), pos.cuda()
    rc = tr.lib.dmg_train_forward(tr.e.h, _ptr(xd), _ptr(pd), _ptr(yd), 2, 0, 1, 0, _stream_ptr())
    assert rc != 0 and b'(1, 1)' in tr.lib.dmg_last_error()
    # a batch without any target: CE is NaN (torch's value), the gradients are zero
    tr.forward(x, torch.full_like(y, PAD), pos)
    tr.backward()
    assert np.isnan(tr.losses()['ce'])
    assert all(torch.count_nonzero(v) == 0 for v in tr.grads().values())
    tr.close()


def _dp_worker(rank, world, port, q):
    os.environ.update(RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE=str(world), MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    from deepmusicgeneration_b200 import sharding
    try:
        sharding.init_distributed(backend='nccl')
        torch.cuda.set_device(rank)
        cfg = small_config(enc_layers=5)
        bptt, per = 128, 2
        torch.manual_seed(0)
        om = obert.get_multitask_model(V, cfg, drop_mult=0., pad_idx=PAD).train()
        pm = get_multitask_model(V, cfg, pad_idx=PAD, dtype='bf16', device=rank, max_batch=per, max_seq=bptt, init=False)
        pm.load_state_dict(om.state_dict())
        tr = RemixTrainer(pm, per, bptt, cfg, pad_idx=PAD, drop_mult=0., distributed=True, bucket_layers=1)
        x, y, pos = masked_batch(torch.Generator().manual_seed(5), world * per, bptt)
        lo, hi = rank * per, (rank + 1) * per
        # the oracle's average of the per-rank gradients (each rank's loss is its own masked mean)
        acc = {}
        for r in range(world):
            for p in otrain.unique_params(om):
                p.grad = None
            sl = slice(r * per, (r + 1) * per)
            obt.masked_ce(om({'msk': {'x': x[sl], 'pos': pos[sl]}})['msk'], y[sl], PAD).backward()
            for n, p in om.state_dict(keep_vars=True).items():
                if getattr(p, 'grad', None) is not None:
                    acc[n] = acc.get(n, 0) + p.grad / world
        for n, p in om.state_dict(keep_vars=True).items():
            if n in acc:
                p.grad = acc[n]
        tr.forward(x[lo:hi], y[lo:hi], pos[lo:hi])
        tr.backward()
        compare_grads(tr.grads(), om, tol=2e-2, world=world)
        tr.close()
        q.put((rank, 'ok'))
    except Exception as e:   # report to the parent
        q.put((rank, repr(e)))
    finally:
        import torch.distributed as dist
        if dist.is_initialized():
            dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs >= 2 GPUs')
def test_two_gpu_gradient_is_the_average_of_rank_gradients():
    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        port = s.getsockname()[1]
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    procs = [ctx.Process(target=_dp_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = dict(q.get(timeout=600) for _ in procs)
    for p in procs:
        p.join(timeout=120)
    assert res == {0: 'ok', 1: 'ok'}, res
