"""GPU checks of validation while training (dmg_train_eval_*, dmg_eval_metrics, TXLTrainer / RemixTrainer.validate, the learners'
validate and fit_one_cycle(valid_batches=..., callbacks=...)) against the float64 reference of validate_ref.py on the oracle models."""
import ctypes as C
import math
import os
import socket

import numpy as np
import pytest
import torch

import validate_ref as ref
from deepmusicgeneration_b200 import training
from deepmusicgeneration_b200._lib import DmgError
from deepmusicgeneration_b200.model import _ptr, _stream_ptr, get_language_model, get_multitask_model
from deepmusicgeneration_b200.training import RemixTrainer, TXLTrainer, one_cycle_lr
from oracle import bert as obert
from oracle import train as otrain
from oracle import txl

pytestmark = pytest.mark.gpu

V, PAD, MASK = 324, 1, 3
CE_TOL = 2e-2          # the CE tolerance of the training-step parity tests (tests/test_gpu_train_step.py)


def txl_config(**kw):
    c = dict(txl.default_config(), n_layers=2, d_model=128, n_heads=2, d_head=64, d_inner=256, mem_len=64, ctx_len=64,
             encode_position=False, mask_steps=1)
    c.update(kw)
    return c


def bert_config(**kw):
    c = dict(obert.multitask_config(), enc_layers=2, d_model=128, n_heads=2, d_head=64, d_inner=256)
    c.update(kw)
    return c


def txl_pair(cfg, bs, bptt, seed=0):
    torch.manual_seed(seed)
    om = txl.get_language_model(V, cfg, drop_mult=0.)
    pm = get_language_model(V, cfg, dtype='bf16', device=0, max_batch=bs, max_seq=max(bptt, 64), keep_hidden=False, init=False)
    pm.load_state_dict(om.state_dict())
    return om, pm, TXLTrainer(pm, bs, bptt, cfg, drop_mult=0., seed=1234, distributed=False)


def bert_pair(cfg, bs, bptt, seed=0, drop_mult=0.):
    torch.manual_seed(seed)
    om = obert.get_multitask_model(V, cfg, drop_mult=drop_mult, pad_idx=PAD)
    pm = get_multitask_model(V, cfg, pad_idx=PAD, dtype='bf16', max_batch=bs, max_seq=bptt, init=False)
    pm.load_state_dict(om.state_dict())
    return om, pm, RemixTrainer(pm, bs, bptt, cfg, pad_idx=PAD, drop_mult=drop_mult, seed=1234, distributed=False)


@pytest.fixture
def fixed_masks(monkeypatch):
    "(1,1) window masks on both sides (the product's training forward and the oracle's train-mode forward)"
    monkeypatch.setattr(training, 'rand_window_mask_size', lambda *a, **k: (1, 1))
    monkeypatch.setattr(txl, 'rand_window_mask', lambda x_len, m_len, device, **kw: txl.window_mask(x_len, device, m_len, size=(1, 1)))


def lm_batches(g, n, bs, bptt):
    """language-model batches whose targets are the input token at half the positions (a freshly initialised tied model often ranks
    its own input first, so the accuracy is far from 0 and from 1) and random elsewhere"""
    out = []
    for _ in range(n):
        x = torch.randint(0, V, (bs, bptt), generator=g)
        y = torch.where(torch.rand(bs, bptt, generator=g) < 0.5, x, torch.randint(0, V, (bs, bptt), generator=g))
        out.append((x, y))
    return out


def masked_batch(g, bs, bptt, p=0.3):
    x = torch.randint(4, V, (bs, bptt), generator=g)
    x[torch.rand(bs, bptt, generator=g) < 0.1] = PAD
    sel = torch.rand(bs, bptt, generator=g) < p
    y = torch.where(sel, x, torch.full_like(x, PAD))
    x = torch.where(sel, torch.full_like(x, MASK), x)
    pos = torch.cumsum(torch.randint(0, 9, (bs, bptt), generator=g), 1)
    return x, y, pos


def oracle_txl_logits(om, batches, reset):
    om.eval()
    if reset:
        om.reset()
    with torch.no_grad():
        return [om(x)[0] for x, _ in batches]


def ambiguous(logits, err):
    """positions whose oracle top-2 margin is below twice the largest logit error `err`: their argmax may go either way (the tie rule
    of DESIGN.md section 6)"""
    top2 = logits.reshape(-1, logits.shape[-1]).float().topk(2, -1).values
    return int(((top2[:, 0] - top2[:, 1]) < 2 * err).sum())


def txl_logit_err(model, om, batches):
    """largest absolute logit error of the product's bf16 weights against the oracle over `batches` (both reset, eval mode, memory
    carried), measured through the inference engine"""
    model.reset()
    return max((model(x.cuda())[0].float().cpu() - lo).abs().max().item() for (x, _), lo in zip(batches, oracle_txl_logits(om, batches, True)))


def remix_logit_err(model, om, batches):
    "the same for the remix encoder over (x, y, pos) batches"
    om.eval()
    with torch.no_grad():
        return max((model({'msk': {'x': x.cuda(), 'pos': p.cuda()}})['msk'].float().cpu() - om({'msk': {'x': x, 'pos': p.clone()}})['msk'])
                   .abs().max().item() for x, _, p in batches)


def remix_ambiguous(om, batches, pad, err):
    "ambiguous predicted positions of the oracle encoder over (x, y, pos) batches"
    om.eval()
    with torch.no_grad():
        return sum(ambiguous(om({'msk': {'x': x, 'pos': p.clone()}})['msk'].reshape(-1, V)[(y != pad).reshape(-1)], err)
                   for x, y, p in batches)


# ---------------------------------------------------------------------------------------------------- 3. the metrics kernel
@pytest.mark.parametrize('Vk', [7, 324, 1000])
@pytest.mark.parametrize('ignore', [None, 2])
def test_eval_metrics_kernel_matches_float64(Vk, ignore):
    from deepmusicgeneration_b200 import _lib
    lib = _lib.load()
    g = torch.Generator().manual_seed(Vk)
    rows, ldl = 1237, Vk + 5                      # rows not a multiple of the 8 rows of a block
    lg = torch.randn(rows, ldl, generator=g) * 3.
    lg[:, Vk:] = 1e30                             # padding columns must not be read
    y = torch.randint(0, Vk, (rows,), generator=g)
    for r in range(0, rows, 5):                   # exact ties of the maximum: the target is the later copy on even r
        a, b = sorted(torch.randperm(Vk, generator=g)[:2].tolist())
        lg[r, a] = lg[r, b] = lg[r, :Vk].max() + 0.5
        y[r] = b if r % 2 == 0 else a
    y[7], y[11] = -4, Vk + 9                      # out of range: clamped as in the training loss
    if ignore is not None:
        y[1::6] = ignore
    lgd, yd = lg.cuda(), y.cuda()
    outs = []
    for _ in range(4):
        out = torch.full((3,), -1., dtype=torch.float64, device='cuda')
        assert lib.dmg_eval_metrics(_ptr(lgd), ldl, _ptr(yd), -1 if ignore is None else ignore, rows, Vk, _ptr(out), _stream_ptr()) == 0
        outs.append(out.cpu())
    want = ref.batch_metrics(lg[:, :Vk], y, ignore)
    got = outs[0].tolist()
    print('metrics kernel', Vk, ignore, got, want)
    assert got[1] == want[1] and got[2] == want[2]
    assert abs(got[0] - want[0]) <= 1e-6 * abs(want[0])
    assert all(torch.equal(o, outs[0]) for o in outs[1:])      # the same bits on every run
    assert lib.dmg_eval_metrics(_ptr(lgd), Vk - 1, _ptr(yd), -1, rows, Vk, _ptr(outs[0]), _stream_ptr()) != 0
    assert b'ldl' in lib.dmg_last_error()


# ---------------------------------------------------------------------------------------------------- 4. TXL validate
def test_txl_validate_after_reset_matches_oracle(fixed_masks):
    cfg = txl_config()
    bs, bptt = 3, 64
    om, pm, tr = txl_pair(cfg, bs, bptt)
    vb = lm_batches(torch.Generator().manual_seed(2), 4, bs, bptt)
    ref_loss, ref_acc, ref_ms = ref.txl_validate(om, vb, reset=True)
    got = tr.validate(vb, reset=True)
    err = txl_logit_err(pm, om, vb)
    amb = sum(ambiguous(lo, err) for lo in oracle_txl_logits(om, vb, True))
    print('txl validate', got, ref_loss, ref_acc, 'logit err', err, 'ambiguous', amb)
    assert abs(got['valid_loss'] - ref_loss) < CE_TOL * max(1., abs(ref_loss))
    assert 0.05 < ref_acc < 0.95
    assert abs(got['accuracy'] - ref_acc) <= amb / (len(vb) * bs * bptt) + 1e-12
    # memory is carried: validating the batches one at a time without reset gives the same table
    tr.reset()
    tab = tr._eval_table(((x, y, None) for x, y in vb), len(vb))
    tr.reset()
    one = np.concatenate([tr._eval_table(iter([(x, y, None)]), 1) for x, y in vb])
    assert np.array_equal(tab, one)
    assert [row[1] for row in ref_ms] == list(tab[:, 1])
    tr.close()


def test_txl_validate_continues_the_training_memory_in_fit_one_cycle(fixed_masks):
    "fit_one_cycle(valid_batches=...): validation straight after an epoch's training batches, memory carried, against the oracle"
    from deepmusicgeneration_b200.codec import MusicDataBunch
    from deepmusicgeneration_b200.learner import music_model_learner
    cfg = txl_config()
    bs, bptt, max_lr = 3, 64, 1e-3
    data = MusicDataBunch.empty('')
    torch.manual_seed(0)
    om = txl.get_language_model(V, cfg, drop_mult=0.)
    learn = music_model_learner(data, config=dict(cfg), drop_mult=0., dtype='bf16', max_batch=bs, max_seq=64, keep_hidden=False, seed=0)
    learn.model.load_state_dict(om.state_dict())
    g = torch.Generator().manual_seed(3)
    tb, vb = lm_batches(g, 3, bs, bptt), lm_batches(g, 3, bs, bptt)
    learn.fit_one_cycle(1, max_lr, tb, drop_mult=0., valid_batches=vb)
    # the oracle: the same one-cycle steps (Adam(true_wd), clip 0.5, eps 1e-8), then validation without a reset
    om.train(); om.reset()
    opt = otrain.AdamTrueWD(otrain.unique_params(om))
    for i, (x, y) in enumerate(tb):
        lr, mom = one_cycle_lr(i, len(tb), max_lr)
        otrain.train_step(om, x, y, opt, lr, wd=0.01, clip=0.5, betas=(mom, 0.99))
    hidden = [h.clone() for h in om[0].hidden]                  # the training memory validation starts from
    ref_loss, ref_acc, _ = ref.txl_validate(om, vb, reset=False)
    om[0].hidden = hidden
    row = learn.recorder[0]
    print('fit_one_cycle validation', row, ref_loss, ref_acc)
    assert len(learn.recorder) == 1 and set(row) == {'epoch', 'train_loss', 'valid_loss', 'accuracy', 'time'}
    assert abs(row['valid_loss'] - ref_loss) < CE_TOL * max(1., abs(ref_loss))
    amb_logits = oracle_txl_logits(om, vb, False)
    err = txl_logit_err(learn.model, om, vb)        # the trained weights of both sides, measured after a reset
    amb = sum(ambiguous(lo, err) for lo in amb_logits)
    print('logit err', err, 'ambiguous', amb)
    assert abs(row['accuracy'] - ref_acc) <= amb / (len(vb) * bs * bptt) + 1e-12
    # validate() resets first: it matches the oracle's validation after a reset
    got = learn.validate(vb)
    ref_loss2, _, _ = ref.txl_validate(om, vb, reset=True)
    assert abs(got[0] - ref_loss2) < CE_TOL * max(1., abs(ref_loss2))


# ---------------------------------------------------------------------------------------------------- 5. remix validate
def test_remix_validate_matches_oracle_with_seeded_masks():
    from deepmusicgeneration_b200.preloader import mask_tfm
    cfg = bert_config()
    bs, bptt = 3, 128
    om, pm, tr = bert_pair(cfg, bs, bptt)
    g = torch.Generator().manual_seed(6)
    vb = []
    for i in range(3):
        x = torch.randint(4, V, (bs, bptt), generator=g).cuda()
        pos = torch.cumsum(torch.randint(0, 9, (bs, bptt), generator=g), 1)
        xm, ym = mask_tfm((x, x), (4, V), MASK, PAD, p=0.3, seed=11 + i)
        vb.append((xm.cpu(), ym.cpu(), pos))
    ref_loss, ref_acc, ref_ms = ref.bert_validate(om, vb, PAD)
    got = tr.validate([({'x': x, 'pos': p}, y) for x, y, p in vb])
    err = remix_logit_err(pm, om, vb)
    amb = remix_ambiguous(om, vb, PAD, err)
    kept = sum(m[1] for m in ref_ms)
    print('remix validate', got, ref_loss, ref_acc, 'logit err', err, 'ambiguous', amb, 'kept', kept)
    assert abs(got['valid_loss'] - ref_loss) < CE_TOL * max(1., abs(ref_loss))
    assert abs(got['mask_acc'] - ref_acc) <= len(vb) * amb / kept + 1e-12    # per batch over ~kept/3 targets
    # a batch with nothing to predict: NaN, and it carries into the epoch value
    x, y, p = vb[0]
    got = tr.validate([(x, y, p), (x, torch.full_like(y, PAD), p)])
    assert math.isnan(got['valid_loss']) and math.isnan(got['mask_acc'])
    tr.close()


def test_remix_validate_over_the_preloader_is_reproducible_with_a_seed():
    from deepmusicgeneration_b200.codec import MusicDataBunch
    from deepmusicgeneration_b200.preloader import MusicPreloader
    from oracle import preloader as opl
    vocab = MusicDataBunch.empty('').vocab
    cfg = bert_config()
    om, pm, tr = bert_pair(cfg, 4, 64)
    rng = np.random.default_rng(0)
    pattern = rng.integers(vocab.note_range[0], vocab.dur_range[1], 48)
    items = [opl.Item(np.tile(pattern, 8)[:int(n)], np.arange(int(n))) for n in rng.integers(160, 380, 6)]
    pl = MusicPreloader(items, vocab, bs=4, bptt=64, shuffle=False, encode_position=True, y_offset=0)
    a = tr.validate(pl, seed=5, vocab=vocab)
    b = tr.validate(pl, seed=5, vocab=vocab)
    c = tr.validate(pl, seed=6, vocab=vocab)
    print('preloader validation', a, c)
    assert a == b and a != c and all(math.isfinite(v) for v in a.values())
    tr.close()


# ---------------------------------------------------------------------------------------------------- 6. eval-only forward
def test_eval_forward_equals_the_training_forward_in_eval_mode(fixed_masks):
    "dmg_train_eval_batch against dmg_train_forward(training=0) + losses()['ce'] on the same batch, both models, at a tcgen05 geometry"
    cfg = txl_config(mem_len=128, ctx_len=128)
    bs, bptt = 2, 128
    _, _, tr = txl_pair(cfg, bs, bptt)
    g = torch.Generator().manual_seed(9)
    diffs = []
    for _ in range(2):          # the second batch attends over the memory of the first
        x, y = lm_batches(g, 1, bs, bptt)[0]
        tr.reset(); tr.eval()
        tr.forward(x, y, mask_size=(1, 1))
        tr.forward(x, y, mask_size=(1, 1))
        want = tr.losses()['ce']
        tr.reset()
        tab = tr._eval_table(iter([(x, y, None), (x, y, None)]), 2)
        diffs.append(abs(tab[1, 0] / (bs * bptt) - want) / want)
    tr.train()
    cfgb = bert_config()
    _, _, trb = bert_pair(cfgb, 2, 128)
    xb, yb, pb = masked_batch(torch.Generator().manual_seed(4), 2, 128)
    trb.eval()
    trb.forward(xb, yb, pb)
    want = trb.losses()['ce']
    got = trb.validate([(xb, yb, pb)])['valid_loss']
    diffs.append(abs(got - want) / want)
    print('eval-only forward vs training forward (training=0), relative CE difference (txl, txl with memory, remix):', diffs)
    assert max(diffs) < 1e-3
    tr.close(); trb.close()


# ---------------------------------------------------------------------------------------------------- 7. training state untouched
def test_validation_leaves_training_state_untouched():
    from deepmusicgeneration_b200 import _lib
    cfg = txl_config()
    bs, bptt = 3, 64
    _, pm, tr = txl_pair(cfg, bs, bptt)
    g = torch.Generator().manual_seed(1)
    tb = lm_batches(g, 2, bs, bptt)
    for x, y in tb:
        tr.step(x, y, lr=1e-3, mask_size=(1, 1))
    before = (pm.state_dict(), tr.opt_state_dict(), tr.step_count, tr.losses())
    tr.validate(lm_batches(g, 2, bs, bptt), reset=False)
    after = (pm.state_dict(), tr.opt_state_dict(), tr.step_count, tr.losses())
    for k in before[0]:
        assert torch.equal(before[0][k], after[0][k]), k
    for i, st in before[1]['state'].items():
        for key in ('exp_avg', 'exp_avg_sq'):
            assert torch.equal(st[key], after[1]['state'][i][key])
        assert st['step'] == after[1]['state'][i]['step']
    assert before[2] == after[2] and before[3] == after[3]
    # a backward after an eval batch is refused, before anything launches
    x, y = tb[0]
    tr.forward(x, y, mask_size=(1, 1))
    tr.validate([(x, y)], reset=False)
    lib = _lib.load()
    torch.cuda.synchronize()
    n0 = lib.dmg_launch_count()
    with pytest.raises(DmgError, match='validation batch'):
        tr.backward()
    assert lib.dmg_launch_count() == n0
    # the next training step works as before
    tr.step(x, y, lr=1e-3, mask_size=(1, 1))
    assert math.isfinite(tr.losses()['ce'])
    tr.close()


# ---------------------------------------------------------------------------------------------------- 8. end to end
def test_fit_one_cycle_with_early_stopping_and_save_model(tmp_path, monkeypatch):
    """Scripted validation values (through a monkeypatched TXLTrainer.validate) plateau after epoch 1: EarlyStopping(patience=1) stops
    after epoch 3 of 8, the recorder has 4 rows, SaveModel kept epoch 1 and the learner ends with exactly those weights and Adam state."""
    from deepmusicgeneration_b200.callbacks import EarlyStoppingCallback, SaveModelCallback
    from deepmusicgeneration_b200.codec import MusicDataBunch
    from deepmusicgeneration_b200.learner import music_model_learner
    cfg = txl_config()
    data = MusicDataBunch.empty(str(tmp_path))
    learn = music_model_learner(data, config=dict(cfg), dtype='bf16', max_batch=4, max_seq=256, keep_hidden=False, seed=0)
    base = (torch.arange(4 * 64 * 6) % 29 + 12).view(4, -1)
    batches = [(base[:, i * 64:(i + 1) * 64], base[:, i * 64 + 1:(i + 1) * 64 + 1]) for i in range(5)]
    script = iter([3.0, 2.0, 2.5, 2.6, 2.7, 2.8, 2.9, 3.0])
    real = TXLTrainer.validate
    snaps = []

    def scripted(self, vb, reset=True):
        r = real(self, vb, reset=reset)            # the real validation runs; its loss is replaced by the script
        snaps.append(self.model.state_dict())
        return {'valid_loss': next(script), 'accuracy': r['accuracy']}
    monkeypatch.setattr(TXLTrainer, 'validate', scripted)
    cbs = [EarlyStoppingCallback(patience=1), SaveModelCallback(name='best')]
    learn.fit_one_cycle(8, 3e-3, batches, valid_batches=batches[:2], callbacks=cbs)
    assert [r['epoch'] for r in learn.recorder] == [0, 1, 2, 3]
    assert [r['valid_loss'] for r in learn.recorder] == [3.0, 2.0, 2.5, 2.6]
    assert all(math.isfinite(r['train_loss']) and 0. <= r['accuracy'] <= 1. for r in learn.recorder)
    best = torch.load(str(tmp_path / 'models' / 'best.pth'), weights_only=False)
    final = learn.model.state_dict()
    assert any(not torch.equal(snaps[1][k], snaps[3][k]) for k in final)       # training moved on after the best epoch
    for k in final:
        assert torch.equal(final[k], best['model'][k]) and torch.equal(final[k], snaps[1][k]), k
    opt = learn._trainer.opt_state_dict()
    assert opt['step_count'] == best['opt']['step_count'] == 2 * len(batches)
    for i, st in best['opt']['state'].items():
        assert torch.equal(st['exp_avg'], opt['state'][i]['exp_avg'])
    # generation runs on the restored weights (a model this small can break the token grammar, which predict reports by raising, as
    # the reference does; generate_batch returns those steps as -2)
    toks = learn.generate_batch(base[:, :64], n_words=16, seed=0).cpu()
    assert toks.shape == (16, 4) and bool((toks[0] != -1).all())


def test_remix_fit_one_cycle_validates_every_epoch_then_predict_mask(tmp_path, golden_dir):
    from deepmusicgeneration_b200.callbacks import EarlyStoppingCallback, SaveModelCallback
    from deepmusicgeneration_b200.codec import MusicDataBunch, MusicItem
    from deepmusicgeneration_b200.learner import multitask_model_learner
    from deepmusicgeneration_b200.preloader import MusicPreloader
    from oracle import preloader as opl
    data = MusicDataBunch.empty(str(tmp_path))
    vocab = data.vocab
    learn = multitask_model_learner(data, config=bert_config(), dtype='bf16', max_batch=4, max_seq=512, seed=0)
    rng = np.random.default_rng(0)
    pattern = rng.integers(vocab.note_range[0], vocab.dur_range[1], 48)
    items = [opl.Item(np.tile(pattern, 8)[:int(n)], np.arange(int(n))) for n in rng.integers(160, 380, 12)]
    pl = MusicPreloader(items, vocab, bs=4, bptt=64, shuffle=True, encode_position=True, y_offset=0)
    pl_valid = MusicPreloader(items[:4], vocab, bs=4, bptt=64, shuffle=False, encode_position=True, y_offset=0)
    cbs = [EarlyStoppingCallback(monitor='mask_acc', patience=3), SaveModelCallback(name='remix_best')]
    learn.fit_one_cycle(3, 3e-3, pl, valid_batches=pl_valid, callbacks=cbs, valid_seed=1)
    print('remix recorder', learn.recorder)
    assert [r['epoch'] for r in learn.recorder] == [0, 1, 2]
    assert all(math.isfinite(r['valid_loss']) and 0. <= r['mask_acc'] <= 1. for r in learn.recorder)
    assert learn.recorder[-1]['valid_loss'] < learn.recorder[0]['valid_loss']
    best = torch.load(str(tmp_path / 'models' / 'remix_best.pth'), weights_only=False)
    for k, v in learn.model.state_dict().items():
        assert torch.equal(v, best['model'][k]), k
    # the reported value is the validation of the weights it belongs to
    i_best = int(np.argmin([r['valid_loss'] for r in learn.recorder]))
    assert learn.validate(pl_valid, seed=1) == pytest.approx([learn.recorder[i_best]['valid_loss'], learn.recorder[i_best]['mask_acc']],
                                                             abs=1e-12)
    item = MusicItem.from_file(os.path.join(golden_dir, 'uploadedMidi.mid'), vocab).trim_to_beat(8)
    notes = [i for i, t in enumerate(item.data) if vocab.note_range[0] <= t < vocab.note_range[1]]
    item.data[notes[::2]] = vocab.mask_idx
    out = learn.predict_mask(item, top_k=1, top_p=0.0)
    assert vocab.mask_idx not in list(out.data)
    # the trained encoder predicts far better than chance: its validation against the oracle on the trained weights
    from deepmusicgeneration_b200.preloader import mask_tfm
    vb = []
    for i, (xb, y) in enumerate(pl_valid):
        xm, ym = mask_tfm((xb['x'], y), (vocab.note_range[0], vocab.dur_range[1]), vocab.mask_idx, vocab.pad_idx, p=0.3, seed=100 + i)
        vb.append((xm.cpu(), ym.cpu(), xb['pos'].cpu()))
    torch.manual_seed(0)
    om = obert.get_multitask_model(len(vocab.itos), bert_config(), pad_idx=vocab.pad_idx)
    om.load_state_dict(learn.model.state_dict(), strict=False)
    ref_loss, ref_acc, ref_ms = ref.bert_validate(om, vb, vocab.pad_idx)
    got = learn._trainer.validate(vb)
    err = remix_logit_err(learn.model, om, vb)
    amb, kept = remix_ambiguous(om, vb, vocab.pad_idx, err), sum(m[1] for m in ref_ms)
    print('trained remix validate', got, ref_loss, ref_acc, 'logit err', err, 'ambiguous', amb, 'kept', kept)
    assert 0.1 < ref_acc < 0.99
    assert abs(got['valid_loss'] - ref_loss) < CE_TOL * max(1., abs(ref_loss))
    assert abs(got['mask_acc'] - ref_acc) <= len(vb) * amb / kept + 1e-12


# ---------------------------------------------------------------------------------------------------- 10. error paths
def test_error_paths_are_rejected_before_any_launch():
    from deepmusicgeneration_b200 import _lib
    lib = _lib.load()
    cfg = txl_config()
    _, _, tr = txl_pair(cfg, 2, 64)
    x, y = lm_batches(torch.Generator().manual_seed(0), 1, 2, 64)[0]
    torch.cuda.synchronize()
    n0 = lib.dmg_launch_count()
    # a bad batch anywhere in a list is refused before the first batch launches (and before the memory reset)
    with pytest.raises(ValueError, match=r'\[2, 64\]'):
        tr.validate([(x, y), (x[:, :32], y[:, :32])])
    with pytest.raises(ValueError, match=r'\[2, 64\]'):
        tr.validate([(x, y), (x, y), (x, y[:1])], reset=False)
    assert lib.dmg_launch_count() == n0
    h = tr.e.h
    xd, yd = x.cuda(), y.cuda()
    torch.cuda.synchronize()
    n0 = lib.dmg_launch_count()
    # a fresh state: close any open table first
    assert lib.dmg_train_eval_begin(h, 1) == 0
    buf = (C.c_double * 6)()
    assert lib.dmg_train_eval_end(h, C.cast(buf, C.c_void_p), 0, _stream_ptr()) == 0
    assert lib.dmg_train_eval_batch(h, _ptr(xd), None, _ptr(yd), _stream_ptr()) != 0
    assert b'dmg_train_eval_begin first' in lib.dmg_last_error()
    assert lib.dmg_train_eval_begin(h, 0) != 0 and b'max_batches' in lib.dmg_last_error()
    assert lib.dmg_train_eval_begin(h, 1) == 0
    assert lib.dmg_train_eval_batch(h, _ptr(xd), None, None, _stream_ptr()) != 0 and b'null' in lib.dmg_last_error()
    n1 = lib.dmg_launch_count()
    assert lib.dmg_train_eval_batch(h, _ptr(xd), None, _ptr(yd), _stream_ptr()) == 0
    assert lib.dmg_launch_count() > n1
    n2 = lib.dmg_launch_count()
    assert lib.dmg_train_eval_batch(h, _ptr(xd), None, _ptr(yd), _stream_ptr()) != 0
    assert b'max_batches' in lib.dmg_last_error()
    assert lib.dmg_train_eval_end(h, C.cast(buf, C.c_void_p), 2, _stream_ptr()) != 0 and b'1 batches' in lib.dmg_last_error()
    assert lib.dmg_launch_count() == n2
    assert n1 == n0
    tr.close()
    cfgb = bert_config()
    _, _, trb = bert_pair(cfgb, 2, 64)
    xb, yb, pb = masked_batch(torch.Generator().manual_seed(1), 2, 64)
    xbd, ybd = xb.cuda(), yb.cuda()
    assert lib.dmg_train_eval_begin(trb.e.h, 2) == 0
    n0 = lib.dmg_launch_count()
    assert lib.dmg_train_eval_batch(trb.e.h, _ptr(xbd), None, _ptr(ybd), _stream_ptr()) != 0
    assert b'pos is required' in lib.dmg_last_error()
    assert lib.dmg_launch_count() == n0
    with pytest.raises(DmgError, match='pos is required'):
        trb.validate([(xb, yb)])
    trb.close()


# ---------------------------------------------------------------------------------------------------- 9. two GPUs
def _dp_worker(rank, world, port, q):
    os.environ.update(RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE=str(world), MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    from deepmusicgeneration_b200 import sharding
    try:
        sharding.init_distributed(backend='nccl')
        torch.cuda.set_device(rank)
        cfg = bert_config()
        torch.manual_seed(0)
        om = obert.get_multitask_model(V, cfg, drop_mult=0., pad_idx=PAD)
        pm = get_multitask_model(V, cfg, pad_idx=PAD, dtype='bf16', device=rank, max_batch=2, max_seq=64, init=False)
        pm.load_state_dict(om.state_dict())
        tr = RemixTrainer(pm, 2, 64, cfg, pad_idx=PAD, drop_mult=0., distributed=True)
        g = torch.Generator().manual_seed(10 + rank)             # every rank validates its own shard
        vb = [masked_batch(g, 2, 64) for _ in range(3)]
        got = tr.validate(vb)
        tr.distributed = False                                   # this rank's own values
        own = tr.validate(vb)
        tr.distributed = True
        try:                                                     # unequal batch counts are refused on every rank, no hang
            tr.validate(vb[:rank + 1])
            raise AssertionError('unequal batch counts were accepted')
        except ValueError as e:
            assert 'same number of batches' in str(e)
        q.put((rank, ([got['valid_loss'], got['mask_acc']], [own['valid_loss'], own['mask_acc']])))
        tr.close()
    except Exception as e:
        q.put((rank, repr(e)))
    finally:
        import torch.distributed as dist
        if dist.is_initialized():
            dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs >= 2 GPUs')
def test_two_gpu_validation_is_identical_on_both_ranks_and_the_mean_of_theirs():
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
    assert all(isinstance(v, tuple) for v in res.values()), res
    (g0, o0), (g1, o1) = res[0], res[1]
    assert g0 == g1                                              # bit-identical (Python floats from the same float64 bits)
    for k in range(2):
        assert g0[k] == pytest.approx((o0[k] + o1[k]) / 2, rel=1e-12)
        assert o0[k] != o1[k]
