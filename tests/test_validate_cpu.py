"""CPU checks of validation while training: the reference's metrics (validate_ref.py) against direct torch computations, the
batch-size weighting, and the product's EarlyStopping / SaveModel callbacks against the reference's restatement of fastai's
TrackerCallback rules on scripted metric sequences."""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import validate_ref as ref
from deepmusicgeneration_b200.callbacks import EarlyStoppingCallback, SaveModelCallback


def test_metrics_match_torch_with_first_index_ties():
    g = torch.Generator().manual_seed(0)
    rows, V = 203, 37
    lg = torch.randn(rows, V, generator=g)
    y = torch.randint(0, V, (rows,), generator=g)
    # exact ties: the maximum appears twice; the target is the LATER copy on even rows, the earlier one on odd rows
    for r in range(0, rows, 3):
        a, b = sorted(torch.randperm(V, generator=g)[:2].tolist())
        lg[r, a] = lg[r, b] = lg[r].max() + 1.
        y[r] = b if r % 2 == 0 else a
    ce, kept, correct = ref.batch_metrics(lg, y)
    assert kept == rows
    assert ce == pytest.approx(F.cross_entropy(lg.double(), y, reduction='sum').item(), rel=1e-12)
    assert correct == (lg.argmax(-1) == y).sum().item()
    tie_rows = list(range(0, rows, 3))
    assert all((lg[r].argmax() != y[r]) == (r % 2 == 0) for r in tie_rows)
    # ignore index: the mean over the kept rows is torch's CrossEntropyFlat(ignore_index)
    y2 = y.clone()
    y2[::4] = 5
    ce, kept, correct = ref.batch_metrics(lg, y2, ignore=5)
    keep = y2 != 5
    assert kept == keep.sum().item()
    loss, acc = ref.batch_values((ce, kept, correct))
    assert loss == pytest.approx(F.cross_entropy(lg.double(), y2, ignore_index=5).item(), rel=1e-12)
    assert acc == pytest.approx((lg.argmax(-1) == y2)[keep].float().mean().item(), rel=1e-6)


def test_all_rows_ignored_gives_nan_like_torch():
    lg = torch.randn(16, 9)
    y = torch.full((16,), 2)
    m = ref.batch_metrics(lg, y, ignore=2)
    assert m[1] == 0 and m[2] == 0
    loss, acc = ref.batch_values(m)
    assert math.isnan(loss) and math.isnan(acc)
    assert math.isnan(F.cross_entropy(lg, y, ignore_index=2).item())
    # and the NaN carries into the epoch average
    assert math.isnan(ref.weighted_mean([1.0, loss], [4, 4]))


def test_out_of_range_targets_are_clamped():
    lg = torch.randn(4, 6)
    y = torch.tensor([-3, 7, 0, 5])
    ce, kept, correct = ref.batch_metrics(lg, y)
    yc = y.clamp(0, 5)
    assert ce == pytest.approx(F.cross_entropy(lg.double(), yc, reduction='sum').item(), rel=1e-12)
    assert correct == (lg.argmax(-1) == yc).sum().item()


def test_unequal_batch_sizes_are_weighted():
    vals, n = [2.0, 3.0, 5.0], [4, 1, 3]
    assert ref.weighted_mean(vals, n) == pytest.approx(np.average(vals, weights=n))
    assert ref.weighted_mean(vals, n) != pytest.approx(np.mean(vals))
    # the language-model validation of two batches of different sizes equals the positions-weighted torch mean
    g = torch.Generator().manual_seed(1)
    batches = [(torch.randn(b, 8, 11, generator=g), torch.randint(0, 11, (b, 8), generator=g)) for b in (3, 1)]
    per = [ref.batch_values(ref.batch_metrics(lg, y), rows=y.numel()) for lg, y in batches]
    loss = ref.weighted_mean([p[0] for p in per], [3, 1])
    all_lg = torch.cat([lg.reshape(-1, 11) for lg, _ in batches]).double()
    all_y = torch.cat([y.reshape(-1) for _, y in batches])
    assert loss == pytest.approx(F.cross_entropy(all_lg, all_y).item(), rel=1e-12)   # equal bptt: weighting by bs = by positions


def test_trainer_average_is_the_weighted_mean():
    from deepmusicgeneration_b200.training import TXLTrainer

    class Stub:
        distributed = False
    per = np.array([[1.0, 0.5], [4.0, 0.25]])
    got = TXLTrainer._average(Stub(), per, [2, 6])
    assert got == pytest.approx([ref.weighted_mean(per[:, 0], [2, 6]), ref.weighted_mean(per[:, 1], [2, 6])], rel=1e-15)
    got = TXLTrainer._average(Stub(), np.array([[1.0, 0.5], [np.nan, np.nan]]), [2, 2])
    assert all(math.isnan(v) for v in got)


class FakeLearner:
    "records what SaveModelCallback saves / loads"
    def __init__(self, path):
        self.data = type('D', (), {'path': str(path)})()
        self.saved, self.saved_at, self.loaded, self.epoch = [], [], [], None

    def save(self, file):
        open(file, 'w').close()
        self.saved.append(file)
        self.saved_at.append(self.epoch)

    def load(self, file):
        self.loaded.append(file)


def run_callbacks(cbs, learn, rows):
    "the learners' epoch loop: callbacks see one recorder row per epoch; returns the epochs run"
    for cb in cbs:
        cb.on_train_begin(learn)
    ran = 0
    for epoch, row in enumerate(rows):
        ran += 1
        learn.epoch = epoch
        stop = False
        for cb in cbs:
            stop = bool(cb.on_epoch_end(epoch, row)) or stop
        if stop:
            break
    for cb in cbs:
        cb.on_train_end()
    return ran


SEQS = {
    'valid_loss': [3.0, 2.5, 2.495, 2.49, 2.6, 2.3, 2.31, 2.32, 2.33, 2.34, 2.2],
    'accuracy': [0.1, 0.2, 0.205, 0.19, 0.3, 0.3, 0.29, 0.31, 0.2, 0.1, 0.1],
}


@pytest.mark.parametrize('monitor', ['valid_loss', 'accuracy'])
@pytest.mark.parametrize('min_delta,patience', [(0., 0), (0., 2), (0.01, 0), (0.01, 1), (0.01, 5), (0.2, 3)])
def test_early_stopping_matches_the_tracker_rules(tmp_path, monitor, min_delta, patience):
    vals = SEQS[monitor]
    rows = [{'epoch': i, 'train_loss': 1., 'valid_loss': SEQS['valid_loss'][i], 'accuracy': SEQS['accuracy'][i], 'time': 0.}
            for i in range(len(vals))]
    want = ref.early_stop_epoch(vals, monitor, 'auto', min_delta, patience)
    ran = run_callbacks([EarlyStoppingCallback(monitor=monitor, min_delta=min_delta, patience=patience)], FakeLearner(tmp_path), rows)
    assert ran == (len(vals) if want is None else want + 1)
    # both ways of stopping occur over the parameter grid
    if (monitor, min_delta, patience) == ('valid_loss', 0.01, 0):
        assert want == 2
    if (monitor, min_delta, patience) == ('valid_loss', 0., 2):
        assert want == 8
    if (monitor, min_delta, patience) == ('valid_loss', 0.01, 5):
        assert want is None


def test_early_stopping_explicit_mode_and_missing_validation(tmp_path):
    vals = [0.5, 0.4, 0.6, 0.7]
    rows = [{'epoch': i, 'valid_loss': 1.0, 'accuracy': v} for i, v in enumerate(vals)]
    ran = run_callbacks([EarlyStoppingCallback(monitor='accuracy', mode='min', patience=0)], FakeLearner(tmp_path), rows)
    assert ran == ref.early_stop_epoch(vals, 'accuracy', 'min', 0., 0) + 1 == 3
    # epochs without validation (valid_loss None) never count
    rows = [{'epoch': i, 'valid_loss': None, 'accuracy': None} for i in range(4)]
    assert run_callbacks([EarlyStoppingCallback(patience=0)], FakeLearner(tmp_path), rows) == 4


@pytest.mark.parametrize('monitor', ['valid_loss', 'accuracy'])
def test_save_model_saves_exactly_at_improvements_and_loads_the_best(tmp_path, monitor):
    vals = SEQS[monitor] + [float('nan')]
    rows = [{'epoch': i, 'valid_loss': v if monitor == 'valid_loss' else 1., 'accuracy': v} for i, v in enumerate(vals)]
    learn = FakeLearner(tmp_path)
    cb = SaveModelCallback(monitor=monitor, name='best')
    run_callbacks([cb], learn, rows)
    want = ref.save_epochs(vals, monitor)
    assert learn.saved_at == want and want[0] == 0 and len(want) >= 3
    assert set(learn.saved) == {str(tmp_path / 'models' / 'best.pth')}
    assert learn.loaded == [str(tmp_path / 'models' / 'best.pth')]
    assert cb.best == (min if monitor == 'valid_loss' else max)(v for v in vals if not math.isnan(v))


def test_save_model_every_epoch(tmp_path):
    learn = FakeLearner(tmp_path)
    run_callbacks([SaveModelCallback(every='epoch', name='m')], learn, [{'valid_loss': 1.}, {'valid_loss': 2.}])
    assert learn.saved == [str(tmp_path / 'models' / 'm_0.pth'), str(tmp_path / 'models' / 'm_1.pth')]
    assert learn.loaded == []


def test_save_model_under_data_parallel_saves_on_rank_0_only_and_waits_before_loading(tmp_path, monkeypatch):
    from deepmusicgeneration_b200 import callbacks
    events = []
    monkeypatch.setattr(callbacks, '_distributed', lambda: True)
    monkeypatch.setattr(torch.distributed, 'barrier', lambda *a, **k: events.append('barrier'))
    rows = [{'valid_loss': v} for v in (3., 2., 2.5)]
    for rank in (0, 1):
        monkeypatch.setattr(torch.distributed, 'get_rank', lambda *a, **k: rank)
        learn = FakeLearner(tmp_path)                    # one shared path: rank 1 reads what rank 0 wrote
        orig_load = learn.load
        learn.load = lambda f: (events.append('load'), orig_load(f))
        events.clear()
        run_callbacks([SaveModelCallback(name='best')], learn, rows)
        assert learn.saved_at == ([0, 1] if rank == 0 else [])
        assert events == ['barrier', 'load']
