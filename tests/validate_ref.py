"""Reference of validation while training: what fastai 1.0.61 does around the reference models, restated from its published source
(fastai is not vendored; the reference repository only calls it).  TEST INFRASTRUCTURE (plain PyTorch, CPU).

- ``basic_train.validate``: model.eval(); per batch ``loss_func(model(xb), yb)`` and ``n = first_el(yb).shape[0]``; the epoch's
  validation loss is ``np.average(losses, weights=n)``.
- ``metrics.accuracy`` (the language model's metric): ``(input.argmax(-1) == targs).float().mean()`` over all positions.
- The remix learner's ``mask_acc`` (deep_music_remix.py:2743-2760) averaged by ``AverageMultiMetric`` (:2762-2779): accuracy over the
  positions whose target is not pad_idx; per batch ``val += n * metric`` (all-reduced over ranks first), epoch value ``val / sum n``.
- ``CrossEntropyFlat(ignore_index=pad_idx)`` gives NaN for a batch with nothing to predict, and the NaN carries into the average.
- ``callbacks/tracker.py``: ``TrackerCallback`` (mode 'auto' = less is better when the name contains "loss"),
  ``EarlyStoppingCallback`` (``operator(current - min_delta, best)`` with min_delta negated for "less"; stop once more than
  `patience` epochs passed without that), ``SaveModelCallback(every='improvement')`` (save when ``operator(current, best)``).

Parity status: unpinned at the fastai boundary (the reference stores no validation artefacts); this file is the definition the
CUDA path is tested against.
"""
import numpy as np
import torch


def batch_metrics(logits, y, ignore=None):
    """(ce_sum, kept, correct) of one batch in float64: ce_sum = sum over kept rows of logsumexp(row) - row[target]; kept = rows whose
    target is not `ignore` (all rows when None); correct = kept rows whose FIRST maximal logit is the target.  Targets outside
    [0, V) are clamped, as the training loss does."""
    lg = logits.reshape(-1, logits.shape[-1]).double()
    V = lg.shape[1]
    t = y.reshape(-1).long()
    keep = torch.ones_like(t, dtype=torch.bool) if ignore is None else t != ignore
    tc = t.clamp(0, V - 1)
    nll = torch.logsumexp(lg, -1) - lg.gather(1, tc[:, None])[:, 0]
    mx = lg.max(-1, keepdim=True).values
    first = torch.where(lg == mx, torch.arange(V)[None, :], torch.full_like(lg, V, dtype=torch.long)).min(-1).values
    return float(nll[keep].sum()), float(keep.sum()), float(((first == tc) & keep).sum())


def batch_values(m, rows=None):
    "(loss, metric) of one batch from its metrics: over `rows` positions (language model), or over the kept ones (rows=None)."
    ce, kept, correct = m
    n = rows if rows is not None else kept
    with np.errstate(invalid='ignore', divide='ignore'):
        return np.float64(ce) / np.float64(n), np.float64(correct) / np.float64(n)


def weighted_mean(values, weights):
    "np.average(values, weights) - NaN in any value gives NaN"
    v, w = np.asarray(values, dtype=np.float64), np.asarray(weights, dtype=np.float64)
    return float((v * w).sum() / w.sum())


def txl_validate(model, batches, reset=True):
    """fastai validate of oracle.txl's SequentialRNN: eval mode, memory carried across batches; returns (valid_loss, accuracy) and the
    per-batch metrics.  batches: (x, y) or ({'x', 'pos'}, y)."""
    model.eval()
    if reset:
        model.reset()
    per, ms = [], []
    with torch.no_grad():
        for xb, y in batches:
            logits = model(xb)[0]
            m = batch_metrics(logits, y)
            ms.append(m)
            per.append(batch_values(m, rows=y.numel()))
    n = [y.shape[0] for _, y in batches]
    return weighted_mean([p[0] for p in per], n), weighted_mean([p[1] for p in per], n), ms


def bert_validate(model, batches, pad_idx):
    """fastai validate of oracle.bert's MultiTransformer on the mask task: eval mode; returns (valid_loss, mask_acc) and the per-batch
    metrics.  batches: (x, y, pos) already masked."""
    model.eval()
    per, ms = [], []
    with torch.no_grad():
        for x, y, pos in batches:
            logits = model({'msk': {'x': x, 'pos': pos.clone()}})['msk']
            m = batch_metrics(logits, y, ignore=pad_idx)
            ms.append(m)
            per.append(batch_values(m))
    n = [y.shape[0] for _, y, _ in batches]
    return weighted_mean([p[0] for p in per], n), weighted_mean([p[1] for p in per], n), ms


def _less(monitor, mode):
    return mode == 'min' or (mode == 'auto' and 'loss' in monitor)


def early_stop_epoch(values, monitor='valid_loss', mode='auto', min_delta=0., patience=0):
    "The epoch after which EarlyStoppingCallback stops training over the monitored `values`, or None."
    less = _less(monitor, mode)
    op = np.less if less else np.greater
    md = -min_delta if less else min_delta
    best, wait = (np.inf if less else -np.inf), 0
    for epoch, cur in enumerate(values):
        if op(cur - md, best):
            best, wait = cur, 0
        else:
            wait += 1
            if wait > patience:
                return epoch
    return None


def save_epochs(values, monitor='valid_loss', mode='auto'):
    "The epochs at which SaveModelCallback(every='improvement') saves over the monitored `values`."
    op = np.less if _less(monitor, mode) else np.greater
    best, out = (np.inf if _less(monitor, mode) else -np.inf), []
    for epoch, cur in enumerate(values):
        if op(cur, best):
            best = cur
            out.append(epoch)
    return out
