"""Epoch-end callbacks of ``fit_one_cycle(..., valid_batches=..., callbacks=[...])``: fastai 1.0.61's ``EarlyStoppingCallback`` and
``SaveModelCallback`` (fastai/callbacks/tracker.py), which the reference's genre notebook trains with
(``EarlyStoppingCallback(monitor='valid_loss', patience=5, min_delta=0.01)``, ``SaveModelCallback(name='lakh_genre_model')``).

fastai builds them with the learner as first argument; here the learner hands itself over in ``on_train_begin``.  The rules are
fastai's ``TrackerCallback``:

- ``mode='auto'`` compares with ``<`` when the monitored name contains "loss", with ``>`` otherwise; ``'min'`` / ``'max'`` force it.
- The monitored value is read from the epoch's recorder row; an epoch without validation (``valid_loss`` None) is skipped.
- A NaN never counts as an improvement (``np.less`` / ``np.greater`` are False for it).
"""
import os
import warnings

import numpy as np
import torch


def _distributed():
    return torch.distributed.is_available() and torch.distributed.is_initialized()


class TrackerCallback:
    "fastai TrackerCallback: the monitored quantity, its comparison and the best value so far."
    def __init__(self, monitor='valid_loss', mode='auto'):
        if mode not in ('auto', 'min', 'max'):
            warnings.warn(f'{type(self).__name__} mode {mode} is invalid, falling back to "auto" mode.')
            mode = 'auto'
        self.monitor, self.mode = monitor, mode
        self.operator = {'min': np.less, 'max': np.greater}.get(mode, np.less if 'loss' in monitor else np.greater)
        self.learn, self.best = None, None

    def on_train_begin(self, learn):
        self.learn = learn
        self.best = float('inf') if self.operator == np.less else -float('inf')

    def get_monitor_value(self, row):
        if row.get('valid_loss') is None:
            return None
        value = row.get(self.monitor)
        if value is None:
            warnings.warn(f'{type(self).__name__} conditioned on metric `{self.monitor}` which is not available. '
                          f'Available metrics are: {", ".join(k for k in row if k not in ("epoch", "time"))}')
        return value

    def on_epoch_end(self, epoch, row):
        "Returns True to stop training."
        return False

    def on_train_end(self):
        pass


class EarlyStoppingCallback(TrackerCallback):
    """Stop when the monitored value has not improved by more than `min_delta` for more than `patience` epochs in a row
    (fastai: ``operator(current - min_delta, best)`` with min_delta negated for "less is better")."""
    def __init__(self, monitor='valid_loss', mode='auto', min_delta=0., patience=0):
        super().__init__(monitor=monitor, mode=mode)
        self.min_delta, self.patience = min_delta, patience
        if self.operator == np.less:
            self.min_delta *= -1
        self.wait = 0

    def on_train_begin(self, learn):
        self.wait = 0
        super().on_train_begin(learn)

    def on_epoch_end(self, epoch, row):
        current = self.get_monitor_value(row)
        if current is None:
            return False
        if self.operator(current - self.min_delta, self.best):
            self.best, self.wait = current, 0
            return False
        self.wait += 1
        if self.wait > self.patience:
            print(f'Epoch {epoch}: early stopping')
            return True
        return False


class SaveModelCallback(TrackerCallback):
    """Save the model and its Adam state (``learn.save``) to ``<data.path>/models/<name>.pth`` whenever the monitored value improves
    (``every='improvement'``), or to ``<name>_<epoch>.pth`` after every epoch (``every='epoch'``).  With 'improvement', the end of
    training loads the best file back into the model and the live trainer (weights and Adam state) and refreshes the inference
    caches.  Data parallel (torch.distributed initialised): as in fastai, only rank 0 writes the file, and every rank waits at a
    barrier before it reads the best file back."""
    def __init__(self, monitor='valid_loss', mode='auto', every='improvement', name='bestmodel'):
        super().__init__(monitor=monitor, mode=mode)
        if every not in ('improvement', 'epoch'):
            warnings.warn(f'SaveModel every {every} is invalid, falling back to "improvement".')
            every = 'improvement'
        self.every, self.name = every, name

    def path(self, name=None):
        root = getattr(getattr(self.learn, 'data', None), 'path', '') or '.'
        return os.path.join(str(root), 'models', f'{name or self.name}.pth')

    def _save(self, name):
        if _distributed() and torch.distributed.get_rank() != 0:
            return
        file = self.path(name)
        os.makedirs(os.path.dirname(file), exist_ok=True)
        self.learn.save(file)

    def on_epoch_end(self, epoch, row):
        if self.every == 'epoch':
            self._save(f'{self.name}_{epoch}')
            return False
        current = self.get_monitor_value(row)
        if current is not None and self.operator(current, self.best):
            print(f'Better model found at epoch {epoch} with {self.monitor} value: {current}.')
            self.best = current
            self._save(self.name)
        return False

    def on_train_end(self):
        if self.every != 'improvement':
            return
        if _distributed():
            torch.distributed.barrier()
        if os.path.isfile(self.path()):
            self.learn.load(self.path())
