"""Training step of the Transformer-XL path on the CUDA library: the host-side mirror of what fastai's ``Learner.fit`` does
for one batch around the reference model (SURVEY.md 3.3, App. A.7):

    model.train(); out = model(x)                      # deep_music_genre.py:1617-1647, dropout + rand_window_mask (:1586-1590)
    loss = CrossEntropyFlat(out[0], y) + AR + TAR      # fastai RNNTrainer(alpha=2, beta=1)
    loss.backward(); clip; Adam(betas=(0.9, 0.99)) with true_wd=0.01; one-cycle schedule

All arithmetic runs in libdmg_b200.so (``dmg_train_*``); PyTorch owns the flat gradient tensor (so that
``torch.distributed`` can all-reduce it over NCCL/NVLink), the streams and the rendezvous.  Data-parallel training shards
the batch over ranks; the only collective is the gradient all-reduce, issued per bucket of layers on a side stream while
the backward pass of the earlier layers is still running.
"""
import ctypes as C
import math

import numpy as np
import torch

from . import _lib
from ._lib import check
from .model import _ptr, _stream_ptr


def rand_window_mask_size(max_size=None, p=0.2, is_eval=False, rng=np.random):
    "The (win_size, k) pair rand_window_mask draws on the host (deep_music_genre.py:1586-1590)."
    if is_eval or rng.rand() >= p or max_size is None:
        return (1, 1)
    return (rng.randint(0, max_size) + 1, 0)


def one_cycle_lr(step, total, lr_max, div_factor=25., pct_start=0.3, final_div=None, moms=(0.95, 0.85)):
    "fastai fit_one_cycle: cosine lr_max/div -> lr_max over pct_start, then cosine down to lr_max/(div*1e4); momentum mirrored."
    final_div = final_div or div_factor * 1e4
    a = int(total * pct_start)
    def cos(start, end, pct): return end + (start - end) / 2 * (math.cos(math.pi * pct) + 1)
    if step < a:
        pct = step / max(1, a)
        return cos(lr_max / div_factor, lr_max, pct), cos(moms[0], moms[1], pct)
    pct = (step - a) / max(1, total - a)
    return cos(lr_max, lr_max / final_div, pct), cos(moms[1], moms[0], pct)


def _tuples(batches):
    """(iterator of (x, y, pos or None), upper bound of its length) for a list of (x, y[, pos]) / ({'x', 'pos'}, y) batches or a
    MusicPreloader (whose len() counts items, not batches)."""
    from .preloader import MusicPreloader
    if isinstance(batches, MusicPreloader):
        n = batches.n_batches
    else:
        batches = batches if hasattr(batches, '__len__') else list(batches)
        n = len(batches)

    def gen():
        for b in batches:
            if isinstance(b[0], dict):
                yield b[0]['x'], b[1], b[0].get('pos')
            else:
                yield b[0], b[1], (b[2] if len(b) > 2 else None)
    return gen(), n


class TXLTrainer:
    """One training step at a time.  ``model`` is the ``SequentialRNN`` mirror from ``model.get_language_model`` (bf16).

    trainer = TXLTrainer(model, bs=32, bptt=512, config=config)       # config carries the *_p dropouts and mask_steps
    trainer.reset()                                                     # RNNTrainer.on_epoch_begin
    trainer.step(x, y, lr=5e-4)                                         # forward + backward + (all-reduce) + Adam
    trainer.losses()                                                    # {'ce':.., 'ar':.., 'tar':.., 'loss':.., 'grad_norm':..}
    """
    def __init__(self, model, bs, bptt, config, drop_mult=1., alpha=2., beta=1., seed=0, process_group=None, bucket_layers=4,
                 distributed=None, wire='bf16', rank_seed=True, pad_idx=0):
        self.model, self.e = model, model._e
        self.lib = self.e.lib
        self.bs, self.bptt = bs, bptt
        self.n_layers = self.e.cfg.n_layers
        self.mask_steps = config.get('mask_steps', 1)
        self.training = True
        self.step_count = 0
        self.pg = process_group
        if distributed is None:
            distributed = torch.distributed.is_available() and torch.distributed.is_initialized() and \
                torch.distributed.get_world_size(process_group) > 1
        self.distributed = distributed
        self.world = torch.distributed.get_world_size(process_group) if distributed else 1
        self.bucket_layers = max(1, bucket_layers)
        self.wire = wire if distributed else 'none'
        assert self.wire in ('bf16', 'f32', 'none')
        if distributed and rank_seed:
            # independent dropout masks per rank, like the reference's DDP processes (each draws from its own generator)
            seed = (int(seed) + 0x9E3779B97F4A7C15 * torch.distributed.get_rank(process_group)) % (1 << 64)
        tc = _lib.TrainConfig()
        tc.batch, tc.bptt = bs, bptt
        for k in ('resid_p', 'attn_p', 'ff_p', 'embed_p', 'output_p'):
            setattr(tc, k, float(config.get(k, 0.)) * drop_mult)
        tc.alpha, tc.beta, tc.seed, tc.pad_idx = alpha, beta, seed, pad_idx
        self.tc = tc
        n = self.lib.dmg_train_param_count(self.e.h)
        if n <= 0:
            raise RuntimeError('dmg_train_param_count failed')
        with torch.cuda.device(self.e.device):
            self.grad = torch.zeros(n, device=self.e.device, dtype=torch.float32)      # torch-owned: NCCL all-reduces it
            check(self.lib.dmg_train_create(self.e.h, C.byref(tc), _ptr(self.grad)), 'dmg_train_create')
            self.comm_stream = torch.cuda.Stream(device=self.e.device) if distributed else None
            self.wire_buf = torch.empty(n, device=self.e.device, dtype=torch.bfloat16) if self.wire == 'bf16' else None
        self._keep = None
        self._comm_events = None
        self.buckets = self._bucket_plan()

    def close(self):
        if self.e.h:
            self.lib.dmg_train_destroy(self.e.h)

    def reset(self):
        check(self.lib.dmg_train_reset(self.e.h), 'dmg_train_reset')

    def train(self, mode=True):
        self.training = bool(mode)
        return self

    def eval(self):
        return self.train(False)

    # ------------------------------------------------------------------ pieces of one step
    def forward(self, x, y=None, pos=None, mask_size=None):
        dev = self.e.device
        x = x.to(dev, torch.int64).contiguous()
        y = y.to(dev, torch.int64).contiguous() if y is not None else None
        pos = pos.to(dev, torch.int64).contiguous() if pos is not None else None
        assert tuple(x.shape) == (self.bs, self.bptt), f'expected [{self.bs}, {self.bptt}] tokens, got {tuple(x.shape)}'
        if mask_size is None:
            mask_size = rand_window_mask_size(self.mask_steps, is_eval=not self.training)
        self._keep = (x, y, pos)            # the library reads ids / pos again in backward
        with torch.cuda.device(dev):
            check(self.lib.dmg_train_forward(self.e.h, _ptr(x), _ptr(pos), _ptr(y), int(mask_size[0]), int(mask_size[1]),
                                             int(self.training), self.step_count, _stream_ptr()), 'dmg_train_forward')
        return mask_size

    def _bucket_plan(self):
        """(layer_hi, layer_lo) slices of one backward pass.  One rank: a single slice.  Data parallel: the head + the two top layers
        go out first (their all-reduce starts while almost the whole backward is still ahead), then `bucket_layers`-layer buckets,
        and the LAST bucket - the only one whose all-reduce nothing is left to hide behind - holds at most two layers."""
        L = self.n_layers
        if not self.distributed:
            return [(L, 0)]
        cuts = [L]
        first = min(2, L)
        if L - first > 0:
            cuts.append(L - first)
        tail = min(2, cuts[-1])
        while cuts[-1] - self.bucket_layers > tail:
            cuts.append(cuts[-1] - self.bucket_layers)
        if cuts[-1] > tail:
            cuts.append(tail)
        if cuts[-1] != 0:
            cuts.append(0)
        return list(zip(cuts[:-1], cuts[1:]))

    def describe_exchange(self):
        if not self.distributed:
            return 'single rank, no gradient exchange'
        return (f'flat gradient all-reduced over NCCL as {self.wire} in {len(self.buckets)} buckets {self.buckets} (layer slices, '
                f'issued on a side stream as each slice of the backward pass completes), 1/{self.world} folded into Adam')

    def _exchange(self, off, cnt):
        "all-reduce (SUM) of grad[off:off+cnt] on the communication stream, in the wire format"
        h, cs = self.e.h, C.c_void_p(self.comm_stream.cuda_stream)
        if self.wire == 'bf16':
            w = self.wire_buf[off:off + cnt]
            check(self.lib.dmg_train_grad_pack(h, off, cnt, _ptr(w), cs), 'dmg_train_grad_pack')
            torch.distributed.all_reduce(w, group=self.pg)
            check(self.lib.dmg_train_grad_unpack(h, off, cnt, _ptr(w), cs), 'dmg_train_grad_unpack')
        else:
            torch.distributed.all_reduce(self.grad[off:off + cnt], group=self.pg)

    def backward(self):
        "loss.backward(); with >1 rank the all-reduce of each bucket of layers overlaps the backward of the next bucket."
        dev = self.e.device
        prof = self._comm_events
        with torch.cuda.device(dev):
            for hi, lo in self.buckets:
                check(self.lib.dmg_train_backward(self.e.h, hi, lo, _stream_ptr()), 'dmg_train_backward')
                if self.distributed:
                    off, cnt = C.c_int64(), C.c_int64()
                    check(self.lib.dmg_train_grad_span(self.e.h, hi, lo, C.byref(off), C.byref(cnt)), 'dmg_train_grad_span')
                    if cnt.value:
                        ev = torch.cuda.Event()
                        ev.record(torch.cuda.current_stream())
                        self.comm_stream.wait_event(ev)
                        with torch.cuda.stream(self.comm_stream):
                            if prof is not None:
                                e0 = torch.cuda.Event(enable_timing=True); e0.record()
                            self._exchange(off.value, cnt.value)
                            if prof is not None:
                                e1 = torch.cuda.Event(enable_timing=True); e1.record()
                                prof['buckets'].append((hi, lo, cnt.value, e0, e1))
            if self.distributed:
                if prof is not None:
                    prof['bwd_end'] = torch.cuda.Event(enable_timing=True); prof['bwd_end'].record()
                torch.cuda.current_stream().wait_stream(self.comm_stream)
                if prof is not None:
                    prof['joined'] = torch.cuda.Event(enable_timing=True); prof['joined'].record()

    def profile_comm(self, step_fn, reps=3):
        """Device-timed view of the gradient exchange over `reps` steps: per bucket the all-reduce time (pack + NCCL + unpack on the
        communication stream) and `exposed_ms` = how long the compute stream waited for the last bucket after backward ended."""
        if not self.distributed:
            return None
        acc, exposed = {}, 0.
        for _ in range(reps):
            self._comm_events = {'buckets': []}
            step_fn()
            torch.cuda.synchronize(self.e.device)
            p = self._comm_events
            for hi, lo, cnt, e0, e1 in p['buckets']:
                a = acc.setdefault((hi, lo), {'layers': [hi, lo], 'elements': cnt, 'ms': 0.})
                a['ms'] += e0.elapsed_time(e1) / reps
            exposed += p['bwd_end'].elapsed_time(p['joined']) / reps
        self._comm_events = None
        bytes_per = 2 if self.wire == 'bf16' else 4
        out = {'wire': self.wire, 'exposed_ms': exposed, 'buckets': list(acc.values()),
               'bytes_per_step': int(sum(a['elements'] for a in acc.values()) * bytes_per)}
        return out

    def optimizer_step(self, lr, betas=(0.9, 0.99), eps=1e-8, wd=0.01, clip=0.5):
        with torch.cuda.device(self.e.device):
            check(self.lib.dmg_train_optimizer_step(self.e.h, lr, betas[0], betas[1], eps, wd, clip if clip else 0.,
                                                    1.0 / self.world, _stream_ptr()), 'dmg_train_optimizer_step')
        self.e.committed = False
        self.step_count += 1

    def step(self, x, y, pos=None, lr=5e-4, betas=(0.9, 0.99), eps=1e-8, wd=0.01, clip=0.5, mask_size=None):
        self.forward(x, y, pos, mask_size)
        self.backward()
        self.optimizer_step(lr, betas, eps, wd, clip)

    def losses(self):
        out = (C.c_float * 4)()
        with torch.cuda.device(self.e.device):
            check(self.lib.dmg_train_losses(self.e.h, out, _stream_ptr()), 'dmg_train_losses')
        ce, ar, tar, gn = (float(v) for v in out)
        return {'ce': ce, 'ar': ar, 'tar': tar, 'loss': ce + ar + tar, 'grad_norm': gn / self.world}

    # ------------------------------------------------------------------ fastai-style loop
    def fit_one_cycle(self, batches, max_lr=5e-4, wd=0.01, clip=0.5, moms=(0.95, 0.85), callback=None):
        "batches: a sequence of (x, y) or (x, y, pos); one pass = one cycle (fastai fit_one_cycle(1, max_lr))."
        total = len(batches)
        self.reset()
        for i, b in enumerate(batches):
            lr, mom = one_cycle_lr(i, total, max_lr, moms=moms)
            x, y = b[0], b[1]
            pos = b[2] if len(b) > 2 else None
            self.step(x, y, pos, lr=lr, betas=(mom, 0.99), wd=wd, clip=clip)
            if callback is not None:
                callback(i, self)

    # ------------------------------------------------------------------ validation
    def _check_shape(self, what, t):
        if t is not None and tuple(t.shape) != (self.bs, self.bptt):
            raise ValueError(f'validation batch: {what} must be [bs, bptt] = [{self.bs}, {self.bptt}] like the training batches, '
                             f'got {list(t.shape)}')

    def _batches(self, batches):
        """_tuples(batches); a list of batches has every shape checked here, before anything is launched (a MusicPreloader's batches
        are checked one by one as they come)."""
        it, n = _tuples(batches)
        from .preloader import MusicPreloader
        if not isinstance(batches, MusicPreloader):
            tuples = list(it)
            for x, y, pos in tuples:
                for what, t in (('x', x), ('y', y), ('pos', pos)):
                    self._check_shape(what, t)
            it = iter(tuples)
        return it, n

    def _eval_table(self, batches, n_max):
        """Forward-only eval-mode batches (x, y, pos) through dmg_train_eval_*: returns the per-batch table, float64 [n, 3] =
        (CE sum, kept targets, correct argmax).  One device-to-host copy at the end, no sync per batch."""
        dev, h = self.e.device, self.e.h
        keep = []
        with torch.cuda.device(dev):
            check(self.lib.dmg_train_eval_begin(h, max(1, n_max)), 'dmg_train_eval_begin')
            n = 0
            for x, y, pos in batches:
                for what, t in (('x', x), ('y', y), ('pos', pos)):
                    self._check_shape(what, t)
                x = x.to(dev, torch.int64).contiguous()
                y = y.to(dev, torch.int64).contiguous()
                pos = pos.to(dev, torch.int64).contiguous() if pos is not None else None
                keep.append((x, y, pos))          # the launches read them asynchronously
                check(self.lib.dmg_train_eval_batch(h, _ptr(x), _ptr(pos), _ptr(y), _stream_ptr()), 'dmg_train_eval_batch')
                n += 1
            tab = np.zeros((n, 3), dtype=np.float64)
            check(self.lib.dmg_train_eval_end(h, tab.ctypes.data_as(C.c_void_p), n, _stream_ptr()), 'dmg_train_eval_end')
        return tab

    def _average(self, per_batch, weights):
        """fastai's validate / AverageMetric: the batch-size-weighted mean of per-batch values ([n, k] float64).  Data parallel: the
        per-batch values are first averaged over the ranks (one all-reduce, as the reference's AverageMultiMetric does for its metric;
        here for the loss too, so that every rank holds the same bits and takes the same early-stopping decision)."""
        vals = torch.from_numpy(np.ascontiguousarray(per_batch, dtype=np.float64))
        if self.distributed:
            # the table all-reduce needs the same number of batches on every rank: check it first (max of n and of -n)
            n = torch.tensor([len(vals), -len(vals)], dtype=torch.int64, device=self.e.device)
            torch.distributed.all_reduce(n, op=torch.distributed.ReduceOp.MAX, group=self.pg)
            hi, lo = int(n[0]), -int(n[1])
            if hi != lo:
                raise ValueError(f'validation: the ranks validated between {lo} and {hi} batches; data-parallel validation needs the '
                                 f'same number of batches on every rank')
            if len(vals):
                d = vals.to(self.e.device)
                torch.distributed.all_reduce(d, group=self.pg)
                vals = (d / self.world).cpu()
        w = torch.as_tensor(np.asarray(weights, dtype=np.float64))
        if len(vals) == 0:
            return [float('nan')] * per_batch.shape[1]
        return [float(v) for v in (vals * w[:, None]).sum(0) / w.sum()]

    def validate(self, batches, reset=True):
        """fastai Learner.validate for the language model: model.eval() over `batches` - (x, y) or (x, y, pos) LongTensors [bs, bptt],
        or a MusicPreloader - with the training memory carried from batch to batch (``reset=True`` forgets it first, as fastai's
        RNNTrainer.on_epoch_begin does).  Returns {'valid_loss': mean CrossEntropyFlat, 'accuracy': fraction of positions whose
        argmax (first maximal logit) is the target}, each the batch-size-weighted mean over the batches.  Weights, optimizer state,
        step_count and losses() are left as they were."""
        it, n_max = self._batches(batches)
        if reset:
            self.reset()
        tab = self._eval_table(it, n_max)
        rows = float(self.bs * self.bptt)
        loss, acc = self._average(np.stack([tab[:, 0] / rows, tab[:, 2] / rows], 1), [self.bs] * len(tab))
        return {'valid_loss': loss, 'accuracy': acc}

    # ------------------------------------------------------------------ test / inspection helpers
    def grads(self):
        "name -> gradient (CPU fp32) in state-dict naming."
        out = {}
        for name, shape in self.e.weight_names().items():
            if name == '1.decoder.weight':
                continue
            a = torch.empty(shape, dtype=torch.float32)
            rc = self.lib.dmg_train_get_grad(self.e.h, name.encode(), C.c_void_p(a.data_ptr()), a.numel())
            if rc == 1:
                continue
            check(rc, f'dmg_train_get_grad({name})')
            out[name] = a
        return out

    def dropout_mask(self, site, layer, shape, step=None):
        "The mask (keep ? 1/(1-p) : 0) the kernels use at `site` of `layer` for step `step`."
        n = int(np.prod(shape))
        out = torch.empty(n, device=self.e.device, dtype=torch.float32)
        with torch.cuda.device(self.e.device):
            check(self.lib.dmg_train_dropout_mask(self.e.h, site, layer, self.step_count if step is None else step, _ptr(out), n,
                                                  _stream_ptr()), 'dmg_train_dropout_mask')
        return out.view(*shape)

    # ------------------------------------------------------------------ optimizer state (checkpoints)
    def opt_state_dict(self):
        """torch.optim.Adam-shaped state ({'state': {i: {'step', 'exp_avg', 'exp_avg_sq'}}, 'param_names': [...]}) - what fastai's
        Learner.save(with_opt=True) stores under 'opt' (deep_music_genre.py:1812-1821); parameters in state-dict order."""
        steps = int(self.lib.dmg_train_opt_steps(self.e.h, -1))
        names, state = [], {}
        for name, shape in self.e.weight_names().items():
            if name == '1.decoder.weight':
                continue
            m1, m2 = torch.empty(shape, dtype=torch.float32), torch.empty(shape, dtype=torch.float32)
            rc = self.lib.dmg_train_opt_state(self.e.h, name.encode(), 1, 0, C.c_void_p(m1.data_ptr()), m1.numel())
            if rc == 1:
                continue
            check(rc, f'dmg_train_opt_state({name})')
            check(self.lib.dmg_train_opt_state(self.e.h, name.encode(), 2, 0, C.c_void_p(m2.data_ptr()), m2.numel()), 'dmg_train_opt_state')
            state[len(names)] = {'step': steps, 'exp_avg': m1, 'exp_avg_sq': m2}
            names.append(name)
        return {'state': state, 'param_names': names, 'step_count': self.step_count}

    def load_opt_state_dict(self, sd):
        "Inverse of opt_state_dict (best effort like the reference, deep_music_genre.py:1802-1803: unknown entries are skipped)."
        steps = 0
        for i, name in enumerate(sd.get('param_names', [])):
            st = sd['state'].get(i)
            if st is None:
                continue
            for which, key in ((1, 'exp_avg'), (2, 'exp_avg_sq')):
                a = st[key].detach().to('cpu', torch.float32).contiguous()
                rc = self.lib.dmg_train_opt_state(self.e.h, name.encode(), which, 1, C.c_void_p(a.data_ptr()), a.numel())
                if rc not in (0, 1):
                    check(rc, f'dmg_train_opt_state({name})')
            steps = max(steps, int(st.get('step', 0)))
        self.lib.dmg_train_opt_steps(self.e.h, steps)
        self.step_count = int(sd.get('step_count', steps))

    def sync_for_inference(self):
        "Re-derive what inference caches from the trained weights (rel-pos key cache)."
        check(self.lib.dmg_commit_weights(self.e.h), 'dmg_commit_weights')
        self.e.committed = True


class RemixTrainer(TXLTrainer):
    """Masked-LM training of the remix encoder: what fastai's ``Learner.fit`` does per batch around ``MultiTransformer`` for the
    ``msk`` task (deep_music_remix.py:1874-1881, 2734-2741)::

        model.train(); logits = head(encoder(x_masked, pos))
        loss = CrossEntropyFlat(ignore_index=pad_idx)(logits, y_masked)      # mean over the positions mask_tfm selected
        loss.backward(); clip; Adam(betas=(0.9, 0.99)) with true_wd

    ``model`` is the ``MultiTransformer`` mirror of ``model.get_multitask_model`` (bf16).  The encoder has no memory (``reset`` is a
    no-op), no AR/TAR terms (``alpha = beta = 0``) and no attention mask.  ``bptt`` must be a multiple of 64.  Every step needs ``pos``;
    ``y`` holds ``pad_idx`` at every position that is not predicted.  Data-parallel training is ``TXLTrainer``'s.
    """
    def __init__(self, model, bs, bptt, config, pad_idx, drop_mult=1., seed=0, **kw):
        super().__init__(model, bs, bptt, config, drop_mult=drop_mult, alpha=0., beta=0., seed=seed, pad_idx=int(pad_idx), **kw)
        self.pad_idx = int(pad_idx)

    def forward(self, x, y=None, pos=None, mask_size=None):
        if pos is None:
            raise ValueError('RemixTrainer: the remix encoder adds beat/bar embeddings, pos is required')
        if mask_size is not None and tuple(mask_size) != (1, 1):
            raise ValueError(f'RemixTrainer: the remix encoder has no attention mask, mask_size must be (1, 1), got {tuple(mask_size)}')
        return super().forward(x, y, pos, (1, 1))

    def validate(self, batches, mask_p=0.3, mask_range=None, seed=None, vocab=None):
        """fastai Learner.validate of the mask task: model.eval() over `batches` - already-masked ({'x', 'pos'}, y) or (x, y, pos)
        batches [bs, bptt], or a MusicPreloader(y_offset=0, encode_position=True) whose batches go through mask_tfm(p=mask_p,
        mask_range) first, as fastai applies the batch transforms to the validation loader too.  `seed` makes those masks (and so the
        result) reproducible: batch i uses a seed derived from (seed, i); None draws them from torch's CPU generator.  `vocab` (default
        MusicVocab.create()) gives mask_idx and the default mask_range (note_range[0], dur_range[1]).  Returns {'valid_loss': mean
        CrossEntropyFlat(ignore_index=pad_idx), 'mask_acc': fraction of the predicted positions whose argmax is the target}: per
        batch over its kept targets (NaN for a batch with none, as torch gives, and the NaN carries into the result), then the
        batch-size-weighted mean.  Weights, optimizer state, step_count and losses() are left as they were."""
        from .preloader import MusicPreloader, mask_tfm
        it, n_max = self._batches(batches)
        if isinstance(batches, MusicPreloader):
            if vocab is None:
                from .codec import MusicVocab
                vocab = MusicVocab.create()
            rng = mask_range or (vocab.note_range[0], vocab.dur_range[1])

            def masked(src):
                for i, (x, y, pos) in enumerate(src):
                    s = None if seed is None else (int(seed) * 1000003 + 7919 * (i + 1)) & 0x7FFFFFFF
                    xm, ym = mask_tfm((x, y), rng, vocab.mask_idx, self.pad_idx, p=mask_p, seed=s)
                    yield xm, ym, pos
            it = masked(it)
        with np.errstate(invalid='ignore', divide='ignore'):
            tab = self._eval_table(it, n_max)
            per = np.stack([tab[:, 0] / tab[:, 1], tab[:, 2] / tab[:, 1]], 1)
        loss, acc = self._average(per, [self.bs] * len(tab))
        return {'valid_loss': loss, 'mask_acc': acc}
