"""Learner-level call surface of the reference on top of the CUDA engine.

``music_model_learner`` / ``MusicLearner.predict`` mirror ``deep_music_genre.py:1784-1972``;
``multitask_model_learner`` / ``MultitaskLearner.predict_mask`` mirror ``deep_music_remix.py:2452-2477,
2563-2613``.  The token loop of ``predict`` (forward -> temperature -> grammar filter -> top-k/top-p ->
multinomial -> bookkeeping) runs on the device without a host round trip per token; ``generate_batch`` is the
same loop over many independent streams (the batched-generation workload of BASELINE.json).
"""
import ctypes as C
import time

import numpy as np
import torch

from . import _lib
from ._lib import check
from .codec import ACCEP_INS, MusicItem, MusicVocab, PAD
from .model import _ptr, _stream_ptr, get_language_model, get_multitask_model


def vocab_layout(vocab):
    v = _lib.VocabLayout()
    v.bos, v.pad, v.eos, v.mask, v.ni, v.sep = (vocab.bos_idx, vocab.pad_idx, vocab.stoi['xxeos'], vocab.mask_idx,
                                                vocab.ni_idx, vocab.sep_idx)
    v.special_lo, v.special_hi = 0, vocab.note_range[0]
    v.note_lo, v.note_hi = vocab.note_range
    v.dur_lo, v.dur_hi = vocab.dur_range
    v.ins_lo, v.ins_hi = vocab.ins_range
    return v


def sampler_params(vocab, n_words, temperatures, min_bars, top_k, top_p, allowed_ins=None, flags=_lib.SAMPLE_EARLY_STOP,
                   seed=None):
    p = _lib.SamplerParams()
    t = tuple(float(x) for x in temperatures)
    if len(t) == 2:
        t = t + (1.0,)
    p.temperatures[0], p.temperatures[1], p.temperatures[2] = t
    p.min_bars, p.top_k, p.top_p, p.n_words = int(min_bars), int(top_k), float(top_p), int(n_words)
    mask = 0
    if allowed_ins is not None:
        for tok in allowed_ins:                       # tokens 'i<k>' after the in-place rewrite below
            mask |= 1 << (vocab.stoi[tok] - vocab.ins_range[0])
    p.allowed_ins_mask, p.flags = mask, flags
    p.seed = int(seed) if seed is not None else int(torch.randint(0, 2 ** 62, (1,)).item())
    return p


def _load_checkpoint(learn, file):
    """fastai Learner.load(with_opt=True) for a file of learn.save: the weights into the model, the Adam state into the live trainer
    (if there is one), then the inference caches."""
    state = torch.load(file, map_location='cpu', weights_only=False)
    learn.model.load_state_dict(state['model'], strict=False)
    tr = getattr(learn, '_trainer', None)
    if tr is not None:
        if state.get('opt'):
            tr.load_opt_state_dict(state['opt'])
        tr.sync_for_inference()
    return learn


def _epoch_end(learn, tr, epoch, t0, validate, metric, callbacks):
    """fastai's end of an epoch in fit(): validate (if there are validation batches), one recorder row, the callbacks.  train_loss is
    the last training batch's loss (dropout on; not fastai's smoothed value).  Returns True when a callback stops training."""
    row = {'epoch': epoch, 'train_loss': tr.losses()['loss'], 'valid_loss': None, metric: None}
    if validate is not None:
        row['valid_loss'], row[metric] = validate()
    row['time'] = time.time() - t0
    learn.recorder.append(row)
    stop = False
    for cb in callbacks:
        stop = bool(cb.on_epoch_end(epoch, row)) or stop
    return stop


def _trainer_for(learn, batches, x_of):
    "the live trainer, or one sized by the first batch of `batches` (a list or a MusicPreloader)"
    from .preloader import MusicPreloader
    tr = getattr(learn, '_trainer', None)
    if tr is not None:
        return tr
    if isinstance(batches, MusicPreloader):
        return learn.trainer(batches.local_bs, batches.bptt)
    x = x_of(batches[0])
    return learn.trainer(x.shape[0], x.shape[1])


class MusicLearner:
    "deep_music_genre.py:1811-1972"
    def __init__(self, data, model, config=None):
        self.data, self.model, self.config = data, model, config
        self.recorder = []         # one row per epoch of fit_one_cycle(valid_batches=... or callbacks=...)

    def load(self, file):
        "Weights and Adam state of a learn.save file (fastai Learner.load)."
        return _load_checkpoint(self, file)

    def validate(self, valid_batches):
        """fastai Learner.validate: [valid_loss, accuracy] of `valid_batches` (a list of (x, y[, pos]) [bs, bptt] or a MusicPreloader) in
        eval mode, on the device (TXLTrainer.validate).  The training memory is reset first (fastai runs on_epoch_begin = RNNTrainer's
        reset there) and carried across the batches.  Uses the live trainer, or creates one sized by the batches."""
        tr = _trainer_for(self, valid_batches, lambda b: b[0]['x'] if isinstance(b[0], dict) else b[0])
        r = tr.validate(valid_batches, reset=True)
        return [r['valid_loss'], r['accuracy']]

    # -- checkpoints: {'model': state_dict (fastai key names), 'config': ...}  (:1812-1821, :1789-1805)
    def save(self, file=None, with_opt=True, config=None):
        """{'model': state_dict (fastai key names), 'opt': Adam state of the live trainer (None before any training), 'config'}: the
        file music_model_learner(pretrained_path=...) / createGenreContinuationModel(ckpt_path=...) reads back."""
        tr = getattr(self, '_trainer', None)
        state = {'model': self.model.state_dict(), 'opt': tr.opt_state_dict() if (with_opt and tr is not None) else None}
        if config or self.config:
            state['config'] = config or self.config
        torch.save(state, file)
        return file

    def load_opt_state(self, opt_state, bs, bptt, **kw):
        "learn.opt.load_state_dict(state['opt']) (deep_music_genre.py:1801-1803) onto the trainer of this (bs, bptt)."
        if opt_state:
            self.trainer(bs, bptt, **kw).load_opt_state_dict(opt_state)

    # -- training: what fastai's Learner.fit_one_cycle does for this learner (notebook cell 70-73, SURVEY.md 3.3)
    def trainer(self, bs, bptt, drop_mult=1., alpha=2., beta=1., seed=0, **kw):
        "The training-step engine for this model (RNNLearner adds RNNTrainer(alpha=2, beta=1)); created once per (bs, bptt)."
        from .training import TXLTrainer
        key = (bs, bptt, float(drop_mult), float(alpha), float(beta), int(seed), tuple(sorted(kw.items())))
        if getattr(self, '_trainer_key', None) != key:
            if getattr(self, '_trainer', None) is not None:
                self._trainer.close()
            self._trainer = TXLTrainer(self.model, bs, bptt, self.config, drop_mult=drop_mult, alpha=alpha, beta=beta, seed=seed, **kw)
            self._trainer_key = key
        return self._trainer

    def fit_one_cycle(self, cyc_len, max_lr, batches, bs=None, bptt=None, wd=0.01, clip=0.5, moms=(0.95, 0.85), drop_mult=1.,
                      callback=None, valid_batches=None, callbacks=None):
        """learner.fit_one_cycle(epochs, lr) over `batches`: a list of (x, y[, pos]) LongTensors [bs, bptt], or a
        deepmusicgeneration_b200.preloader.MusicPreloader (the reference's contiguous streams with per-item random transpose,
        deep_music_genre.py:1001-1125, assembled on the GPU; every pass is a new epoch = new shuffle / transposes, like the
        reference's DataLoader): one-cycle LR / momentum schedule over all cyc_len passes, memory reset at every epoch start
        (RNNTrainer.on_epoch_begin), Adam(true_wd), gradient clipping.

        valid_batches (same forms, same [bs, bptt]): after every epoch the model is validated on them in eval mode, straight after
        the training batches and without a memory reset, as fastai's fit loop does.  With valid_batches or callbacks
        (callbacks.EarlyStoppingCallback, callbacks.SaveModelCallback), every epoch appends {'epoch', 'train_loss', 'valid_loss',
        'accuracy', 'time'} to self.recorder (train_loss: the epoch's last batch loss, dropout on, read once per epoch - not
        fastai's smoothed loss; time: seconds) and the callbacks may stop training early.  Without either, nothing is added to
        the loop.  `callback(i, trainer)` still runs after every step."""
        from .training import one_cycle_lr
        from .preloader import MusicPreloader
        is_pl = isinstance(batches, MusicPreloader)
        n_b = batches.n_batches if is_pl else len(batches)
        tr = self.trainer(bs or (batches.local_bs if is_pl else batches[0][0].shape[0]),
                          bptt or (batches.bptt if is_pl else batches[0][0].shape[1]), drop_mult=drop_mult)
        if getattr(self, 'pretrained_opt_state', None):
            try:    tr.load_opt_state_dict(self.pretrained_opt_state)     # try / except: pass, like the reference
            except Exception: pass
            self.pretrained_opt_state = None
        track = valid_batches is not None or bool(callbacks)
        cbs = list(callbacks or [])
        if track:
            self.recorder = []
            for cb in cbs:
                cb.on_train_begin(self)
        validate = (lambda: list(tr.validate(valid_batches, reset=False).values())) if valid_batches is not None else None
        total, i = cyc_len * n_b, 0
        for epoch in range(cyc_len):
            t0 = time.time()
            tr.reset()
            for b in batches:
                if is_pl:                           # (x, y) or ({'x', 'pos'}, y)
                    b = (b[0]['x'], b[1], b[0]['pos']) if isinstance(b[0], dict) else b
                lr, mom = one_cycle_lr(i, total, max_lr, moms=moms)
                tr.step(b[0], b[1], b[2] if len(b) > 2 else None, lr=lr, betas=(mom, 0.99), wd=wd, clip=clip)
                if callback is not None:
                    callback(i, tr)
                i += 1
            if track and _epoch_end(self, tr, epoch, t0, validate, 'accuracy', cbs):
                break
        for cb in cbs:
            cb.on_train_end()
        tr.sync_for_inference()
        return tr.losses()

    def _prefill(self, x, pos):
        max_seq = self.model._e.cfg.max_seq
        if x.shape[1] > max_seq:
            # the reference runs the whole seed as ONE forward (memory-less attention over every seed token); splitting it into
            # segments would change the result, so the engine has to be built large enough
            raise ValueError(f'seed of {x.shape[1]} tokens exceeds max_seq={max_seq}: build the learner with '
                             f'music_model_learner(..., max_seq=<longest seed>) or cut the seed with item.trim_to_beat(...)')
        enc = self.model[0]
        enc._bs = x.shape[0]
        self.model._e.forward(x, pos if enc.encode_position else None, _lib.LOGITS_LAST)

    def _run_loop(self, n_words, prev_idx, last_pos, params):
        e = self.model._e
        bs = len(prev_idx)
        prev = np.ascontiguousarray(np.asarray(prev_idx, dtype=np.int32))
        lp = np.ascontiguousarray(np.asarray(last_pos, dtype=np.int64))
        vl = vocab_layout(self.data.vocab)
        check(e.lib.dmg_sampler_init(e.h, C.byref(vl), C.byref(params), prev.ctypes.data_as(C.c_void_p),
                                     lp.ctypes.data_as(C.c_void_p), bs), 'dmg_sampler_init')
        toks = torch.empty(n_words, bs, dtype=torch.int32, device=e.device)
        with torch.cuda.device(e.device):
            check(e.lib.dmg_generate(e.h, n_words, _ptr(toks), _stream_ptr()), 'dmg_generate')
        return toks

    def predict(self, item, n_words=128, temperatures=(1.0, 1.0, 1.0), min_bars=4, top_k=30, top_p=0.6, allowed_ins=None,
                seed=None):
        "Return the `n_words` that come after `item` -> (pred, full).  Signature of deep_music_genre.py:1853-1855."
        self.model.reset()
        vocab = self.data.vocab
        x, pos = item.to_tensor(), item.get_pos_tensor()
        last_pos = int(pos[-1]) if len(pos) else 0
        if allowed_ins is not None:                   # the reference rewrites the caller's list in place (:1878-1880)
            for i, ins in enumerate(allowed_ins):
                allowed_ins[i] = 'i' + str(ACCEP_INS[ins])
        prev_idx = int(item.data[-1])
        print('Init prev_idx = ', prev_idx)
        self._prefill(x[None], pos[None])
        params = sampler_params(vocab, n_words, temperatures, min_bars, top_k, top_p, allowed_ins, seed=seed)
        toks = self._run_loop(n_words, [prev_idx], [last_pos], params).cpu().numpy()[:, 0]
        new_idx = []
        for t in toks:
            if t == -2:
                bad = new_idx[-1] if new_idx else prev_idx
                print(item.to_text())
                print(f'Assertion error: prev_idx = {vocab.itos[bad]}')
                raise AssertionError
            if t < 0:
                break
            new_idx.append(int(t))
        pred = vocab.to_music_item(np.array(new_idx, dtype=np.int64), item.ins)
        full = item.append(pred)
        return pred, full

    def generate_batch(self, x, pos=None, n_words=128, temperatures=(1.0, 1.0, 1.0), min_bars=4, top_k=30, top_p=0.6,
                       seed=0, early_stop=False, mask_unused=False):
        """`predict` over B independent streams: x LongTensor [B, T] of seeds (equal length), returns int32
        [n_words, B] on the device (-1 = stream stopped, -2 = stream hit the reference's AssertionError case)."""
        self.model.reset()
        x = x.to(self.model._e.device)
        B, T = x.shape
        if pos is None:
            pos = torch.zeros_like(x)
        self._prefill(x, pos)
        flags = (_lib.SAMPLE_EARLY_STOP if early_stop else 0) | (_lib.SAMPLE_MASK_UNUSED if mask_unused else 0)
        params = sampler_params(self.data.vocab, n_words, temperatures, min_bars, top_k, top_p, None, flags=flags, seed=seed)
        return self._run_loop(n_words, x[:, -1].cpu().numpy(), pos[:, -1].cpu().numpy(), params)

    def beam_search(self, xb, n_words, top_k=10, beam_sz=10, temperature=1., return_beams=False):
        """Return the `n_words` that come after `xb` using beam search (signature of deep_music_genre.py:1823-1851).

        The beams live on the device: the K/V rings of the `top_k` copies of the seed are permuted by ``select_hidden`` (one
        ``dmg_select_hidden`` per step), each step's log-softmax / per-beam top-k / global selection is one kernel
        (``dmg_beam_step``) and only the survivors' (parent, token) pairs - a few dozen integers - come back to the host, which
        keeps the token history.  Like the reference the final node is drawn with ``multinomial(exp(-scores / temperature))``."""
        e = self.model._e
        self.model.reset()
        self.model.eval()
        xb = xb.to(e.device)
        seed_len = xb.shape[-1]
        if xb.shape[0] > 1: xb = xb[0][None]
        nb = top_k                                               # the reference starts from top_k identical copies of the seed
        assert max(top_k, beam_sz) <= e.cfg.max_batch, f'beam search over {max(top_k, beam_sz)} beams needs max_batch >= that'
        x = xb.repeat(nb, 1)
        self.model[0]._bs = nb
        e.forward(x, torch.zeros_like(x) if self.model[0].encode_position else None, _lib.LOGITS_LAST)
        scores = torch.zeros(1, dtype=torch.float32, device=e.device)
        new_scores = torch.empty(beam_sz, dtype=torch.float32, device=e.device)
        parents = torch.empty(beam_sz, dtype=torch.int32, device=e.device)
        tokens = torch.empty(beam_sz, dtype=torch.int32, device=e.device)
        history = np.zeros((nb, 0), dtype=np.int64)
        for step in range(n_words):
            with torch.cuda.device(e.device):
                check(e.lib.dmg_beam_step(e.h, _ptr(scores), scores.numel(), nb, top_k, beam_sz, _ptr(new_scores), _ptr(parents),
                                          _ptr(tokens), _stream_ptr()), 'dmg_beam_step')
            par, tok = parents.cpu().numpy(), tokens.cpu().numpy().astype(np.int64)
            history = np.concatenate([history[par], tok[:, None]], axis=1)
            self.model[0].select_hidden(par)                     # the survivors inherit their parents' memory (:1847)
            nb = beam_sz
            scores = new_scores.clone()
            if step + 1 < n_words:
                xs = torch.from_numpy(tok).to(e.device)[:, None]
                e.forward(xs, torch.zeros_like(xs) if self.model[0].encode_position else None, _lib.LOGITS_LAST)
        if temperature != 1.: scores.div_(temperature)
        if return_beams:
            return history, scores.cpu()
        node_idx = torch.multinomial(torch.exp(-scores), 1).item()
        return [int(i) for i in history[node_idx]]


def music_model_learner(data, arch=None, config=None, drop_mult=1., pretrained_path=None, encode_position=True,
                        dtype='bf16', device=0, max_batch=None, max_seq=None, keep_hidden=True, seed=None, **learn_kwargs):
    "Create a learner with a language model from `data` and `config` (deep_music_genre.py:1784-1807)."
    state = None
    if pretrained_path:
        state = torch.load(pretrained_path, map_location='cpu', weights_only=False)
        if config is None: config = state['config']
    config = dict(config)
    beam = max_batch or 10                             # beam_search repeats the seed top_k (default 10) times
    model = get_language_model(len(data.vocab.itos), config, drop_mult=drop_mult, dtype=dtype, device=device,
                               max_batch=beam, max_seq=max_seq, keep_hidden=keep_hidden, seed=seed,
                               init=state is None)
    learn = MusicLearner(data, model, config=config)
    if state is not None:
        model.load_state_dict(state['model'], strict=False)
        learn.pretrained_opt_state = state.get('opt')      # applied by fit_one_cycle to the trainer it creates (:1801-1803)
    return learn


def predict_from_midi(learn, midi=None, n_words=400, temperatures=(1.0, 1.0), top_k=30, top_p=0.6, seed_len=None, **kwargs):
    "deep_music_genre.py:1975-1982"
    vocab = learn.data.vocab
    seed = MusicItem.from_file(midi, vocab)
    if seed_len is not None: seed = seed.trim_to_beat(seed_len)
    pred, full = learn.predict(seed, n_words=n_words, temperatures=temperatures, top_k=top_k, top_p=top_p, **kwargs)
    return full


class MultitaskLearner:
    "deep_music_remix.py:2479-2613 (mask task)."
    def __init__(self, data, model, config=None):
        self.data, self.model, self.config = data, model, config
        self.recorder = []         # one row per epoch of fit_one_cycle(valid_batches=... or callbacks=...)

    def load(self, file):
        "Weights and Adam state of a learn.save file (fastai Learner.load)."
        return _load_checkpoint(self, file)

    def validate(self, valid_batches, mask_p=0.3, mask_range=None, seed=None):
        """fastai Learner.validate of the mask task: [valid_loss, mask_acc] of `valid_batches` (already-masked ({'x', 'pos'}, y)
        batches, or a MusicPreloader whose batches go through mask_tfm first; see RemixTrainer.validate), in eval mode on the device.
        Uses the live trainer, or creates one sized by the batches."""
        tr = _trainer_for(self, valid_batches, lambda b: b[0]['x'])
        r = tr.validate(valid_batches, mask_p=mask_p, mask_range=mask_range, seed=seed, vocab=self.data.vocab)
        return [r['valid_loss'], r['mask_acc']]

    def save(self, file=None, with_opt=True, config=None):
        """{'model': state_dict, 'opt': Adam state of the live trainer (None before any training or with with_opt=False)[, 'config']}:
        the file multitask_model_learner(pretrained_path=...) reads back."""
        tr = getattr(self, '_trainer', None)
        state = {'model': self.model.state_dict(), 'opt': tr.opt_state_dict() if (with_opt and tr is not None) else None}
        if config: state['config'] = config
        torch.save(state, file)
        return file

    # -- training of the mask task: what fastai's Learner.fit_one_cycle does for this learner (MTTrainer, SURVEY.md App. D.8)
    def trainer(self, bs, bptt, drop_mult=1., seed=0, **kw):
        "The training-step engine for this model (masked cross entropy, ignore index = the vocabulary's pad); created once per (bs, bptt)."
        from .training import RemixTrainer
        key = (bs, bptt, float(drop_mult), int(seed), tuple(sorted(kw.items())))
        if getattr(self, '_trainer_key', None) != key:
            if getattr(self, '_trainer', None) is not None:
                self._trainer.close()
            self._trainer = RemixTrainer(self.model, bs, bptt, self.config, pad_idx=self.data.vocab.pad_idx, drop_mult=drop_mult,
                                         seed=seed, **kw)
            self._trainer_key = key
        return self._trainer

    def load_opt_state(self, opt_state, bs, bptt, **kw):
        "learn.opt.load_state_dict(state['opt']) onto the trainer of this (bs, bptt)."
        if opt_state:
            self.trainer(bs, bptt, **kw).load_opt_state_dict(opt_state)

    def fit_one_cycle(self, cyc_len, max_lr, batches, bs=None, bptt=None, wd=0.01, clip=0.5, moms=(0.95, 0.85), drop_mult=1.,
                      mask_p=0.3, mask_range=None, callback=None, valid_batches=None, callbacks=None, valid_seed=None):
        """learner.fit_one_cycle(epochs, lr) of the mask task over `batches`: either a list of already-masked ({'x', 'pos'}, y)
        batches (LongTensors [bs, bptt], y = pad_idx where nothing is predicted), or a deepmusicgeneration_b200.preloader.MusicPreloader
        built with y_offset=0 and encode_position=True, whose every batch goes through mask_tfm(p=mask_p, mask_range) on the device
        (deep_music_remix.py:1208-1223).  The default mask_range is (vocab.note_range[0], vocab.dur_range[1]), the range the
        preloader golden (tests/golden/make_preloader_golden.py) was generated with.  One-cycle LR / momentum schedule over all
        cyc_len passes, Adam(true_wd), gradient clipping; returns the last step's losses.

        valid_batches (same forms, same [bs, bptt]; a preloader's batches are masked with mask_p / mask_range, seeded by valid_seed):
        validated in eval mode after every epoch.  With valid_batches or callbacks (callbacks.EarlyStoppingCallback,
        callbacks.SaveModelCallback), every epoch appends {'epoch', 'train_loss', 'valid_loss', 'mask_acc', 'time'} to self.recorder
        (train_loss: the epoch's last batch loss, dropout on, read once per epoch - not fastai's smoothed loss; time: seconds) and
        the callbacks may stop training early.  Without either, nothing is added to the loop."""
        from .training import one_cycle_lr
        from .preloader import MusicPreloader, mask_tfm
        vocab = self.data.vocab
        if mask_range is None:
            mask_range = (vocab.note_range[0], vocab.dur_range[1])
        is_pl = isinstance(batches, MusicPreloader)
        n_b = batches.n_batches if is_pl else len(batches)
        tr = self.trainer(bs or (batches.local_bs if is_pl else batches[0][0]['x'].shape[0]),
                          bptt or (batches.bptt if is_pl else batches[0][0]['x'].shape[1]), drop_mult=drop_mult)
        if getattr(self, 'pretrained_opt_state', None):
            try:    tr.load_opt_state_dict(self.pretrained_opt_state)     # try / except: pass, like the reference
            except Exception: pass
            self.pretrained_opt_state = None
        track = valid_batches is not None or bool(callbacks)
        cbs = list(callbacks or [])
        if track:
            self.recorder = []
            for cb in cbs:
                cb.on_train_begin(self)
        validate = (lambda: list(tr.validate(valid_batches, mask_p=mask_p, mask_range=mask_range, seed=valid_seed,
                                             vocab=vocab).values())) if valid_batches is not None else None
        total, i = cyc_len * n_b, 0
        for epoch in range(cyc_len):
            t0 = time.time()
            for xb, y in batches:
                if not isinstance(xb, dict):
                    raise ValueError('the remix encoder needs ({"x", "pos"}, y) batches (MusicPreloader(encode_position=True))')
                x, pos = xb['x'], xb['pos']
                if is_pl:
                    x, y = mask_tfm((x, y), mask_range, vocab.mask_idx, vocab.pad_idx, p=mask_p)
                lr, mom = one_cycle_lr(i, total, max_lr, moms=moms)
                tr.step(x, y, pos, lr=lr, betas=(mom, 0.99), wd=wd, clip=clip)
                if callback is not None:
                    callback(i, tr)
                i += 1
            if track and _epoch_end(self, tr, epoch, t0, validate, 'mask_acc', cbs):
                break
        for cb in cbs:
            cb.on_train_end()
        tr.sync_for_inference()
        return tr.losses()

    def pred_batch(self, batch):
        "fastai Learner.pred_batch: eval-mode forward of one batch."
        xb, _ = batch
        return self.model.eval()(xb)

    def predict_mask(self, masked_item, temperatures=(1.0, 1.0), top_k=20, top_p=0.8, seed=None):
        "One full encoder forward per masked position, sampled on the device (deep_music_remix.py:2563-2613)."
        e = self.model._e
        vocab = self.data.vocab
        x = masked_item.to_tensor().to(e.device)
        pos = masked_item.get_pos_tensor().to(e.device)
        self.model.reset()
        mask_idxs = (x == vocab.mask_idx).nonzero().view(-1)
        vl = vocab_layout(vocab)
        params = sampler_params(vocab, 1, temperatures, 0, top_k, top_p, None, flags=_lib.SAMPLE_REMIX_FILTER, seed=seed)
        rc_dev = torch.zeros(1, dtype=torch.int32, device=e.device)
        out_dev = torch.zeros(1, dtype=torch.int32, device=e.device)
        nc_dev = torch.zeros(1, dtype=torch.int32, device=e.device)
        repeat_count = 0
        for n, midx in enumerate(mask_idxs.tolist()):
            prev = x[midx - 1:midx].to(torch.int32) if midx > 0 else x[-1:].to(torch.int32)   # x[-1] wraps like the reference
            logits = self.pred_batch(batch=({'msk': {'x': x[None], 'pos': pos[None]}}, None))['msk'][0][midx].contiguous()
            rc_dev.fill_(repeat_count)
            with torch.cuda.device(e.device):
                check(e.lib.dmg_sample_logits(e.h, _ptr(logits), _ptr(prev), _ptr(rc_dev), 1, C.byref(vl), C.byref(params),
                                              n, _ptr(out_dev), _ptr(nc_dev), _stream_ptr()), 'dmg_sample_logits')
            idx, num_choices = int(out_dev.item()), int(nc_dev.item())
            repeat_count = repeat_count + 1 if num_choices <= 2 else repeat_count // 2
            x[midx] = idx
        return vocab.to_music_item(x.cpu().numpy())

    def predict_mask_batch(self, items, temperatures=(1.0, 1.0), top_k=20, top_p=0.8, seed=None):
        """predict_mask over many items at once: returns one MusicItem per item.  The items (of any lengths up to max_seq) run as
        padded batches of up to max_batch items through dmg_predict_mask_batch: every step is one encoder forward over the batch and
        one sampled token per item that still has masks, with no host round trip.  Item i draws from Philox stream i of `seed` (its
        n-th mask uses counter n), so item 0 makes the draws of predict_mask(items[0], ..., seed=seed).  Its logit row is summed in another
        order than the head GEMM's, so a near-tie can still go the other way.  In fp32 no result depends on how the items are grouped;
        in bf16 the GEMM kernel follows the row count of a group (max_batch / max_rows), which can likewise flip a near-tie.  Items
        are sorted by length before they are grouped, which keeps the padding small."""
        e = self.model._e
        vocab = self.data.vocab
        cfg = e.cfg
        max_rows = cfg.max_rows if cfg.max_rows > 0 else cfg.max_batch * cfg.max_seq
        datas = [np.asarray(it.data, dtype=np.int64) for it in items]
        poss = [np.asarray(it.position, dtype=np.int64) for it in items]
        for i, x in enumerate(datas):
            if len(x) > cfg.max_seq:
                raise ValueError(f'item {i} has {len(x)} tokens and exceeds max_seq={cfg.max_seq}: build the learner with '
                                 f'multitask_model_learner(..., max_seq=<longest item>) or cut the item with item.trim_to_beat(...)')
            if len(x) == 0:
                raise ValueError(f'item {i} is empty')
        vl = vocab_layout(vocab)
        params = sampler_params(vocab, 1, temperatures, 0, top_k, top_p, None, flags=_lib.SAMPLE_REMIX_FILTER, seed=seed)
        out = [None] * len(items)
        order = sorted(range(len(items)), key=lambda i: len(datas[i]))
        k = 0
        while k < len(order):
            chunk = [order[k]]                         # ascending lengths: the last item of a chunk sets its padded length
            while (k + len(chunk) < len(order) and len(chunk) < cfg.max_batch and
                   (len(chunk) + 1) * len(datas[order[k + len(chunk)]]) <= max_rows):
                chunk.append(order[k + len(chunk)])
            k += len(chunk)
            B, T = len(chunk), max(len(datas[i]) for i in chunk)
            lens = np.array([len(datas[i]) for i in chunk], dtype=np.int32)
            x = np.full((B, T), vocab.pad_idx, dtype=np.int64)
            pos = np.zeros((B, T), dtype=np.int64)
            masks = [np.flatnonzero(datas[i] == vocab.mask_idx).astype(np.int32) for i in chunk]
            n_max = max(1, max(len(mp) for mp in masks))
            mask_pos = np.zeros((B, n_max), dtype=np.int32)
            for j, i in enumerate(chunk):
                x[j, :lens[j]] = datas[i]
                pos[j, :lens[j]] = poss[i]
                mask_pos[j, :len(masks[j])] = masks[j]
            n_masks = np.array([len(mp) for mp in masks], dtype=np.int32)
            streams = np.array(chunk, dtype=np.int32)
            xd = torch.from_numpy(x).to(e.device)
            pd = torch.from_numpy(pos).to(e.device)
            with torch.cuda.device(e.device):
                check(e.lib.dmg_predict_mask_batch(e.h, _ptr(xd), _ptr(pd), lens.ctypes.data_as(C.c_void_p),
                                                   mask_pos.ctypes.data_as(C.c_void_p), n_masks.ctypes.data_as(C.c_void_p),
                                                   streams.ctypes.data_as(C.c_void_p), B, T, n_max, C.byref(vl), C.byref(params),
                                                   _stream_ptr()), 'dmg_predict_mask_batch')
            res = xd.cpu().numpy()
            for j, i in enumerate(chunk):
                out[i] = vocab.to_music_item(res[j, :lens[j]].copy())
        return out


def multitask_model_learner(data, config=None, drop_mult=1., pretrained_path=None, dtype='bf16', device=0, max_batch=1,
                            max_seq=1024, seed=None, **learn_kwargs):
    "deep_music_remix.py:2452-2477"
    vocab = data.vocab
    state = None
    if pretrained_path:
        state = torch.load(pretrained_path, map_location='cpu', weights_only=False)
        if config is None: config = state['config']
    config = dict(config)
    model = get_multitask_model(len(vocab), config, drop_mult=drop_mult, pad_idx=vocab.pad_idx, dtype=dtype, device=device,
                                max_batch=max_batch, max_seq=max_seq, seed=seed, init=state is None)
    learn = MultitaskLearner(data, model, config=config)
    if state is not None:
        model.load_state_dict(state['model'], strict=False)
        learn.pretrained_opt_state = state.get('opt')      # applied by fit_one_cycle to the trainer it creates
    return learn
