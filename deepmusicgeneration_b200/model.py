"""Host-side mirrors of the reference's model objects, backed by libdmg_b200.so.

``get_language_model`` returns a ``SequentialRNN``-like object whose call surface is the reference's
(``deep_music_genre.py:1886-1889``, fastai ``SequentialRNN``/``TransformerXL``/``LinearDecoder``):

    decoded, raw_outputs, outputs = model(x)          # x: LongTensor [bs, x_len] or {'x':.., 'pos':..}
    model.reset(); model[0].hidden; model[0].select_hidden(idxs); model[0].mem_len; model.eval()

``get_multitask_model`` returns the ``MultiTransformer`` mirror for the mask task
(``deep_music_remix.py:1874-1881``): ``model({'msk': {'x':.., 'pos':..}}) -> {'msk': logits}``.

All arithmetic runs in the CUDA library; PyTorch here only owns device buffers and the stream.
"""
import ctypes as C
import math

import numpy as np
import torch

from . import _lib
from ._lib import check


def tfmerXL_lm_config():
    "fastai.text.models.transformer.tfmerXL_lm_config"
    return dict(ctx_len=150, n_layers=12, n_heads=10, d_model=410, d_head=41, d_inner=2100, resid_p=0.1, attn_p=0.1,
                ff_p=0.1, embed_p=0.1, output_p=0.1, bias=False, scale=True, act='gelu', double_drop=True,
                tie_weights=True, out_bias=True, mem_len=150, mask=True)


def _stream_ptr():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


class _Engine:
    "Owns one dmg_model handle."
    def __init__(self, arch, vocab_sz, config, dtype, device, max_batch, max_seq, max_rows, keep_hidden, gemm_backend=0, kernel_flags=0):
        self.lib = _lib.load()
        if not torch.cuda.is_available():
            raise RuntimeError('deepmusicgeneration_b200 needs a CUDA device (B200, sm_100a); there is no CPU path')
        self.device = torch.device('cuda', device if isinstance(device, int) else torch.device(device).index or 0)
        bert = arch == _lib.ARCH_BERT
        cfg = _lib.Config()
        cfg.arch, cfg.dtype = arch, {'f32': _lib.F32, 'fp32': _lib.F32, 'bf16': _lib.BF16}[dtype]
        cfg.vocab = vocab_sz
        cfg.d_model, cfg.n_heads, cfg.d_head = config['d_model'], config['n_heads'], config['d_head']
        cfg.n_layers = config['enc_layers'] if bert else config['n_layers']
        cfg.d_inner = config['d_inner']
        cfg.mem_len = 0 if bert else config['mem_len']
        cfg.attn_bias = int(bool(config.get('bias', False)))
        cfg.encode_position = 1 if bert else int(bool(config.get('encode_position', True)))
        cfg.max_batch, cfg.max_seq, cfg.max_rows = max_batch, max_seq, max_rows
        cfg.keep_hidden = int(keep_hidden and not bert)
        cfg.gemm_backend = gemm_backend
        cfg.kernel_flags = kernel_flags
        self.cfg, self.dtype = cfg, dtype
        h = C.c_void_p()
        check(self.lib.dmg_create(C.byref(cfg), self.device.index, C.byref(h)), 'dmg_create')
        self.h = h
        self.committed = False

    def __del__(self):
        h, self.h = getattr(self, 'h', None), None
        if h:
            self.lib.dmg_destroy(h)

    # ---- weights
    def weight_names(self):
        c, bert = self.cfg, self.cfg.arch == _lib.ARCH_BERT
        HD, d, V = c.n_heads * c.d_head, c.d_model, c.vocab
        names = {}
        if bert:
            names.update({'encoder.embed.embed.weight': (V, d), 'head.decoder.weight': (V, d), 'head.decoder.bias': (V,),
                          'encoder.u': (c.n_heads, 1, c.d_head), 'encoder.v': (c.n_heads, 1, c.d_head),
                          'encoder.embed.beat_enc.weight': (32, d), 'encoder.embed.bar_enc.weight': (1024, d)})
            for l in range(c.n_layers):
                p = f'encoder.layers.{l}.mha1.'
                for w in ('q_wgt', 'k_wgt', 'v_wgt', 'r_attn'):
                    names[p + w + '.weight'] = (HD, d)
                    if c.attn_bias: names[p + w + '.bias'] = (HD,)
                names[p + 'ln.weight'] = (d,); names[p + 'ln.bias'] = (d,)
        else:
            names.update({'0.encoder.weight': (V, d), '1.decoder.weight': (V, d), '1.decoder.bias': (V,),
                          '0.u': (c.n_heads, 1, c.d_head), '0.v': (c.n_heads, 1, c.d_head)})
            if c.encode_position:
                names.update({'0.beat_enc.beat_enc.weight': (32, d), '0.beat_enc.bar_enc.weight': (1024, d)})
            for l in range(c.n_layers):
                p, f = f'0.layers.{l}.mhra.', f'0.layers.{l}.ff.layers.'
                names[p + 'attention.weight'] = (3 * HD, d); names[p + 'out.weight'] = (d, HD)
                names[p + 'r_attn.weight'] = (HD, d)
                if c.attn_bias:
                    names[p + 'attention.bias'] = (3 * HD,); names[p + 'out.bias'] = (d,); names[p + 'r_attn.bias'] = (HD,)
                names[p + 'ln.weight'] = (d,); names[p + 'ln.bias'] = (d,)
                names[f + '0.weight'] = (c.d_inner, d); names[f + '0.bias'] = (c.d_inner,)
                names[f + '3.weight'] = (d, c.d_inner); names[f + '3.bias'] = (d,)
                names[f + '6.weight'] = (d,); names[f + '6.bias'] = (d,)
        return names

    def load_state_dict(self, state, strict=False):
        known = self.weight_names()
        missing = [k for k in known if k not in state]
        if strict and missing:
            raise KeyError(f'missing keys: {missing[:5]}...')
        for name, t in state.items():
            if name not in known:
                continue                                        # strict=False: e.g. pos_enc.freq, mha2.*, decoder.*
            a = t.detach().to('cpu', torch.float32).contiguous()
            check(self.lib.dmg_set_weight(self.h, name.encode(), C.c_void_p(a.data_ptr()), a.numel()), f'set_weight({name})')
        check(self.lib.dmg_commit_weights(self.h), 'dmg_commit_weights')
        self.committed = True
        return missing

    def state_dict(self):
        out = {}
        for name, shape in self.weight_names().items():
            a = torch.empty(shape, dtype=torch.float32)
            check(self.lib.dmg_get_weight(self.h, name.encode(), C.c_void_p(a.data_ptr()), a.numel()), f'get_weight({name})')
            out[name] = a
        return out

    # ---- forward
    def forward(self, ids, pos, logits_mode, want_core=False, mask=(1, 1), lens=None):
        """One forward over ids [bs, T].  lens: the length of every row, a padded batch of sequences that are each computed as if alone
        at their length (dmg_forward_varlen).  BERT encoder: logits_mode LOGITS_NONE or LOGITS_ALL.  Transformer-XL: the prefill of
        bs seeds after reset() (every stream then holds its own seed as memory); LOGITS_LAST gives the logits of row lens[b] - 1."""
        assert ids.dim() == 2
        ids = ids.to(self.device, torch.int64).contiguous()
        if pos is not None:
            pos = pos.to(self.device, torch.int64).contiguous()
        bs, T = ids.shape
        V, d = self.cfg.vocab, self.cfg.d_model
        logits = None
        if logits_mode == _lib.LOGITS_ALL:
            logits = torch.empty(bs, T, V, device=self.device, dtype=torch.float32)
        elif logits_mode == _lib.LOGITS_LAST:
            logits = torch.empty(bs, V, device=self.device, dtype=torch.float32)
        core = torch.empty(bs, T, d, device=self.device, dtype=torch.float32) if want_core else None
        with torch.cuda.device(self.device):
            if lens is not None:
                ln = np.ascontiguousarray(np.asarray(lens, dtype=np.int32))
                if ln.shape != (bs,):
                    raise ValueError(f'lens must hold one length per row ({bs}), got shape {ln.shape}')
                check(self.lib.dmg_forward_varlen(self.h, _ptr(ids), _ptr(pos), ln.ctypes.data_as(C.c_void_p), bs, T, logits_mode,
                                                  _ptr(logits), _ptr(core), _stream_ptr()), 'dmg_forward_varlen')
            else:
                check(self.lib.dmg_forward(self.h, _ptr(ids), _ptr(pos), bs, T, int(mask[0]), int(mask[1]), logits_mode,
                                           _ptr(logits), _ptr(core), _stream_ptr()), 'dmg_forward')
        return logits, core

    def reset(self, batch=0):
        check(self.lib.dmg_reset(self.h, batch), 'dmg_reset')

    def mem_count(self):
        "memory positions held by every stream (ValueError when the streams hold memories of different lengths: see mem_counts)"
        m = self.lib.dmg_mem_count(self.h)
        if m < 0:
            raise ValueError(self.lib.dmg_last_error().decode())
        return m

    def mem_counts(self, n=None):
        "memory positions held by each of the first n streams (default: max_batch), a list"
        n = self.cfg.max_batch if n is None else n
        out = np.zeros(n, dtype=np.int32)
        check(self.lib.dmg_mem_counts(self.h, out.ctypes.data_as(C.c_void_p), n), 'dmg_mem_counts')
        return out.tolist()

    def hidden(self, level, bs):
        m = self.mem_count()
        if m == 0:
            return torch.empty(0, device=self.device)
        out = torch.empty(bs, m, self.cfg.d_model, device=self.device, dtype=torch.float32)
        with torch.cuda.device(self.device):
            check(self.lib.dmg_get_hidden(self.h, level, _ptr(out), _stream_ptr()), 'dmg_get_hidden')
        return out

    def select_hidden(self, idxs):
        idx = np.ascontiguousarray(torch.as_tensor(idxs).cpu().numpy().astype(np.int32))
        torch.cuda.synchronize(self.device)
        check(self.lib.dmg_select_hidden(self.h, idx.ctypes.data_as(C.c_void_p), len(idx)), 'dmg_select_hidden')


# ------------------------------------------------------------------------------------------ init (fastai init_transformer)
def init_state_dict(engine, seed=None):
    """Random-init weights with the distributions fastai's ``model.apply(init_transformer)`` leaves behind
    (SURVEY.md App. A.6): Linear W ~ N(0, .02), b = 0; LayerNorm w ~ N(1, .02), b = 0; u, v ~ N(0, .02); the tied
    embedding ~ N(0, .02); beat/bar embeddings ~ N(0, 1) with row 0 = 0."""
    g = torch.Generator().manual_seed(seed if seed is not None else int(torch.randint(0, 2 ** 31 - 1, (1,))))
    sd = {}
    for name, shape in engine.weight_names().items():
        if name in ('1.decoder.weight', 'head.decoder.weight'):
            continue
        if 'beat_enc' in name or 'bar_enc' in name:
            w = torch.randn(shape, generator=g)
            w[0] = 0
        elif name.endswith('.bias'):
            w = torch.zeros(shape)
        elif '.ln.' in name or '.ff.layers.6.' in name:          # LayerNorms: mhra.ln / mha1.ln and SequentialEx index 6 of the FFN
            w = torch.randn(shape, generator=g) * 0.02 + 1.0
        else:
            w = torch.randn(shape, generator=g) * 0.02
        sd[name] = w
    return sd


# ------------------------------------------------------------------------------------------ reference-shaped objects
class MusicTransformerXL:
    "model[0] of the reference (deep_music_genre.py:1603-1647 on fastai TransformerXL)."
    def __init__(self, engine, config):
        self._e = engine
        self.mem_len = config['mem_len']
        self.n_layers, self.d_model = config['n_layers'], config['d_model']
        self.encode_position = bool(config.get('encode_position', True))
        self.mask_steps = config.get('mask_steps', 1)
        self.mask = config.get('mask', True)
        self.training = False
        self.init = False
        self._bs = 0

    def reset(self):
        self._e.reset(0)
        self._bs = 0

    @property
    def hidden(self):
        "List of L+1 tensors [bs, <=mem_len, d] (empty 1-D tensors right after reset), fetched from the device rings."
        if not self._e.cfg.keep_hidden:
            raise RuntimeError('model was built with keep_hidden=False (generation-only engine)')
        counts = self._e.mem_counts(self._bs)
        if len(set(counts)) > 1:
            raise ValueError(f'the {self._bs} streams hold memories of different lengths (per-stream counts {counts}), which one '
                             f'[bs, mem, d] tensor per layer cannot hold; read them with the engine\'s mem_counts()')
        return [self._e.hidden(l, self._bs) for l in range(self.n_layers + 1)]

    def select_hidden(self, idxs):
        self._e.select_hidden(idxs)
        self._bs = len(idxs)

    def forward(self, x, logits_mode=_lib.LOGITS_NONE, mask_size=None):
        pos = None
        if self.encode_position:
            x, pos = x['x'], x['pos']
        if mask_size is None:
            mask_size = (1, 1)          # eval: causal with all memory visible (rand_window_mask(is_eval=True))
        self._bs = x.shape[0]
        return self._e.forward(x, pos, logits_mode, want_core=True, mask=mask_size)

    __call__ = forward


class LinearDecoder:
    "model[1] of the reference: tied decoder; its GEMM is fused into the engine's forward."
    def __init__(self, engine):
        self._e = engine


class SequentialRNN:
    "fastai SequentialRNN(MusicTransformerXL, LinearDecoder) mirror."
    def __init__(self, engine, config):
        self._e = engine
        self._mods = [MusicTransformerXL(engine, config), LinearDecoder(engine)]
        self.training = False

    def __getitem__(self, i): return self._mods[i]
    def __len__(self): return 2

    def reset(self):
        self._mods[0].reset()

    def eval(self):
        self.training = self._mods[0].training = False
        return self

    def train(self, mode=True):
        # Dropout is not implemented in the CUDA forward (parity is defined in eval mode, SURVEY.md App. D.12);
        # train() only records the flag so reference call sites keep working.
        self.training = self._mods[0].training = bool(mode)
        return self

    def __call__(self, x, mask_size=None):
        enc = self._mods[0]
        logits, core = enc.forward(x, logits_mode=_lib.LOGITS_ALL, mask_size=mask_size)
        raw_outputs = _LazyHidden(enc) if enc.mem_len > 0 else [core]
        return logits, raw_outputs, [core]

    def load_state_dict(self, state, strict=False): return self._e.load_state_dict(state, strict=strict)
    def state_dict(self): return self._e.state_dict()
    def parameters_count(self):
        return sum(int(np.prod(s)) for n, s in self._e.weight_names().items() if n != '1.decoder.weight')


class _LazyHidden:
    "raw_outputs of the reference forward: materialised from the device rings only when somebody looks."
    def __init__(self, enc): self._enc, self._val = enc, None
    def _get(self):
        if self._val is None: self._val = self._enc.hidden
        return self._val
    def __getitem__(self, i): return self._get()[i]
    def __len__(self): return self._enc.n_layers + 1
    def __iter__(self): return iter(self._get())


def get_language_model(vocab_sz, config, drop_mult=1., dtype='bf16', device=0, max_batch=1, max_seq=None, max_rows=0,
                       keep_hidden=True, seed=None, init=True, gemm_backend=0, kernel_flags=0):
    "fastai get_language_model(MusicTransformerXL, vocab_sz, config, drop_mult) (deep_music_genre.py:1793)."
    config = dict(config)
    max_seq = max_seq or max(config.get('ctx_len', 512), config['mem_len'], 1024)
    eng = _Engine(_lib.ARCH_TXL, vocab_sz, config, dtype, device, max_batch, max_seq, max_rows, keep_hidden, gemm_backend, kernel_flags)
    model = SequentialRNN(eng, config)
    if init:
        eng.load_state_dict(init_state_dict(eng, seed))
    return model


class MultiTransformer:
    "deep_music_remix.py:1864-1902, mask task (encoder + head)."
    def __init__(self, engine, config):
        self._e = engine
        self.default_mem_len = config.get('mem_len', 512)
        self.training = False

    def __call__(self, inp):
        out = {}
        msk = inp.get('msk')
        if msk is not None:
            logits, _ = self._e.forward(msk['x'], msk['pos'], _lib.LOGITS_ALL)
            out['msk'] = logits
        for key in ('lm', 's2f', 'f2s'):
            if inp.get(key) is not None:
                raise NotImplementedError(f'task {key!r}: decoder / seq2seq branches are outside the B200 hot path')
        return out

    def reset(self): pass
    def eval(self): self.training = False; return self
    def train(self, mode=True): self.training = bool(mode); return self
    def load_state_dict(self, state, strict=False): return self._e.load_state_dict(state, strict=strict)
    def state_dict(self): return self._e.state_dict()


def get_multitask_model(vocab_size, config, drop_mult=1., pad_idx=None, dtype='bf16', device=0, max_batch=1, max_seq=1024,
                        max_rows=0, seed=None, init=True, gemm_backend=0, kernel_flags=0):
    "deep_music_remix.py:1851-1862 (encoder + head; the decoder is not built)."
    config = dict(config)
    eng = _Engine(_lib.ARCH_BERT, vocab_size, config, dtype, device, max_batch, max_seq, max_rows, False, gemm_backend, kernel_flags)
    model = MultiTransformer(eng, config)
    if init:
        eng.load_state_dict(init_state_dict(eng, seed))
    return model
