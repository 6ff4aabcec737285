"""ctypes binding of libdmg_b200.so (the C ABI declared in include/dmg_b200.h).

There is no CPU path and no fallback: if the library is missing or cannot be loaded, importing the
symbols raises.  The .so is built in-tree by ``deepmusicgeneration_b200.build`` (nvcc, sm_100a).
"""
import ctypes as C
import os

from . import build as _build

_LIB = None

c_i32, c_i64, c_u32, c_u64, c_f32, c_f64, c_vp = C.c_int32, C.c_int64, C.c_uint32, C.c_uint64, C.c_float, C.c_double, C.c_void_p

ARCH_TXL, ARCH_BERT = 0, 1
F32, BF16 = 0, 1
GEMM_AUTO, GEMM_SIMT, GEMM_TC_TILE = 0, 1, 2
LOGITS_NONE, LOGITS_ALL, LOGITS_LAST = 0, 1, 2
SAMPLE_EARLY_STOP, SAMPLE_MASK_UNUSED, SAMPLE_REMIX_FILTER = 1, 2, 4
# dmg_config.kernel_flags (DMG_KF_*): non-default kernels for parity tests / reproducing measurements; 0 = the product path
(KF_NO_DECODE_KERNEL, KF_NO_FLASH, KF_NO_GRAPH, KF_BERT_MMA_SYNC, KF_BERT_FP32_STRIP, KF_NO_SPLITK, KF_NO_BIG_GEMM, KF_GEMM_SIMT,
 KF_NO_FUSED_DECODE, KF_NO_DUAL_DECODE, KF_ATTN_DECODE_V2) = (1, 2, 4, 8, 16, 32, 64, 128, 256, 512, 1024)


class Config(C.Structure):
    _fields_ = [(n, c_i32) for n in ('arch', 'dtype', 'vocab', 'd_model', 'n_layers', 'n_heads', 'd_head', 'd_inner',
                                     'mem_len', 'attn_bias', 'encode_position', 'max_batch', 'max_seq', 'max_rows',
                                     'keep_hidden', 'gemm_backend', 'kernel_flags')] + [('reserved', c_i32 * 3)]


class VocabLayout(C.Structure):
    _fields_ = [(n, c_i32) for n in ('bos', 'pad', 'eos', 'mask', 'ni', 'sep', 'special_lo', 'special_hi', 'note_lo',
                                     'note_hi', 'dur_lo', 'dur_hi', 'ins_lo', 'ins_hi')]


class SamplerParams(C.Structure):
    _fields_ = [('temperatures', c_f64 * 3), ('min_bars', c_i32), ('top_k', c_i32), ('top_p', c_f32),
                ('n_words', c_i32), ('allowed_ins_mask', c_u32), ('flags', c_i32), ('seed', c_u64)]


class TrainConfig(C.Structure):
    _fields_ = [('batch', c_i32), ('bptt', c_i32), ('resid_p', c_f32), ('attn_p', c_f32), ('ff_p', c_f32), ('embed_p', c_f32),
                ('output_p', c_f32), ('alpha', c_f32), ('beta', c_f32), ('seed', c_u64), ('pad_idx', c_i32),
                ('reserved', c_i32 * 3)]


# name -> (restype, argtypes): every symbol include/dmg_b200.h declares
SYMBOLS = {
    'dmg_last_error': (C.c_char_p, []),
    'dmg_abi_version': (c_i32, []),
    'dmg_create': (c_i32, [C.POINTER(Config), c_i32, C.POINTER(c_vp)]),
    'dmg_destroy': (None, [c_vp]),
    'dmg_set_weight': (c_i32, [c_vp, C.c_char_p, c_vp, c_i64]),
    'dmg_get_weight': (c_i32, [c_vp, C.c_char_p, c_vp, c_i64]),
    'dmg_commit_weights': (c_i32, [c_vp]),
    'dmg_reset': (c_i32, [c_vp, c_i32]),
    'dmg_select_hidden': (c_i32, [c_vp, c_vp, c_i32]),
    'dmg_mem_count': (c_i32, [c_vp]),
    'dmg_forward': (c_i32, [c_vp, c_vp, c_vp, c_i32, c_i32, c_i32, c_i32, c_i32, c_vp, c_vp, c_vp]),
    'dmg_get_hidden': (c_i32, [c_vp, c_i32, c_vp, c_vp]),
    'dmg_sampler_init': (c_i32, [c_vp, C.POINTER(VocabLayout), C.POINTER(SamplerParams), c_vp, c_vp, c_i32]),
    'dmg_generate': (c_i32, [c_vp, c_i32, c_vp, c_vp]),
    'dmg_generate_step_host': (c_i32, [c_vp, c_vp, c_vp, c_vp]),
    'dmg_sample_logits': (c_i32, [c_vp, c_vp, c_vp, c_vp, c_i32, C.POINTER(VocabLayout), C.POINTER(SamplerParams),
                                  c_u64, c_vp, c_vp, c_vp]),
    'dmg_beam_step': (c_i32, [c_vp, c_vp, c_i32, c_i32, c_i32, c_i32, c_vp, c_vp, c_vp, c_vp]),
    'dmg_sample_probs': (c_i32, [c_vp, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_i32, C.POINTER(VocabLayout), C.POINTER(SamplerParams),
                                 c_u64, c_vp, c_vp, c_vp, c_vp]),
    'dmg_device_bytes': (c_i64, [c_vp]),
    'dmg_launch_count': (c_i64, []),
    'dmg_uses_tcgen05': (c_i32, [c_vp]),
    'dmg_attn_decode_layer': (c_i32, [c_vp, c_i32, c_vp]),
    'dmg_decode_dual_launch': (c_i32, [c_vp, c_i32, c_vp]),
    'dmg_decode_timeline': (c_i32, [c_vp, c_vp]),
    'dmg_gemm_bf16': (c_i32, [c_vp, c_vp, c_vp, c_vp, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_vp]),
    # training step
    'dmg_train_param_count': (c_i64, [c_vp]),
    'dmg_train_create': (c_i32, [c_vp, C.POINTER(TrainConfig), c_vp]),
    'dmg_train_destroy': (None, [c_vp]),
    'dmg_train_reset': (c_i32, [c_vp]),
    'dmg_train_forward': (c_i32, [c_vp, c_vp, c_vp, c_vp, c_i32, c_i32, c_i32, c_i64, c_vp]),
    'dmg_train_backward': (c_i32, [c_vp, c_i32, c_i32, c_vp]),
    'dmg_train_grad_span': (c_i32, [c_vp, c_i32, c_i32, C.POINTER(c_i64), C.POINTER(c_i64)]),
    'dmg_train_grad_pack': (c_i32, [c_vp, c_i64, c_i64, c_vp, c_vp]),
    'dmg_train_grad_unpack': (c_i32, [c_vp, c_i64, c_i64, c_vp, c_vp]),
    'dmg_train_optimizer_step': (c_i32, [c_vp, c_f32, c_f32, c_f32, c_f32, c_f32, c_f32, c_f32, c_vp]),
    'dmg_train_opt_state': (c_i32, [c_vp, C.c_char_p, c_i32, c_i32, c_vp, c_i64]),
    'dmg_train_opt_steps': (c_i64, [c_vp, c_i64]),
    'dmg_train_losses': (c_i32, [c_vp, c_vp, c_vp]),
    'dmg_train_get_grad': (c_i32, [c_vp, C.c_char_p, c_vp, c_i64]),
    'dmg_train_dropout_mask': (c_i32, [c_vp, c_i32, c_i32, c_i64, c_vp, c_i64, c_vp]),
    'dmg_train_grad_buffer': (c_vp, [c_vp]),
    'dmg_gemm_train': (c_i32, [c_vp, c_i32, c_i64, c_vp, c_i32, c_i64, c_i32, c_i32, c_i32, c_i32, c_vp, c_i32, c_vp, c_i64,
                               c_i32, c_vp, c_i64, c_i32, c_vp, c_i64, c_f32, c_u32, c_vp]),
    'dmg_preload_fill': (c_i32, [c_vp, c_vp, c_vp, c_vp, c_i32, c_i32, c_vp, c_i32, c_i32, c_vp, c_vp, c_i32, c_i32, c_i32, c_vp, c_vp, c_vp,
                                 c_vp]),
    'dmg_mask_tfm': (c_i32, [c_vp, c_vp, c_i64, c_i32, c_i32, c_i32, c_i32, C.c_double, c_u32, c_vp, c_vp, c_vp]),
    'dmg_attn_train_fwd': (c_i32, [c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_i32, c_i32, c_i32, c_i32, c_i32,
                                   c_i32, c_i32, c_f32, c_u32, c_vp, c_vp, c_vp]),
    'dmg_attn_train_bwd': (c_i32, [c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i32, c_i32, c_i32, c_i32,
                                   c_i32, c_i32, c_i32, c_f32, c_u32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
}


def lib_path():
    return _build.LIB


def load():
    "Load (building first if the sources changed and nvcc is around) and type every exported symbol."
    global _LIB
    if _LIB is not None:
        return _LIB
    path = lib_path()
    if not _build.is_current():
        try:
            _build.build()
        except Exception as e:   # no nvcc on the box: use the shipped .so if there is one
            if not os.path.exists(path):
                raise RuntimeError(f'libdmg_b200.so is missing and could not be built: {e}') from e
    if not os.path.exists(path):
        raise RuntimeError(f'{path} not found: the CUDA extension is required, there is no fallback path')
    lib = C.CDLL(path)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)     # AttributeError if the library does not export it
        fn.restype, fn.argtypes = res, args
    _LIB = lib
    return lib


class DmgError(RuntimeError):
    pass


def check(rc, what=''):
    if rc != 0:
        msg = load().dmg_last_error()
        raise DmgError(f'{what}: {msg.decode() if msg else "error"} (rc={rc})')
