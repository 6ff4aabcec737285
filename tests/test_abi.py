"""CPU checks of the C-ABI boundary: the library builds/loads, exports every symbol include/dmg_b200.h declares, the
ctypes structs match the header, and the product path fails loudly without a GPU (no CPU fallback)."""
import ctypes as C
import os
import re

import pytest
import torch

from deepmusicgeneration_b200 import _lib, build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_functions():
    src = open(os.path.join(ROOT, 'include', 'dmg_b200.h')).read()
    src = re.sub(r'/\*.*?\*/', '', src, flags=re.S)
    return sorted(set(re.findall(r'\b(dmg_[a-z0-9_]+)\s*\(', src)))


def test_library_builds_for_sm100a_and_loads():
    path = build.build()
    assert os.path.exists(path)
    assert 'arch=compute_100a,code=sm_100a' in ' '.join(build.NVCC_FLAGS) and '-lineinfo' in build.NVCC_FLAGS
    lib = _lib.load()
    assert lib.dmg_abi_version() == 1


def test_every_declared_symbol_is_exported_and_bound():
    lib = C.CDLL(build.LIB)
    declared = _header_functions()
    assert len(declared) >= 18
    for name in declared:
        assert hasattr(lib, name), f'{name} declared in include/dmg_b200.h but not exported'
        assert name in _lib.SYMBOLS, f'{name} has no ctypes signature in _lib.SYMBOLS'
    assert sorted(_lib.SYMBOLS) == declared


def test_struct_layouts_match_header():
    assert C.sizeof(_lib.Config) == 20 * 4
    assert C.sizeof(_lib.VocabLayout) == 14 * 4
    assert C.sizeof(_lib.SamplerParams) == 3 * 8 + 4 * 4 + 2 * 4 + 8
    assert _lib.SamplerParams.seed.offset == 48
    assert C.sizeof(_lib.DecodeAttnArgs) == 8 * 8 + 8 + 8 * 4
    assert _lib.DecodeAttnArgs.pos_total.offset == 64 and _lib.DecodeAttnArgs.kernel.offset == 100
    assert C.sizeof(_lib.DecodeLayerArgs) == 17 * 8 + 8 + 8 * 4
    assert _lib.DecodeLayerArgs.pp_stride.offset == 136 and _lib.DecodeLayerArgs.d_inner.offset == 172


@pytest.mark.skipif(torch.cuda.is_available(), reason='CPU-only check')
def test_no_cpu_fallback():
    lib = _lib.load()
    cfg, h = _lib.Config(), C.c_void_p()
    assert lib.dmg_create(C.byref(cfg), 0, C.byref(h)) != 0
    assert b'no CUDA device' in lib.dmg_last_error()
    from deepmusicgeneration_b200.model import get_language_model
    from deepmusicgeneration_b200.app_utils import default_config
    with pytest.raises(RuntimeError):
        get_language_model(324, default_config())


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, 'deepmusicgeneration_b200')
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(('.py', '.cu', '.cuh', '.h')):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r'^\s*(from|import)\s+oracle\b', src, flags=re.M), f
                assert 'oracle/' not in src or f.endswith('.md'), f
