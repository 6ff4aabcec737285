"""Builds libdmg_b200.so (hand-written sm_100a CUDA + the C ABI of include/dmg_b200.h) in-tree with nvcc.

nvcc cross-compiles without a GPU; the built .so travels to the GPU box with the repo snapshot.
Every .cu is compiled to its own object (in parallel, cached by a digest of the source + headers + flags) and the
objects are linked into one shared library.
"""
import hashlib
import os
import subprocess
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
OBJDIR = os.path.join(HERE, 'build')
LIB = os.path.join(HERE, 'libdmg_b200.so')
SOURCES = ['gemm.cu', 'gemm_train.cu', 'elementwise.cu', 'attention.cu', 'attention_decode2.cu', 'decode_layer.cu', 'attention_flash.cu', 'attention_train.cu', 'attention_train_tc.cu', 'attention_bert_tc.cu', 'attention_bert_train.cu',
           'sampling.cu', 'train_kernels.cu', 'preload.cu', 'model.cu', 'train.cu']
HEADERS = ['common.cuh', 'kernels.cuh', 'attention_decode2.cuh', 'attention_decode3.cuh', 'sampling.cuh', 'launch.cuh', 'attention_bert_tc_common.cuh', 'model.cuh', 'train_kernels.cuh', 'mma_sync.cuh', 'attention_train_common.cuh',
           os.path.join('..', '..', 'include', 'dmg_b200.h')]
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17',
              '-Xcompiler', '-fPIC']


def _nvcc():
    for cand in (os.environ.get('NVCC'), '/usr/local/cuda/bin/nvcc', 'nvcc'):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return 'nvcc'


def _existing(files):
    return [f for f in files if os.path.exists(os.path.join(CSRC, f))]


def _header_digest():
    h = hashlib.sha256()
    for f in _existing(HEADERS):
        with open(os.path.join(CSRC, f), 'rb') as fh:
            h.update(fh.read())
    h.update(' '.join(NVCC_FLAGS).encode())
    return h.hexdigest()


def _file_digest(src, hd):
    h = hashlib.sha256(hd.encode())
    with open(os.path.join(CSRC, src), 'rb') as fh:
        h.update(fh.read())
    return h.hexdigest()


def source_digest():
    hd = _header_digest()
    h = hashlib.sha256()
    for s in _existing(SOURCES):
        h.update(_file_digest(s, hd).encode())
    return h.hexdigest()


def is_current():
    stamp = LIB + '.digest'
    return os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read().strip() == source_digest()


def _compile_one(src, hd, verbose):
    obj = os.path.join(OBJDIR, src.replace('.cu', '.o'))
    stamp = obj + '.digest'
    dg = _file_digest(src, hd)
    if os.path.exists(obj) and os.path.exists(stamp) and open(stamp).read().strip() == dg:
        return obj, ''
    cmd = [_nvcc()] + NVCC_FLAGS + (['-Xptxas=-v'] if verbose else []) + ['-c', '-o', obj, os.path.join(CSRC, src)]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError('nvcc failed on %s:\n%s%s' % (src, res.stdout, res.stderr))
    with open(stamp, 'w') as fh:
        fh.write(dg)
    return obj, res.stderr


def build(force=False, verbose=False):
    "Compile every CUDA source for sm_100a into libdmg_b200.so; no-op when the sources have not changed."
    if not force and is_current():
        return LIB
    os.makedirs(OBJDIR, exist_ok=True)
    if force:
        for f in os.listdir(OBJDIR):
            os.remove(os.path.join(OBJDIR, f))
    hd = _header_digest()
    srcs = _existing(SOURCES)
    with ThreadPoolExecutor(max_workers=min(8, len(srcs))) as ex:
        results = list(ex.map(lambda s: _compile_one(s, hd, verbose), srcs))
    if verbose:
        for _, log in results:
            if log:
                print(log)
    cmd = [_nvcc(), '-shared', '-gencode', 'arch=compute_100a,code=sm_100a', '-o', LIB] + [o for o, _ in results]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError('link failed:\n' + res.stdout + res.stderr)
    with open(LIB + '.digest', 'w') as fh:
        fh.write(source_digest())
    return LIB


if __name__ == '__main__':
    import sys
    print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))
