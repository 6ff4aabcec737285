"Times the training attention forward / backward (C3 geometry: 32 streams x 8 heads, T = M = 512) through the C ABI with CUDA events."
import ctypes as C, os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from deepmusicgeneration_b200 import _lib
from deepmusicgeneration_b200._lib import check
B, T, H, M = int(os.environ.get('B', 32)), 512, 8, 512
HD, S = H * 64, M + T
lib = _lib.load()
g = torch.Generator(device='cuda').manual_seed(0)
p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)
st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
NB = 4   # rotate buffers (> L2)
qkv = [(torch.randn(B * T, 3 * HD, device='cuda', generator=g) * 0.8).bfloat16() for _ in range(NB)]
kvm = [(torch.randn(B * M, 2 * HD, device='cuda', generator=g) * 0.8).bfloat16() for _ in range(NB)]
rk = (torch.randn(S, HD, device='cuda', generator=g) * 0.8).bfloat16()
u = torch.randn(HD, device='cuda', generator=g) * 0.3
v = torch.randn(HD, device='cuda', generator=g) * 0.3
out = torch.zeros(B * T, HD, device='cuda', dtype=torch.bfloat16)
lse = torch.zeros(B, H, T, device='cuda')
dout = (torch.randn(B * T, HD, device='cuda', generator=g) * 0.5).bfloat16()
delta = torch.zeros(B, H, T, device='cuda')
dqkv = torch.zeros_like(qkv[0]); dkvm = torch.zeros_like(kvm[0])
dsd = torch.zeros(B * T, H * S, device='cuda', dtype=torch.bfloat16)
du = torch.zeros(HD, device='cuda'); dv = torch.zeros(HD, device='cuda')
psave = torch.zeros(B * H, T, S, device='cuda', dtype=torch.bfloat16)
msave = torch.zeros(B * H, T, S // 64, device='cuda')
def fwd(i, pdrop, save):
    check(lib.dmg_attn_train_fwd(p(qkv[i % NB]), 3 * HD, p(kvm[i % NB]), 2 * HD, p(rk), p(u), p(v), p(out), p(lse), B, T, H, M, M, 1, 1, pdrop, 99,
                                 p(psave if save else None), p(msave if save else None), st), 'fwd')
def bwd(i, pdrop, save):
    check(lib.dmg_attn_train_bwd(p(qkv[i % NB]), 3 * HD, p(kvm[i % NB]), 2 * HD, p(rk), p(u), p(v), p(out), p(lse), p(dout), B, T, H, M, M, 1, 1,
                                 pdrop, 99, p(delta), p(dqkv), p(dkvm), p(dsd), p(du), p(dv), p(psave if save else None), p(msave if save else None), st), 'bwd')
def timeit(fn, R=20):
    for i in range(3): fn(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(R): fn(i)
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / R * 1e3
for pdrop in (0.1, 0.0):
    for save in (False, True):
        us = timeit(lambda i: fwd(i, pdrop, save))
        print(f'attn_train_fwd p={pdrop} save={save}: {us:.1f} us  {3 * 2 * B * T * HD * S / us / 1e6:.0f} TFLOP/s dense-count')
        fwd(0, pdrop, save)
        if os.environ.get('BWD', '1') == '1':
            us = timeit(lambda i: bwd(0, pdrop, save), R=10)
            print(f'attn_train_bwd p={pdrop} saved={save}: {us:.1f} us (delta + dQ + dK/dV kernels)')
