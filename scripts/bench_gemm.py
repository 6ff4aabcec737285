"Times the training GEMM shapes of C3 through dmg_gemm_train (CUDA events, L2 flushed by rotating buffers)."
import ctypes as C, sys, os, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from deepmusicgeneration_b200 import _lib
lib = _lib.load()
def P(t): return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)
st = C.c_void_p(0)
dev = 'cuda'
rows = 16384
def run(name, M, N, K, a_mn, b_mn, out_mode, splitk=1, bias=False, gelu=0, aux_mode=0, pre=False, drop=0.0, reps=20):
    nb = 4
    As = [(torch.randn((K, M) if a_mn else (M, K), device=dev) * 0.1).bfloat16() for _ in range(nb)]
    Bs = [(torch.randn((K, N) if b_mn else (N, K), device=dev) * 0.1).bfloat16() for _ in range(nb)]
    outs = [torch.zeros(M, N, device=dev, dtype=torch.bfloat16 if out_mode == 1 else torch.float32) for _ in range(nb)]
    pres = [torch.zeros(M, N, device=dev, dtype=torch.bfloat16) for _ in range(nb)] if pre else [None] * nb
    b = torch.randn(N, device=dev) if bias else None
    aux = None
    if aux_mode in (2, 4): aux = torch.randn(M, N, device=dev).bfloat16()
    if aux_mode == 3: aux = torch.randn(M, N, device=dev)
    def call(i):
        rc = lib.dmg_gemm_train(P(As[i]), a_mn, As[i].stride(0), P(Bs[i]), b_mn, Bs[i].stride(0), M, N, K, splitk, P(b), gelu, P(aux),
                                aux.stride(0) if aux is not None else 0, aux_mode, P(outs[i]), N, out_mode, P(pres[i]), N if pre else 0,
                                drop, 7, st)
        assert rc == 0, lib.dmg_last_error()
    for i in range(nb): call(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for r in range(reps): call(r % nb)
    e1.record(); torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / reps
    print(f'{name:28s} M={M:6d} N={N:5d} K={K:6d}  {us:8.1f} us  {2*M*N*K/us/1e6:7.1f} TFLOP/s')
if os.environ.get('GEMM_MAJORS'):
    for a_mn, b_mn in ((0, 0), (1, 0), (0, 1), (1, 1)):
        run(f'4096^3 a_mn={a_mn} b_mn={b_mn}', 4096, 4096, 4096, a_mn, b_mn, 1, reps=10)
    run('dW2 shape, K=4096 only (no split)', 512, 2048, 4096, 1, 1, 2, splitk=1)
    run('dW2 shape K-major operands', 512, 2048, 16384, 0, 0, 2, splitk=4)
    for sk in (2, 4, 8, 9):
        run(f'dW2 atomic sk{sk}', 512, 2048, rows, 1, 1, 2, splitk=sk)
    for sk in (3, 6, 12):
        run(f'dWqkv atomic sk{sk}', 1536, 512, rows, 1, 1, 2, splitk=sk)
    for sk in (9, 18, 37):
        run(f'dWo atomic sk{sk}', 512, 512, rows, 1, 1, 2, splitk=sk)
    sys.exit(0)
only = os.environ.get('GEMM_ONLY')
if only:
    run('QKV fwd', rows, 1536, 512, 0, 0, 1, reps=2)
    run('FF1 fwd (bias gelu drop gfac)', rows, 2048, 512, 0, 0, 1, bias=True, gelu=2, pre=True, drop=0.1, reps=2)
    sys.exit(0)
run('QKV fwd', rows, 1536, 512, 0, 0, 1)
run('KVmem fwd', rows, 1024, 512, 0, 0, 1)
run('out-proj fwd', rows, 512, 512, 0, 0, 1)
run('FF1 fwd (bias gelu drop gfac)', rows, 2048, 512, 0, 0, 1, bias=True, gelu=2, pre=True, drop=0.1)
run('FF2 fwd (bias)', rows, 512, 2048, 0, 0, 1, bias=True)
run('dh = dY W2 (x gfac)', rows, 2048, 512, 0, 1, 1, aux_mode=4)
run('dbranch = dh W1 (bf16)', rows, 512, 2048, 0, 1, 1)
run('dbranch = dqkv Wqkv (bf16)', rows, 512, 1536, 0, 1, 1)
run('dattn = dY Wo (bf16)', rows, 512, 512, 0, 1, 1)
run('dW2 = dY^T h (atomic sk4)', 512, 2048, rows, 1, 1, 2, splitk=4)
run('dW1 = dh^T x (atomic sk4)', 2048, 512, rows, 1, 1, 2, splitk=4)
run('dWqkv (atomic sk6)', 1536, 512, rows, 1, 1, 2, splitk=6)
run('dWo (atomic sk18)', 512, 512, rows, 1, 1, 2, splitk=18)
run('plain 8192^3', 8192, 8192, 8192, 0, 0, 1, reps=5)
