"""Developer timing of the train step's GEMMs (zf_selftest_umma_gemm -> launch_gemm) at the conditioner's shapes.
   python scripts/gemm_perf.py [legacy|simt]: no argument times the default choice (tcgen05, fed by the copy engine where
   the operands allow), 'legacy' the tcgen05 GEMM with register-path loaders, 'simt' the fp32 FFMA GEMM."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
if os.environ.get("ZF_LIB"):
    from zenflow_b200 import build as _zb
    _zb.LIB_PATH = os.path.abspath(os.environ["ZF_LIB"]); os.environ["ZENFLOW_B200_NO_BUILD"] = "1"
from zenflow_b200 import _lib
lib = _lib.load()
if len(sys.argv) > 1:
    _lib.set_impl(None, sys.argv[1])
M = 262144
dev = "cuda"
def t(fn, n=5):
    fn(); torch.cuda.synchronize()
    best = 1e9
    for _ in range(n):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record(); torch.cuda.synchronize(); best = min(best, a.elapsed_time(b))
    return best
def run(mode, I, J, R, a_swish=0, with_z=False):
    if mode == 0:
        A = torch.randn(I, R, device=dev); B = torch.randn(R, J, device=dev) * 0.1; C = torch.empty(I, J, device=dev)
        lda, ldb, ldc = R, J, J
    elif mode == 1:
        A = torch.randn(I, R, device=dev); B = torch.randn(J, R, device=dev) * 0.1; C = torch.empty(I, J, device=dev)
        lda, ldb, ldc = R, R, J
    else:
        A = torch.randn(R, I, device=dev); B = torch.randn(R, J, device=dev); C = torch.zeros(I, J, device=dev)
        lda, ldb, ldc = I, J, J
    bias = torch.randn(J, device=dev) if mode == 0 else None
    colsum = torch.zeros(J, device=dev) if mode == 2 else None
    Z = torch.randn(I, J, device=dev) if with_z else None
    p = lambda x: 0 if x is None else x.data_ptr()
    s = torch.cuda.current_stream().cuda_stream
    def fn():
        rc = lib.zf_selftest_umma_gemm(s, mode, p(A), lda, p(B), ldb, p(C), ldc, p(bias), p(colsum), p(Z), J, a_swish, I, J, R, 2048)
        _lib.check(rc, "gemm")
    ms = t(fn)
    fl = 2.0 * I * J * R
    print(f"mode {mode} I={I:7d} J={J:4d} R={R:7d}: {ms*1e3:8.1f} us ({fl/ms/1e9:6.1f} TFLOP/s algorithmic)")
run(0, M, 128, 8, 0)          # first Dense (F = 8)
run(0, M, 128, 128, 1)        # hidden
run(0, M, 760, 128, 1)        # last layer (8 dims x 95)
run(1, M, 128, 760, 0, True)  # grad-input through the last layer
run(1, M, 128, 128, 0, True)  # grad-input through a hidden layer
run(1, M, 8, 128, 0, False)   # grad wrt the BatchNorm output
run(2, 128, 760, M, 1)        # grad-weight last layer
run(2, 128, 128, M, 1)        # grad-weight hidden
run(2, 8, 128, M, 0)          # grad-weight first layer
