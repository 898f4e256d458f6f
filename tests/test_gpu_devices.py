"""Per-device state of the native library: device properties and every kernel's dynamic shared-memory opt-in are kept
per device, so one process runs the same kernels on device 0 and then on device 1."""
import numpy as np
import pytest
import torch

from oracle import zenflow_oracle as zo
from tests.helpers import assert_fp32_parity, product_chain, to64, trained_variables

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")]

CHAINS = [
    # name, D, C, K, layers, n_couplings, roll shift, M
    ("two_moons_conditional", 2, 1, 16, (128, 128), None, 1, 4096),   # chain_umma_pp_kernel
    ("cond16", 16, 4, 32, (128, 128), 8, 2, 1500),                    # chain_umma_kernel, tensor-core first Dense
]


def _wide_gemm_err(seed):
    """Dense forward with 256 output columns and aligned operands: the copy-engine-fed tcgen05 GEMM with 256-column
    tiles.  Returns max |C - C64| / max |C64|."""
    from zenflow_b200 import _lib

    lib = _lib.load()
    I, J, R = 300, 256, 128
    rng = np.random.default_rng(seed)
    A = rng.normal(size=(I, R)); B = rng.normal(size=(R, J)) / np.sqrt(R); bias = rng.normal(size=J)
    ref = (A / (1 + np.exp(-A))) @ B + bias
    cu = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).cuda()
    At, Bt, bt = cu(A), cu(B), cu(bias)
    Ct = torch.full((I, J), float("nan"), device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    _lib.check(lib.zf_selftest_umma_gemm(st, 0, At.data_ptr(), R, Bt.data_ptr(), J, Ct.data_ptr(), J, bt.data_ptr(),
                                         None, None, 0, 1, I, J, R, 0))
    torch.cuda.synchronize()
    return np.abs(Ct.cpu().numpy() - ref).max() / np.abs(ref).max()


def test_gemm_and_chain_on_device_0_then_1():
    from zenflow_b200 import Flow

    cases = []
    for name, D, C, K, layers, ncoup, shift, M in CHAINS:
        ops = zo.make_chain(D, K, layers, n_couplings=ncoup, roll_shift=shift)
        rng = np.random.default_rng(M)
        x = rng.normal(0.3, 1.2, (M, D)).astype(np.float32)
        c = rng.uniform(0, 1, (M, C)).astype(np.float32)
        v = trained_variables(ops, x, c, seed=1)
        lp64, _ = zo.flow_log_prob(ops, to64(v), x.astype(np.float64), c.astype(np.float64))
        lpo, _ = zo.flow_log_prob(ops, v, x, c)
        cases.append((name, ops, v, x, c, lp64, lpo))
    for dev in (0, 1):
        with torch.cuda.device(dev):
            err = _wide_gemm_err(dev)
            print(f"\ncuda:{dev} GEMM 300x256x128: max err / max|ref| = {err:.2e}")
            assert err < 5e-6
            for name, ops, v, x, c, lp64, lpo in cases:
                fv = {"params": {"bijector": v["params"]}, "batch_stats": {"bijector": v["batch_stats"]}}
                lp = Flow(product_chain(ops)).apply(fv, x, c)
                # tensor-core chain kernels: the tolerances of test_gpu_chain.py's tensor-core cases
                assert_fp32_parity(lp, lp64, lpo, f"cuda:{dev} {name} log_prob", atol=5e-5, slack=4.0)
