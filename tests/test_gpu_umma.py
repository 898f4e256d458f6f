"""tcgen05 building blocks: the 3xTF32 split GEMM (A in tensor memory, B image in shared memory,
fp32 accumulator in tensor memory) must be fp32-accurate."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("N,K", [(128, 128), (96, 128), (48, 128), (16, 8), (64, 32)])
def test_umma_3xtf32_gemm(N, K):
    from zenflow_b200 import _lib

    lib = _lib.load()
    rng = np.random.default_rng(N + K)
    A = rng.normal(size=(128, K)).astype(np.float32)
    B = (rng.normal(size=(N, K)) / np.sqrt(K)).astype(np.float32)
    At, Bt = torch.from_numpy(A).cuda(), torch.from_numpy(B).cuda()
    out = torch.full((128, N), float("nan"), device="cuda")
    _lib.check(lib.zf_selftest_umma(torch.cuda.current_stream().cuda_stream, At.data_ptr(), Bt.data_ptr(), N, K,
                                    out.data_ptr(), 0))
    torch.cuda.synchronize()
    got = out.cpu().numpy()
    ref64 = A.astype(np.float64) @ B.astype(np.float64).T
    ref32 = A @ B.T
    err = np.abs(got - ref64).max()
    err32 = np.abs(ref32 - ref64).max()
    print(f"\nN={N} K={K}: 3xTF32 max err {err:.2e}, fp32 sgemm max err {err32:.2e}")
    assert err <= 4 * err32 + 2e-6


def test_umma_error_budget():
    """Diagnostic: where the 3xTF32 error comes from.  With operands that are exactly representable in
    tf32 (lo parts zero) the only error left is the tensor core's fp32 accumulation."""
    from zenflow_b200 import _lib

    lib = _lib.load()
    rng = np.random.default_rng(7)
    N = K = 128

    def run(A, B):
        At, Bt = torch.from_numpy(A).cuda(), torch.from_numpy(B).cuda()
        out = torch.empty((128, N), device="cuda")
        _lib.check(lib.zf_selftest_umma(torch.cuda.current_stream().cuda_stream, At.data_ptr(), Bt.data_ptr(), N, K,
                                        out.data_ptr(), 0))
        return out.cpu().numpy()

    def tf32(a):
        b = a.view(np.uint32).astype(np.uint64)
        b = ((b + 0x1000) & 0xFFFFE000).astype(np.uint32)
        return b.view(np.float32)

    A = np.abs(rng.normal(size=(128, K))).astype(np.float32)  # all positive: truncation shows up as bias
    B = np.abs(rng.normal(size=(N, K)) / np.sqrt(K)).astype(np.float32)
    for name, (a, b) in {"full fp32 operands": (A, B), "tf32-exact operands": (tf32(A.copy()), tf32(B.copy()))}.items():
        got = run(a, b)
        ref = a.astype(np.float64) @ b.astype(np.float64).T
        rel = (got - ref) / np.abs(ref)
        rel32 = ((a @ b.T) - ref) / np.abs(ref)
        print(f"\n{name}: 3xTF32 rel err max {np.abs(rel).max():.2e} mean {rel.mean():+.2e} rms {rel.std():.2e} | "
              f"fp32 sgemm max {np.abs(rel32).max():.2e} mean {rel32.mean():+.2e} rms {rel32.std():.2e}")


def _swish(x):
    return x / (1 + np.exp(-x))


def _swish_grad(z):
    s = 1 / (1 + np.exp(-z))
    return s * (1 + z * (1 - s))


GEMM_SHAPES = [
    (0, 300, 760, 128, 1), (0, 1000, 128, 12, 0), (0, 129, 47, 128, 1), (0, 64, 128, 2, 0),
    (1, 300, 128, 760, 0), (1, 777, 12, 128, 0), (1, 130, 128, 47, 0),
    (2, 128, 760, 5000, 1), (2, 12, 128, 4097, 0), (2, 128, 47, 300, 1), (2, 2, 128, 31, 0),
]
GEMMS = ["", "legacy", "simt"]


# the default GEMM ("") keeps the shape-only test ids
@pytest.mark.parametrize("mode,I,J,R,a_swish,gemm", [s + (g,) for g in GEMMS for s in GEMM_SHAPES],
                         ids=["-".join(map(str, s + ((g,) if g else ()))) for g in GEMMS for s in GEMM_SHAPES])
def test_umma_gemm_family(mode, I, J, R, a_swish, gemm, request):
    """The three GEMM shapes of the conditioner VJP, incl. ragged sizes, vs float64, on each train GEMM: "" = tcgen05
    fed by the copy engine where the operands allow (else register-path loaders), "legacy" = tcgen05 with
    register-path loaders, "simt" = the fp32 FFMA GEMM."""
    from zenflow_b200 import _lib

    _lib.set_impl(None, gemm or None)
    request.addfinalizer(lambda: _lib.set_impl(None))
    lib = _lib.load()
    rng = np.random.default_rng(mode * 1000 + I + J + R)
    st = torch.cuda.current_stream().cuda_stream
    cu = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).cuda()
    if mode == 0:
        A = rng.normal(size=(I, R)); B = rng.normal(size=(R, J)) / np.sqrt(R); bias = rng.normal(size=J)
        ref = (_swish(A) if a_swish else A) @ B + bias
        At, Bt, bt = cu(A), cu(B), cu(bias)
        Ct = torch.full((I, J), float("nan"), device="cuda")
        _lib.check(lib.zf_selftest_umma_gemm(st, 0, At.data_ptr(), R, Bt.data_ptr(), J, Ct.data_ptr(), J, bt.data_ptr(),
                                             None, None, 0, a_swish, I, J, R, 0))
    elif mode == 1:
        A = rng.normal(size=(I, R)); B = rng.normal(size=(J, R)) / np.sqrt(R); Z = rng.normal(size=(I, J))
        ref = (A @ B.T) * _swish_grad(Z)
        At, Bt, Zt = cu(A), cu(B), cu(Z)
        Ct = torch.full((I, J), float("nan"), device="cuda")
        _lib.check(lib.zf_selftest_umma_gemm(st, 1, At.data_ptr(), R, Bt.data_ptr(), R, Ct.data_ptr(), J, None, None,
                                             Zt.data_ptr(), J, 0, I, J, R, 0))
    else:
        A = rng.normal(size=(R, I)); B = rng.normal(size=(R, J)) / np.sqrt(R)
        C0 = rng.normal(size=(I, J)); cs0 = rng.normal(size=J)
        ref = C0 + (_swish(A) if a_swish else A).T @ B
        ref_cs = cs0 + B.sum(0)
        At, Bt, Ct, cst = cu(A), cu(B), cu(C0), cu(cs0)
        _lib.check(lib.zf_selftest_umma_gemm(st, 2, At.data_ptr(), I, Bt.data_ptr(), J, Ct.data_ptr(), J, None,
                                             cst.data_ptr(), None, 0, a_swish, I, J, R, 1024))
        np.testing.assert_allclose(cst.cpu().numpy(), ref_cs, rtol=1e-5, atol=1e-5)
    torch.cuda.synchronize()
    got = Ct.cpu().numpy()
    scale = np.abs(ref).max()
    err = np.abs(got - ref).max() / scale
    print(f"\nmode {mode} I={I} J={J} R={R}: max err / max|ref| = {err:.2e}")
    assert err < 5e-6


@pytest.mark.parametrize("mask_mode", [1, 2])
def test_umma_output_lane_mask(mask_mode):
    """The MMA's output-lane mask: masked tensor-memory lanes keep their previous contents (the half-tile
    chain kernel relies on it to run two 64-event pipelines on disjoint lanes of the same columns)."""
    from zenflow_b200 import _lib

    lib = _lib.load()
    rng = np.random.default_rng(3)
    N = K = 64
    A = rng.normal(size=(128, K)).astype(np.float32)
    B = (rng.normal(size=(N, K)) / np.sqrt(K)).astype(np.float32)
    At, Bt = torch.from_numpy(A).cuda(), torch.from_numpy(B).cuda()
    out = torch.zeros((128, N), device="cuda")
    _lib.check(lib.zf_selftest_umma(torch.cuda.current_stream().cuda_stream, At.data_ptr(), Bt.data_ptr(), N, K,
                                    out.data_ptr(), mask_mode))
    got = out.cpu().numpy()
    ref = A.astype(np.float64) @ B.astype(np.float64).T
    live = slice(0, 64) if mask_mode == 1 else slice(64, 128)
    kept = slice(64, 128) if mask_mode == 1 else slice(0, 64)
    assert np.abs(got[live] - ref[live]).max() < 1e-5
    assert (got[kept] == 777.0).all()


@pytest.mark.parametrize("N,K", [(128, 64), (96, 32), (16, 128)])
@pytest.mark.parametrize("flags", [0, 1, 2, 3])
def test_bf16x2_split_with_k_major_and_mn_major_operands(N, K, flags):
    """The train step's image GEMMs (csrc/zf_img_gemm.cu): kind::f16 on bf16 hi/lo parts, both operands in shared
    memory, each either K-major or MN-major (flags bit 0 / 1).  For an MN-major operand the descriptor's SBO is the
    stride between core matrices along MN and its LBO the stride along K; every combination gives the same product,
    at the 2^-17 relative accuracy of the two-part split."""
    from zenflow_b200 import _lib

    torch.manual_seed(N * 7 + K + flags)
    A = torch.randn(128, K, device="cuda")
    B = torch.randn(N, K, device="cuda")
    out = torch.full((128, N), float("nan"), device="cuda")
    _lib.check(_lib.load().zf_selftest_umma_bf16(torch.cuda.current_stream().cuda_stream, A.data_ptr(), B.data_ptr(), N, K,
                                                 out.data_ptr(), flags), "zf_selftest_umma_bf16")
    torch.cuda.synchronize()
    ref = A.double() @ B.double().T
    err = (out.double() - ref).abs().max().item() / ref.abs().max().item()
    assert err < 3e-5, err
