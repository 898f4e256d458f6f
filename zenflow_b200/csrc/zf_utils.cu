// The reference's L0 public functions on NORMALISED spline parameters (zenflow/utils.py):
//   zf_squareplus                  <- squareplus                          utils.py:18-20
//   zf_normalize_spline_params     <- normalize_spline_params             utils.py:37-62 (softmax_with_threshold :23-34)
//   zf_rqs_forward_normalized      <- rational_quadratic_spline_forward   utils.py:65-141
//   zf_rqs_inverse_normalized      <- rational_quadratic_spline_inverse   utils.py:144-202
// The hot path never materialises dx / dy / slope (zf_rqs_forward fuses the normalisation, zf_stage.cu); these
// entry points exist so that code written against zenflow.utils runs unchanged.  One thread per (event, dim) row,
// reference operation order with IEEE-rounded intrinsics: bin indices are bit-exact given the same dx / dy.
#include "zf_common.cuh"
#include "zf_math.cuh"

namespace zf {

__global__ void __launch_bounds__(256) squareplus_kernel(const float* __restrict__ x, long long n, float* __restrict__ y) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        y[i] = squareplus_rn(x[i]);
}

// theta row (3K-1 raw values) -> dx (K), dy (K), slope (K-1)
__global__ void __launch_bounds__(128) normalize_params_kernel(const float* __restrict__ theta, long long rows, int K,
                                                               float* __restrict__ dx, float* __restrict__ dy,
                                                               float* __restrict__ slope) {
    const KnotNorm kn = make_knot_norm(K);
    const int P = 3 * K - 1;
    for (long long r = blockIdx.x * (long long)blockDim.x + threadIdx.x; r < rows; r += (long long)gridDim.x * blockDim.x) {
        const float* th = theta + r * P;
#pragma unroll 1
        for (int blk = 0; blk < 2; ++blk) {
            const float* ps = th + blk * K;
            float* out = (blk == 0 ? dx : dy) + r * K;
            float sum = 0.f;
            for (int j = 0; j < K; ++j) {
                const float t = squareplus_rn(ps[j]);
                sum = j == 0 ? t : __fadd_rn(sum, t);
            }
            for (int j = 0; j < K; ++j) out[j] = knot_normalise_safe(squareplus_rn(ps[j]), sum, kn);
        }
        for (int j = 0; j < K - 1; ++j) slope[r * (K - 1) + j] = squareplus_rn(th[2 * K + j]);
    }
}

// _compute_rqs_input (utils.py:205-232) on normalised parameters: knots by sequential cumsum, bin by counting the
// knots <= v, gathers with JAX's fill-mode semantics for idx == K.
__device__ __forceinline__ void locate_normalized(const float* __restrict__ dxs, const float* __restrict__ dys,
                                                  const float* __restrict__ sl, int K, bool forward, float v, RqsBin& o) {
    const float* ps = forward ? dxs : dys;   // searched axis
    const float* po = forward ? dys : dxs;
    float acc = 0.f, acc_o = 0.f, ks = 0.f, ko = 0.f, bs = 0.f, bo = 0.f;
    int idx = 0;
    for (int j = 0; j < K; ++j) {
        const bool in = (j == 0) || (acc <= v);   // knot_j <= v (utils.py:246); knot_0 = 0 always counts via the clip
        if (in) { idx = j; ks = acc; ko = acc_o; bs = ps[j]; bo = po[j]; }
        acc = __fadd_rn(acc, ps[j]);
        acc_o = __fadd_rn(acc_o, po[j]);
    }
    if (acc <= v) { idx = K; ks = acc; ko = acc_o; bs = CUDART_NAN_F; bo = CUDART_NAN_F; }
    float dk = 1.0f, dkp1 = 1.0f;            // dk = pad(slope, 1 | 1, value 1)   (utils.py:211-216)
    if (idx >= 1 && idx <= K - 1) dk = sl[idx - 1];
    if (idx + 1 <= K - 1) dkp1 = sl[idx];
    else if (idx + 1 > K) dkp1 = CUDART_NAN_F;
    o.idx = idx; o.ks = ks; o.bs = bs; o.ko = ko; o.bo = bo; o.dk = dk; o.dkp1 = dkp1;
}

template <bool INVERSE>
__global__ void __launch_bounds__(128) rqs_normalized_kernel(const float* __restrict__ v_in, const float* __restrict__ dx,
                                                             const float* __restrict__ dy, const float* __restrict__ slope,
                                                             long long M, int d, int K, float* __restrict__ out,
                                                             float* __restrict__ log_det, int* __restrict__ idx_out) {
    // one thread per event: the log-det is the sum over the event's dims in order (utils.py:139)
    for (long long m = blockIdx.x * (long long)blockDim.x + threadIdx.x; m < M; m += (long long)gridDim.x * blockDim.x) {
        float ld_sum = 0.f;
        for (int j = 0; j < d; ++j) {
            const long long r = m * d + j;
            const float v = v_in[r];
            RqsBin b;
            locate_normalized(dx + r * K, dy + r * K, slope + r * (K - 1), K, !INVERSE, v, b);
            if (idx_out) idx_out[r] = b.idx;
            if (!INVERSE) {
                float y, ld;
                rqs_eval_forward(v, b, y, ld);
                out[r] = y;
                ld_sum = j == 0 ? ld : ld_sum + ld;
            } else {
                out[r] = rqs_eval_inverse(v, b);
            }
        }
        if (!INVERSE && log_det) log_det[m] = ld_sum;
    }
}

static unsigned util_grid(long long n, int per_block) {
    long long b = (n + per_block - 1) / per_block;
    if (b < 1) b = 1;
    if (b > 148 * 16) b = 148 * 16;
    return (unsigned)b;
}

}  // namespace zf

using namespace zf;

extern "C" int zf_squareplus(void* stream, const float* x, int64_t n, float* y) {
    ZF_REQUIRE(n >= 0 && (n == 0 || (x && y)), "squareplus: bad argument");
    if (n == 0) return ZF_OK;
    squareplus_kernel<<<util_grid(n, 256 * 4), 256, 0, (cudaStream_t)stream>>>(x, n, y);
    count_launch();
    ZF_CUDA_CHECK(cudaGetLastError());
    return ZF_OK;
}

extern "C" int zf_normalize_spline_params(void* stream, const float* theta, int64_t rows, int32_t K, float* dx, float* dy,
                                          float* slope) {
    ZF_REQUIRE(rows >= 0 && K >= 1 && (rows == 0 || (theta && dx && dy && (slope || K == 1))), "normalize_spline_params: bad argument");
    if (rows == 0) return ZF_OK;
    normalize_params_kernel<<<util_grid(rows, 128), 128, 0, (cudaStream_t)stream>>>(theta, rows, K, dx, dy, slope);
    count_launch();
    ZF_CUDA_CHECK(cudaGetLastError());
    return ZF_OK;
}

extern "C" int zf_rqs_forward_normalized(void* stream, const float* x, const float* dx, const float* dy, const float* slope,
                                         int64_t M, int32_t d, int32_t K, float* y, float* log_det, int32_t* idx) {
    ZF_REQUIRE(M >= 0 && d >= 1 && K >= 1, "rqs_forward_normalized: bad shape");
    if (M == 0) return ZF_OK;
    ZF_REQUIRE(x && dx && dy && (slope || K == 1) && y, "rqs_forward_normalized: null argument");
    rqs_normalized_kernel<false><<<util_grid(M, 128), 128, 0, (cudaStream_t)stream>>>(x, dx, dy, slope, M, d, K, y, log_det, idx);
    count_launch();
    ZF_CUDA_CHECK(cudaGetLastError());
    return ZF_OK;
}

extern "C" int zf_rqs_inverse_normalized(void* stream, const float* y, const float* dx, const float* dy, const float* slope,
                                         int64_t M, int32_t d, int32_t K, float* x, int32_t* idx) {
    ZF_REQUIRE(M >= 0 && d >= 1 && K >= 1, "rqs_inverse_normalized: bad shape");
    if (M == 0) return ZF_OK;
    ZF_REQUIRE(y && dx && dy && (slope || K == 1) && x, "rqs_inverse_normalized: null argument");
    rqs_normalized_kernel<true><<<util_grid(M, 128), 128, 0, (cudaStream_t)stream>>>(y, dx, dy, slope, M, d, K, x, nullptr, idx);
    count_launch();
    ZF_CUDA_CHECK(cudaGetLastError());
    return ZF_OK;
}
