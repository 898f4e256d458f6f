// Deep-Set conditioner Phi (examples/deep_set.ipynb:138-160): the step on the other side of `c` in
// BASELINE config "deep_set" (SURVEY.md 8f-4):
//     BatchNorm -> NNBlock(out, depth, width) = (Dense + swish) x depth, Dense(out) -> Dropout(rate) -> sum_matrix @ .
// sum_matrix is the notebook's BCOO matrix of ones (deep_set.ipynb:60-74): a COO list (set, row) that sum-pools the
// per-element embeddings of each set; rows outside every set (the padding to 50,000 rows) contribute nothing to c but
// DO enter the train-mode BatchNorm moments, exactly as in the notebook.
//
//   zf_phi_forward   c (S, out) from x (N, in); train mode uses batch moments, updates the running statistics and
//                    keeps the layer pre-activations in the workspace for zf_phi_backward
//   zf_phi_backward  parameter cotangents (+=) from gc (S, out) = d loss / d c (what zf_flow_value_and_grad returns)
// The Dense layers run on the train step's tcgen05 GEMM family (zf_umma_gemm.cu); BatchNorm, dropout and the pooling
// are small SIMT kernels.  Dropout draws its keep-mask from Philox keyed by (seed, row, column) (jax's threefry
// stream cannot be reproduced without JAX) or takes an explicit multiplier matrix (parity tests).
#include "zf_common.cuh"
#include "zf_math.cuh"
#include "zf_rng.cuh"

#include <algorithm>

namespace zf {

// sums[f] = sum_n x[n][f], sums[F + f] = sum_n x[n][f]^2 (double)
__global__ void __launch_bounds__(256) phi_moments_kernel(const float* __restrict__ x, long long N, int F, double* sums) {
    extern __shared__ double sh[];
    for (int i = threadIdx.x; i < 2 * F; i += blockDim.x) sh[i] = 0.0;
    __syncthreads();
    const int R = blockDim.x / F, r = threadIdx.x / F, f = threadIdx.x - r * F;
    if (r < R) {
        double s1 = 0.0, s2 = 0.0;
        for (long long n = (long long)blockIdx.x * R + r; n < N; n += (long long)gridDim.x * R) {
            const double v = (double)x[n * F + f];
            s1 += v;
            s2 += v * v;
        }
        atomicAdd(&sh[f], s1);
        atomicAdd(&sh[F + f], s2);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 2 * F; i += blockDim.x) atomicAdd(&sums[i], sh[i]);
}

// flax BatchNorm: (x - mean) * (rsqrt(var + eps) * scale) + bias
__global__ void __launch_bounds__(256) phi_bn_apply_kernel(const float* __restrict__ x, long long N, int F,
                                                           const float* __restrict__ scale, const float* __restrict__ bias,
                                                           const float* __restrict__ mean, const float* __restrict__ var,
                                                           float* __restrict__ h0) {
    const long long n = N * F;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
        const int f = (int)(e % F);
        const float mul = __fdiv_rn(1.0f, __fsqrt_rn(__fadd_rn(var[f], 1e-5f))) * scale[f];
        h0[e] = (x[e] - mean[f]) * mul + bias[f];
    }
}

// d/d(scale), d/d(bias) of the train-mode BatchNorm: sum g * xhat, sum g  (x itself is data: no cotangent needed)
__global__ void __launch_bounds__(256) phi_bn_param_grads_kernel(const float* __restrict__ x, const float* __restrict__ g,
                                                                 long long N, int F, const float* __restrict__ mean,
                                                                 const float* __restrict__ var, double* sums) {
    extern __shared__ double sh[];
    for (int i = threadIdx.x; i < 2 * F; i += blockDim.x) sh[i] = 0.0;
    __syncthreads();
    const int R = blockDim.x / F, r = threadIdx.x / F, f = threadIdx.x - r * F;
    if (r < R) {
        const float mu = mean[f], rstd = __fdiv_rn(1.0f, __fsqrt_rn(__fadd_rn(var[f], 1e-5f)));
        double s1 = 0.0, s2 = 0.0;
        for (long long n = (long long)blockIdx.x * R + r; n < N; n += (long long)gridDim.x * R) {
            const float gg = g[n * F + f];
            s1 += (double)gg;
            s2 += (double)gg * (double)((x[n * F + f] - mu) * rstd);
        }
        atomicAdd(&sh[f], s1);
        atomicAdd(&sh[F + f], s2);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 2 * F; i += blockDim.x) atomicAdd(&sums[i], sh[i]);
}

__device__ __forceinline__ float dropout_mult(const float* __restrict__ mask, long long row, int col, int O, int train,
                                              float rate, unsigned long long seed) {
    if (mask) return mask[row * O + col];
    if (!train || rate <= 0.f) return 1.0f;
    LatentRng rng(seed ^ 0xD509A7E5C3B1F00Dull, row, col);
    return rng.uniform() >= rate ? 1.0f / (1.0f - rate) : 0.0f;   // keep with probability 1 - rate, flax scaling
}

// c[set] += dropout(o[row])   over the COO entries of the sum matrix
__global__ void __launch_bounds__(256) phi_pool_kernel(const float* __restrict__ o, const int* __restrict__ set_idx,
                                                       const int* __restrict__ row_idx, long long nnz, int O, long long N,
                                                       long long S, const float* __restrict__ mask, int train, float rate,
                                                       unsigned long long seed, float* __restrict__ c) {
    const long long n = nnz * O;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
        const long long k = e / O;
        const int col = (int)(e - k * O);
        const long long row = row_idx[k], set = set_idx[k];
        if (row < 0 || row >= N || set < 0 || set >= S) continue;
        atomicAdd(&c[set * O + col], o[row * O + col] * dropout_mult(mask, row, col, O, train, rate, seed));
    }
}

// go[row] += dropout multiplier * gc[set]   (the transpose of the pooling)
__global__ void __launch_bounds__(256) phi_unpool_kernel(const float* __restrict__ gc, const int* __restrict__ set_idx,
                                                         const int* __restrict__ row_idx, long long nnz, int O, long long N,
                                                         long long S, const float* __restrict__ mask, int train, float rate,
                                                         unsigned long long seed, float* __restrict__ go) {
    const long long n = nnz * O;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
        const long long k = e / O;
        const int col = (int)(e - k * O);
        const long long row = row_idx[k], set = set_idx[k];
        if (row < 0 || row >= N || set < 0 || set >= S) continue;
        atomicAdd(&go[row * O + col], gc[set * O + col] * dropout_mult(mask, row, col, O, train, rate, seed));
    }
}

__global__ void phi_bn_grads_add_kernel(const double* sums, int F, float* gscale, float* gbias) {
    const int f = threadIdx.x;
    if (f < F) {
        gbias[f] += (float)sums[f];
        gscale[f] += (float)sums[F + f];
    }
}

static unsigned phi_grid(long long n, int per_block, int cap) {
    long long b = (n + per_block - 1) / per_block;
    return (unsigned)std::min<long long>(std::max<long long>(b, 1), cap);
}

struct PhiPlan {
    int L;                       // hidden layers
    int widths[ZF_MAX_LAYERS + 2];   // in, hidden..., out
    size_t off_act[ZF_MAX_LAYERS + 2];   // floats: H0 | Z_1 .. Z_L | O
    size_t off_g[2];             // two gradient ping-pong buffers (N x max width)
    size_t off_stats;            // bmean[F] bvar[F] (float) then 2F doubles
    size_t total_bytes;
};

static int phi_plan(const zf_phi* phi, long long N, PhiPlan& p) {
    ZF_REQUIRE(phi != nullptr, "phi is NULL");
    ZF_REQUIRE(phi->in_dim >= 1 && phi->in_dim <= 256 && phi->out_dim >= 1, "phi: bad in_dim / out_dim");
    ZF_REQUIRE(phi->n_hidden >= 0 && phi->n_hidden <= ZF_MAX_LAYERS, "phi: at most %d hidden layers", ZF_MAX_LAYERS);
    ZF_REQUIRE(N >= 1, "phi: N must be >= 1");
    p.L = phi->n_hidden;
    p.widths[0] = phi->in_dim;
    int wmax = std::max(phi->in_dim, phi->out_dim);
    for (int l = 0; l < p.L; ++l) {
        ZF_REQUIRE(phi->hidden[l] >= 1, "phi: layer width must be positive");
        p.widths[l + 1] = phi->hidden[l];
        wmax = std::max(wmax, phi->hidden[l]);
    }
    p.widths[p.L + 1] = phi->out_dim;
    size_t off = 0;
    auto take = [&](size_t floats) { size_t o = off; off += (floats + 63) / 64 * 64; return o; };
    for (int l = 0; l <= p.L + 1; ++l) p.off_act[l] = take((size_t)N * p.widths[l]);
    p.off_g[0] = take((size_t)N * wmax);
    p.off_g[1] = take((size_t)N * wmax);
    p.off_stats = take((size_t)2 * phi->in_dim + (size_t)4 * phi->in_dim + 16);
    p.total_bytes = off * sizeof(float);
    return ZF_OK;
}

}  // namespace zf

using namespace zf;

extern "C" size_t zf_phi_workspace_bytes(const zf_phi* phi, int64_t N) {
    PhiPlan p;
    if (phi_plan(phi, N, p) != ZF_OK) return 0;
    return p.total_bytes;
}

extern "C" int zf_phi_forward(void* stream, const zf_phi* phi, const float* x, int64_t N, const int32_t* set_idx,
                              const int32_t* row_idx, int64_t nnz, int64_t S, int32_t train, float dropout_rate,
                              uint64_t dropout_seed, const float* dropout_mask, float* c_out, void* workspace,
                              size_t workspace_bytes) {
    PhiPlan p;
    if (int rc = phi_plan(phi, N, p)) return rc;
    ZF_REQUIRE(x && c_out && workspace && (nnz == 0 || (set_idx && row_idx)) && S >= 1 && nnz >= 0, "phi_forward: bad argument");
    ZF_REQUIRE(dropout_rate >= 0.f && dropout_rate < 1.f, "phi_forward: dropout rate must be in [0, 1)");
    ZF_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "phi_forward: workspace must be 256-byte aligned");
    if (workspace_bytes < p.total_bytes) return fail(ZF_ERR_WORKSPACE, "phi_forward: workspace too small");
    ZF_REQUIRE(phi->bn_scale && phi->bn_bias && phi->bn_mean && phi->bn_var, "phi_forward: BatchNorm leaf is NULL");
    cudaStream_t st = (cudaStream_t)stream;
    float* ws = static_cast<float*>(workspace);
    const int F = phi->in_dim, O = phi->out_dim, L = p.L;
    float* bmean = ws + p.off_stats;
    float* bvar = bmean + F;
    double* sums = reinterpret_cast<double*>(ws + p.off_stats + 2 * F + ((2 * F) & 1));
    const float *mean = phi->bn_mean, *var = phi->bn_var;
    if (train) {   // batch moments over ALL rows (the notebook normalises the padded array), running stats updated
        ZF_CUDA_CHECK(cudaMemsetAsync(sums, 0, 2 * F * sizeof(double), st));
        phi_moments_kernel<<<phi_grid(N, (256 / F) * 64, 148 * 4), 256, 2 * F * sizeof(double), st>>>(x, N, F, sums);
        count_launch();
        if (int rc = zf_bn_finalize(st, sums, (double)N, F, 0.99f, bmean, bvar, phi->bn_mean, phi->bn_var)) return rc;
        mean = bmean;
        var = bvar;
    }
    phi_bn_apply_kernel<<<phi_grid(N * F, 256 * 8, 148 * 8), 256, 0, st>>>(x, N, F, phi->bn_scale, phi->bn_bias, mean, var,
                                                                           ws + p.off_act[0]);
    count_launch();
    for (int l = 0; l <= L; ++l) {   // Z_{l+1} = act(Z_l) W_l + b_l (pre-activations are kept)
        ZF_REQUIRE(phi->kernel[l] && phi->bias[l], "phi_forward: Dense_%d leaf is NULL", l);
        if (int rc = launch_umma_gemm(st, 0, ws + p.off_act[l], p.widths[l], phi->kernel[l], p.widths[l + 1],
                                      ws + p.off_act[l + 1], p.widths[l + 1], phi->bias[l], nullptr, nullptr, 0, l > 0, N,
                                      p.widths[l + 1], p.widths[l], 0))
            return rc;
    }
    ZF_CUDA_CHECK(cudaMemsetAsync(c_out, 0, (size_t)S * O * sizeof(float), st));
    if (nnz > 0) {
        phi_pool_kernel<<<phi_grid(nnz * O, 256 * 4, 148 * 8), 256, 0, st>>>(ws + p.off_act[L + 1], set_idx, row_idx, nnz, O, N, S,
                                                                             dropout_mask, train, dropout_rate, dropout_seed,
                                                                             c_out);
        count_launch();
    }
    ZF_CUDA_CHECK(cudaGetLastError());
    return ZF_OK;
}

extern "C" int zf_phi_backward(void* stream, const zf_phi* phi, const zf_coupling_grads* grads, const float* x, int64_t N,
                               const int32_t* set_idx, const int32_t* row_idx, int64_t nnz, int64_t S, float dropout_rate,
                               uint64_t dropout_seed, const float* dropout_mask, const float* gc, void* workspace,
                               size_t workspace_bytes) {
    PhiPlan p;
    if (int rc = phi_plan(phi, N, p)) return rc;
    ZF_REQUIRE(x && gc && grads && workspace && (nnz == 0 || (set_idx && row_idx)) && S >= 1, "phi_backward: bad argument");
    if (workspace_bytes < p.total_bytes) return fail(ZF_ERR_WORKSPACE, "phi_backward: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    float* ws = static_cast<float*>(workspace);
    const int F = phi->in_dim, O = phi->out_dim, L = p.L;
    float* bmean = ws + p.off_stats;
    float* bvar = bmean + F;
    double* sums = reinterpret_cast<double*>(ws + p.off_stats + 2 * F + ((2 * F) & 1));
    float* gcur = ws + p.off_g[0];
    float* gnext = ws + p.off_g[1];
    // cotangent of the Dense(out) output: the transpose of the pooling, through the same dropout multipliers
    ZF_CUDA_CHECK(cudaMemsetAsync(gcur, 0, (size_t)N * O * sizeof(float), st));
    if (nnz > 0) {
        phi_unpool_kernel<<<phi_grid(nnz * O, 256 * 4, 148 * 8), 256, 0, st>>>(gc, set_idx, row_idx, nnz, O, N, S, dropout_mask, 1,
                                                                               dropout_rate, dropout_seed, gcur);
        count_launch();
    }
    for (int l = L; l >= 0; --l) {
        ZF_REQUIRE(grads->kernel[l] && grads->bias[l], "phi_backward: Dense_%d gradient leaf is NULL", l);
        // dW_l += act(Z_l)^T dZ_{l+1}, db_l += colsum(dZ_{l+1})
        if (int rc = launch_umma_gemm(st, 2, ws + p.off_act[l], p.widths[l], gcur, p.widths[l + 1], grads->kernel[l],
                                      p.widths[l + 1], nullptr, grads->bias[l], nullptr, 0, l > 0, p.widths[l], p.widths[l + 1],
                                      N, 2048))
            return rc;
        // dZ_l = (dZ_{l+1} W_l^T) * swish'(Z_l)   (l = 0: d/d(BatchNorm output), no activation)
        if (int rc = launch_umma_gemm(st, 1, gcur, p.widths[l + 1], phi->kernel[l], p.widths[l + 1], gnext, p.widths[l], nullptr,
                                      nullptr, l == 0 ? nullptr : ws + p.off_act[l], p.widths[l], 0, N, p.widths[l],
                                      p.widths[l + 1], 0))
            return rc;
        std::swap(gcur, gnext);
    }
    // BatchNorm parameters (train-mode statistics of the matching forward are still in the workspace)
    ZF_REQUIRE(grads->bn_scale && grads->bn_bias, "phi_backward: BatchNorm gradient leaf is NULL");
    ZF_CUDA_CHECK(cudaMemsetAsync(sums, 0, 2 * F * sizeof(double), st));
    phi_bn_param_grads_kernel<<<phi_grid(N, (256 / F) * 64, 148 * 4), 256, 2 * F * sizeof(double), st>>>(x, gcur, N, F, bmean, bvar,
                                                                                                        sums);
    phi_bn_grads_add_kernel<<<1, 256, 0, st>>>(sums, F, grads->bn_scale, grads->bn_bias);
    count_launch(); count_launch();
    ZF_CUDA_CHECK(cudaGetLastError());
    return ZF_OK;
}
