// Train-mode kernels: everything train.py:64-86 (loss_fn + jax.grad + optax update) needs
// beyond the eval chain kernel.  The reference has no hand-written backward (jax.grad does it);
// the derivatives here follow the as-computed forward expressions incl. every +EPS
// (SURVEY.md Appendix A) and are checked against float64 autograd of the oracle.
//
// The batch couples samples in train mode (BatchNorm batch moments, ShiftBounds batch
// min/max), so the step is a sequence of phases; between phases the host may all-reduce the
// small statistics across ranks (NCCL) - see zenflow_b200/_train.py.
//
//   zf_shift_bounds_minmax / _update   <- bijectors.py:250-260
//   zf_bn_moments / zf_bn_finalize      <- flax BatchNorm(use_running_average=False), bijectors.py:342
//   zf_flow_loss_grad                   <- flow.py:46-47 + train.py:73 (-mean) and d/dz of the latent
//   zf_coupling_backward                <- VJP of bijectors.py:329-365 (conditioner recompute + spline VJP)
//   zf_bn_backward_apply                <- VJP of train-mode BatchNorm into x and c
//   zf_nadamw_update                    <- optax.nadamw / adamw (train.py:12-15,84-85)
#include "zf_common.cuh"
#include "zf_math.cuh"
#include "zf_vjp.cuh"

#include <float.h>
#include <stdlib.h>
#include <algorithm>

namespace zf {

// ---------------------------------------------------------------------------------------------
// ShiftBounds batch min/max
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned f2ord(float f) {
    unsigned u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ord2f(unsigned u) {
    return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}

struct SbCols {
    int kind[ZF_MAX_DIM];
    float lo[ZF_MAX_DIM], hi[ZF_MAX_DIM];
};

__global__ void minmax_init_kernel(unsigned* enc, int D) {
    int i = threadIdx.x;
    if (i < D) { enc[i] = 0xffffffffu; enc[D + i] = 0u; }
}

__global__ void __launch_bounds__(256) minmax_kernel(const __grid_constant__ SbCols cols, const float* __restrict__ x,
                                                     long long M, int D, unsigned* enc) {
    __shared__ unsigned smin[ZF_MAX_DIM], smax[ZF_MAX_DIM];
    if (threadIdx.x < D) { smin[threadIdx.x] = 0xffffffffu; smax[threadIdx.x] = 0u; }
    __syncthreads();
    const long long n = M * D;
    const long long gtid = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const long long gsz = (long long)gridDim.x * blockDim.x;
    // coalesced sweep over the row-major batch; per-column results meet in shared-memory atomics
    // (this pass is tiny next to the conditioner GEMMs)
    for (long long e = gtid; e < n; e += gsz) {
        const int j = (int)(e % D);
        float v = x[e];
        const int kind = cols.kind[j];
        if (kind == ZF_BOUND_BOTH) continue;
        if (kind == ZF_BOUND_LOWER) v = logf(__fadd_rn(__fsub_rn(v, cols.lo[j]), FLT_MIN));
        if (kind == ZF_BOUND_UPPER) v = logf(__fadd_rn(__fsub_rn(cols.hi[j], v), FLT_MIN));
        if (v != v) continue;
        const unsigned o = f2ord(v);
        atomicMin(&smin[j], o);
        atomicMax(&smax[j], o);
    }
    __syncthreads();
    if (threadIdx.x < D) {
        atomicMin(&enc[threadIdx.x], smin[threadIdx.x]);
        atomicMax(&enc[D + threadIdx.x], smax[threadIdx.x]);
    }
}

__global__ void minmax_decode_kernel(const unsigned* enc, float* out, int D) {
    int i = threadIdx.x;
    if (i < 2 * D) out[i] = ord2f(enc[i]);
}

// bijectors.py:250-260: widen by the margin, merge with the running values, store.
__global__ void sb_update_kernel(const __grid_constant__ SbCols cols, float margin, const float* minmax, float* xmin,
                                 float* xmax, int D) {
    int i = threadIdx.x;
    if (i >= D || cols.kind[i] == ZF_BOUND_BOTH) return;
    float lo = minmax[i], hi = minmax[D + i];
    float delta = __fmul_rn(__fmul_rn(0.5f, __fsub_rn(hi, lo)), margin);
    lo = __fsub_rn(lo, delta);
    hi = __fadd_rn(hi, delta);
    xmin[i] = fminf(xmin[i], lo);
    xmax[i] = fmaxf(xmax[i], hi);
}

// ---------------------------------------------------------------------------------------------
// BatchNorm train statistics: h = hstack(x[:, d:], c)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float cond_feature(const float* __restrict__ x, const float* __restrict__ c, long long m,
                                              int f, int D, int d, int C) {
    return (f < D - d) ? x[m * D + d + f] : c[m * C + (f - (D - d))];
}

// (s1, s2) of the threads that share feature f -> sh[f], sh[F + f].  Shared-memory double atomics are
// compare-and-swap loops, so 256 / F threads on one address serialise: when F is a power of two the lanes of a
// warp that hold the same feature (F apart) are summed with shuffles first.  Every thread of the block must call.
__device__ __forceinline__ void feature_sums_to_shared(double s1, double s2, int f, int F, bool valid, double* sh) {
    if (F <= 32 && (F & (F - 1)) == 0) {
        for (int o = F; o < 32; o <<= 1) {
            s1 += __shfl_xor_sync(0xffffffffu, s1, o);
            s2 += __shfl_xor_sync(0xffffffffu, s2, o);
        }
        valid = valid && (threadIdx.x & 31) < F;
    }
    if (valid) {
        atomicAdd(&sh[f], s1);
        atomicAdd(&sh[F + f], s2);
    }
}

// sums[f] += sum_m h, sums[F+f] += sum_m h^2 (double)
__global__ void __launch_bounds__(256) bn_moments_kernel(const float* __restrict__ x, const float* __restrict__ c,
                                                         long long M, int D, int C, double* sums) {
    const int d = D / 2, F = D - d + C;
    extern __shared__ double sh[];  // [2][F]
    for (int i = threadIdx.x; i < 2 * F; i += blockDim.x) sh[i] = 0.0;
    __syncthreads();
    const int R = blockDim.x / F;  // rows per pass
    const int r = threadIdx.x / F, f = threadIdx.x - r * F;
    double s1 = 0.0, s2 = 0.0;
    if (r < R) {
        const long long step = (long long)gridDim.x * R;
        long long m = (long long)blockIdx.x * R + r;
        for (; m + 3 * step < M; m += 4 * step) {   // four rows in flight per thread (the loads are the whole cost)
            float h[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) h[k] = cond_feature(x, c, m + k * step, f, D, d, C);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                s1 += (double)h[k];
                s2 += (double)h[k] * (double)h[k];
            }
        }
        for (; m < M; m += step) {
            const float h = cond_feature(x, c, m, f, D, d, C);
            s1 += (double)h;
            s2 += (double)h * (double)h;
        }
    }
    feature_sums_to_shared(s1, s2, f, F, r < R, sh);
    __syncthreads();
    for (int i = threadIdx.x; i < 2 * F; i += blockDim.x) atomicAdd(&sums[i], sh[i]);
}

// mean, biased variance via E[x^2]-E[x]^2 clipped at 0, running update with momentum
__global__ void bn_finalize_kernel(const double* sums, double count, int F, float momentum, float* bmean, float* bvar,
                                   float* ra_mean, float* ra_var) {
    int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= F) return;
    const float mean = (float)(sums[f] / count);
    const float mean2 = (float)(sums[F + f] / count);
    const float var = fmaxf(0.f, __fsub_rn(mean2, __fmul_rn(mean, mean)));
    bmean[f] = mean;
    bvar[f] = var;
    if (ra_mean) ra_mean[f] = __fadd_rn(__fmul_rn(momentum, ra_mean[f]), __fmul_rn((float)(1.0 - (double)momentum), mean));
    if (ra_var) ra_var[f] = __fadd_rn(__fmul_rn(momentum, ra_var[f]), __fmul_rn((float)(1.0 - (double)momentum), var));
}

// H0[m][f] = (h - mean) * (rsqrt(var+eps)*scale) + bias      (row stride F)
__global__ void __launch_bounds__(256) bn_apply_kernel(const float* __restrict__ x, const float* __restrict__ c,
                                                       long long M, int D, int C, const float* __restrict__ scale,
                                                       const float* __restrict__ bias, const float* __restrict__ mean,
                                                       const float* __restrict__ var, float* __restrict__ H0) {
    const int d = D / 2, F = D - d + C;
    const long long n = M * F;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
        const long long m = e / F;
        const int f = (int)(e - m * F);
        const float h = cond_feature(x, c, m, f, D, d, C);
        const float mul = __fdiv_rn(1.0f, __fsqrt_rn(__fadd_rn(var[f], 1e-5f))) * scale[f];
        H0[e] = (h - mean[f]) * mul + bias[f];
    }
}

// sums[f] += sum_m g, sums[F+f] += sum_m g*xhat   (xhat = (h-mean)*rstd)
__global__ void __launch_bounds__(256) bn_bwd_sums_kernel(const float* __restrict__ x, const float* __restrict__ c,
                                                          const float* __restrict__ g, long long M, int D, int C,
                                                          const float* __restrict__ mean, const float* __restrict__ var,
                                                          double* sums) {
    const int d = D / 2, F = D - d + C;
    extern __shared__ double sh[];
    for (int i = threadIdx.x; i < 2 * F; i += blockDim.x) sh[i] = 0.0;
    __syncthreads();
    const int R = blockDim.x / F;
    const int r = threadIdx.x / F, f = threadIdx.x - r * F;
    double s1 = 0.0, s2 = 0.0;
    if (r < R) {
        const float mu = mean[f];
        const float rstd = __fdiv_rn(1.0f, __fsqrt_rn(__fadd_rn(var[f], 1e-5f)));
        const long long step = (long long)gridDim.x * R;
        long long m = (long long)blockIdx.x * R + r;
        for (; m + 3 * step < M; m += 4 * step) {   // four rows in flight per thread (the loads are the whole cost)
            float h[4], gg[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                h[k] = cond_feature(x, c, m + k * step, f, D, d, C);
                gg[k] = g[(m + k * step) * F + f];
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                s1 += (double)gg[k];
                s2 += (double)gg[k] * (double)((h[k] - mu) * rstd);
            }
        }
        for (; m < M; m += step) {
            const float h = cond_feature(x, c, m, f, D, d, C);
            const float gg = g[m * F + f];
            s1 += (double)gg;
            s2 += (double)gg * (double)((h - mu) * rstd);
        }
    }
    feature_sums_to_shared(s1, s2, f, F, r < R, sh);
    __syncthreads();
    for (int i = threadIdx.x; i < 2 * F; i += blockDim.x) atomicAdd(&sums[i], sh[i]);
}

// dh = scale*rstd*(g - S1/N - xhat*S2/N); gx[:, d+f] += dh (f < D-d), gc[:, f-(D-d)] += dh
__global__ void __launch_bounds__(256) bn_bwd_apply_kernel(const float* __restrict__ x, const float* __restrict__ c,
                                                           const float* __restrict__ g, long long M, int D, int C,
                                                           const float* __restrict__ scale, const float* __restrict__ mean,
                                                           const float* __restrict__ var, const double* __restrict__ sums,
                                                           double count, float* __restrict__ gx, float* __restrict__ gc) {
    const int d = D / 2, F = D - d + C;
    // per-feature constants once per block: scale * rstd, mean, rstd, sum(g) / count, sum(g xhat) / count
    extern __shared__ float shc[];
    for (int f = threadIdx.x; f < F; f += blockDim.x) {
        const float rstd = __fdiv_rn(1.0f, __fsqrt_rn(__fadd_rn(var[f], 1e-5f)));
        shc[f] = scale[f] * rstd;
        shc[F + f] = mean[f];
        shc[2 * F + f] = rstd;
        shc[3 * F + f] = (float)(sums[f] / count);
        shc[4 * F + f] = (float)(sums[F + f] / count);
    }
    __syncthreads();
    // thread = (row r of the pass, feature f): consecutive threads read consecutive elements of g
    const int R = blockDim.x / F;
    const int r = threadIdx.x / F, f = threadIdx.x - r * F;
    if (r >= R) return;
    const float a = shc[f], mu = shc[F + f], rstd = shc[2 * F + f], s1 = shc[3 * F + f], s2 = shc[4 * F + f];
    const bool to_x = f < D - d;
    const long long step = (long long)gridDim.x * R;
    auto apply = [&](long long m, float h, float gg) {
        const float xhat = (h - mu) * rstd;
        const float dh = a * (gg - s1 - xhat * s2);
        if (to_x) gx[m * D + d + f] += dh;
        else if (gc) gc[m * C + (f - (D - d))] += dh;
    };
    long long m = (long long)blockIdx.x * R + r;
    for (; m + 3 * step < M; m += 4 * step) {   // four rows in flight per thread
        float h[4], gg[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            h[k] = cond_feature(x, c, m + k * step, f, D, d, C);
            gg[k] = g[(m + k * step) * F + f];
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) apply(m + k * step, h[k], gg[k]);
    }
    for (; m < M; m += step) apply(m, cond_feature(x, c, m, f, D, d, C), g[m * F + f]);
}

// ---------------------------------------------------------------------------------------------
// loss and latent gradient
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) loss_grad_kernel(LatentConst lc, const float* __restrict__ z,
                                                        const float* __restrict__ log_det, long long M, int D,
                                                        float wgt, const float* __restrict__ cot,
                                                        float* __restrict__ lp_out, float* __restrict__ gz,
                                                        float* __restrict__ glp, double* lp_sum) {
    __shared__ double red[256];
    double local = 0.0;
    for (long long m = blockIdx.x * (long long)blockDim.x + threadIdx.x; m < M; m += (long long)gridDim.x * blockDim.x) {
        float lat = 0.f;
        for (int j = 0; j < D; ++j) lat += latent_logpdf(z[m * D + j], lc);
        const float raw = lat + log_det[m];
        const float lp = nan_to_num_lp(raw);
        const bool fin = (raw == raw) && fabsf(raw) <= FLT_MAX;
        const float w = fin ? (cot ? cot[m] : wgt) : 0.f;   // nan_to_num replaces non-finite lp by constants: zero gradient
        if (lp_out) lp_out[m] = lp;
        glp[m] = w;
        local += (double)lp;
        for (int j = 0; j < D; ++j) {
            const float v = z[m * D + j];
            float dl = 0.f;
            if (lc.kind == kLatentBeta) dl = (v > 1.f || v < 0.f) ? 0.f : (lc.p1 / v - lc.p1 / (1.f - v));
            else if (lc.kind == kLatentNormal) dl = -(v - 0.5f) / 0.01f;
            else if (lc.kind == kLatentTruncNormal) dl = (v > 1.f || v < 0.f) ? 0.f : -(v - 0.5f) / 0.01f;
            gz[m * D + j] = w * dl;
        }
    }
    red[threadIdx.x] = local;
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) {
        if (threadIdx.x < s) red[threadIdx.x] += red[threadIdx.x + s];
        __syncthreads();
    }
    if (threadIdx.x == 0) atomicAdd(lp_sum, red[0]);
}

// ---------------------------------------------------------------------------------------------
// generic fp32 GEMM family for the conditioner recompute / backward (64x64x16 tiles, 4x4 per thread)
//   mode 0 (NN): C[m][n]  = sum_k opA(A[m][k]) * B[k][n] + bias[n]
//   mode 1 (NT): C[m][k]  = (sum_n A[m][n] * B[k][n]) * swish'(Z[m][k])          (Z optional)
//   mode 2 (TN): C[k][n] += sum_m opA(A[m][k]) * B[m][n];  colsum[n] += sum_m B[m][n]
// opA = the activation `act` (swish by default) when a_swish: stored pre-activations are re-activated on load.
// ---------------------------------------------------------------------------------------------
struct GemmArgs {
    const float* A; long long lda;
    const float* B; long long ldb;
    float* C; long long ldc;
    const float* bias;
    float* colsum;
    const float* Z; long long ldz;
    int a_swish;         // apply the activation to A on load
    int act;             // zf_act_kind (0 = swish) of opA and of the derivative that multiplies mode 1's product
    long long I, J, R;   // output rows, output cols, reduction length
    long long r_slab;    // mode 2: reduction rows per CTA (gridDim.z slabs)
};

constexpr int GT = 64, GK = 16, GS = 68;


// pattern T: S[r][t] = X[(t0+t)*ld + r0+r]   (r contiguous in memory)
__device__ __forceinline__ void load_T(float (*S)[GS], const float* __restrict__ X, long long ld, long long t0,
                                       long long tmax, long long r0, long long rmax, int act, int tid) {
#pragma unroll
    for (int q = 0; q < (GT * GK) / 256; ++q) {
        const int e = tid + q * 256;
        const int r = e % GK, t = e / GK;
        float v = 0.f;
        if (t0 + t < tmax && r0 + r < rmax) {
            v = X[(t0 + t) * ld + r0 + r];
            if (act >= 0) v = act_apply(act, v);
        }
        S[r][t] = v;
    }
}
// pattern D: S[r][t] = X[(r0+r)*ld + t0+t]   (t contiguous in memory)
__device__ __forceinline__ void load_D(float (*S)[GS], const float* __restrict__ X, long long ld, long long t0,
                                       long long tmax, long long r0, long long rmax, int act, int tid) {
#pragma unroll
    for (int q = 0; q < (GT * GK) / 256; ++q) {
        const int e = tid + q * 256;
        const int t = e % GT, r = e / GT;
        float v = 0.f;
        if (t0 + t < tmax && r0 + r < rmax) {
            v = X[(r0 + r) * ld + t0 + t];
            if (act >= 0) v = act_apply(act, v);
        }
        S[r][t] = v;
    }
}

template <int MODE>
__global__ void __launch_bounds__(256) gemm_kernel(const __grid_constant__ GemmArgs g) {
    __shared__ __align__(16) float As[GK][GS];
    __shared__ __align__(16) float Bs[GK][GS];
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const long long i0 = (long long)blockIdx.x * GT, j0 = (long long)blockIdx.y * GT;
    long long rbeg = 0, rend = g.R;
    if (MODE == 2) {
        rbeg = (long long)blockIdx.z * g.r_slab;
        rend = rbeg + g.r_slab < g.R ? rbeg + g.r_slab : g.R;
    }
    float acc[4][4];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) acc[a][b] = 0.f;
    float csum = 0.f;

    for (long long r0 = rbeg; r0 < rend; r0 += GK) {
        if (MODE == 0) {
            load_T(As, g.A, g.lda, i0, g.I, r0, rend, g.a_swish ? g.act : -1, tid);
            load_D(Bs, g.B, g.ldb, j0, g.J, r0, rend, -1, tid);
        } else if (MODE == 1) {
            load_T(As, g.A, g.lda, i0, g.I, r0, rend, -1, tid);
            load_T(Bs, g.B, g.ldb, j0, g.J, r0, rend, -1, tid);
        } else {
            load_D(As, g.A, g.lda, i0, g.I, r0, rend, g.a_swish ? g.act : -1, tid);
            load_D(Bs, g.B, g.ldb, j0, g.J, r0, rend, -1, tid);
        }
        __syncthreads();
        if (MODE == 2 && g.colsum && blockIdx.x == 0 && tid < GT) {
#pragma unroll
            for (int r = 0; r < GK; ++r) csum += Bs[r][tid];
        }
#pragma unroll
        for (int r = 0; r < GK; ++r) {
            const float4 a = *reinterpret_cast<const float4*>(&As[r][tx * 4]);
            const float4 b = *reinterpret_cast<const float4*>(&Bs[r][ty * 4]);
            const float a_[4] = {a.x, a.y, a.z, a.w}, b_[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int p = 0; p < 4; ++p)
#pragma unroll
                for (int q = 0; q < 4; ++q) acc[p][q] = fmaf(a_[p], b_[q], acc[p][q]);
        }
        __syncthreads();
    }

#pragma unroll
    for (int p = 0; p < 4; ++p) {
        const long long i = i0 + tx * 4 + p;
        if (i >= g.I) continue;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const long long j = j0 + ty * 4 + q;
            if (j >= g.J) continue;
            float v = acc[p][q];
            if (MODE == 0) {
                if (g.bias) v += g.bias[j];
                g.C[i * g.ldc + j] = v;
            } else if (MODE == 1) {
                if (g.Z) v *= act_grad(g.act, g.Z[i * g.ldz + j]);
                g.C[i * g.ldc + j] = v;
            } else {
                atomicAdd(&g.C[i * g.ldc + j], v);
            }
        }
    }
    if (MODE == 2 && g.colsum && blockIdx.x == 0 && tid < GT && j0 + tid < g.J) atomicAdd(&g.colsum[j0 + tid], csum);
}

static int launch_gemm(cudaStream_t st, int mode, const GemmArgs& g) {
    // tensor-core (tcgen05, 3xTF32) GEMM by default; ZF_GEMM_IMPL=simt, or an activation other than swish,
    // keeps the fp32 FFMA kernel
    const char* impl = impl_switch().gemm;
    if (impl[0] != 's' && g.act == ZF_ACT_SWISH)
        return launch_umma_gemm(st, mode, g.A, g.lda, g.B, g.ldb, g.C, g.ldc, g.bias, g.colsum, g.Z, g.ldz, g.a_swish,
                                g.I, g.J, g.R, mode == 2 ? 4096 : 0);
    dim3 grid((unsigned)((g.I + GT - 1) / GT), (unsigned)((g.J + GT - 1) / GT), 1);
    if (mode == 2) grid.z = (unsigned)((g.R + g.r_slab - 1) / g.r_slab);
    if (grid.x == 0 || grid.y == 0) return ZF_OK;
    if (mode == 0) gemm_kernel<0><<<grid, 256, 0, st>>>(g);
    else if (mode == 1) gemm_kernel<1><<<grid, 256, 0, st>>>(g);
    else gemm_kernel<2><<<grid, 256, 0, st>>>(g);
    count_launch();
    ZF_CUDA_CHECK(cudaGetLastError());
    return ZF_OK;
}

// ---------------------------------------------------------------------------------------------
// spline VJP: theta row -> d(theta) row in place; d/dx of the transformed columns; pass-through
// of the conditioning columns' cotangent
// ---------------------------------------------------------------------------------------------
struct SplineBwdArgs {
    float* theta;          // (Mb, d, P) in: raw params, out: their cotangent
    const float* x_in;     // (M, D) rows m0..m0+Mb of the coupling input
    const float* gy;       // (M, D) cotangent of the coupling output, column (j + rot) % D
    const float* glp;      // (M,) cotangent of the log-det
    float* gx;             // (M, D) out
    long long m0, Mb;
    int D, d, K, rot;
    int TS;                // samples per tile (multiple of 4: tiles are 16-byte multiples)
    int stages;
    int use_bulk;
};

__device__ __forceinline__ void bulk_copy_s2g(void* dst_gmem, const void* src_smem, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(smem_u32(src_smem)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }

// theta tiles stream HBM -> smem ring (bulk copies) -> in-place VJP, one thread per (sample, dim) row ->
// HBM (bulk store); same pipeline shape as rqs_stage_kernel.
template <int KT>
__global__ void __launch_bounds__(256) spline_bwd_kernel(const __grid_constant__ SplineBwdArgs a) {
    extern __shared__ __align__(128) float sm[];
    const int tid = threadIdx.x;
    const int K = KT > 0 ? KT : a.K;
    const int P = 3 * K - 1, d = a.d, D = a.D, S = a.stages;
    const int R = a.TS * d;
    const int tile_floats = R * P;
    uint64_t* bars = reinterpret_cast<uint64_t*>(sm + (size_t)S * tile_floats);
    const KnotNorm kn = make_knot_norm(K);
    const long long n_tiles = (a.Mb + a.TS - 1) / a.TS;

    if (tid == 0) {
        for (int s = 0; s < S; ++s) mbar_init(&bars[s], 1);
        mbar_fence_init();
    }
    __syncthreads();
    auto tile_rows = [&](long long tile) { return (int)min((long long)a.TS, a.Mb - tile * a.TS) * d; };
    auto issue = [&](long long tile, int stage) {
        const uint32_t bytes = (uint32_t)tile_rows(tile) * P * 4u;
        if (a.use_bulk && (bytes & 15u) == 0u) {
            mbar_arrive_expect_tx(&bars[stage], bytes);
            bulk_copy_g2s(sm + (size_t)stage * tile_floats, a.theta + tile * (long long)R * P, bytes, &bars[stage]);
        }
    };
    if (tid == 0)
        for (int s = 0; s < S; ++s) {
            const long long t = (long long)blockIdx.x + (long long)s * gridDim.x;
            if (t < n_tiles) issue(t, s);
        }

    int it = 0;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
        const int stage = it % S;
        const uint32_t parity = (uint32_t)(it / S) & 1u;
        const long long s0 = tile * a.TS;
        const int rows = tile_rows(tile);
        const int ns = rows / d;
        const uint32_t bytes = (uint32_t)rows * P * 4u;
        const bool bulk = a.use_bulk && (bytes & 15u) == 0u;
        float* buf = sm + (size_t)stage * tile_floats;
        float* src = a.theta + s0 * d * P;
        if (bulk) {
            mbar_wait(&bars[stage], parity);
        } else {
            for (int e = tid; e < rows * P; e += 256) buf[e] = src[e];
            __syncthreads();
        }
        for (int r = tid; r < rows; r += 256) {
            const int sidx = r / d, jj = r - sidx * d;
            const long long m = a.m0 + s0 + sidx;
            const float x = a.x_in[m * D + jj];
            const float gy = a.gy[m * D + (jj + a.rot) % D];
            a.gx[m * D + jj] = rqs_row_backward<KT>(buf + (size_t)r * P, K, x, gy, a.glp[m], kn);
        }
        // conditioning columns pass through unchanged: d y[:, j] / d x[:, j] = 1   (bijectors.py:364)
        for (int e = tid; e < ns * (D - d); e += 256) {
            const int sidx = e / (D - d), j = d + (e - sidx * (D - d));
            const long long m = a.m0 + s0 + sidx;
            a.gx[m * D + j] = a.gy[m * D + (j + a.rot) % D];
        }
        fence_proxy_async_smem();
        __syncthreads();
        if (bulk) {
            if (tid == 0) {
                bulk_copy_s2g(src, buf, bytes);
                bulk_commit();
                bulk_wait_read<0>();   // the store has read the buffer: it may be refilled
                const long long next = tile + (long long)S * gridDim.x;
                if (next < n_tiles) issue(next, stage);
            }
        } else {
            for (int e = tid; e < rows * P; e += 256) src[e] = buf[e];
            __syncthreads();
            if (tid == 0) {
                const long long next = tile + (long long)S * gridDim.x;
                if (next < n_tiles) issue(next, stage);
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// optimiser: optax.nadamw / adamw on a flat parameter buffer
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) nadamw_kernel(long long n, float* __restrict__ p, const float* __restrict__ g,
                                                     float* __restrict__ mu, float* __restrict__ nu, float lr, float b1,
                                                     float b2, float eps, float wd, float bc1_t, float bc1_t1, float bc2_t,
                                                     int nesterov) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const float gi = g[i];
        const float m = b1 * mu[i] + (1.0f - b1) * gi;
        const float v = b2 * nu[i] + (1.0f - b2) * gi * gi;
        mu[i] = m;
        nu[i] = v;
        float mhat;
        if (nesterov) mhat = b1 * (m / bc1_t1) + (1.0f - b1) * (gi / bc1_t);
        else mhat = m / bc1_t;
        const float vhat = v / bc2_t;
        const float upd = mhat / (sqrtf(vhat) + eps) + wd * p[i];
        p[i] = p[i] - lr * upd;
    }
}

// The same update with the step counter in device memory: bias corrections from count[0] (updates done so far),
// then count[0] += 1.  Nothing on the host changes from step to step, so a captured train step can be replayed.
__global__ void nadamw_bias_kernel(long long* count, float b1, float b2, float* bc) {
    const double t = (double)count[0] + 1.0;
    bc[0] = (float)(1.0 - pow((double)b1, t));
    bc[1] = (float)(1.0 - pow((double)b1, t + 1.0));
    bc[2] = (float)(1.0 - pow((double)b2, t));
    count[0] += 1;
}

__global__ void __launch_bounds__(256) nadamw_dev_kernel(long long n, float* __restrict__ p, const float* __restrict__ g,
                                                         float* __restrict__ mu, float* __restrict__ nu, float lr, float b1,
                                                         float b2, float eps, float wd, const float* __restrict__ bc,
                                                         int nesterov) {
    const float bc1_t = bc[0], bc1_t1 = bc[1], bc2_t = bc[2];
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const float gi = g[i];
        const float m = b1 * mu[i] + (1.0f - b1) * gi;
        const float v = b2 * nu[i] + (1.0f - b2) * gi * gi;
        mu[i] = m;
        nu[i] = v;
        float mhat;
        if (nesterov) mhat = b1 * (m / bc1_t1) + (1.0f - b1) * (gi / bc1_t);
        else mhat = m / bc1_t;
        const float vhat = v / bc2_t;
        const float upd = mhat / (sqrtf(vhat) + eps) + wd * p[i];
        p[i] = p[i] - lr * upd;
    }
}

// ---------------------------------------------------------------------------------------------
// epoch shuffle (train.py:104-108): X_perm = X_train[perm].  perm is a keyed pseudo-random
// permutation of [0, N): a 4-round balanced Feistel network on 2h >= log2(N) bits with cycle
// walking, so row i of the output can be located without materialising or sorting anything.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t mix32(uint32_t x, uint32_t k) {
    x ^= k;
    x *= 0x9E3779B1u; x ^= x >> 15;
    x *= 0x85EBCA77u; x ^= x >> 13;
    x *= 0xC2B2AE3Du; x ^= x >> 16;
    return x;
}
__device__ __forceinline__ unsigned long long feistel_perm(unsigned long long i, unsigned long long N, int h, uint4 keys) {
    const uint32_t mask = (h >= 32) ? 0xffffffffu : ((1u << h) - 1u);
    unsigned long long v = i;
    do {
        uint32_t L = (uint32_t)(v >> h) & mask, R = (uint32_t)v & mask;
        uint32_t t;
        t = L ^ (mix32(R, keys.x) & mask); L = R; R = t;
        t = L ^ (mix32(R, keys.y) & mask); L = R; R = t;
        t = L ^ (mix32(R, keys.z) & mask); L = R; R = t;
        t = L ^ (mix32(R, keys.w) & mask); L = R; R = t;
        v = ((unsigned long long)L << h) | R;
    } while (v >= N);
    return v;
}

__global__ void __launch_bounds__(256) permute_rows_kernel(const float* __restrict__ x, long long N, int D, int h, uint4 keys,
                                                           float* __restrict__ out) {
    const long long n = N * D;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
        const long long i = e / D;
        const int j = (int)(e - i * D);
        out[e] = x[feistel_perm((unsigned long long)i, (unsigned long long)N, h, keys) * D + j];
    }
}

// -mean over finite-or-not entries exactly as jnp.mean would see them (train.py:73,78)
__global__ void __launch_bounds__(256) neg_sum_kernel(const float* __restrict__ lp, long long M, double* out) {
    __shared__ double red[256];
    double local = 0.0;
    for (long long m = blockIdx.x * (long long)blockDim.x + threadIdx.x; m < M; m += (long long)gridDim.x * blockDim.x)
        local -= (double)lp[m];
    red[threadIdx.x] = local;
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) {
        if (threadIdx.x < s) red[threadIdx.x] += red[threadIdx.x + s];
        __syncthreads();
    }
    if (threadIdx.x == 0) atomicAdd(out, red[0]);
}

static unsigned grid_for(long long n, int per_block, int cap) {
    long long b = (n + per_block - 1) / per_block;
    if (b < 1) b = 1;
    if (b > cap) b = cap;
    return (unsigned)b;
}

// passes per block of the row-strided statistics kernels: the tuned figure for big batches, 4 for the small batches of
// a reference-style train() (a step of 1,000 rows is latency-bound: one block walking them serially costs ~10 us)
static int small_batch_rows(long long M, int big) { return M <= (1 << 16) ? 4 : big; }

static void fill_cols(const zf_shift_bounds* sb, int D, SbCols& c) {
    for (int i = 0; i < D; ++i) {
        c.kind[i] = sb->kind[i];
        c.lo[i] = (float)sb->lo[i];
        c.hi[i] = (float)sb->hi[i];
    }
}

}  // namespace zf

using namespace zf;

extern "C" int zf_selftest_umma_gemm(void* stream, int32_t mode, const float* A, int64_t lda, const float* B, int64_t ldb,
                                     float* C, int64_t ldc, const float* bias, float* colsum, const float* Z, int64_t ldz,
                                     int32_t a_swish, int64_t I, int64_t J, int64_t R, int64_t r_slab) {
    ZF_REQUIRE(A && B && C && mode >= 0 && mode <= 2 && I >= 1 && J >= 1 && R >= 1, "selftest_umma_gemm: bad argument");
    ZF_REQUIRE(mode != 2 || (I <= 128 && r_slab >= 32 && r_slab % 32 == 0), "selftest_umma_gemm: mode 2 needs I <= 128 and r_slab % 32 == 0");
    const GemmArgs g{A, lda, B, ldb, C, ldc, bias, colsum, Z, ldz, a_swish, ZF_ACT_SWISH, I, J, R, r_slab};
    return launch_gemm((cudaStream_t)stream, mode, g);
}

extern "C" int zf_shift_bounds_minmax(void* stream, const zf_shift_bounds* sb, const float* x, int64_t M, int32_t D,
                                      float* minmax, void* scratch) {
    ZF_REQUIRE(sb && x && minmax && scratch, "shift_bounds_minmax: null argument");
    ZF_REQUIRE(D >= 1 && D <= ZF_MAX_DIM && M >= 1, "shift_bounds_minmax: bad shape");
    cudaStream_t st = (cudaStream_t)stream;
    SbCols cols{};
    fill_cols(sb, D, cols);
    unsigned* enc = static_cast<unsigned*>(scratch);
    minmax_init_kernel<<<1, 2 * ZF_MAX_DIM, 0, st>>>(enc, D);
    minmax_kernel<<<grid_for(M * D, 256 * 16, 148 * 8), 256, 0, st>>>(cols, x, M, D, enc);
    minmax_decode_kernel<<<1, 2 * ZF_MAX_DIM, 0, st>>>(enc, minmax, D);
    count_launch(); count_launch(); count_launch();
    ZF_CUDA_CHECK(cudaGetLastError());
    return ZF_OK;
}

extern "C" int zf_shift_bounds_update(void* stream, const zf_shift_bounds* sb, int32_t D, const float* minmax) {
    ZF_REQUIRE(sb && minmax && sb->xmin && sb->xmax, "shift_bounds_update: null argument");
    SbCols cols{};
    fill_cols(sb, D, cols);
    sb_update_kernel<<<1, ZF_MAX_DIM, 0, (cudaStream_t)stream>>>(cols, (float)sb->margin, minmax, sb->xmin, sb->xmax, D);
    count_launch();
    ZF_CUDA_CHECK(cudaGetLastError());
    return ZF_OK;
}

extern "C" int zf_bn_moments(void* stream, const float* x, const float* c, int64_t M, int32_t D, int32_t C, double* sums) {
    const int d = D / 2, F = D - d + C;
    ZF_REQUIRE(x && sums && (C == 0 || c) && M >= 1 && d > 0 && F <= 256, "bn_moments: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    ZF_CUDA_CHECK(cudaMemsetAsync(sums, 0, 2 * F * sizeof(double), st));
    const int R = 256 / F;
    bn_moments_kernel<<<grid_for(M, R * small_batch_rows(M, 64), 148 * 8), 256, 2 * F * sizeof(double), st>>>(x, c, M, D, C, sums);
    count_launch();
    ZF_CUDA_CHECK(cudaGetLastError());
    return ZF_OK;
}

extern "C" int zf_bn_finalize(void* stream, const double* sums, double count, int32_t F, float momentum,
                              float* batch_mean, float* batch_var, float* ra_mean, float* ra_var) {
    ZF_REQUIRE(sums && batch_mean && batch_var && F >= 1 && count >= 1, "bn_finalize: bad argument");
    bn_finalize_kernel<<<(F + 127) / 128, 128, 0, (cudaStream_t)stream>>>(sums, count, F, momentum, batch_mean, batch_var,
                                                                           ra_mean, ra_var);
    count_launch();
    ZF_CUDA_CHECK(cudaGetLastError());
    return ZF_OK;
}

extern "C" int zf_flow_loss_grad_ct(void* stream, int32_t latent_kind, float peakness, const float* z, const float* log_det,
                                    int64_t M, int32_t D, double global_count, const float* lp_cotangent, float* lp,
                                    float* gz, float* glp, double* lp_sum) {
    ZF_REQUIRE(z && log_det && gz && glp && lp_sum && M >= 1 && D >= 1 && global_count >= 1, "flow_loss_grad: bad argument");
    LatentConst lc{};
    lc.kind = latent_kind;
    lc.p1 = (float)((double)peakness - 1.0);
    lc.betaln = (float)(2.0 * lgamma((double)peakness) - lgamma(2.0 * (double)peakness));
    lc.lognorm = (float)log(2.0 * M_PI * 0.1 * 0.1);
    lc.logmass = (float)log(0.5 * (erf(5.0 / sqrt(2.0)) - erf(-5.0 / sqrt(2.0))));
    loss_grad_kernel<<<grid_for(M, 256, 148 * 8), 256, 0, (cudaStream_t)stream>>>(lc, z, log_det, M, D,
                                                                                  (float)(-1.0 / global_count),
                                                                                  lp_cotangent, lp, gz, glp, lp_sum);
    count_launch();
    ZF_CUDA_CHECK(cudaGetLastError());
    return ZF_OK;
}

extern "C" int zf_flow_loss_grad(void* stream, int32_t latent_kind, float peakness, const float* z, const float* log_det,
                                 int64_t M, int32_t D, double global_count, float* lp, float* gz, float* glp,
                                 double* lp_sum) {
    return zf_flow_loss_grad_ct(stream, latent_kind, peakness, z, log_det, M, D, global_count, nullptr, lp, gz, glp, lp_sum);
}

// Workspace of zf_coupling_backward.
// Fused path (hidden width 128, K in {16, 32}: the tensor-core kernels): the cotangent of theta has each dim's 3K-1
// columns padded to NL = a multiple of 16 and the last Dense is differentiated in that padded column space.
//   fixed   [packed parameters | weight images of every Dense | dW_L padded | db_L padded]
//   per micro-batch   images: dTheta, swish(Z_l), H0 (+ bias column), two dZ buffers;  fp32: swish'(Z_l)
// Otherwise: per micro-batch H0 | Z_1 .. Z_L | Theta in fp32.
struct CplBwdLayout {
    bool fused;
    int NL, TW, WH, WF0;  // columns per dim / of the theta block; widths of the H0 image and of the first Dense's weight image
    size_t pack_floats;
    size_t fixed_bytes;
    size_t off_wimg[ZF_MAX_LAYERS + 1], off_gwp, off_gbp;
};
static size_t up256(size_t v) { return (v + 255) / 256 * 256; }
static CplBwdLayout cpl_bwd_layout(const zf_coupling* cp, int D, int C) {
    const int d = D / 2, F = D - d + C, P = 3 * cp->knots - 1, L = cp->n_hidden;
    CplBwdLayout lay{};
    lay.pack_floats = coupling_vjp_ws_floats(cp, D, C);
    lay.fused = lay.pack_floats > 0;
    lay.NL = lay.fused ? (P + 15) / 16 * 16 : P;
    lay.TW = d * lay.NL;
    lay.WH = (F + 1 + 15) / 16 * 16;
    lay.WF0 = (F + 15) / 16 * 16;
    if (lay.fused) {
        size_t off = up256(lay.pack_floats * 4);
        for (int l = 0; l <= L; ++l) {
            lay.off_wimg[l] = off;
            off += up256(l == 0 ? zf::w_image_bytes(lay.WF0, 128) : l == L ? zf::w_image_bytes(128, lay.TW) : zf::w_image_bytes(128, 128));
        }
        lay.off_gwp = off; off += up256((size_t)128 * lay.TW * 4);
        lay.off_gbp = off; off += up256((size_t)lay.TW * 4);
        lay.fixed_bytes = off;
    }
    return lay;
}
static size_t cpl_bwd_batch_bytes(const zf_coupling* cp, const CplBwdLayout& lay, int D, int C, long long Mb) {
    const int d = D / 2, F = D - d + C, L = cp->n_hidden;
    if (!lay.fused) {
        size_t n = F;
        for (int l = 0; l < L; ++l) n += cp->hidden[l];
        n += (size_t)d * lay.NL;
        return (n * (size_t)Mb + 64) * sizeof(float);
    }
    size_t b = up256(zf::img_bytes(Mb, lay.TW)) + up256(zf::img_bytes(Mb, lay.WH)) + 2 * up256(zf::img_bytes(Mb, 128));
    b += (size_t)L * (up256(zf::img_bytes(Mb, 128)) + up256(zf::img_bytes(Mb, 128)));   // activation image + swish' tile image (same size)
    return b;
}

extern "C" size_t zf_coupling_backward_workspace_bytes(const zf_coupling* cp, int32_t D, int32_t C, int64_t micro_batch) {
    if (!cp || D < 2 || micro_batch < 1) return 0;
    const CplBwdLayout lay = cpl_bwd_layout(cp, D, C);
    return lay.fixed_bytes + cpl_bwd_batch_bytes(cp, lay, D, C, micro_batch) + 256;
}

// gW (Hin, d P) += gWp (Hin, d NL) without the padding; gb (d P) += gbp (d NL)
__global__ void __launch_bounds__(256) unpad_add_kernel(const float* __restrict__ gWp, const float* __restrict__ gbp, int Hin, int d, int P,
                                                        int NL, float* __restrict__ gW, float* __restrict__ gb) {
    const int n = (Hin + 1) * d * P;
    for (int e = blockIdx.x * 256 + threadIdx.x; e < n; e += gridDim.x * 256) {
        const int h = e / (d * P), r = e - h * (d * P), jj = r / P, p = r - jj * P;
        if (h < Hin) gW[e] += gWp[(size_t)h * d * NL + jj * NL + p];
        else gb[r] += gbp[jj * NL + p];
    }
}

// Fused path of zf_coupling_backward (see CplBwdLayout).
static int coupling_backward_fused(cudaStream_t st, const zf_coupling* cp, const zf_coupling_grads* gr, int D, int C, const float* x_in,
                                   const float* c, const float* gy, int gy_rot, const float* glp, long long M, float* gx, float* gh0,
                                   double* bn_sums, char* ws, long long micro_batch, const CplBwdLayout& lay) {
    const int d = D / 2, F = D - d + C, K = cp->knots, P = 3 * K - 1, L = cp->n_hidden, NL = lay.NL, TW = lay.TW;
    float* pack = reinterpret_cast<float*>(ws);
    float* gWp = reinterpret_cast<float*>(ws + lay.off_gwp);
    float* gbp = reinterpret_cast<float*>(ws + lay.off_gbp);
    if (int rc = coupling_vjp_pack(st, cp, D, C, pack)) return rc;
    {   // Dense_l kernel (in, out) as the image [n = in][k = out], every layer in one launch
        PackWJob jobs[ZF_MAX_LAYERS + 1];
        for (int l = 0; l <= L; ++l) {
            if (l == 0) jobs[l] = PackWJob{cp->kernel[0], ws + lay.off_wimg[0], 128, F, lay.WF0, 128, 128, 128, 0, 0};
            else if (l == L) jobs[l] = PackWJob{cp->kernel[L], ws + lay.off_wimg[L], d * P, 128, 128, TW, P, NL, 0, 0};
            else jobs[l] = PackWJob{cp->kernel[l], ws + lay.off_wimg[l], 128, 128, 128, 128, 128, 128, 0, 0};
        }
        if (int rc = pack_w_images(st, jobs, L + 1)) return rc;
    }
    ZF_CUDA_CHECK(cudaMemsetAsync(gWp, 0, lay.fixed_bytes - lay.off_gwp, st));
    char* wb = ws + lay.fixed_bytes;
    for (long long m0 = 0; m0 < M; m0 += micro_batch) {
        const long long Mb = std::min<long long>(micro_batch, M - m0);
        char* p = wb;
        auto take = [&](size_t bytes) { char* o = p; p += up256(bytes); return o; };
        void* img_dt = take(img_bytes(Mb, TW));
        void* img_h0 = take(img_bytes(Mb, lay.WH));
        void* img_dz[2] = {take(img_bytes(Mb, 128)), take(img_bytes(Mb, 128))};
        void* img_act[ZF_MAX_LAYERS];
        float* act_g[ZF_MAX_LAYERS];
        for (int l = 0; l < L; ++l) {
            img_act[l] = take(img_bytes(Mb, 128));
            act_g[l] = reinterpret_cast<float*>(take(img_bytes(Mb, 128)));   // fp32 tile image: whole tiles
        }
        // BatchNorm, conditioner (theta in tensor memory), spline VJP: writes gx and the images
        if (int rc = coupling_vjp_run(st, cp, D, C, pack, x_in + m0 * D, c ? c + m0 * C : nullptr, gy + m0 * D, gy_rot, glp + m0, Mb,
                                      gx + m0 * D, img_h0, lay.WH, img_act, act_g, img_dt))
            return rc;
        // last Dense (padded column space): dW_L, db_L, dZ_L = (dTheta W_L^T) swish'(Z_L)
        if (int rc = launch_img_tn(st, img_act[L - 1], img_dt, TW, gWp, TW, 1, 128, TW, gbp, nullptr, -1, Mb)) return rc;
        if (int rc = launch_img_nt(st, img_dt, TW, ws + lay.off_wimg[L], 128, act_g[L - 1], -1, img_dz[0], nullptr, 0, 0, Mb)) return rc;
        int cur = 0;
        for (int l = L - 1; l >= 1; --l) {   // hidden Dense_l: input swish(Z_l), output cotangent dZ_{l+1}
            if (int rc = launch_img_tn(st, img_act[l - 1], img_dz[cur], 128, gr->kernel[l], 128, 1, 128, 128, gr->bias[l], nullptr, -1, Mb))
                return rc;
            if (int rc = launch_img_nt(st, img_dz[cur], 128, ws + lay.off_wimg[l], 128, act_g[l - 1], -1, img_dz[cur ^ 1], nullptr, 0, 0, Mb))
                return rc;
            cur ^= 1;
        }
        // first Dense: dW_0[f][h] = sum_e H0[e][f] dZ_1[e][h] (transposed product; H0's bias column gives db_0), d/dH0
        if (int rc = launch_img_tn(st, img_dz[cur], img_h0, lay.WH, gr->kernel[0], 1, 128, 128, F, nullptr, gr->bias[0], F, Mb)) return rc;
        if (int rc = launch_img_nt(st, img_dz[cur], 128, ws + lay.off_wimg[0], lay.WF0, nullptr, 0, nullptr, gh0 + m0 * F, F, F, Mb)) return rc;
        const int R = 256 / F;
        bn_bwd_sums_kernel<<<grid_for(Mb, R * small_batch_rows(Mb, 64), 148 * 4), 256, 2 * F * sizeof(double), st>>>(
            x_in + m0 * D, c ? c + m0 * C : nullptr, gh0 + m0 * F, Mb, D, C, cp->bn_mean, cp->bn_var, bn_sums);
        count_launch();
    }
    unpad_add_kernel<<<grid_for((long long)(128 + 1) * d * P, 256, 148 * 4), 256, 0, st>>>(gWp, gbp, 128, d, P, NL, gr->kernel[L], gr->bias[L]);
    count_launch();
    ZF_CUDA_CHECK(cudaGetLastError());
    return ZF_OK;
}

extern "C" int zf_coupling_backward(void* stream, const zf_coupling* cp, const zf_coupling_grads* gr, int32_t D, int32_t C,
                                    const float* x_in, const float* c, const float* gy, int32_t gy_rot, const float* glp,
                                    int64_t M, float* gx, float* gh0, double* bn_sums, void* workspace,
                                    size_t workspace_bytes, int64_t micro_batch) {
    ZF_REQUIRE(cp && gr && x_in && gy && glp && gx && gh0 && bn_sums && workspace, "coupling_backward: null argument");
    const int d = D / 2, F = D - d + C;
    ZF_REQUIRE(d > 0 && d < D && (C == 0 || c) && M >= 1 && micro_batch >= 1, "coupling_backward: bad shape");
    ZF_REQUIRE(F <= 256, "coupling_backward: at most 256 conditioner inputs");
    const int K = cp->knots, P = 3 * K - 1, L = cp->n_hidden;
    const CplBwdLayout lay = cpl_bwd_layout(cp, D, C);
    if (workspace_bytes < lay.fixed_bytes + cpl_bwd_batch_bytes(cp, lay, D, C, std::min<long long>(micro_batch, M)))
        return fail(ZF_ERR_WORKSPACE, "coupling_backward: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    ZF_CUDA_CHECK(cudaMemsetAsync(bn_sums, 0, 2 * F * sizeof(double), st));
    if (lay.fused) {
        ZF_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "coupling_backward: workspace must be 256-byte aligned");
        return coupling_backward_fused(st, cp, gr, D, C, x_in, c, gy, gy_rot, glp, M, gx, gh0, bn_sums, static_cast<char*>(workspace),
                                       micro_batch, lay);
    }
    DeviceInfo di;
    if (int rc = get_device_info(&di)) return rc;

    // spline tile: TS samples (multiple of 4) x d rows, ~256 rows; two or three ring stages
    int TS = std::max(4, (256 / d) & ~3);
    while (TS > 4 && (size_t)TS * d * P * 4 > 96 * 1024) TS -= 4;
    const size_t tile_bytes = (size_t)TS * d * P * 4;
    int sp_stages = (int)std::min<size_t>(3, ((size_t)di.max_smem_optin - 256) / tile_bytes);
    int sp_bps = 1;
    if (2 * (2 * tile_bytes + 256) + 2048 <= (size_t)di.max_smem_optin) { sp_stages = 2; sp_bps = 2; }
    if (sp_stages < 1) return fail(ZF_ERR_UNSUPPORTED, "coupling_backward: spline tile does not fit shared memory");
    const size_t sp_smem = (size_t)sp_stages * tile_bytes + 64;
    auto sp_kernel = (K == 16) ? spline_bwd_kernel<16> : (K == 32) ? spline_bwd_kernel<32> : spline_bwd_kernel<0>;
    if (int rc = smem_optin((const void*)sp_kernel, sp_smem)) return rc;

    float* ws = static_cast<float*>(workspace);
    int widths[ZF_MAX_LAYERS + 2];
    widths[0] = F;
    for (int l = 0; l < L; ++l) widths[l + 1] = cp->hidden[l];
    widths[L + 1] = d * P;

    for (long long m0 = 0; m0 < M; m0 += micro_batch) {
        const long long Mb = std::min<long long>(micro_batch, M - m0);
        // activations of this micro-batch: H0 | Z_1 .. Z_L | Theta
        float* act[ZF_MAX_LAYERS + 2];
        size_t off = 0;
        for (int l = 0; l <= L + 1; ++l) {
            act[l] = ws + off;
            off += (size_t)widths[l] * Mb;
        }
        bn_apply_kernel<<<grid_for(Mb * F, 256 * 8, 148 * 16), 256, 0, st>>>(x_in + m0 * D, c ? c + m0 * C : nullptr, Mb, D, C,
                                                                             cp->bn_scale, cp->bn_bias, cp->bn_mean,
                                                                             cp->bn_var, act[0]);
        count_launch();
        // forward recompute: Z_{l+1} = act(Z_l) W_l + b_l   (pre-activations are stored)
        for (int l = 0; l <= L; ++l) {
            GemmArgs g{};
            g.A = act[l]; g.lda = widths[l];
            g.B = cp->kernel[l]; g.ldb = widths[l + 1];
            g.C = act[l + 1]; g.ldc = widths[l + 1];
            g.bias = cp->bias[l];
            g.a_swish = l > 0; g.act = cp->act;
            g.I = Mb; g.J = widths[l + 1]; g.R = widths[l];
            if (int rc = launch_gemm(st, 0, g)) return rc;
        }
        // spline VJP: Theta -> dTheta in place, gx for all columns
        {
            SplineBwdArgs a{};
            a.theta = act[L + 1]; a.x_in = x_in; a.gy = gy; a.glp = glp; a.gx = gx;
            a.m0 = m0; a.Mb = Mb; a.D = D; a.d = d; a.K = K; a.rot = ((gy_rot % D) + D) % D; a.TS = TS;
            a.stages = sp_stages;
            a.use_bulk = ((reinterpret_cast<uintptr_t>(a.theta) & 15) == 0) ? 1 : 0;
            const long long tiles = (Mb + TS - 1) / TS;
            sp_kernel<<<(unsigned)std::min<long long>(tiles, (long long)di.sm_count * sp_bps), 256, sp_smem, st>>>(a);
            count_launch();
        }
        // backward through the dense layers
        for (int l = L; l >= 0; --l) {
            GemmArgs gw{};  // dW_l += act(Z_l)^T dZ_{l+1}; db_l += colsum(dZ_{l+1})
            gw.A = act[l]; gw.lda = widths[l];
            gw.B = act[l + 1]; gw.ldb = widths[l + 1];
            gw.C = gr->kernel[l]; gw.ldc = widths[l + 1];
            gw.colsum = gr->bias[l];
            gw.a_swish = l > 0; gw.act = cp->act;
            gw.I = widths[l]; gw.J = widths[l + 1]; gw.R = Mb; gw.r_slab = 2048;
            if (int rc = launch_gemm(st, 2, gw)) return rc;
            GemmArgs ga{};  // dZ_l = (dZ_{l+1} W_l^T) * swish'(Z_l)   (l = 0: d/d(BN output), no activation)
            ga.A = act[l + 1]; ga.lda = widths[l + 1];
            ga.B = cp->kernel[l]; ga.ldb = widths[l + 1];
            ga.C = (l == 0) ? gh0 + m0 * F : act[l]; ga.ldc = widths[l];
            ga.Z = (l == 0) ? nullptr : act[l]; ga.ldz = widths[l]; ga.act = cp->act;
            ga.I = Mb; ga.J = widths[l]; ga.R = widths[l + 1];
            if (int rc = launch_gemm(st, 1, ga)) return rc;
        }
        const int R = 256 / F;
        bn_bwd_sums_kernel<<<grid_for(Mb, R * small_batch_rows(Mb, 64), 148 * 4), 256, 2 * F * sizeof(double), st>>>(
            x_in + m0 * D, c ? c + m0 * C : nullptr, gh0 + m0 * F, Mb, D, C, cp->bn_mean, cp->bn_var, bn_sums);
        count_launch();
    }
    ZF_CUDA_CHECK(cudaGetLastError());
    return ZF_OK;
}

__global__ void bn_param_grads_kernel(const double* sums, int F, float* gscale, float* gbias) {
    int f = threadIdx.x;
    if (f < F) {
        gbias[f] += (float)sums[f];
        gscale[f] += (float)sums[F + f];
    }
}

extern "C" int zf_bn_param_grads(void* stream, const double* bn_sums, int32_t F, float* g_scale, float* g_bias) {
    ZF_REQUIRE(bn_sums && g_scale && g_bias && F >= 1 && F <= 256, "bn_param_grads: bad argument");
    bn_param_grads_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(bn_sums, F, g_scale, g_bias);
    count_launch();
    ZF_CUDA_CHECK(cudaGetLastError());
    return ZF_OK;
}

extern "C" int zf_bn_backward_apply(void* stream, const zf_coupling* cp, int32_t D, int32_t C, const float* x_in,
                                    const float* c, const float* gh0, const double* bn_sums, double global_count, int64_t M,
                                    float* gx, float* gc) {
    ZF_REQUIRE(cp && x_in && gh0 && bn_sums && gx && M >= 1 && global_count >= 1, "bn_backward_apply: bad argument");
    const int d = D / 2, F = D - d + C;
    const int R = 256 / F;
    bn_bwd_apply_kernel<<<grid_for(M, R * small_batch_rows(M, 16), 148 * 16), 256, 5 * F * sizeof(float), (cudaStream_t)stream>>>(
        x_in, c, gh0, M, D, C, cp->bn_scale, cp->bn_mean, cp->bn_var, bn_sums, global_count, gx, gc);
    count_launch();
    ZF_CUDA_CHECK(cudaGetLastError());
    return ZF_OK;
}

extern "C" int zf_nadamw_update(void* stream, int64_t n, float* params, const float* grads, float* mu, float* nu,
                                int64_t count, float lr, float b1, float b2, float eps, float weight_decay,
                                int32_t nesterov) {
    ZF_REQUIRE(params && grads && mu && nu && n >= 0 && count >= 0, "nadamw_update: bad argument");
    if (n == 0) return ZF_OK;
    const double t = (double)count + 1.0;
    const float bc1_t = (float)(1.0 - pow((double)b1, t));
    const float bc1_t1 = (float)(1.0 - pow((double)b1, t + 1.0));
    const float bc2_t = (float)(1.0 - pow((double)b2, t));
    nadamw_kernel<<<grid_for(n, 256 * 4, 148 * 8), 256, 0, (cudaStream_t)stream>>>(n, params, grads, mu, nu, lr, b1, b2, eps,
                                                                                  weight_decay, bc1_t, bc1_t1, bc2_t, nesterov);
    count_launch();
    ZF_CUDA_CHECK(cudaGetLastError());
    return ZF_OK;
}

extern "C" int zf_nadamw_update_dev(void* stream, int64_t n, float* params, const float* grads, float* mu, float* nu,
                                    int64_t* count_dev, float* bias_scratch, float lr, float b1, float b2, float eps,
                                    float weight_decay, int32_t nesterov) {
    ZF_REQUIRE(params && grads && mu && nu && count_dev && bias_scratch && n >= 0, "nadamw_update_dev: bad argument");
    nadamw_bias_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(reinterpret_cast<long long*>(count_dev), b1, b2, bias_scratch);
    count_launch();
    if (n > 0) {
        nadamw_dev_kernel<<<grid_for(n, 256 * 4, 148 * 8), 256, 0, (cudaStream_t)stream>>>(n, params, grads, mu, nu, lr, b1, b2,
                                                                                          eps, weight_decay, bias_scratch, nesterov);
        count_launch();
    }
    ZF_CUDA_CHECK(cudaGetLastError());
    return ZF_OK;
}

extern "C" int zf_permute_rows(void* stream, const float* x, int64_t N, int32_t D, uint64_t seed, float* out) {
    ZF_REQUIRE(N >= 0 && D >= 1, "permute_rows: bad shape");
    if (N == 0) return ZF_OK;
    ZF_REQUIRE(x && out && x != out, "permute_rows: null or aliased tensors (the gather is out of place)");
    int bits = 1;
    while ((1ull << bits) < (unsigned long long)N) ++bits;
    const int h = (bits + 1) / 2;
    // four round keys from the seed (splitmix64)
    unsigned long long z = seed + 0x9E3779B97F4A7C15ull;
    auto next = [&]() {
        unsigned long long r = (z += 0x9E3779B97F4A7C15ull);
        r = (r ^ (r >> 30)) * 0xBF58476D1CE4E5B9ull;
        r = (r ^ (r >> 27)) * 0x94D049BB133111EBull;
        return (unsigned)((r ^ (r >> 31)) >> 16);
    };
    uint4 keys = make_uint4(next(), next(), next(), next());
    permute_rows_kernel<<<grid_for(N * D, 256 * 4, 148 * 16), 256, 0, (cudaStream_t)stream>>>(x, N, D, h, keys, out);
    count_launch();
    ZF_CUDA_CHECK(cudaGetLastError());
    return ZF_OK;
}

extern "C" int zf_neg_sum(void* stream, const float* lp, int64_t M, double* out) {
    ZF_REQUIRE(out != nullptr && M >= 0 && (lp || M == 0), "neg_sum: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    ZF_CUDA_CHECK(cudaMemsetAsync(out, 0, sizeof(double), st));
    if (M == 0) return ZF_OK;
    neg_sum_kernel<<<grid_for(M, 256 * 8, 148 * 4), 256, 0, st>>>(lp, M, out);
    count_launch();
    ZF_CUDA_CHECK(cudaGetLastError());
    return ZF_OK;
}
