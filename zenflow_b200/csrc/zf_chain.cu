// Whole-chain eval passes: one kernel applies every bijector of a Chain to a tile of samples
// that stays in shared memory from the first ShiftBounds to the latent log-pdf.
//
//   zf_chain_forward  <- Chain.__call__(train=False)        bijectors.py:104-111
//   zf_chain_inverse  <- Chain.inverse                      bijectors.py:113-116
//   zf_flow_log_prob  <- Flow.__call__(train=False)         flow.py:22-48
// per step:
//   ShiftBounds.__call__/inverse                            bijectors.py:164-240
//   Roll                                                    bijectors.py:288-297 (column renaming only)
//   NeuralSplineCoupling._spline_params/__call__/inverse    bijectors.py:329-371
//     eval BatchNorm -> Dense+swish ... -> Dense            (fp32 FFMA register-tiled GEMM)
//     -> normalize_spline_params + rqs forward/inverse      (zf_math.cuh), theta never leaves smem
//
// Data layout: the tile is feature-major in shared memory (xs[col][m]) in *physical* column
// order; a Roll only changes the logical->physical rotation carried by the following steps.
// Parameters are re-packed per call by a tiny kernel into zero-padded, 16-byte aligned blocks
// in the caller's workspace (the FLAX leaves themselves are never modified).
#include "zf_common.cuh"
#include "zf_math.cuh"
#include "zf_umma.cuh"
#include "zf_rng.cuh"
#include "zf_vjp.cuh"

#include <float.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <vector>

namespace zf {

constexpr int TM = 64;        // samples per tile
constexpr int KC = 16;        // k rows per staged weight chunk
constexpr int NCOL = 128;     // output columns per GEMM pass
constexpr int kChainThreads = 256;
constexpr int kStepKindShiftBounds = 0, kStepKindCoupling = 2;

__host__ __device__ inline int ru(int x, int m) { return (x + m - 1) / m * m; }

// Device-side description of one non-Roll step; lives at the head of the workspace.
struct StepDesc {
    int kind;
    int rot;       // logical column j is physical column (j - rot) mod D while this step runs
    int K, n_hidden, F, d;
    int hidden[ZF_MAX_LAYERS];
    int off_bn;                     // float offsets into the workspace
    int off_W[ZF_MAX_LAYERS + 1];
    int off_b[ZF_MAX_LAYERS + 1];
    int off_sb;
    int off_U[ZF_MAX_LAYERS + 1];   // tensor-core weight images (3xTF32 hi|lo, K-major core matrices), layers 1..L
    int umma_ok;                    // this coupling fits the tensor-core kernel
    int off_C;                      // tensor-core kernel: this coupling's small constants as one contiguous block
    int cidx;                       // ordinal of this coupling among the chain's couplings (bin-index output)
    int act;                        // zf_act_kind of the hidden layers (the tensor-core kernels take swish only)
    int pad[1];
};
static_assert(sizeof(StepDesc) % 16 == 0, "StepDesc must keep the packed blocks 16-byte aligned");

struct UCst { int bn, w0, b0, bh, bl, w0i, total; };   // float offsets inside a constant block (ucst_layout); w0i < 0: no image

struct PackJob {
    StepDesc desc;
    UCst cst;
    int step_index;
    int D;
    // coupling
    const float *bn_scale, *bn_bias, *bn_mean, *bn_var;
    const float* kernel[ZF_MAX_LAYERS + 1];
    const float* bias[ZF_MAX_LAYERS + 1];
    int Kin[ZF_MAX_LAYERS + 1];
    int N[ZF_MAX_LAYERS + 1];
    // shift bounds
    int sb_kind[ZF_MAX_DIM];
    double lo[ZF_MAX_DIM], hi[ZF_MAX_DIM];
    const float *xmin, *xmax;
};

constexpr int kSbStride = 8;  // floats per column: kind, a, b, xmin, xmax, mul, log(mul), -

// Up to kPackBatch steps per launch (blockIdx.y = step of the batch): kernel parameters may be 32 KB since CUDA 12.1,
// so a whole chain's jobs travel in one launch instead of one launch per step.
constexpr int kPackBatch = 16;
struct PackBatch { PackJob jobs[kPackBatch]; };
static_assert(sizeof(PackBatch) <= 32000, "PackBatch must fit the kernel parameter space");

__global__ void __launch_bounds__(256) pack_step_kernel(const __grid_constant__ PackBatch batch, float* ws) {
    const PackJob& job = batch.jobs[blockIdx.y];
    const int gtid = blockIdx.x * blockDim.x + threadIdx.x;
    const int gsz = gridDim.x * blockDim.x;
    const StepDesc& s = job.desc;
    if (gtid == 0) reinterpret_cast<StepDesc*>(ws)[job.step_index] = s;

    if (s.kind == kStepKindShiftBounds) {
        for (int i = gtid; i < job.D; i += gsz) {
            float* t = ws + s.off_sb + i * kSbStride;
            const int kind = job.sb_kind[i];
            float a = (float)job.lo[i], b = (float)job.hi[i];
            float xmin = 0.f, xmax = 0.f, mul;
            if (kind == ZF_BOUND_BOTH) {
                mul = (float)(1.0 / (job.hi[i] - job.lo[i]));      // bijectors.py:189
            } else {
                xmin = job.xmin[i];
                xmax = job.xmax[i];
                mul = __fdiv_rn(1.0f, __fsub_rn(xmax, xmin));      // bijectors.py:265
            }
            t[0] = (float)kind; t[1] = a; t[2] = b; t[3] = xmin; t[4] = xmax;
            t[5] = mul; t[6] = logf(mul); t[7] = 0.f;
        }
        return;
    }

    // BatchNorm (eval): y = (x - mean) * (rsqrt(var + eps) * scale) + bias
    const int F = s.F, F_p = ru(F, KC);
    for (int f = gtid; f < F_p; f += gsz) {
        float mul = 0.f, mean = 0.f, bias = 0.f;
        if (f < F) {
            mul = __fdiv_rn(1.0f, __fsqrt_rn(__fadd_rn(job.bn_var[f], 1e-5f))) * job.bn_scale[f];
            mean = job.bn_mean[f];
            bias = job.bn_bias[f];
        }
        ws[s.off_bn + f] = mul;
        ws[s.off_bn + F_p + f] = mean;
        ws[s.off_bn + 2 * F_p + f] = bias;
    }
    // hidden layers: W (Kin, N) -> [Kin_p][N_p] zero padded
    for (int l = 0; l < s.n_hidden; ++l) {
        const int Kin = job.Kin[l], N = job.N[l];
        const int Kin_p = ru(Kin, KC), N_p = ru(N, KC);
        const float* W = job.kernel[l];
        for (int e = gtid; e < Kin_p * N_p; e += gsz) {
            int k = e / N_p, n = e - k * N_p;
            ws[s.off_W[l] + e] = (k < Kin && n < N) ? W[(size_t)k * N + n] : 0.f;
        }
        for (int n = gtid; n < N_p; n += gsz) ws[s.off_b[l] + n] = n < N ? job.bias[l][n] : 0.f;
    }
    // last layer: (Kin, d*P) -> [d][Kin_p][Pp]
    {
        const int L = s.n_hidden;
        const int Kin = job.Kin[L], Kin_p = ru(Kin, KC);
        const int P = 3 * s.K - 1, Pp = ru(P, 4), d = s.d;
        const float* W = job.kernel[L];
        const int per = Kin_p * Pp;
        for (int e = gtid; e < d * per; e += gsz) {
            int jj = e / per, r = e - jj * per;
            int k = r / Pp, p = r - k * Pp;
            ws[s.off_W[L] + e] = (k < Kin && p < P) ? W[(size_t)k * (d * P) + jj * P + p] : 0.f;
        }
        for (int e = gtid; e < d * Pp; e += gsz) {
            int jj = e / Pp, p = e - jj * Pp;
            ws[s.off_b[L] + e] = p < P ? job.bias[L][jj * P + p] : 0.f;
        }
    }
    // tensor-core images: per unit (hidden layer l >= 1, or one transformed dim of the last layer)
    // 4 K-chunks of 32, each [hi image | lo image] in fp16 (3xFP16 split, zf_umma.cuh), image = [k/8][n/8][n%8][k%8]
    if (s.umma_ok) {
        const int L = s.n_hidden, P = 3 * s.K - 1, NL = ru(P, 16), d = s.d;
        {   // the constant block the producer warp fetches with one bulk copy per coupling
            float* cb = ws + s.off_C;
            const UCst& cl = job.cst;
            const int n_plain = cl.w0i >= 0 ? cl.w0i : cl.total;
            if (cl.w0i >= 0) {
                // first Dense as a K = 16 operand image.  The BatchNorm scale is NOT folded in here: the tensor-core path
                // multiplies it into the A operand ((x - mean) * mul is O(1) whatever the scale of the raw inputs, so the
                // fp16 hi / lo' split neither overflows nor goes subnormal on un-normalised conditioning features)
                __half* dst = reinterpret_cast<__half*>(cb + cl.w0i);
                for (int e = gtid; e < 16 * 128; e += gsz) {
                    const int k = e >> 7, n = e & 127;
                    const float val = k < F ? job.kernel[0][k * 128 + n] : 0.f;
                    const __half hi = __float2half_rn(val);
                    const __half lo = __float2half_rn((val - __half2float(hi)) * umma::kF16LoScale);
                    const int ii = umma::b_image_index_f16(n, k, 128);
                    dst[ii] = hi;
                    dst[16 * 128 + ii] = lo;
                }
            }
            for (int i = gtid; i < n_plain; i += gsz) {
                float v = 0.f;
                if (i < cl.w0) {                       // BatchNorm [mul | mean | bias], F_p each
                    const int part = i / F_p, f = i - part * F_p;
                    if (part < 3 && f < F) {
                        if (part == 0) v = __fdiv_rn(1.0f, __fsqrt_rn(__fadd_rn(job.bn_var[f], 1e-5f))) * job.bn_scale[f];
                        else v = part == 1 ? job.bn_mean[f] : job.bn_bias[f];
                    }
                } else if (i < cl.b0) {                // first Dense kernel [F][128] with the BatchNorm scale folded in:
                    const int e = i - cl.w0;           // the kernels compute sum_f (x_f - mean_f) * (mul_f W0[f][n]) + b0'[n]
                    if (e < F * 128) {
                        const int f = e >> 7;
                        const float mul = __fdiv_rn(1.0f, __fsqrt_rn(__fadd_rn(job.bn_var[f], 1e-5f))) * job.bn_scale[f];
                        v = __fmul_rn(mul, job.kernel[0][e]);
                    }
                } else if (i < cl.bh) {                // first Dense bias + (BatchNorm bias) . W0
                    const int n = i - cl.b0;
                    v = job.bias[0][n];
                    for (int f = 0; f < F; ++f) v = fmaf(job.bn_bias[f], job.kernel[0][f * 128 + n], v);
                } else if (i < cl.bl) {                // hidden biases, layers 1..L-1
                    const int e = i - cl.bh, l = 1 + (e >> 7);
                    if (l < L) v = job.bias[l][e & 127];
                } else {                               // last-layer bias [d][NL], zero padded
                    const int e = i - cl.bl, jj = e / NL, pp = e - jj * NL;
                    if (jj < d && pp < P) v = job.bias[L][jj * P + pp];
                }
                cb[i] = v;
            }
        }
        for (int l = 1; l <= L; ++l) {
            const float* W = job.kernel[l];
            const int units = (l < L) ? 1 : d;
            const int N = (l < L) ? 128 : NL;
            const int ldw = (l < L) ? 128 : d * P;
            for (int e = gtid; e < units * N * 128; e += gsz) {
                const int u = e / (N * 128), r = e - u * (N * 128);
                const int k = r / N, n = r - k * N;
                float val = 0.f;
                if (l < L) val = W[(size_t)k * ldw + n];
                else if (n < P) val = W[(size_t)k * ldw + u * P + n];
                const __half hi = __float2half_rn(val);
                const __half lo = __float2half_rn((val - __half2float(hi)) * umma::kF16LoScale);
                __half* dst = reinterpret_cast<__half*>(ws + s.off_U[l] + (size_t)u * N * 128 + (size_t)(k >> 5) * N * 32);
                const int ii = umma::b_image_index_f16(n, k & 31, N);
                dst[ii] = hi;
                dst[N * 32 + ii] = lo;
            }
        }
    }
}

enum ChainMode : int { kModeForward = 0, kModeLogProb = 1, kModeInverse = 2, kModeVjp = 3 };

struct ChainArgs {
    const float* x;     // (M, D) input (x for forward/log_prob, z for inverse)
    const float* c;     // (M, C) or null
    float* y;           // (M, D) output or null
    float* log_det;     // (M,) or null (forward)
    float* lp;          // (M,) (log_prob)
    const float* ws;    // workspace: StepDesc[n_steps] then packed parameters
    long long M;
    int D, C;
    int n_steps;
    int rot_total;      // rotation after the last step
    int act_rows;
    int mode;
    int acc_log_det;    // log_det[m] += instead of =
    int sample;         // inverse mode: draw z from the latent (seed) instead of reading a.x
    unsigned long long seed;
    float peakness;
    LatentConst lc;
    int u_fmax, u_hmax, u_blmax;   // tensor-core kernel: max conditioner inputs / hidden biases / last-layer bias floats
    int u_w0img;        // the constant blocks carry the first Dense's operand image (first Dense on the tensor cores)
    int* idx_out;       // (M, n_couplings, d) bin indices of every spline evaluation, or null (parity evidence)
    int n_couplings;
    // kModeVjp (chain_umma_kernel<false, true>, a chain of ONE coupling): conditioner recompute + spline VJP
    const float* gy;    // (M, D) cotangent of the coupling's output; logical column j is read at (j + gy_rot) % D
    const float* glp;   // (M,) cotangent of the log-det
    float* gx;          // (M, D) out: d/dx of the transformed columns, pass-through cotangent of the others
    // outputs for the Dense VJPs, as event-row images (bf16 x 2, csrc/zf_img_gemm.cu) of whole 128-event tiles
    char* img_h0;       // width wh0: BatchNorm output, feature F = 1 (the bias column), zero padding
    char* img_act[ZF_MAX_LAYERS];   // width 128: swish of the hidden pre-activations
    float* act_g[ZF_MAX_LAYERS];    // swish' of the hidden pre-activations, fp32 tile images [tile][n / 4][event % 128][n % 4]
    char* img_dtheta;   // width d NL: cotangent of theta, dim j in columns [j NL, j NL + 3K-1), padding zero
    int wh0, gy_rot;
};

// bin index of event m, coupling s.cidx, transformed dim jj (zf_chain_bin_indices)
__device__ __forceinline__ void put_idx(const ChainArgs& a, const StepDesc& s, long long m, int jj, int idx) {
    if (a.idx_out) a.idx_out[(m * a.n_couplings + s.cidx) * s.d + jj] = idx;
}

__device__ __forceinline__ int pmod(int a, int D) {
    int r = a % D;
    return r < 0 ? r + D : r;
}

// acc[4][8] += act_in[Kin_p][TM]^T (samples tx*4..+3) x W[Kin_p][ncols] (cols ty*4..+3, 64+ty*4..+3)
// W rows are streamed from global (L2) through a cp.async double buffer.
__device__ __forceinline__ void gemm_pass(const float* __restrict__ act_in, int Kin_p,
                                          const float* __restrict__ Wg, int ldw, int ncols,
                                          float* __restrict__ wst, float (&acc)[4][8], int tid) {
    const int tx = tid & 15, ty = tid >> 4;
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
    const int nchunks = Kin_p / KC;
    const int c4 = ncols >> 2;
    auto load_chunk = [&](int c, int buf) {
        const float* src = Wg + (size_t)c * KC * ldw;
        float* dst = wst + buf * (KC * NCOL);
        for (int q = tid; q < KC * c4; q += kChainThreads) {
            int row = q / c4, col = (q - row * c4) << 2;
            cp_async_16(dst + row * NCOL + col, src + (size_t)row * ldw + col);
        }
    };
    load_chunk(0, 0);
    cp_async_commit();
    for (int c = 0; c < nchunks; ++c) {
        if (c + 1 < nchunks) {
            load_chunk(c + 1, (c + 1) & 1);
            cp_async_commit();
            cp_async_wait<1>();
        } else {
            cp_async_wait<0>();
        }
        __syncthreads();
        const float* wb = wst + (c & 1) * (KC * NCOL);
        const float* ab = act_in + c * KC * TM;
#pragma unroll
        for (int kk = 0; kk < KC; ++kk) {
            const float4 av = *reinterpret_cast<const float4*>(ab + kk * TM + tx * 4);
            const float4 b0 = *reinterpret_cast<const float4*>(wb + kk * NCOL + ty * 4);
            const float4 b1 = *reinterpret_cast<const float4*>(wb + kk * NCOL + 64 + ty * 4);
            const float a_[4] = {av.x, av.y, av.z, av.w};
            const float b_[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a_[i], b_[j], acc[i][j]);
        }
        __syncthreads();
    }
}

template <bool INVERSE>
__device__ __forceinline__ int spline_rows(float* th, int Pst, int K, const KnotNorm& kn, float* xcol,
                                           float& ldc, int tid) {
    // one thread per sample of the tile (tid < TM): theta row -> bin -> transform
    float* row = th + tid * Pst;
    const float v = xcol[tid];
    RqsBin b;
    switch (K) {
        case 16: rqs_locate<16>(row, K, !INVERSE, v, kn, b); break;
        case 32: rqs_locate<32>(row, K, !INVERSE, v, kn, b); break;
        default: rqs_locate<0>(row, K, !INVERSE, v, kn, b); break;
    }
    if (!INVERSE) {
        float y, ld;
        rqs_eval_forward(v, b, y, ld);
        xcol[tid] = y;
        ldc += ld;
    } else {
        xcol[tid] = rqs_eval_inverse(v, b);
    }
    return b.idx;
}

template <bool INVERSE>
__device__ __forceinline__ void run_coupling(const ChainArgs& a, long long m0, int nm, const StepDesc& s,
                                             const float* __restrict__ wsf, int D, int C,
                                             float* xs, const float* cs, float* act0, float* act1,
                                             float* wst, float& ld_acc, int tid) {
    const int d = s.d, F = s.F, F_p = ru(F, KC), rot = s.rot;
    // ---- conditioner input: hstack(xc, c) then eval BatchNorm (bijectors.py:341-342)
    {
        const float* bn = wsf + s.off_bn;
        for (int e = tid; e < F_p * TM; e += kChainThreads) {
            const int f = e / TM, m = e - f * TM;
            float h = 0.f;
            if (f < F) {
                const float v = (f < D - d) ? xs[pmod(d + f - rot, D) * TM + m] : cs[(f - (D - d)) * TM + m];
                h = (v - bn[F_p + f]) * bn[f] + bn[2 * F_p + f];
            }
            act0[e] = h;
        }
    }
    __syncthreads();

    float* cur = act0;
    float* nxt = act1;
    const int tx = tid & 15, ty = tid >> 4;
    float acc[4][8];
    int Kin_p = F_p;
    // ---- hidden layers: Dense + act (swish unless the coupling says otherwise; bijectors.py:343-345)
    for (int l = 0; l < s.n_hidden; ++l) {
        const int N_p = ru(s.hidden[l], KC);
        const float* W = wsf + s.off_W[l];
        const float* bias = wsf + s.off_b[l];
        for (int n0 = 0; n0 < N_p; n0 += NCOL) {
            const int ncols = min(NCOL, N_p - n0);
            gemm_pass(cur, Kin_p, W + n0, N_p, ncols, wst, acc, tid);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int n = (j < 4) ? (ty * 4 + j) : (64 + ty * 4 + (j - 4));
                if (n < ncols) {
                    const float bj = bias[n0 + n];
                    float4 o;
                    o.x = act_apply(s.act, acc[0][j] + bj);
                    o.y = act_apply(s.act, acc[1][j] + bj);
                    o.z = act_apply(s.act, acc[2][j] + bj);
                    o.w = act_apply(s.act, acc[3][j] + bj);
                    *reinterpret_cast<float4*>(nxt + (n0 + n) * TM + tx * 4) = o;
                }
            }
        }
        __syncthreads();
        float* t = cur; cur = nxt; nxt = t;
        Kin_p = N_p;
    }
    // ---- last Dense, one transformed dim at a time; theta rows go to the dead buffer
    const int K = s.K, P = 3 * K - 1, Pp = ru(P, 4), Pst = P | 1;
    const KnotNorm kn = make_knot_norm(K);
    const int L = s.n_hidden;
    float ldc = 0.f;
    for (int jj = 0; jj < d; ++jj) {
        const float* W = wsf + s.off_W[L] + (size_t)jj * Kin_p * Pp;
        const float* bias = wsf + s.off_b[L] + jj * Pp;
        gemm_pass(cur, Kin_p, W, Pp, Pp, wst, acc, tid);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int p = (j < 4) ? (ty * 4 + j) : (64 + ty * 4 + (j - 4));
            if (p < P) {
                const float bj = bias[p];
#pragma unroll
                for (int i = 0; i < 4; ++i) nxt[(tx * 4 + i) * Pst + p] = acc[i][j] + bj;
            }
        }
        __syncthreads();
        if (tid < TM) {
            const int idx = spline_rows<INVERSE>(nxt, Pst, K, kn, xs + pmod(jj - rot, D) * TM, ldc, tid);
            if (tid < nm) put_idx(a, s, m0 + tid, jj, idx);
        }
        __syncthreads();
    }
    ld_acc += ldc;  // Chain: log_det += ld   (bijectors.py:110)
}

// ShiftBounds for one event m of a tile held as xs[col][stride] (bijectors.py:183-207 / :214-238)
template <bool INVERSE>
__device__ __forceinline__ void shift_bounds_row(const StepDesc& s, const float* __restrict__ wsf, int D, float* xs,
                                                 int stride, int m, float& ld_acc, int i0 = 0, int istep = 1) {
    float ldc = 0.f;
    for (int i = i0; i < D; i += istep) {
        const float* t = wsf + s.off_sb + i * kSbStride;
        const int kind = (int)t[0];
        const float a = t[1], b = t[2], xmin = t[3], xmax = t[4], mul = t[5], logmul = t[6];
        float* px = xs + pmod(i - s.rot, D) * stride + m;
        const float v = *px;
        if (!INVERSE) {
            float z, ld;
            if (kind == ZF_BOUND_BOTH) {
                z = __fmul_rn(__fsub_rn(v, a), mul);
                ld = logmul;
            } else {
                float u = v;
                if (kind == ZF_BOUND_LOWER) u = logf(__fadd_rn(__fsub_rn(v, a), FLT_MIN));
                if (kind == ZF_BOUND_UPPER) u = logf(__fadd_rn(__fsub_rn(b, v), FLT_MIN));
                z = clip_nanprop(__fmul_rn(__fsub_rn(u, xmin), mul), 0.f, 1.f);
                ld = (kind == ZF_BOUND_NONE) ? logmul : (logmul - u);
            }
            *px = z;
            ldc += ld;
        } else {
            float x;
            if (kind == ZF_BOUND_BOTH) {
                x = __fadd_rn(__fmul_rn(v, b), __fmul_rn(__fsub_rn(1.f, v), a));
            } else {
                float u = __fadd_rn(__fmul_rn(v, xmax), __fmul_rn(__fsub_rn(1.f, v), xmin));
                if (kind == ZF_BOUND_LOWER) x = expf(u) + a;
                else if (kind == ZF_BOUND_UPPER) x = b - expf(u);
                else x = u;
            }
            *px = x;
        }
    }
    ld_acc += ldc;
}

template <bool INVERSE>
__device__ __forceinline__ void run_shift_bounds(const StepDesc& s, const float* __restrict__ wsf, int D,
                                                 float* xs, float& ld_acc, int tid) {
    if (tid < TM) shift_bounds_row<INVERSE>(s, wsf, D, xs, TM, tid, ld_acc);
    __syncthreads();
}

template <bool INVERSE>
__global__ void __launch_bounds__(kChainThreads, 2) chain_kernel(const __grid_constant__ ChainArgs a) {
    extern __shared__ __align__(128) float smem[];
    const int tid = threadIdx.x;
    const int D = a.D, C = a.C;
    float* xs = smem;
    float* cs = xs + D * TM;
    float* act0 = cs + C * TM;
    float* act1 = act0 + a.act_rows * TM;
    float* wst = act1 + a.act_rows * TM;
    const StepDesc* steps = reinterpret_cast<const StepDesc*>(a.ws);
    const float* wsf = a.ws;

    const long long n_tiles = (a.M + TM - 1) / TM;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const long long m0 = tile * TM;
        const int nm = (int)min((long long)TM, a.M - m0);
        // ---- load the tile, feature-major; padding samples sit at 0.5 and are never stored
        const int rot_in = INVERSE ? a.rot_total : 0;
        for (int e = tid; e < TM * D; e += kChainThreads) {
            const int m = e / D, j = e - m * D;
            const float v = (m < nm) ? (a.sample ? latent_draw(a.lc.kind, a.peakness, a.seed, m0 + m, j) : a.x[m0 * D + e]) : 0.5f;
            xs[pmod(j - rot_in, D) * TM + m] = v;
        }
        for (int e = tid; e < TM * C; e += kChainThreads) {
            const int m = e / C, j = e - m * C;
            cs[j * TM + m] = (m < nm) ? a.c[m0 * C + e] : 0.f;
        }
        __syncthreads();

        float ld_acc = 0.f;  // Chain: log_det = zeros(M)   (bijectors.py:107)
        for (int si = 0; si < a.n_steps; ++si) {
            const StepDesc& s = steps[INVERSE ? (a.n_steps - 1 - si) : si];
            if (s.kind == kStepKindShiftBounds) run_shift_bounds<INVERSE>(s, wsf, D, xs, ld_acc, tid);
            else run_coupling<INVERSE>(a, m0, nm, s, wsf, D, C, xs, cs, act0, act1, wst, ld_acc, tid);
        }

        // ---- store
        if (a.mode == kModeLogProb) {
            if (tid < nm) {  // flow.py:46-47
                float lat = 0.f;
                for (int j = 0; j < D; ++j) lat += latent_logpdf(xs[pmod(j - a.rot_total, D) * TM + tid], a.lc);
                a.lp[m0 + tid] = nan_to_num_lp(lat + ld_acc);
            }
        } else {
            const int rot_out = INVERSE ? 0 : a.rot_total;
            if (a.y) {
                for (int e = tid; e < nm * D; e += kChainThreads) {
                    const int m = e / D, j = e - m * D;
                    a.y[m0 * D + e] = xs[pmod(j - rot_out, D) * TM + m];
                }
            }
            if (!INVERSE && a.log_det && tid < nm) a.log_det[m0 + tid] = a.acc_log_det ? a.log_det[m0 + tid] + ld_acc : ld_acc;
        }
        __syncthreads();
    }
}

// =============================================================================================
// Tensor-core chain kernel (tcgen05, 3xTF32): same program, same outputs as chain_kernel.
//
// One CTA per SM, 128 events per tile, 10 warps:
//   warps 0-7  epilogue / SIMT: ShiftBounds, BatchNorm + first Dense (K = F is tiny), bias+swish+split of
//              every hidden layer, the spline rows, latent log-pdf.  Thread (q*32+lane, half): TMEM lane
//              quarter q = warp%4 (hardware rule), column half = warp/4.
//   warp 8     weight producer: 1-D bulk copies of pre-split K-major weight images L2 -> 4-stage smem ring
//   warp 9     MMA issuer: tcgen05.mma kind::tf32, A (activations) in tensor memory, B from the ring,
//              fp32 accumulators in tensor memory; also owns the TMEM allocation.
// Tensor memory (512 columns): A_hi [0,128) | A_lo [128,256) | D0 [256,384) | D1 [384,512).
// Hidden layers accumulate into D0; the last layer runs one transformed dim at a time, alternating
// D0/D1 so that the spline rows of dim j (warps 0-3 for even j, 4-7 for odd j) overlap the MMAs of j+1.
// 3xFP16 split on kind::f16 (zf_umma.cuh): x = hi + lo' * 2^-11 (fp16 each), main = A_hi*B_hi and
// cross = A_lo'*B_hi + A_hi*B_lo' in separate accumulators, theta = main + cross * 2^-11: fp32-class accuracy
// (measured: below fp32 sgemm's error) at twice the tensor rate and half the operand bytes of the 3xTF32 split
// it replaces; a single TF32/BF16 pass would break the rel-1e-5 parity (SURVEY H2).  Valid while the
// conditioner's activations and weights stay below 65504 in magnitude (beyond that the event's result is NaN).
// Tensor memory (512 columns): A_hi [0,64) | A_lo [64,128) as fp16 pairs; hidden layers main [256,384), cross
// [384,512); last layer, buffer b: main [128 + 192 b, +96), cross 96 columns further.
// =============================================================================================
#ifdef ZF_TRACE   // developer build only (scripts/trace_chain.py): per-phase clock64 stamps of one steady-state tile
__device__ long long g_zf_trace[4][64];
#define ZF_TR_DECL int titer_ = -1, tev_ = 0
#define ZF_TR_TILE do { ++titer_; tev_ = 0; } while (0)
#define ZF_TRV(slot, v) do { if (blockIdx.x == 0 && titer_ == 8 && lane == 0 && tev_ < 64) g_zf_trace[slot][tev_++] = (v); } while (0)
#define ZF_TR(slot) do { if (blockIdx.x == 0 && titer_ == 8 && lane == 0 && tev_ < 64) g_zf_trace[slot][tev_++] = clock64(); } while (0)
#else
#define ZF_TR_DECL
#define ZF_TR_TILE
#define ZF_TR(slot)
#define ZF_TRV(slot, v)
#endif
constexpr int UM = 128;
#ifndef ZF_URING
#define ZF_URING 4
#endif
constexpr int URING = ZF_URING;   // <= 8 (barrier numbering below)
constexpr int URING_FLOATS = 4096;  // 16 KB: one K-chunk (32) of a 128-column unit, fp16 hi|lo
constexpr uint32_t TC_ALO = 64, TC_XOFF = 96;
// Hidden accumulators.  Single-tile kernel: main [256,384), cross [384,512) - theta buffer 0 = [128,320) then only
// overlaps the hidden main columns of K-chunks 0 and 1, so the first last-layer unit starts while the hidden epilogue
// is still draining chunks 2 and 3.  Two-tile kernel: main [128,256), cross [256,384).
constexpr uint32_t TC_HMAIN = 256, TC_HCROSS = 384, TC_PP_HMAIN = 128, TC_PP_HCROSS = 256;
// first Dense on the tensor cores (K = 16): ONE accumulator [128,256) - cross products first, then the main product on
// top as D = A B + D 2^-11 (scale-input-d); it is drained before the first theta unit overwrites the columns
constexpr uint32_t TC_FD = 128;
// Two-tile kernel, theta columns of the (single) transformed dim.  K = 16 (48 + 48 columns): [384, 480), clear of the
// hidden accumulators, so the theta unit runs under the hidden epilogue of its own slot and the other slot's hidden
// GEMM does not have to wait for the row warps.  K = 32 (96 + 96 columns) only fits on top of them: [128, 320).
__host__ __device__ constexpr uint32_t tc_pp_theta(int NL) { return NL == 48 ? 384u : 128u; }
__host__ __device__ constexpr uint32_t tc_pp_xoff(int NL) { return NL == 48 ? 48u : 96u; }
__host__ __device__ constexpr uint32_t tc_dmain(int b) { return 128u + 192u * (uint32_t)b; }
constexpr int UFMAX = 32;           // conditioner inputs handled by the SIMT first layer
constexpr int UDMAX = 32;           // transformed dims
// B_AREADY + c: K-chunk c (32 columns) of the current activation version is in tensor memory AND the
// accumulator columns it was computed from have been read (so they may be overwritten)
// B_CFULL/B_CEMPTY + b: constant block buffer b;  B_XFULL/B_XEMPTY: the raw rows of the next input tile
enum UBar : int { B_FULL = 0, B_EMPTY = 8, B_AREADY = 16, B_DFULL_H = 20, B_DFULL_D = 21, B_DEMPTY_D = 23,
                  B_CFULL = 25, B_CEMPTY = 27, B_XFULL = 29, B_XEMPTY = 30, B_A0READY = 31, B_COUNT = 32 };

// per-coupling constants (BatchNorm affine, first Dense, biases), double-buffered: the next coupling's set is
// fetched with cp.async while the current one computes
// img: the block also carries the first Dense as a 3xFP16 operand image (K = 16 x N = 128: hi 4 KB | lo' 4 KB), for the
// kernels that run the first Dense on the tensor cores
constexpr int UW0IMG_FLOATS = 2048;
__host__ __device__ inline UCst ucst_layout(int Fmax, int Hmax, int BLmax, bool img = false) {
    UCst l;
    l.bn = 0;
    l.w0 = ru(3 * ru(Fmax, KC), 32);
    l.b0 = l.w0 + Fmax * 128;
    l.bh = l.b0 + 128;
    l.bl = l.bh + Hmax * 128;
    l.total = ru(l.bl + BLmax, 32);
    l.w0i = -1;
    if (img) { l.w0i = l.total; l.total += UW0IMG_FLOATS; }
    return l;
}
constexpr int USTEPS = 40;   // step descriptors kept in shared memory (longer programs read them from global)
constexpr int VJP_ROW = 97;   // floats per theta row of the VJP kernel (odd: one thread per row without bank conflicts)
__host__ __device__ inline size_t umma_hs_floats(int Fmax) { return (size_t)Fmax * UM; }   // x - mean, [Fmax][UM]
__host__ __device__ inline size_t umma_smem_floats(int D, int C, int Fmax, int Hmax, int BLmax, bool vjp = false, bool img = false) {
    return 2 * (size_t)UM * (D + C) + umma_hs_floats(Fmax) + (vjp ? 1 : 2) * (size_t)ucst_layout(Fmax, Hmax, BLmax, img).total + 3 * UM +
           (vjp ? 2 * UM * VJP_ROW : 2 * 8 * UM * 4) +
           (size_t)URING * URING_FLOATS + 2 * B_COUNT + 32 + USTEPS * sizeof(StepDesc) / sizeof(float);
}

__device__ __forceinline__ void epi_barrier() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

// swish with the SFU exp2 / reciprocal: the absolute error stays below ~1e-7 (the exponent's argument
// rounding only matters where exp(-x) is negligible against 1, or where swish itself is ~0); measured
// on log_prob it is indistinguishable from expf + IEEE division and costs a quarter of the instructions
// The reciprocal is taken with rcp.approx directly: __fdividef adds a compare and two predicated multiplies per
// element to rescale denominators above 2^126, where swish is below 1e-36 anyway (3 of ~20 instructions per element
// in the activation phases, which are issue-bound).
__device__ __forceinline__ float swish_fast(float x) {
    float e, r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * -1.4426950408889634f));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(1.0f + e));
    return x * r;
}

// ---- theta row of this thread's event from a D buffer in tensor memory ---------------------------
// issue the TMEM loads of one raw K-block (main accumulator and the cross accumulator cross_off columns further);
// tcgen05.wait::ld must follow before the registers are read
template <int KT>
__device__ __forceinline__ void theta_block_issue(uint32_t dbase, uint32_t cross_off, int col, float (&p)[KT], float (&w)[KT]) {
#pragma unroll
    for (int c0 = 0; c0 < KT; c0 += 16) umma::ld16(dbase + col + c0, p + c0);
#pragma unroll
    for (int c0 = 0; c0 < KT; c0 += 16) umma::ld16(dbase + cross_off + col + c0, w + c0);
}
// main + cross * 2^-11 + bias; returns max |theta| of the block (NaN-poisoned to +inf)
template <int KT>
__device__ __forceinline__ float theta_block_finish(int col, const float* __restrict__ bias, float (&p)[KT],
                                                    const float (&w)[KT]) {
    float amax = 0.f;
    bool nan = false;
#pragma unroll
    for (int j = 0; j < KT; ++j) {
        p[j] = fmaf(w[j], umma::kF16LoUnscale, p[j]) + bias[col + j];
        amax = fmaxf(amax, fabsf(p[j]));
        nan = nan || (p[j] != p[j]);
    }
    return nan ? CUDART_INF_F : amax;
}


// One spline row of this thread's event from a D buffer in tensor memory, with the lean block forms of zf_math.cuh
// (rows are issue-bound: ~1.3k instead of ~1.9k instructions for K = 32).  The three raw blocks are loaded in a software
// pipeline (the next block's TMEM load is in flight while the current one is processed) and the D buffer is handed
// back to the MMA warp (release()) right after the last load.  Bins are bit-identical to the IEEE path
// (rqs_block_search<KT>); the other-axis knot, the bin height / width and the knot derivatives are
// fp32-tolerance quantities either way.  scr: this thread's scratch column (float4, stride apart, KT / 4 entries).
// Rows with |theta| >= kThetaFastBound (or inf) take the IEEE path (rqs_block_search / rqs_block_other).
template <int KT>
__device__ __forceinline__ float theta_block_finish_lean(int col, const float* __restrict__ bias, float (&p)[KT],
                                                         const float (&w)[KT]) {
    float amax = 0.f;   // NaN entries are not tracked: they poison the row's sums identically on either path
#pragma unroll
    for (int j = 0; j < KT; ++j) {
        p[j] = fmaf(w[j], umma::kF16LoUnscale, p[j]) + bias[col + j];
        amax = fmaxf(amax, fabsf(p[j]));
    }
    return amax;
}
template <int KT, bool INVERSE, class Release>
__device__ __forceinline__ void spline_row_tmem_lean(uint32_t dbase, uint32_t cross_off, const float* __restrict__ bias, float v,
                                                     RqsBin& b, float4* scr, int stride, Release release) {
    constexpr int cs_ = INVERSE ? KT : 0, co_ = INVERSE ? 0 : KT;
    const KnotNorm kn = make_knot_norm(KT);
    float pa[KT], pb[KT], wa[KT], wb[KT];
    theta_block_issue<KT>(dbase, cross_off, cs_, pa, wa);
    umma::wait_ld();
    const float amax_s = theta_block_finish_lean<KT>(cs_, bias, pa, wa);
    theta_block_issue<KT>(dbase, cross_off, co_, pb, wb);          // in flight during the search pass
    const bool slow_s = __any_sync(0xffffffffu, !(amax_s < kThetaFastBound));
    if (slow_s) rqs_block_search<KT>(pa, v, kn, b.idx, b.ks, b.bs);
    else rqs_block_search_lean<KT>(pa, v, kn, b.idx, b.ks, b.bs);
    umma::wait_ld();
    const float amax_o = theta_block_finish_lean<KT>(co_, bias, pb, wb);
    theta_block_issue<KT>(dbase, cross_off, 2 * KT, pa, wa);       // raw slopes reuse the searched block's registers
    umma::wait_ld();
    release();                                          // every TMEM read of this row is done
    if (__any_sync(0xffffffffu, !(amax_o < kThetaFastBound))) rqs_block_other<KT>(pb, b.idx, kn, b.ko, b.bo);
    else rqs_block_other_lean<KT>(pb, b.idx, kn, scr, stride, b.ko, b.bo);
    rqs_block_slopes_lean<KT>(pa, wa, umma::kF16LoUnscale, bias + 2 * KT, b.idx, scr, stride, b.dk, b.dkp1);
}

// Activation phase of the VJP kernel: swish for the next GEMM (fp16 x 3 split into tensor memory, as in the eval
// kernels) plus what the Dense VJPs need of this layer: the activations as an event-row image (bf16 x 2) and
// swish' of the pre-activations (fp32).  Rows beyond the batch are written as zeros.
template <int CW>
__device__ __forceinline__ void vjp_activation(const ChainArgs& a, int layer, long long tile, long long m0, int m, int nm, int n0,
                                               const float (&z)[CW], uint32_t (&ahi)[CW / 2], uint32_t (&alo)[CW / 2]) {
    float sw[CW], gs[CW];
    const bool valid = m < nm;
#pragma unroll
    for (int j = 0; j < CW; ++j) {
        float e, r;
        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(z[j] * -1.4426950408889634f));
        asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(1.0f + e));
        sw[j] = z[j] * r;                       // swish(z) = z sigmoid(z)
        gs[j] = fmaf(sw[j], 1.0f - r, r);       // swish'(z) = sigmoid(z) (1 + z (1 - sigmoid(z)))
    }
#pragma unroll
    for (int i = 0; i < CW / 2; ++i) umma::split_f16x2(sw[2 * i], sw[2 * i + 1], ahi[i], alo[i]);
    if (valid) {   // fp32 tile image [tile][n / 4][event][n % 4]: a warp writes 512 contiguous bytes per 4-column unit
        char* go = reinterpret_cast<char*>(a.act_g[layer]) + (size_t)tile * (128 * 128 * 4) + (size_t)(n0 >> 2) * 2048 + (size_t)m * 16;
#pragma unroll
        for (int g4 = 0; g4 < CW / 4; ++g4)
            *reinterpret_cast<float4*>(go + (size_t)g4 * 2048) = make_float4(gs[g4 * 4], gs[g4 * 4 + 1], gs[g4 * 4 + 2], gs[g4 * 4 + 3]);
    }
    char* it = a.img_act[layer] + (size_t)tile * 2 * 128 * 256 + (size_t)(m >> 3) * 128 + (size_t)(m & 7) * 16;
#pragma unroll
    for (int u = 0; u < CW / 8; ++u) {
        uint32_t hi[4], lo[4];
#pragma unroll
        for (int q2 = 0; q2 < 4; ++q2)
            umma::split_bf16x2(valid ? sw[8 * u + 2 * q2] : 0.f, valid ? sw[8 * u + 2 * q2 + 1] : 0.f, hi[q2], lo[q2]);
        char* dst = it + (size_t)((n0 >> 3) + u) * 2048;
        *reinterpret_cast<uint4*>(dst) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
        *reinterpret_cast<uint4*>(dst + 128 * 256) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
    }
}

// ---- VJP row of the fused train kernel: theta from tensor memory -> cotangent of theta in this thread's row buffer
// (row[0, 3 KT - 1), row[3 KT - 1] = 0).  Fast path: theta stays in registers (rqs_row_vjp_regs); rows with
// |theta| >= kThetaFastBound, inf or NaN go through the IEEE path on the row buffer (rqs_row_backward).
// INVERSE: the VJP of the spline inverse at y = x (no log-det), always on the row buffer (rqs_row_inverse_backward).
template <int KT, bool INVERSE, class Release>
__device__ __forceinline__ float vjp_row_tmem(uint32_t dbase, const float* __restrict__ bias, float* row, float x, float gy,
                                              float gld, Release release) {
    const KnotNorm kn = make_knot_norm(KT);
    if constexpr (INVERSE) {
        // the inverse row works on the row buffer: theta goes there one block at a time (three blocks of KT columns)
        float p[KT], w[KT];
#pragma unroll
        for (int blk = 0; blk < 3; ++blk) {
            theta_block_issue<KT>(dbase, TC_XOFF, blk * KT, p, w);
            umma::wait_ld();
            if (blk == 2) release();                                  // every TMEM read of this row is done
#pragma unroll
            for (int j = 0; j < KT; ++j) row[blk * KT + j] = fmaf(w[j], umma::kF16LoUnscale, p[j]) + bias[blk * KT + j];
        }
        const float g = rqs_row_inverse_backward<KT>(row, KT, x, gy, kn);
        row[3 * KT - 1] = 0.f;
        return g;
    } else {
        float pa[KT], pb[KT], wa[KT], wb[KT];
        theta_block_issue<KT>(dbase, TC_XOFF, 0, pa, wa);
        theta_block_issue<KT>(dbase, TC_XOFF, KT, pb, wb);
        umma::wait_ld();
        const float amax_w = theta_block_finish<KT>(0, bias, pa, wa);
        const float amax_h = theta_block_finish<KT>(KT, bias, pb, wb);
        theta_block_issue<KT>(dbase, TC_XOFF, 2 * KT, wa, wb);       // slopes: main in wa, cross in wb
        umma::wait_ld();
        release();                                                    // every TMEM read of this row is done
        float amax_s = 0.f;
#pragma unroll
        for (int j = 0; j < KT; ++j) {
            wa[j] = fmaf(wb[j], umma::kF16LoUnscale, wa[j]) + bias[2 * KT + j];
            if (j < KT - 1) amax_s = fmaxf(amax_s, fabsf(wa[j]));
        }
        const bool slow = !(fmaxf(fmaxf(amax_w, amax_h), amax_s) < kThetaFastBound) || !(amax_s == amax_s);
        if (__any_sync(0xffffffffu, slow)) {
#pragma unroll
            for (int j = 0; j < KT; ++j) { row[j] = pa[j]; row[KT + j] = pb[j]; row[2 * KT + j] = wa[j]; }
            const float g = rqs_row_backward<KT>(row, KT, x, gy, gld, kn);
            row[3 * KT - 1] = 0.f;
            return g;
        }
#pragma unroll
        for (int j = 0; j < KT - 1; ++j) row[j] = wa[j];
        const float g = rqs_row_vjp_regs<KT>(pa, pb, row, x, gy, gld, kn);
        row[3 * KT - 1] = 0.f;
        return g;
    }
}

// ---- the epilogue / SIMT role of the tensor-core chain kernel ------------------------------------------------
// NG column groups of 4 warps each (group g = warp / 4 owns CW = 32 / NG columns of every 32-column K-chunk and
// every NG-th feature / bounded column); TMEM lane quarter = warp % 4 (hardware rule).  Spline rows are run by
// groups 0 and 1 (one transformed dim each, alternating accumulator buffers; one thread per row, so a single-dim
// coupling's row runs on group 0 alone).
struct UCtx {
    const ChainArgs& a;
    float *xs, *cs, *xraw, *hs, *cst, *ldx;
    float4* scratch;   // per-thread scratch columns of the lean spline row: [2][8][UM] float4 (32 KB)
    uint64_t* bars;
    const StepDesc* steps;
    uint32_t tb;
    long long n_tiles;
    UCst cl;
    int cst_stride;   // floats between the two constant buffers (0 in the VJP kernel: one coupling, one buffer)
    bool in16;
    uint32_t in_bytes;
};
template <int ET>
__device__ __forceinline__ void epi_barrier() { asm volatile("bar.sync 1, %0;" ::"n"(ET) : "memory"); }
template <int CW>
__device__ __forceinline__ void tmem_load(uint32_t addr, float (&v)[CW]) {
    if constexpr (CW == 16) umma::ld16(addr, v);
    else umma::ld8(addr, v);
}
// swish + 3xFP16 split of CW consecutive activations (k = n0 .. n0 + CW) -> CW / 2 words of fp16 pairs each
template <int CW>
__device__ __forceinline__ void activation_compute(const float (&v)[CW], uint32_t (&hi)[CW / 2], uint32_t (&lo)[CW / 2]) {
#pragma unroll
    for (int i = 0; i < CW / 2; ++i) umma::split_f16x2(swish_fast(v[2 * i]), swish_fast(v[2 * i + 1]), hi[i], lo[i]);
}
template <int CW>
__device__ __forceinline__ void activation_store(uint32_t tb, uint32_t lane_base, int n0, const uint32_t (&hi)[CW / 2],
                                                 const uint32_t (&lo)[CW / 2]) {
    static_assert(CW == 16, "one tcgen05.st.x8 per part");
    umma::st8u(umma::taddr(tb, lane_base, n0 >> 1), hi);
    umma::st8u(umma::taddr(tb, lane_base, TC_ALO + (n0 >> 1)), lo);
}

// Act: the activation of one chunk, act(layer, n0, z, hi, lo) - swish + split (activation_compute) in the eval passes,
// vjp_activation in the VJP kernel.
// FFMA first Dense (K = F), output straight into tensor memory: K-chunk c of the next GEMM = columns [32c, 32c+32), of
// which column group `half` owns CW.  The event's first four inputs stay in registers for all chunks, the rest are read
// from hs ([F][UM], x - mean) in a loop.  before_store() runs once, ahead of the first tcgen05.st.
template <int CW, class Act, class BeforeStore>
__device__ __forceinline__ void first_dense_ffma(const float* hs, int F, int m, int half, const float* w0s, const float* b0s,
                                                 uint32_t tb, uint32_t lane_base, uint64_t* aready, Act act,
                                                 BeforeStore before_store) {
    float hreg[4];
#pragma unroll
    for (int f = 0; f < 4; ++f) hreg[f] = f < F ? hs[f * UM + m] : 0.f;
#pragma unroll 1
    for (int c = 0; c < 4; ++c) {
        const int n0 = c * 32 + half * CW;
        float acc[CW];
        uint32_t ahi[CW / 2], alo[CW / 2];
        {
            const float4* bv = reinterpret_cast<const float4*>(b0s + n0);
#pragma unroll
            for (int g4 = 0; g4 < CW / 4; ++g4) {
                const float4 t = bv[g4];
                acc[g4 * 4 + 0] = t.x; acc[g4 * 4 + 1] = t.y; acc[g4 * 4 + 2] = t.z; acc[g4 * 4 + 3] = t.w;
            }
        }
        auto fma_row = [&](float h, int f) {
            const float4* w = reinterpret_cast<const float4*>(w0s + f * 128 + n0);
#pragma unroll
            for (int g4 = 0; g4 < CW / 4; ++g4) {
                const float4 wv = w[g4];
                acc[g4 * 4 + 0] = fmaf(h, wv.x, acc[g4 * 4 + 0]);
                acc[g4 * 4 + 1] = fmaf(h, wv.y, acc[g4 * 4 + 1]);
                acc[g4 * 4 + 2] = fmaf(h, wv.z, acc[g4 * 4 + 2]);
                acc[g4 * 4 + 3] = fmaf(h, wv.w, acc[g4 * 4 + 3]);
            }
        };
#pragma unroll
        for (int f = 0; f < 4; ++f)
            if (f < F) fma_row(hreg[f], f);
        for (int f = 4; f < F; ++f) fma_row(hs[f * UM + m], f);
        act(0, n0, acc, ahi, alo);
        if (c == 0) before_store();
        activation_store<CW>(tb, lane_base, n0, ahi, alo);
        umma::wait_st();
        umma::fence_before_sync();
        umma::mbar_arrive(&aready[c]);
    }
}

// Hidden-layer drain: accumulator -> main + cross * 2^-11 + bias -> act -> the next activations, chunk c = accumulator
// columns [32c + CW half, +CW) -> the same columns of the A operand, then aready[c].  The TMEM loads of chunk c+1 are in
// flight during the arithmetic of chunk c.  FD: the one merged accumulator of the tensor-core first Dense (bias b0').
template <int CW, bool FD, class Act>
__device__ __forceinline__ void hidden_drain(uint32_t cmain, uint32_t ccross, const float* bh, int layer, int half,
                                             uint32_t tb, uint32_t lane_base, uint64_t* aready, Act act) {
    float vn[CW], wn[FD ? 1 : CW];
    tmem_load<CW>(umma::taddr(tb, lane_base, cmain + half * CW), vn);                     // main products
    if constexpr (!FD) tmem_load<CW>(umma::taddr(tb, lane_base, ccross + half * CW), wn);  // cross products (scale 2^11)
#pragma unroll 1
    for (int c = 0; c < 4; ++c) {
        const int n0 = c * 32 + half * CW;
        float v[CW];
        uint32_t ahi[CW / 2], alo[CW / 2];
        umma::wait_ld();
        {
            const float4* bv = reinterpret_cast<const float4*>(bh + n0);
#pragma unroll
            for (int g4 = 0; g4 < CW / 4; ++g4) {
                const float4 t = bv[g4];
                if constexpr (FD) {
                    v[g4 * 4 + 0] = vn[g4 * 4 + 0] + t.x;
                    v[g4 * 4 + 1] = vn[g4 * 4 + 1] + t.y;
                    v[g4 * 4 + 2] = vn[g4 * 4 + 2] + t.z;
                    v[g4 * 4 + 3] = vn[g4 * 4 + 3] + t.w;
                } else {
                    v[g4 * 4 + 0] = fmaf(wn[g4 * 4 + 0], umma::kF16LoUnscale, vn[g4 * 4 + 0]) + t.x;
                    v[g4 * 4 + 1] = fmaf(wn[g4 * 4 + 1], umma::kF16LoUnscale, vn[g4 * 4 + 1]) + t.y;
                    v[g4 * 4 + 2] = fmaf(wn[g4 * 4 + 2], umma::kF16LoUnscale, vn[g4 * 4 + 2]) + t.z;
                    v[g4 * 4 + 3] = fmaf(wn[g4 * 4 + 3], umma::kF16LoUnscale, vn[g4 * 4 + 3]) + t.w;
                }
            }
        }
        if (c < 3) {
            tmem_load<CW>(umma::taddr(tb, lane_base, cmain + n0 + 32), vn);
            if constexpr (!FD) tmem_load<CW>(umma::taddr(tb, lane_base, ccross + n0 + 32), wn);
        }
        act(layer, n0, v, ahi, alo);
        activation_store<CW>(tb, lane_base, n0, ahi, alo);
        umma::wait_st();
        umma::fence_before_sync();
        umma::mbar_arrive(&aready[c]);
    }
}

// Producer: one unit's weight image (N columns x 4 K-chunks of 32, fp16 hi | lo each) into the 4-stage ring
__device__ __forceinline__ void stream_unit(uint64_t* full, uint64_t* empty, float* ring, const float* base, int N,
                                            uint32_t& stage, uint32_t& phase) {
    const uint32_t bytes = (uint32_t)N * 128u;   // one K-chunk (32): fp16 hi | lo images
    for (int c = 0; c < 4; ++c) {
        mbar_wait(&empty[stage], phase ^ 1u);
        mbar_arrive_expect_tx(&full[stage], bytes);
        bulk_copy_g2s(ring + (size_t)stage * URING_FLOATS, base + (size_t)c * N * 32, bytes, &full[stage]);
        if (++stage == URING) { stage = 0; phase ^= 1u; }
    }
}

// MMA issuer: the MMAs of one unit (N = 128 for a hidden layer, NL for one transformed dim of the last layer) into the
// main (dmain) and cross (dcross) accumulators, then `done` is committed.  newver: the unit reads a new version of the
// activations, whose K-chunk c is waited for (aready[c], phase p_ar) before chunk c's MMAs, and chunks [0, nfree) before
// the first (the chunks whose accumulator columns this unit overwrites).  Advances the ring phase, and p_ar if newver.
// One unit = 4 K-chunks = one lap of the 4-stage ring, so chunk c always sits in stage c and every descriptor is (a
// hoisted ring address) + (a compile-time offset): the issuing thread's per-MMA work is what bounds the small-N units,
// keep it to a couple of instructions.
// wait (trace build only, may be null): cycles spent waiting for the activations ([0]) and the weights ([1]) are added.
template <int N>
__device__ __forceinline__ void issue_unit(uint64_t* full, uint64_t* empty, uint64_t* aready, uint64_t* done, const float* ring,
                                           uint32_t tb, uint32_t dmain, uint32_t dcross, bool newver, int nfree,
                                           uint32_t& phase, uint32_t& p_ar, long long* wait = nullptr) {
    static_assert(URING == 4, "the MMA issuer maps chunk c to ring stage c");
    constexpr uint32_t lbo = (uint32_t)(N >> 3) * 128u;
    constexpr uint32_t idesc = umma::instr_desc_f16(N);
    constexpr uint32_t desc_hi = (128u >> 4) | (1u << 14);   // SBO, descriptor version
    const uint32_t ring16 = (smem_u32(ring) >> 4) | ((lbo >> 4) << 16);
    int waited = 0;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
#ifdef ZF_TRACE
        const long long t_a = wait ? clock64() : 0;
#endif
        if (newver) {
            const int need = max(c + 1, nfree);
#pragma unroll
            for (int w = 0; w < 4; ++w)
                if (w >= waited && w < need) mbar_wait(&aready[w], p_ar);
            waited = max(waited, need);
        }
#ifdef ZF_TRACE
        const long long t_f = wait ? clock64() : 0;
        if (wait) wait[0] += t_f - t_a;
#endif
        mbar_wait(&full[c], phase);
#ifdef ZF_TRACE
        if (wait) wait[1] += clock64() - t_f;
#endif
        umma::fence_after_sync();
        if (umma::elect_one()) {
#pragma unroll
            for (int ks = 0; ks < 2; ++ks) {   // K = 16 per kind::f16 instruction
                const uint32_t off_hi = (uint32_t)(c * URING_FLOATS * 4 + ks * 2 * (int)lbo) >> 4;
                const uint32_t off_lo = off_hi + ((uint32_t)N * 64u >> 4);   // lo image follows the hi image
                const uint64_t dhi = ((uint64_t)desc_hi << 32) | (uint64_t)(ring16 + off_hi);
                const uint64_t dlo = ((uint64_t)desc_hi << 32) | (uint64_t)(ring16 + off_lo);
                const uint32_t acol = (uint32_t)(c * 16 + ks * 8);   // fp16 pairs: 8 columns per k-step
                const bool first = (c | ks) == 0;
                umma::mma_f16_ts(dcross, tb + TC_ALO + acol, dhi, idesc, !first);   // A_lo' * B_hi
                umma::mma_f16_ts(dcross, tb + acol, dlo, idesc, true);              // A_hi * B_lo'
                umma::mma_f16_ts(dmain, tb + acol, dhi, idesc, !first);             // A_hi * B_hi
            }
            umma::commit(&empty[c]);
            if (c == 3) umma::commit(done);
        }
        __syncwarp();
    }
    phase ^= 1u;
    if (newver) p_ar ^= 1u;
}

template <bool INVERSE, bool VJP = false>
__device__ __forceinline__ void umma_epilogue_role(const UCtx& cx) {
    constexpr int NG = 2;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int q = warp & 3, half = warp >> 2, m = q * 32 + lane;   // half = column group g in [0, NG)
    constexpr int ET = NG * 128, CW = 32 / NG;                    // epilogue threads; columns per thread and K-chunk
    const ChainArgs& a = cx.a;
    const int D = a.D, C = a.C;
    const UCst cl = cx.cl;
    float *xs = cx.xs, *cs = cx.cs, *xraw = cx.xraw, *hs = cx.hs, *cst = cx.cst, *ldx = cx.ldx;
    uint64_t* bars = cx.bars;
    const StepDesc* steps = cx.steps;
    const float* wsf = a.ws;
    const uint32_t tb = cx.tb;
    const long long n_tiles = cx.n_tiles;
    auto tile_by_bulk = [&](long long t) { return cx.in16 && cx.in_bytes != 0 && (t + 1) * UM <= a.M; };
    const uint32_t lane_base = (uint32_t)(q * 32);
    uint32_t p_fh = 0, p_fd = 0;
    ZF_TR_DECL;
#ifdef ZF_TRACE
    const int trs = (warp == 0) ? 0 : (warp == 4 ? 1 : 3);
#endif
    const int rot_in = INVERSE ? a.rot_total : 0;
    uint32_t ke = 0, xk = 0;   // couplings / bulk-fetched tiles consumed so far (barrier phases)
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        ZF_TR_TILE;
        ZF_TR(trs);
        const long long m0 = tile * UM;
        const int nm = (int)min((long long)UM, a.M - m0);
        // rows -> feature-major tile; padding events sit at 0.5 / 0 and are never stored
        const bool bulk = tile_by_bulk(tile);
        if (bulk) mbar_wait(&bars[B_XFULL], xk & 1u);
        const float* xsrc = bulk ? xraw : a.x + m0 * D;
        const float* csrc = bulk ? xraw + UM * D : a.c + m0 * C;
        const bool xs16 = (D & 3) == 0 && (a.sample || (reinterpret_cast<uintptr_t>(xsrc) & 15) == 0);
        const bool cs16 = C > 0 && (C & 3) == 0 && (reinterpret_cast<uintptr_t>(csrc) & 15) == 0;
        if (xs16) {
            // this thread: every second group of four columns of its own event, one 16-byte read per group and
            // conflict-free writes into the feature-major tile
            const float4* xr = reinterpret_cast<const float4*>(xsrc + (size_t)m * D);
            for (int q = half; q < (D >> 2); q += NG) {
                float4 v = make_float4(0.5f, 0.5f, 0.5f, 0.5f);
                if (m < nm) {
                    if (a.sample) {   // counter-based draws: the value of (event, column) does not depend on who computes it
                        float dr[4];
#pragma unroll 1
                        for (int i = 0; i < 4; ++i) dr[i] = latent_draw(a.lc.kind, a.peakness, a.seed, m0 + m, 4 * q + i);
                        v = make_float4(dr[0], dr[1], dr[2], dr[3]);
                    } else {
                        v = xr[q];
                    }
                }
                int col = pmod(4 * q - rot_in, D);
                const float o[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    xs[col * UM + m] = o[i];
                    if (++col == D) col = 0;
                }
            }
        } else {   // element e = mm * D + j, advanced by 256 per round without dividing
            int mm = tid / D, j = tid - mm * D;
            const int dm = ET / D, dj = ET - dm * D;
            for (int e = tid; e < UM * D; e += ET) {
                int col = j - rot_in;
                if (col < 0) col += D;
                xs[col * UM + mm] =
                    (mm < nm) ? (a.sample ? latent_draw(a.lc.kind, a.peakness, a.seed, m0 + mm, j) : xsrc[e]) : 0.5f;
                mm += dm; j += dj;
                if (j >= D) { j -= D; ++mm; }
            }
        }
        if (cs16) {
            const float4* cr = reinterpret_cast<const float4*>(csrc + (size_t)m * C);
            for (int q = half; q < (C >> 2); q += NG) {
                const float4 v = (m < nm) ? cr[q] : make_float4(0.f, 0.f, 0.f, 0.f);
                cs[(4 * q + 0) * UM + m] = v.x; cs[(4 * q + 1) * UM + m] = v.y;
                cs[(4 * q + 2) * UM + m] = v.z; cs[(4 * q + 3) * UM + m] = v.w;
            }
        } else if (C) {
            int mm = tid / C, j = tid - mm * C;
            const int dm = ET / C, dj = ET - dm * C;
            for (int e = tid; e < UM * C; e += ET) {
                cs[j * UM + mm] = (mm < nm) ? csrc[e] : 0.f;
                mm += dm; j += dj;
                if (j >= C) { j -= C; ++mm; }
            }
        }
        if (bulk) { umma::mbar_arrive(&bars[B_XEMPTY]); ++xk; }
        // the log-det this tile accumulates onto (train forward: one launch per coupling) is requested now, not at the end
        float ld_prev = 0.f;
        if (!VJP && !INVERSE && a.mode != kModeLogProb && a.log_det && a.acc_log_det && half == 0 && m < nm) ld_prev = a.log_det[m0 + m];
        epi_barrier<ET>();
        ZF_TR(trs);   // 1: inputs loaded

        float ld_acc = 0.f;
        for (int si = 0; si < a.n_steps; ++si) {
            const StepDesc& s = steps[INVERSE ? (a.n_steps - 1 - si) : si];
            if (s.kind == kStepKindShiftBounds) {
                // columns split between the groups; groups 1.. hand their log-det share over through ldx
                float ld_sb = 0.f;
                shift_bounds_row<INVERSE>(s, wsf, D, xs, UM, m, ld_sb, half, NG);
                if (half > 0) ldx[(half - 1) * UM + m] = ld_sb;
                epi_barrier<ET>();
                if (half == 0) {
#pragma unroll
                    for (int g = 1; g < NG; ++g) ld_sb += ldx[(g - 1) * UM + m];
                    ld_acc += ld_sb;
                }
                epi_barrier<ET>();
                ZF_TR(trs);   // shift bounds done
                continue;
            }
            const int d = s.d, F = s.F, F_p = ru(F, KC), L = s.n_hidden, rot = s.rot;
            const int K = s.K, P = 3 * K - 1, NL = ru(P, 16);
            // ---- this coupling's constants: fetched by the producer warp into buffer ke & 1
            const uint32_t cb = ke & 1u;
            const float* cc = cst + (size_t)cb * cx.cst_stride;
            const float *bns = cc + cl.bn, *w0s = cc + cl.w0, *b0s = cc + cl.b0, *bhs = cc + cl.bh, *bls = cc + cl.bl;
            mbar_wait(&bars[B_CFULL + cb], (ke >> 1) & 1u);
            ZF_TR(trs);   // constants staged
            // ---- hstack(xc, c) + eval BatchNorm (bijectors.py:341-342).  Scale and bias are folded into the first
            // Dense at pack time, what is left is x - mean: when the first Dense runs on the tensor cores every thread takes
            // it straight from the tile (no staging, no barrier); otherwise the halves share the features
            const bool tcfd = a.u_w0img && F <= 16;   // first Dense on the tensor cores (see below)
            const bool direct = tcfd;
            if (!direct) {
                for (int f = half; f < F; f += NG) {
                    const float v = (f < D - d) ? xs[pmod(d + f - rot, D) * UM + m] : cs[(f - (D - d)) * UM + m];
                    hs[f * UM + m] = v - bns[F_p + f];
                }
                epi_barrier<ET>();
            }
            ZF_TR(trs);   // batch norm done
            auto vjp_side_outputs = [&]() {
                // BatchNorm output for the grad-weight GEMM of the first Dense; the conditioning columns' cotangent
                // passes through unchanged (d y[:, j] / d x[:, j] = 1, bijectors.py:364)
                {
                    char* ht = a.img_h0 + (size_t)tile * 2 * a.wh0 * 256 + (size_t)(m >> 3) * 128 + (size_t)(m & 7) * 16;
                    for (int g8 = half; g8 < (a.wh0 >> 3); g8 += NG) {
                        float hv[8];
                        int col = pmod(d + g8 * 8 - rot, D);
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            const int f = g8 * 8 + i;
                            float v = f == F ? 1.0f : 0.f;
                            if (f < F) {
                                const float xm = ((f < D - d) ? xs[col * UM + m] : cs[(f - (D - d)) * UM + m]) - bns[F_p + f];
                                v = fmaf(xm, bns[f], bns[2 * F_p + f]);
                            }
                            hv[i] = (m < nm) ? v : 0.f;
                            if (++col == D) col = 0;
                        }
                        uint32_t hi[4], lo[4];
#pragma unroll
                        for (int q2 = 0; q2 < 4; ++q2) umma::split_bf16x2(hv[2 * q2], hv[2 * q2 + 1], hi[q2], lo[q2]);
                        *reinterpret_cast<uint4*>(ht + (size_t)g8 * 2048) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                        *reinterpret_cast<uint4*>(ht + (size_t)a.wh0 * 256 + (size_t)g8 * 2048) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
                    }
                }
                if (m < nm) {   // this thread: every second conditioning column of its own event, four loads in flight
                    const float* gyr = a.gy + (m0 + m) * D;
                    float* gxr = a.gx + (m0 + m) * D;
                    int src = pmod(d + half + a.gy_rot, D);
                    for (int j0 = d + half; j0 < D; j0 += 8) {
                        float gv[4];
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            gv[k] = (j0 + 2 * k < D) ? gyr[src] : 0.f;
                            src += 2;
                            if (src >= D) src -= D;
                        }
#pragma unroll
                        for (int k = 0; k < 4; ++k)
                            if (j0 + 2 * k < D) gxr[j0 + 2 * k] = gv[k];
                    }
                }
            };
            if (VJP && !tcfd) vjp_side_outputs();
            auto act = [&](int l, int n0, const float (&z)[CW], uint32_t (&hi)[CW / 2], uint32_t (&lo)[CW / 2]) {
                if (VJP) vjp_activation<CW>(a, l, tile, m0, m, nm, n0, z, hi, lo);
                else activation_compute<CW>(z, hi, lo);
            };
            if (tcfd) {
                // ---- first Dense on the tensor cores: (x - mean) * mul of the event's inputs (3xFP16 split) as a K = 16 A operand
                // in tensor memory, columns [0, 8) (hi) and [TC_ALO, +8) (lo'); this thread writes inputs [8 half, +8) of
                // its event = 4 columns of each.  The MMA warp multiplies it with the W0 image of the constant block
                // into columns [TC_FD, +128); the epilogue below treats the result like a hidden layer.
                float hv[8];
                {
                    const int f0 = 8 * half;
                    int col = pmod(d + f0 - rot, D);
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const int f = f0 + i;
                        float v = 0.f;
                        if (f < F) v = (((f < D - d) ? xs[col * UM + m] : cs[(f - (D - d)) * UM + m]) - bns[F_p + f]) * bns[f];
                        hv[i] = v;
                        if (++col == D) col = 0;
                    }
                }
                uint32_t hi[4], lo[4];
#pragma unroll
                for (int q2 = 0; q2 < 4; ++q2) umma::split_f16x2(hv[2 * q2], hv[2 * q2 + 1], hi[q2], lo[q2]);
                umma::st4u(umma::taddr(tb, lane_base, 4 * half), hi);
                umma::st4u(umma::taddr(tb, lane_base, TC_ALO + 4 * half), lo);
                umma::wait_st();
                umma::fence_before_sync();
                umma::mbar_arrive(&bars[B_A0READY]);
                if (VJP) vjp_side_outputs();   // under the first Dense's MMAs
            } else {
                // first Dense on the FFMA pipe: couplings with more than 16 conditioner inputs, and flows of single-dim
                // couplings run through this kernel (F is 2 or 3 there)
                first_dense_ffma<CW>(hs, F, m, half, w0s, b0s, tb, lane_base, &bars[B_AREADY], act, [] {});
            }
            ZF_TR(trs);   // first dense done
            // ---- hidden layers 1..L-1 (and the tensor-core first Dense's accumulator): drain -> next activations
            auto hidden_epilogue = [&](auto fdtag, int l) {
                constexpr bool FD = decltype(fdtag)::value;
                mbar_wait(&bars[B_DFULL_H], p_fh);
                p_fh ^= 1u;
                umma::fence_after_sync();
                ZF_TR(trs);   // hidden accumulator ready
                hidden_drain<CW, FD>(FD ? TC_FD : TC_HMAIN, TC_HCROSS, FD ? b0s : bhs + (l - 1) * 128, l, half, tb, lane_base,
                                     &bars[B_AREADY], act);
                ZF_TR(trs);   // hidden epilogue done
            };
            if (tcfd) hidden_epilogue(std::true_type{}, 0);
            for (int l = 1; l < L; ++l) hidden_epilogue(std::false_type{}, l);
            // ---- last layer: theta of one transformed dim at a time, read from tensor memory
            float ldc = 0.f;
            if (VJP) {
                // theta row -> this thread's row buffer in shared memory -> cotangent of theta in place (zf_vjp.cuh)
                // -> global, one transformed dim per column group at a time
                float* wrows = reinterpret_cast<float*>(cx.scratch) + ((size_t)half * UM + q * 32) * VJP_ROW;   // this warp's 32 rows
                float* row = wrows + lane * VJP_ROW;
                const KnotNorm kn = make_knot_norm(K);
                const float gld = (!INVERSE && m < nm) ? a.glp[m0 + m] : 0.f;   // the inverse has no log-det
                float gy_next = (half < d && m < nm) ? a.gy[(m0 + m) * D + pmod(half + a.gy_rot, D)] : 0.f;
                for (int jj = half; jj < d; jj += 2) {
                    const float gyv = gy_next;
                    if (jj + 2 < d && m < nm) gy_next = a.gy[(m0 + m) * D + pmod(jj + 2 + a.gy_rot, D)];   // under this row's work
                    mbar_wait(&bars[B_DFULL_D + half], p_fd);
                    p_fd ^= 1u;
                    umma::fence_after_sync();
                    ZF_TR(trs);   // theta ready
                    const uint32_t dbase = umma::taddr(tb, lane_base, tc_dmain(half));
                    auto release = [&]() {
                        umma::fence_before_sync();
                        umma::mbar_arrive(&bars[B_DEMPTY_D + half]);
                        ZF_TR(trs);   // released
                    };
                    const float xv = xs[pmod(jj - rot, D) * UM + m];
                    float g_x;
                    if (K == 16) g_x = vjp_row_tmem<16, INVERSE>(dbase, bls + jj * NL, row, xv, gyv, gld, release);
                    else g_x = vjp_row_tmem<32, INVERSE>(dbase, bls + jj * NL, row, xv, gyv, gld, release);
                    ZF_TR(trs);   // row cotangent done
                    if (m < nm) a.gx[(m0 + m) * D + jj] = g_x;
                    {   // this thread's row -> the event-row image: 16-byte units of 8 columns, hi and lo parts; the 32 lanes of a
                        // warp write 512 contiguous bytes per unit
                        const int TW = d * NL;
                        char* dt = a.img_dtheta + (size_t)tile * 2 * TW * 256 + (size_t)(m >> 3) * 128 + (size_t)(m & 7) * 16 +
                                   (size_t)(jj * NL >> 3) * 2048;
                        const bool valid = m < nm;
                        for (int u = 0; u < (NL >> 3); ++u) {
                            uint32_t hi[4], lo[4];
#pragma unroll
                            for (int q2 = 0; q2 < 4; ++q2)
                                umma::split_bf16x2(valid ? row[8 * u + 2 * q2] : 0.f, valid ? row[8 * u + 2 * q2 + 1] : 0.f, hi[q2], lo[q2]);
                            *reinterpret_cast<uint4*>(dt + (size_t)u * 2048) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                            *reinterpret_cast<uint4*>(dt + (size_t)TW * 256 + (size_t)u * 2048) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
                        }
                    }
                }
            } else {
                for (int jj = half; jj < d && half < 2; jj += 2) {
                    mbar_wait(&bars[B_DFULL_D + half], p_fd);
                    p_fd ^= 1u;
                    umma::fence_after_sync();
                    ZF_TR(trs);   // theta ready
                    const uint32_t dbase = umma::taddr(tb, lane_base, tc_dmain(half));
                    float* px = xs + pmod(jj - rot, D) * UM + m;
                    const float v = *px;
                    RqsBin bin;
                    auto release = [&]() {
                        umma::fence_before_sync();
                        umma::mbar_arrive(&bars[B_DEMPTY_D + half]);
                        ZF_TR(trs);   // released
                    };
                    float4* scr = cx.scratch + (size_t)half * 8 * UM + m;   // [half][K / 4][UM] float4
                    if (K == 16) spline_row_tmem_lean<16, INVERSE>(dbase, TC_XOFF, bls + jj * NL, v, bin, scr, UM, release);
                    else spline_row_tmem_lean<32, INVERSE>(dbase, TC_XOFF, bls + jj * NL, v, bin, scr, UM, release);
                    if (m < nm) put_idx(a, s, m0 + m, jj, bin.idx);
                    if (!INVERSE) {
                        float y, ld;
                        rqs_eval_forward(v, bin, y, ld);
                        *px = y;
                        ldc += ld;
                    } else {
                        *px = rqs_eval_inverse(v, bin);
                    }
                }
            }
            ZF_TR(trs);   // spline rows done
            umma::mbar_arrive(&bars[B_CEMPTY + cb]);   // last read of this coupling's constants
            ++ke;
            if (half == 1) ldx[m] = ldc;
            epi_barrier<ET>();
            if (half == 0) ld_acc += ldc + ldx[m];
            epi_barrier<ET>();
            ZF_TR(trs);   // coupling done
        }

        // ---- store
        if (VJP) {
        } else if (a.mode == kModeLogProb) {
            if (half == 0 && m < nm) {
                float lat = 0.f;
                for (int j = 0; j < D; ++j) lat += latent_logpdf(xs[pmod(j - a.rot_total, D) * UM + m], a.lc);
                a.lp[m0 + m] = nan_to_num_lp(lat + ld_acc);
            }
        } else {
            const int rot_out = INVERSE ? 0 : a.rot_total;
            if (a.y) {
                if ((D & 3) == 0 && (reinterpret_cast<uintptr_t>(a.y) & 15) == 0) {
                    // this thread: every second group of four columns of its own event (conflict-free reads of the
                    // feature-major tile, one 16-byte store per group)
                    if (m < nm) {
                        float4* yr = reinterpret_cast<float4*>(a.y + (m0 + m) * D);
                        for (int q = half; q < (D >> 2); q += NG) {
                            int col = pmod(4 * q - rot_out, D);
                            float o[4];
#pragma unroll
                            for (int i = 0; i < 4; ++i) {
                                o[i] = xs[col * UM + m];
                                if (++col == D) col = 0;
                            }
                            yr[q] = make_float4(o[0], o[1], o[2], o[3]);
                        }
                    }
                } else {
                    for (int e = tid; e < nm * D; e += ET) {
                        const int mm = e / D, j = e - mm * D;
                        a.y[m0 * D + e] = xs[pmod(j - rot_out, D) * UM + mm];
                    }
                }
            }
            if (!INVERSE && a.log_det && half == 0 && m < nm)
                a.log_det[m0 + m] = a.acc_log_det ? ld_prev + ld_acc : ld_acc;
        }
        epi_barrier<ET>();
        ZF_TR(trs);   // tile stored
    }
}

template <int N> __device__ __forceinline__ void reg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N)); }
template <int N> __device__ __forceinline__ void reg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N)); }

// 8 epilogue warps (two column groups) + producer + MMA issuer (320 threads).
template <bool INVERSE, bool VJP = false>
__global__ void __launch_bounds__(320, 1) chain_umma_kernel(const __grid_constant__ ChainArgs a) {
    constexpr int NG = 2;
    extern __shared__ __align__(128) float smem[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    constexpr int ET = NG * 128, PW = NG * 4, MW = NG * 4 + 1;   // epilogue threads, producer warp, MMA warp
    const int D = a.D, C = a.C;
    const UCst cl = ucst_layout(a.u_fmax, a.u_hmax, a.u_blmax, a.u_w0img != 0);
    float* xs = smem;                         // [D][UM]  the tile, feature-major
    float* cs = xs + D * UM;                  // [C][UM]
    float* xraw = cs + C * UM;                // [UM][D] | [UM][C]  next tile as it lies in global memory (cp.async)
    float* hs = xraw + UM * (D + C);          // [Fmax][UM]  x - mean (couplings whose first Dense reads it from shared memory)
    float* cst = hs + umma_hs_floats(a.u_fmax);   // [2][cl.total] per-coupling constants
    // the VJP kernel runs ONE coupling: its constants are fetched once and both buffer indices name the same block
    const int cst_stride = VJP ? 0 : cl.total;
    float* ldx = cst + (VJP ? 1 : 2) * cl.total;
    float* scratch = ldx + 3 * UM;            // [2][8][UM] float4: scratch columns of the lean spline rows
    float* ring = scratch + (VJP ? 2 * UM * VJP_ROW : 2 * 8 * UM * 4);   // VJP: [2][UM][VJP_ROW] theta rows instead
    uint64_t* bars = reinterpret_cast<uint64_t*>(ring + (size_t)URING * URING_FLOATS);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + B_COUNT);
    StepDesc* steps_s = reinterpret_cast<StepDesc*>(tmem_slot + 32);
    const float* wsf = a.ws;
    // the step program is read at every phase boundary by every role: keep it in shared memory
    const bool steps_fit = a.n_steps <= USTEPS;
    if (steps_fit) {
        const int4* src = reinterpret_cast<const int4*>(a.ws);
        int4* dst = reinterpret_cast<int4*>(steps_s);
        for (int i = tid; i < a.n_steps * (int)(sizeof(StepDesc) / 16); i += (int)blockDim.x) dst[i] = src[i];
    }
    const StepDesc* steps = steps_fit ? steps_s : reinterpret_cast<const StepDesc*>(a.ws);

    if (tid == 0) {
        for (int i = 0; i < URING; ++i) { mbar_init(&bars[B_FULL + i], 1); mbar_init(&bars[B_EMPTY + i], 1); }
        for (int i = 0; i < 4; ++i) mbar_init(&bars[B_AREADY + i], ET);
        mbar_init(&bars[B_DFULL_H], 1);
        mbar_init(&bars[B_DFULL_D + 0], 1);
        mbar_init(&bars[B_DFULL_D + 1], 1);
        mbar_init(&bars[B_DEMPTY_D + 0], 128);
        mbar_init(&bars[B_DEMPTY_D + 1], 128);
        for (int i = 0; i < 2; ++i) { mbar_init(&bars[B_CFULL + i], 1); mbar_init(&bars[B_CEMPTY + i], ET); }
        mbar_init(&bars[B_XFULL], 1);
        mbar_init(&bars[B_XEMPTY], ET);
        mbar_init(&bars[B_A0READY], ET);
        mbar_fence_init();
    }
    if (warp == MW) umma::tmem_alloc(tmem_slot, 512);
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tb = *tmem_slot;
    const long long n_tiles = (a.M + UM - 1) / UM;
    // Full tiles of 16-byte-aligned inputs are fetched one tile ahead by the producer warp (bulk copies of the raw
    // rows); the tail tile and unaligned inputs are read by the epilogue warps themselves.
    const uint32_t in_bytes = (a.sample ? 0u : (uint32_t)(UM * D * 4)) + (uint32_t)(UM * C * 4);
    const bool in16 = ((reinterpret_cast<uintptr_t>(a.x) | reinterpret_cast<uintptr_t>(a.c)) & 15) == 0;
    auto tile_by_bulk = [&](long long t) { return in16 && in_bytes != 0 && (t + 1) * UM <= a.M; };
    // the coupling that follows step position `si` in processing order, cyclically (the next tile starts over)
    auto next_coupling = [&](int si) -> const StepDesc& {
        for (int k = 1; k <= a.n_steps; ++k) {
            const int sj = (si + k) % a.n_steps;
            const StepDesc& t = steps[INVERSE ? (a.n_steps - 1 - sj) : sj];
            if (t.kind == kStepKindCoupling) return t;
        }
        return steps[0];   // not reached: this kernel is only launched for chains with a coupling
    };
    int last_coupling_si = 0;
    for (int si = 0; si < a.n_steps; ++si)
        if (steps[INVERSE ? (a.n_steps - 1 - si) : si].kind == kStepKindCoupling) last_coupling_si = si;

    auto producer_role = [&]() {
        // ------------------------------------------------------------------ producer: weights, constants, inputs
        if (lane == 0) {
            uint32_t stage = 0, phase = 0, kc = 0, xk = 0;
            auto issue_consts = [&](const StepDesc& sn) {   // constant block of the kc-th coupling of this CTA
                const uint32_t b = kc & 1u;
                mbar_wait(&bars[B_CEMPTY + b], ((kc >> 1) & 1u) ^ 1u);
                if (VJP && kc > 0) {
                    umma::mbar_arrive(&bars[B_CFULL + b]);   // already resident
                } else {
                    mbar_arrive_expect_tx(&bars[B_CFULL + b], (uint32_t)cl.total * 4u);
                    bulk_copy_g2s(cst + (size_t)b * cst_stride, wsf + sn.off_C, (uint32_t)cl.total * 4u, &bars[B_CFULL + b]);
                }
                ++kc;
            };
            auto issue_inputs = [&](long long t) {
                if (!tile_by_bulk(t)) return;
                mbar_wait(&bars[B_XEMPTY], (xk & 1u) ^ 1u);
                mbar_arrive_expect_tx(&bars[B_XFULL], in_bytes);
                if (!a.sample) bulk_copy_g2s(xraw, a.x + t * UM * D, (uint32_t)(UM * D * 4), &bars[B_XFULL]);
                if (C) bulk_copy_g2s(xraw + UM * D, a.c + t * UM * C, (uint32_t)(UM * C * 4), &bars[B_XFULL]);
                ++xk;
            };
            if ((long long)blockIdx.x < n_tiles) {
                issue_inputs(blockIdx.x);
                issue_consts(next_coupling(a.n_steps - 1));
            }
            for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
                const bool more_tiles = tile + gridDim.x < n_tiles;
                bool inputs_pending = more_tiles;
                for (int si = 0; si < a.n_steps; ++si) {
                    const StepDesc& s = steps[INVERSE ? (a.n_steps - 1 - si) : si];
                    if (s.kind != kStepKindCoupling) continue;
                    const int L = s.n_hidden, NL = ru(3 * s.K - 1, 16);
                    for (int u = 0; u < (L - 1) + s.d; ++u) {
                        const bool hid = u < L - 1;
                        const int N = hid ? 128 : NL;
                        const float* base = hid ? wsf + s.off_U[u + 1] : wsf + s.off_U[L] + (size_t)(u - (L - 1)) * NL * 128;
                        stream_unit(&bars[B_FULL], &bars[B_EMPTY], ring, base, N, stage, phase);
                        if (u == 0) {
                            // behind this coupling's first unit: the next coupling's constants (their buffer is
                            // released when the previous coupling ends) and, once per tile, the next tile's rows
                            if (si != last_coupling_si || more_tiles) issue_consts(next_coupling(si));
                            if (inputs_pending) { issue_inputs(tile + gridDim.x); inputs_pending = false; }
                        }
                    }
                }
            }
        }
        __syncwarp();
    };
    auto mma_role = [&]() {
        // ------------------------------------------------------------------ MMA issuer
        // Main and cross products go to separate accumulators (the cross products carry the 2^11 scale of the lo'
        // parts; the tensor core's fp32 accumulator also truncates at every accumulate step - measured -2.3e-8
        // relative per step, tests/test_gpu_umma.py - which the small cross terms would otherwise suffer at the
        // main product's magnitude): hidden layers main [256,384), cross [384,512); last-layer dim in buffer
        // b = dim & 1: main [128 + 192 b, +NL), cross 96 columns further.
        // The epilogue publishes a new activation version one 32-column K-chunk at a time (B_AREADY + c), and the
        // MMAs of chunk c are issued as soon as it has arrived, so the layer's GEMM runs underneath the
        // bias/swish/split of the chunks behind it.  The arrival of chunk c also says that accumulator columns
        // [32c, 32c+32) of D0 and D1 have been drained, which is what lets the first last-layer unit start
        // before the hidden epilogue has finished (it only needs the columns it overwrites to be free).
        uint32_t phase = 0, p_ar = 0, p_ed0 = 0, p_ed1 = 0, p_a0 = 0, kcm = 0;
        bool dim_pending0 = false, dim_pending1 = false;
        ZF_TR_DECL;
        for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            ZF_TR_TILE;
            for (int si = 0; si < a.n_steps; ++si) {
                const StepDesc& s = steps[INVERSE ? (a.n_steps - 1 - si) : si];
                if (s.kind != kStepKindCoupling) continue;
                const int L = s.n_hidden, NL = ru(3 * s.K - 1, 16);
                const bool tcfd = a.u_w0img && s.F <= 16;
                if (tcfd) {
                    // first Dense: A = the epilogue's (x - mean) operand in tensor memory, B = the W0 image of this
                    // coupling's constant block; one k-step (K = 16), three products into ONE accumulator [TC_FD, +128):
                    // the two cross products (scale 2^11) first, then the main product as D = A_hi B_hi + D 2^-11
                    if (dim_pending0) { mbar_wait(&bars[B_DEMPTY_D + 0], p_ed0); p_ed0 ^= 1u; dim_pending0 = false; }
                    if (dim_pending1) { mbar_wait(&bars[B_DEMPTY_D + 1], p_ed1); p_ed1 ^= 1u; dim_pending1 = false; }
                    const uint32_t cbm = kcm & 1u;
                    mbar_wait(&bars[B_CFULL + cbm], (kcm >> 1) & 1u);
                    mbar_wait(&bars[B_A0READY], p_a0);
                    p_a0 ^= 1u;
                    umma::fence_after_sync();
                    if (umma::elect_one()) {
                        const uint32_t w0 = smem_u32(cst + (size_t)cbm * cst_stride + cl.w0i);
                        const uint64_t b_hi = umma::smem_desc_kmajor(w0, 2048u, 128u), b_lo = umma::smem_desc_kmajor(w0 + 4096u, 2048u, 128u);
                        constexpr uint32_t idesc = umma::instr_desc_f16(128);
                        umma::mma_f16_ts(tb + TC_FD, tb + TC_ALO, b_hi, idesc, false);
                        umma::mma_f16_ts(tb + TC_FD, tb, b_lo, idesc, true);
                        umma::mma_f16_ts_scaled<11>(tb + TC_FD, tb, b_hi, idesc);
                        umma::commit(&bars[B_DFULL_H]);
                    }
                    __syncwarp();
                }
                ++kcm;
                for (int u = 0; u < (L - 1) + s.d; ++u) {
                    const bool hid = u < L - 1;
                    const int b = hid ? 0 : ((u - (L - 1)) & 1);
                    ZF_TR(2);
                    const bool newver = hid || u == L - 1;   // this unit reads a new version of the activations
                    // chunks that must have arrived before the first MMA: those whose accumulator columns this unit
                    // overwrites (u == 0 follows the SIMT first layer: nothing to drain); a hidden unit overwrites all of
                    // them, the first last-layer unit (theta buffer 0) only the hidden main columns of chunks 0 and 1
                    // (a tensor-core first Dense accumulates in [TC_FD, +128): only a theta unit right behind it overlaps)
                    const int nfree = (u == 0) ? ((tcfd && !hid) ? 4 : 0) : (hid ? 4 : 2);
                    long long w_ab[2] = {0, 0};   // trace build: cycles waited for the activations / the weights
#ifdef ZF_TRACE
                    long long w_pend = clock64();
#endif
                    if ((hid || b == 0) && dim_pending0) { mbar_wait(&bars[B_DEMPTY_D + 0], p_ed0); p_ed0 ^= 1u; dim_pending0 = false; }
                    if ((hid || b == 1) && dim_pending1) { mbar_wait(&bars[B_DEMPTY_D + 1], p_ed1); p_ed1 ^= 1u; dim_pending1 = false; }
                    umma::fence_after_sync();
#ifdef ZF_TRACE
                    w_pend = clock64() - w_pend;
#endif
                    const uint32_t dmain = hid ? tb + TC_HMAIN : tb + tc_dmain(b);
                    const uint32_t dcross = hid ? tb + TC_HCROSS : dmain + TC_XOFF;
                    uint64_t* done = &bars[hid ? B_DFULL_H : (B_DFULL_D + b)];
                    auto unit = [&](auto n) {
                        issue_unit<decltype(n)::value>(&bars[B_FULL], &bars[B_EMPTY], &bars[B_AREADY], done, ring, tb, dmain,
                                                       dcross, newver, nfree, phase, p_ar, w_ab);
                    };
                    if (hid) unit(std::integral_constant<int, 128>{});
                    else if (NL == 48) unit(std::integral_constant<int, 48>{});
                    else unit(std::integral_constant<int, 96>{});
                    ZF_TR(2);
                    ZF_TRV(2, -w_pend); ZF_TRV(2, -w_ab[0]); ZF_TRV(2, -w_ab[1]);
                    if (!hid) { if (b) dim_pending1 = true; else dim_pending0 = true; }
                }
            }
        }
    };
    // ------------------------------------------------------------------ role dispatch
    const UCtx cx{a, xs, cs, xraw, hs, cst, ldx, reinterpret_cast<float4*>(scratch), bars, steps, tb, n_tiles, cl, cst_stride, in16, in_bytes};
    if (warp == PW) producer_role();
    else if (warp == MW) mma_role();
    else umma_epilogue_role<INVERSE, VJP>(cx);

    umma::fence_before_sync();
    __syncthreads();
    if (warp == MW) umma::tmem_dealloc(tb, 512);
}

// =============================================================================================
// Two tiles in flight for flows whose couplings transform ONE dim (every 2-D / 3-D flow: the headline config).
//
// The single-tile kernel above is a serial chain per tile: activation phases (SFU / issue bound), GEMM tails, the
// spline row, the tile's load / ShiftBounds / store, each waiting for the previous one, because tensor memory is full
// and a second tile cannot simply be added.  But the chain only needs the activations (A) and the hidden
// accumulators (D0, D1) during the conditioner, and only the theta columns during the spline - so two tiles can
// share the same tensor memory if they are half a coupling apart.  Warps are specialised by PHASE instead of by
// column group:
//   warps 0-7   "activation" warps (S1): BatchNorm, first Dense, hidden epilogues, for slot 0 and slot 1 in turn
//   warps 8-11  "row" warps (S2): tile load, ShiftBounds, the spline row (theta from tensor memory), latent + store
//   warp 12     producer (weights ring, per-(coupling, slot) constants, next tile's raw rows)
//   warp 13     MMA issuer (same unit logic as above, in the interleaved order)
// Every role walks the same static schedule: for each pair of tiles, for each step, slot 0 then slot 1.  While S2 runs
// the spline of slot X, S1 is already in the next activation phase of slot Y, and the MMA tails of one slot hide under
// the other slot's work.  setmaxnreg gives S2 the registers of the spline code and S1 a small budget.
// =============================================================================================
enum PpBar : int { PP_FULL = 0, PP_EMPTY = 4, PP_AREADY = 8, PP_DFULL_H = 12, PP_DFULL_D = 13, PP_DEMPTY_D = 14,
                   PP_CFULL = 15, PP_CEMPTY = 19, PP_XFULL = 23, PP_XEMPTY = 25, PP_XSREADY = 27, PP_COUNT = 32 };
constexpr int PP_TBUF = 4;   // tile-state buffers: the row warps prepare the next pair's tiles while the current pair runs
constexpr int PP_THREADS = 512;
constexpr int PP_CBUF = 4;   // constant-block buffers: one (coupling, slot) occurrence each, fetched one occurrence ahead

__host__ __device__ inline size_t umma_pp_smem_floats(int D, int C, int Fmax, int Hmax, int BLmax) {
    return (PP_TBUF + 2) * (size_t)UM * (D + C) + 2 * (size_t)Fmax * UM + PP_CBUF * (size_t)ucst_layout(Fmax, Hmax, BLmax).total +
           PP_TBUF * UM + 8 * UM * 4 +
           (size_t)URING * URING_FLOATS + 2 * PP_COUNT + 32 + USTEPS * sizeof(StepDesc) / sizeof(float) + USTEPS;
}

__device__ __forceinline__ void s1_barrier() { asm volatile("bar.sync 1, 256;" ::: "memory"); }
__device__ __forceinline__ void s2_barrier() { asm volatile("bar.sync 2, 128;" ::: "memory"); }

template <bool INVERSE>
__global__ void __launch_bounds__(PP_THREADS, 1) chain_umma_pp_kernel(const __grid_constant__ ChainArgs a) {
    extern __shared__ __align__(128) float smem[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    constexpr int PW = 12, MW = 13;
    const int D = a.D, C = a.C;
    const UCst cl = ucst_layout(a.u_fmax, a.u_hmax, a.u_blmax);
    float* xsb = smem;                          // [PP_TBUF][D][UM]  tile state (tile k in buffer k % PP_TBUF), feature-major
    float* csb = xsb + PP_TBUF * D * UM;        // [PP_TBUF][C][UM]
    float* xraw = csb + PP_TBUF * C * UM;       // [2]{[UM][D] | [UM][C]}  raw rows of upcoming tiles (bulk copy)
    float* hs2 = xraw + 2 * UM * (D + C);       // [2][Fmax][UM]  BatchNorm output by occurrence parity (S1 only)
    float* cst = hs2 + 2 * a.u_fmax * UM;       // [PP_CBUF][cl.total]
    float* ldacc = cst + PP_CBUF * cl.total;    // [PP_TBUF][UM]  log-det accumulator per tile (S2 only)
    float* scratch = ldacc + PP_TBUF * UM;      // [8][UM] float4: scratch columns of the lean spline rows (S2 only)
    float* ring = scratch + 8 * UM * 4;
    uint64_t* bars = reinterpret_cast<uint64_t*>(ring + (size_t)URING * URING_FLOATS);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + PP_COUNT);
    StepDesc* steps_s = reinterpret_cast<StepDesc*>(tmem_slot + 32);
    int* coup_si = reinterpret_cast<int*>(steps_s + USTEPS);   // processing positions of the coupling steps
    const float* wsf = a.ws;

    {   // step program -> shared memory (the host only launches this kernel when it fits)
        const int4* src = reinterpret_cast<const int4*>(a.ws);
        int4* dst = reinterpret_cast<int4*>(steps_s);
        for (int i = tid; i < a.n_steps * (int)(sizeof(StepDesc) / 16); i += PP_THREADS) dst[i] = src[i];
    }
    const StepDesc* steps = steps_s;
    if (tid == 0) {
        for (int i = 0; i < URING; ++i) { mbar_init(&bars[PP_FULL + i], 1); mbar_init(&bars[PP_EMPTY + i], 1); }
        for (int i = 0; i < 4; ++i) mbar_init(&bars[PP_AREADY + i], 256);
        mbar_init(&bars[PP_DFULL_H], 1);
        mbar_init(&bars[PP_DFULL_D], 1);
        mbar_init(&bars[PP_DEMPTY_D], 128);
        for (int i = 0; i < PP_CBUF; ++i) { mbar_init(&bars[PP_CFULL + i], 1); mbar_init(&bars[PP_CEMPTY + i], 256 + 128); }
        for (int i = 0; i < 2; ++i) { mbar_init(&bars[PP_XFULL + i], 1); mbar_init(&bars[PP_XEMPTY + i], 128); }
        for (int i = 0; i < PP_TBUF; ++i) mbar_init(&bars[PP_XSREADY + i], 128);
        mbar_fence_init();
    }
    if (warp == MW) umma::tmem_alloc(tmem_slot, 512);
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tb = *tmem_slot;
    if (tid == 0) {
        int n = 0;
        for (int si = 0; si < a.n_steps; ++si)
            if (steps[INVERSE ? (a.n_steps - 1 - si) : si].kind == kStepKindCoupling) coup_si[n++] = si;
    }
    __syncthreads();
    int ncoup = 0;
    for (int si = 0; si < a.n_steps; ++si)
        if (steps[si].kind == kStepKindCoupling) ++ncoup;
    auto step_at = [&](int si) -> const StepDesc& { return steps[INVERSE ? (a.n_steps - 1 - si) : si]; };

    const long long n_tiles = (a.M + UM - 1) / UM;
    const long long n_my = ((long long)blockIdx.x < n_tiles) ? (n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    const long long n_occ = n_my * ncoup;       // (coupling, tile) occurrences of this CTA, in schedule order
    auto tile_of = [&](long long k) { return (long long)blockIdx.x + k * gridDim.x; };
    const uint32_t in_bytes = (a.sample ? 0u : (uint32_t)(UM * D * 4)) + (uint32_t)(UM * C * 4);
    const bool in16 = ((reinterpret_cast<uintptr_t>(a.x) | reinterpret_cast<uintptr_t>(a.c)) & 15) == 0;
    auto tile_by_bulk = [&](long long t) { return in16 && in_bytes != 0 && (t + 1) * UM <= a.M; };
    // the coupling step of occurrence n: pairs of tiles, coupling-major, slot-minor
    auto occ_step = [&](long long n) -> const StepDesc& {
        const long long per_pair = 2LL * ncoup;
        const long long p = n / per_pair;
        const long long r = n - p * per_pair;
        const int nslots = (2 * p + 1 < n_my) ? 2 : 1;
        return step_at(coup_si[(int)(r / nslots)]);
    };

    // ------------------------------------------------------------------------------------------------ roles
    auto producer_role = [&]() {
        if (lane != 0) return;
        uint32_t stage = 0, phase = 0;
        long long kc = 0;   // constant blocks issued
        auto issue_consts = [&]() {
            if (kc >= n_occ) return;
            const uint32_t b = (uint32_t)(kc % PP_CBUF);
            mbar_wait(&bars[PP_CEMPTY + b], (uint32_t)((kc / PP_CBUF) & 1) ^ 1u);
            mbar_arrive_expect_tx(&bars[PP_CFULL + b], (uint32_t)cl.total * 4u);
            bulk_copy_g2s(cst + (size_t)b * cl.total, wsf + occ_step(kc).off_C, (uint32_t)cl.total * 4u, &bars[PP_CFULL + b]);
            ++kc;
        };
        // tile k (slot k & 1, pair k >> 1) is staged in raw buffer k & 1; its previous user was tile k - 2.  Only full
        // tiles of aligned inputs come this way, and only the globally last tile can be ragged, so the use count of a
        // buffer is the pair index on both sides.
        auto issue_inputs = [&](long long k) {
            if (k >= n_my) return;
            const long long t = tile_of(k);
            if (!tile_by_bulk(t)) return;
            const int b = (int)(k & 1);
            const uint32_t use = (uint32_t)(k >> 1);
            float* dst = xraw + (size_t)b * UM * (D + C);
            mbar_wait(&bars[PP_XEMPTY + b], (use & 1u) ^ 1u);
            mbar_arrive_expect_tx(&bars[PP_XFULL + b], in_bytes);
            if (!a.sample) bulk_copy_g2s(dst, a.x + t * UM * D, (uint32_t)(UM * D * 4), &bars[PP_XFULL + b]);
            if (C) bulk_copy_g2s(dst + UM * D, a.c + t * UM * C, (uint32_t)(UM * C * 4), &bars[PP_XFULL + b]);
        };
        issue_inputs(0);
        issue_inputs(1);
        issue_consts();
        for (long long p = 0; 2 * p < n_my; ++p) {
            const int nslots = (2 * p + 1 < n_my) ? 2 : 1;
            for (int si = 0; si < a.n_steps; ++si) {
                const StepDesc& s = step_at(si);
                if (s.kind != kStepKindCoupling) continue;
                const int L = s.n_hidden, NL = ru(3 * s.K - 1, 16);
                for (int slot = 0; slot < nslots; ++slot) {
                    for (int u = 0; u < L; ++u) {   // L - 1 hidden units + one last-layer unit (d == 1)
                        const bool hid = u < L - 1;
                        const int N = hid ? 128 : NL;
                        const float* base = hid ? wsf + s.off_U[u + 1] : wsf + s.off_U[L];
                        stream_unit(&bars[PP_FULL], &bars[PP_EMPTY], ring, base, N, stage, phase);
                        if (u == 0) {
                            issue_consts();                       // the next occurrence's constants
                            // once per tile: the rows of the tile that takes this slot in the next pair
                            if (si == coup_si[0]) issue_inputs(2 * (p + 1) + slot);
                        }
                    }
                }
            }
        }
    };

    auto mma_role = [&]() {
        uint32_t phase = 0, p_ar = 0, p_ed = 0;
        bool theta_pending = false;   // the theta columns hold a row that the row warps may still be reading
        int pending_nl = 0;           // its width (decides whether the hidden accumulators overlap it)
        for (long long p = 0; 2 * p < n_my; ++p) {
            const int nslots = (2 * p + 1 < n_my) ? 2 : 1;
            for (int si = 0; si < a.n_steps; ++si) {
                const StepDesc& s = step_at(si);
                if (s.kind != kStepKindCoupling) continue;
                const int L = s.n_hidden, NL = ru(3 * s.K - 1, 16);
                for (int slot = 0; slot < nslots; ++slot) {
                    for (int u = 0; u < L; ++u) {
                        const bool hid = u < L - 1;
                        // a theta row at [384, 480) (K = 16) overlaps nothing but the next theta row
                        const bool clear = !hid && NL == 48;
                        const int nfree = (u == 0 || clear) ? 0 : 4;
                        if (theta_pending && (!hid || pending_nl != 48)) {
                            mbar_wait(&bars[PP_DEMPTY_D], p_ed); p_ed ^= 1u; theta_pending = false;
                        }
                        umma::fence_after_sync();
                        const uint32_t dmain = hid ? tb + TC_PP_HMAIN : tb + tc_pp_theta(NL);
                        const uint32_t dcross = hid ? tb + TC_PP_HCROSS : dmain + tc_pp_xoff(NL);
                        uint64_t* done = &bars[hid ? PP_DFULL_H : PP_DFULL_D];
                        // every unit reads a new version of the activations (d == 1)
                        auto unit = [&](auto n) {
                            issue_unit<decltype(n)::value>(&bars[PP_FULL], &bars[PP_EMPTY], &bars[PP_AREADY], done, ring, tb, dmain,
                                                           dcross, true, nfree, phase, p_ar);
                        };
                        if (hid) unit(std::integral_constant<int, 128>{});
                        else if (NL == 48) unit(std::integral_constant<int, 48>{});
                        else unit(std::integral_constant<int, 96>{});
                        if (!hid) { theta_pending = true; pending_nl = NL; }
                    }
                }
            }
        }
    };

    // S1: BatchNorm + first Dense + hidden epilogues of one (coupling, slot) occurrence after the other
    auto activation_role = [&]() {
        const int q = warp & 3, half = warp >> 2, m = q * 32 + lane;
        const uint32_t lane_base = (uint32_t)(q * 32);
        constexpr int CW = 16;
        auto act = [](int, int, const float (&z)[CW], uint32_t (&hi)[CW / 2], uint32_t (&lo)[CW / 2]) {
            activation_compute<CW>(z, hi, lo);
        };
        uint32_t p_fh = 0;
        long long n1 = 0;
        long long bn_done = -1;   // occurrence whose BatchNorm output is already in hs2[n & 1]
        // waits + hstack(xc, c) + eval BatchNorm (bijectors.py:341-342) of occurrence n = (pair p, coupling cj, slot)
        auto batch_norm = [&](long long n, long long p, int cj, int slot) {
            const StepDesc& s = step_at(coup_si[cj]);
            const int d = s.d, F = s.F, F_p = ru(F, KC), rot = s.rot;
            const long long k = 2 * p + slot;
            const int tbuf = (int)(k % PP_TBUF);
            const float* xs = xsb + tbuf * D * UM;
            const float* cs = csb + tbuf * C * UM;
            const uint32_t cb = (uint32_t)(n % PP_CBUF);
            const float* bns = cst + (size_t)cb * cl.total + cl.bn;
            float* hs = hs2 + (size_t)(n & 1) * a.u_fmax * UM;
            mbar_wait(&bars[PP_CFULL + cb], (uint32_t)((n / PP_CBUF) & 1));
            // the cj-th signal of the (k / PP_TBUF)-th tile that uses this state buffer
            mbar_wait(&bars[PP_XSREADY + tbuf], (uint32_t)(((k / PP_TBUF) * ncoup + cj) & 1));
            for (int f = half; f < F; f += 2) {
                const float v = (f < D - d) ? xs[pmod(d + f - rot, D) * UM + m] : cs[(f - (D - d)) * UM + m];
                hs[f * UM + m] = v - bns[F_p + f];   // scale and bias are folded into the first Dense (pack_step_kernel)
            }
            bn_done = n;
        };
        for (long long p = 0; 2 * p < n_my; ++p) {
            const int nslots = (2 * p + 1 < n_my) ? 2 : 1;
            int cj = -1;   // ordinal of the coupling inside the step program
            for (int si = 0; si < a.n_steps; ++si) {
                const StepDesc& s = step_at(si);
                if (s.kind != kStepKindCoupling) continue;
                ++cj;
                const int F = s.F, L = s.n_hidden;
#pragma unroll 1
                for (int slot = 0; slot < nslots; ++slot, ++n1) {
                    const uint32_t cb = (uint32_t)(n1 % PP_CBUF);
                    const float* cc = cst + (size_t)cb * cl.total;
                    const float *w0s = cc + cl.w0, *b0s = cc + cl.b0, *bhs = cc + cl.bh;
                    const float* hs = hs2 + (size_t)(n1 & 1) * a.u_fmax * UM;
                    if (bn_done != n1) batch_norm(n1, p, cj, slot);
                    s1_barrier();   // hs of this occurrence complete; every read of the other parity's hs is over
                    // the activations of the previous occurrence are still the A operand of its last-layer MMAs: wait
                    // for their completion (the accumulator-full barrier the row warps also wait on) before the first
                    // store; the first chunk's arithmetic has already run underneath that tail
                    first_dense_ffma<CW>(hs, F, m, half, w0s, b0s, tb, lane_base, &bars[PP_AREADY], act, [&] {
                        if (n1 > 0) {
                            mbar_wait(&bars[PP_DFULL_D], (uint32_t)((n1 - 1) & 1));
                            umma::fence_after_sync();
                        }
                    });
                    for (int l = 1; l < L; ++l) {
                        if (l == 1 && nslots == 2) {
                            // While the first hidden GEMM finishes: the BatchNorm of the next occurrence.  It belongs
                            // to the other tile of the pair (or to the next pair), whose state does not depend on
                            // anything this occurrence still has to produce, so waiting for it here cannot deadlock
                            // (the row warps publish a tile of the next pair as soon as they are through the first
                            // coupling of the tile it replaces).
                            long long pn = p;
                            int cjn = cj, sn = 1;
                            if (slot == 1) { sn = 0; if (++cjn == ncoup) { cjn = 0; ++pn; } }
                            if (2 * pn < n_my) batch_norm(n1 + 1, pn, cjn, sn);
                        }
                        mbar_wait(&bars[PP_DFULL_H], p_fh);
                        p_fh ^= 1u;
                        umma::fence_after_sync();
                        hidden_drain<CW, false>(TC_PP_HMAIN, TC_PP_HCROSS, bhs + (l - 1) * 128, l, half, tb, lane_base,
                                                &bars[PP_AREADY], act);
                    }
                    umma::mbar_arrive(&bars[PP_CEMPTY + cb]);   // S1 is done with this occurrence's constants
                }
            }
        }
    };

    // S2: one thread per event: tile load, ShiftBounds, spline row, latent + store.  The load and the leading
    // non-coupling steps of the NEXT pair's tiles are done in the middle of the current pair (right after its first
    // coupling), so the activation warps never wait for a tile at a pair boundary.
    auto row_role = [&]() {
        const int q = warp & 3, m = q * 32 + lane, t2 = tid - 256;   // t2: index inside S2
        const uint32_t lane_base = (uint32_t)(q * 32);
        const int rot_in = INVERSE ? a.rot_total : 0;
        const int fc = coup_si[0];                                   // position of the first coupling
        uint32_t p_fd = 0;
        long long n2 = 0;
        auto tile_ptrs = [&](long long k, float*& xs, float*& cs, float*& lda) {
            const int tbuf = (int)(k % PP_TBUF);
            xs = xsb + tbuf * D * UM; cs = csb + tbuf * C * UM; lda = ldacc + tbuf * UM;
        };
        auto signal_ready = [&](long long k) { umma::mbar_arrive(&bars[PP_XSREADY + (int)(k % PP_TBUF)]); };
        auto preamble = [&](long long k) {
            if (k >= n_my) return;
            float *xs, *cs, *lda;
            tile_ptrs(k, xs, cs, lda);
            const long long tile = tile_of(k), m0 = tile * UM;
            const int nm = (int)min((long long)UM, a.M - m0);
            const int rb = (int)(k & 1);
            // rows -> feature-major tile; padding events sit at 0.5 / 0 and are never stored
            const bool bulk = tile_by_bulk(tile);
            const float* raw = xraw + (size_t)rb * UM * (D + C);
            if (bulk) mbar_wait(&bars[PP_XFULL + rb], (uint32_t)((k >> 1) & 1));
            const float* xsrc = bulk ? raw : a.x + m0 * D;
            const float* csrc = bulk ? raw + UM * D : a.c + m0 * C;
            {
                int mm = t2 / D, j = t2 - mm * D;
                const int dm = 128 / D, dj = 128 - dm * D;
                for (int e = t2; e < UM * D; e += 128) {
                    int col = j - rot_in;
                    if (col < 0) col += D;
                    xs[col * UM + mm] =
                        (mm < nm) ? (a.sample ? latent_draw(a.lc.kind, a.peakness, a.seed, m0 + mm, j) : xsrc[e]) : 0.5f;
                    mm += dm; j += dj;
                    if (j >= D) { j -= D; ++mm; }
                }
            }
            if (C) {
                int mm = t2 / C, j = t2 - mm * C;
                const int dm = 128 / C, dj = 128 - dm * C;
                for (int e = t2; e < UM * C; e += 128) {
                    cs[j * UM + mm] = (mm < nm) ? csrc[e] : 0.f;
                    mm += dm; j += dj;
                    if (j >= C) { j -= C; ++mm; }
                }
            }
            if (bulk) umma::mbar_arrive(&bars[PP_XEMPTY + rb]);
            s2_barrier();
            float ld0 = 0.f;
            for (int si = 0; si < fc; ++si) shift_bounds_row<INVERSE>(step_at(si), wsf, D, xs, UM, m, ld0);   // only non-coupling kind
            lda[m] = ld0;
            signal_ready(k);   // the tile state is complete for the first coupling
        };
        preamble(0);
        preamble(1);
        for (long long p = 0; 2 * p < n_my; ++p) {
            const int nslots = (2 * p + 1 < n_my) ? 2 : 1;
            for (int si = fc; si < a.n_steps; ++si) {
                const StepDesc& s = step_at(si);
#pragma unroll 1
                for (int slot = 0; slot < nslots; ++slot) {
                    const long long k = 2 * p + slot;
                    float *xs, *cs, *lda;
                    tile_ptrs(k, xs, cs, lda);
                    const long long m0 = tile_of(k) * UM;
                    const int nm = (int)min((long long)UM, a.M - m0);
                    if (s.kind == kStepKindShiftBounds) {
                        float ld_sb = 0.f;
                        shift_bounds_row<INVERSE>(s, wsf, D, xs, UM, m, ld_sb);
                        lda[m] += ld_sb;
                    } else {
                        const int K = s.K, rot = s.rot;
                        const uint32_t cb = (uint32_t)(n2 % PP_CBUF);
                        const float* bls = cst + (size_t)cb * cl.total + cl.bl;
                        mbar_wait(&bars[PP_CFULL + cb], (uint32_t)((n2 / PP_CBUF) & 1));
                        mbar_wait(&bars[PP_DFULL_D], p_fd);
                        p_fd ^= 1u;
                        umma::fence_after_sync();
                        const int NLr = ru(3 * K - 1, 16);
                        const uint32_t dbase = umma::taddr(tb, lane_base, tc_pp_theta(NLr));
                        float* px = xs + pmod(0 - rot, D) * UM + m;
                        const float v = *px;
                        RqsBin bin;
                        auto release = [&]() {
                            umma::fence_before_sync();
                            umma::mbar_arrive(&bars[PP_DEMPTY_D]);
                        };
                        float4* scr = reinterpret_cast<float4*>(scratch) + m;
                        if (K == 16) spline_row_tmem_lean<16, INVERSE>(dbase, tc_pp_xoff(48), bls, v, bin, scr, UM, release);
                        else spline_row_tmem_lean<32, INVERSE>(dbase, tc_pp_xoff(96), bls, v, bin, scr, UM, release);
                        if (m < nm) put_idx(a, s, m0 + m, 0, bin.idx);
                        umma::mbar_arrive(&bars[PP_CEMPTY + cb]);   // last read of this occurrence's constants by S2
                        if (!INVERSE) {
                            float y, ld;
                            rqs_eval_forward(v, bin, y, ld);
                            *px = y;
                            lda[m] += ld;
                        } else {
                            *px = rqs_eval_inverse(v, bin);
                        }
                        ++n2;
                    }
                    // as soon as this tile's state is complete for its next coupling, tell the activation warps
                    if (si + 1 < a.n_steps && step_at(si + 1).kind == kStepKindCoupling) signal_ready(k);
                    // the tile that takes this slot in the next pair: its buffers were released two pairs ago.  It is
                    // published here, not after both slots: the activation warps may wait for it while they still owe
                    // this pair's other slot (in a chain of one coupling, before that slot's spline rows can run).
                    if (si == fc) preamble(k + 2);
                    if (si == a.n_steps - 1) {
                        // ---- store this tile
                        if (a.mode == kModeLogProb) {
                            if (m < nm) {
                                float lat = 0.f;
                                for (int j = 0; j < D; ++j) lat += latent_logpdf(xs[pmod(j - a.rot_total, D) * UM + m], a.lc);
                                a.lp[m0 + m] = nan_to_num_lp(lat + lda[m]);
                            }
                        } else {
                            const int rot_out = INVERSE ? 0 : a.rot_total;
                            s2_barrier();
                            if (a.y) {
                                for (int e = t2; e < nm * D; e += 128) {
                                    const int mm = e / D, j = e - mm * D;
                                    a.y[m0 * D + e] = xs[pmod(j - rot_out, D) * UM + mm];
                                }
                            }
                            if (!INVERSE && a.log_det && m < nm)
                                a.log_det[m0 + m] = a.acc_log_det ? a.log_det[m0 + m] + lda[m] : lda[m];
                            s2_barrier();
                        }
                    }
                }
            }
        }
    };

    // Each setmaxnreg dominates exactly its warpgroup's role: 2 x 96 (S1) + 184 (S2) + 104 (producer, MMA issuer, idle)
    static_assert(256 * 96 + 128 * 184 + 128 * 104 <= 512 * 128, "register split exceeds the launch allocation");
    if (warp < 8) {
        reg_dec<96>();
        activation_role();
    } else if (warp < 12) {
        reg_inc<184>();
        row_role();
    } else {
        reg_dec<104>();
        if (warp == PW) producer_role();
        else if (warp == MW) mma_role();
    }
    umma::fence_before_sync();
    __syncthreads();
    if (warp == MW) umma::tmem_dealloc(tb, 512);
}

// ---- host side ------------------------------------------------------------------------

struct Plan {
    int D = 0, C = 0;                     // chain dim and conditioning dim
    std::vector<PackJob> jobs;
    int rot_total = 0;
    int act_rows = KC;
    size_t ws_floats = 0;
    bool umma_ok = true;   // every coupling fits the tensor-core kernel
    int n_couplings = 0;
    int Fmax = 1, Hmax = 1, BLmax = 32;   // shared-memory sizing of the two-pipeline kernel
    bool all_d1 = true;                   // every coupling transforms a single dim
    bool w0img = false;                   // constant blocks carry the first Dense's operand image (choose_chain_kernel)
};

// for_vjp: the plan of the fused VJP kernel (a chain of one coupling, multi-dim or not)
static int build_plan(const zf_chain* chain, Plan& plan, bool for_vjp = false) {
    ZF_REQUIRE(chain != nullptr, "chain is NULL");
    const int D = chain->dim, C = chain->cdim;
    ZF_REQUIRE(D >= 1 && D <= ZF_MAX_DIM, "dim must be in [1, %d] (got %d)", ZF_MAX_DIM, D);
    ZF_REQUIRE(C >= 0 && C <= 1024, "cdim must be in [0, 1024] (got %d)", C);
    ZF_REQUIRE(chain->n_ops >= 0 && (chain->n_ops == 0 || chain->ops), "ops is NULL");
    plan.D = D;
    plan.C = C;
    int rot = 0;
    for (int i = 0; i < chain->n_ops; ++i) {
        const zf_op& op = chain->ops[i];
        if (op.kind == ZF_OP_ROLL) {
            rot = ((rot + op.shift) % D + D) % D;
            continue;
        }
        PackJob job{};
        job.D = D;
        job.desc.rot = rot;
        if (op.kind == ZF_OP_SHIFT_BOUNDS) {
            ZF_REQUIRE(op.shift_bounds, "op %d: shift_bounds is NULL", i);
            const zf_shift_bounds& sb = *op.shift_bounds;
            job.desc.kind = kStepKindShiftBounds;
            bool need_stats = false;
            for (int j = 0; j < D; ++j) {
                ZF_REQUIRE(sb.kind[j] >= 0 && sb.kind[j] <= 3, "op %d: bad bound kind for column %d", i, j);
                job.sb_kind[j] = sb.kind[j];
                job.lo[j] = sb.lo[j];
                job.hi[j] = sb.hi[j];
                if (sb.kind[j] != ZF_BOUND_BOTH) need_stats = true;
            }
            ZF_REQUIRE(!need_stats || (sb.xmin && sb.xmax), "op %d: xmin/xmax are NULL", i);
            job.xmin = sb.xmin;
            job.xmax = sb.xmax;
        } else if (op.kind == ZF_OP_COUPLING) {
            ZF_REQUIRE(op.coupling, "op %d: coupling is NULL", i);
            const zf_coupling& cp = *op.coupling;
            const int d = D / 2;
            ZF_REQUIRE(d > 0 && d < D, "NeuralSplineCoupling needs dim >= 2 (bijectors.py:326)");
            ZF_REQUIRE(cp.knots >= 1, "op %d: knots must be >= 1", i);
            ZF_REQUIRE(cp.n_hidden >= 0 && cp.n_hidden <= ZF_MAX_LAYERS, "op %d: at most %d hidden layers", i,
                       ZF_MAX_LAYERS);
            const int P = 3 * cp.knots - 1;
            if (ru(P, 4) > NCOL)
                return fail(ZF_ERR_UNSUPPORTED, "op %d: knots=%d needs %d columns per dim; the fused kernel holds %d",
                            i, cp.knots, P, NCOL);
            job.desc.kind = kStepKindCoupling;
            job.desc.cidx = plan.n_couplings;
            plan.n_couplings++;
            ZF_REQUIRE(cp.act >= ZF_ACT_SWISH && cp.act <= ZF_ACT_LEAKY_RELU, "op %d: unknown activation %d", i, cp.act);
            job.desc.act = cp.act;
            {   // tensor-core kernel: swish, hidden width 128 throughout, K in {16, 32}, small first layer
                bool ok = cp.n_hidden >= 1 && (cp.knots == 16 || cp.knots == 32) && (D - d + C) <= UFMAX && d <= UDMAX &&
                          cp.act == ZF_ACT_SWISH;
                for (int l = 0; l < cp.n_hidden; ++l) ok = ok && cp.hidden[l] == 128;
                job.desc.umma_ok = ok ? 1 : 0;
                plan.umma_ok = plan.umma_ok && ok;
                plan.Fmax = std::max(plan.Fmax, D - d + C);
                plan.Hmax = std::max(plan.Hmax, std::max(1, cp.n_hidden - 1));
                plan.BLmax = std::max(plan.BLmax, d * ru(3 * cp.knots - 1, 16));
                plan.all_d1 = plan.all_d1 && d == 1;
            }
            job.desc.K = cp.knots;
            job.desc.n_hidden = cp.n_hidden;
            job.desc.F = D - d + C;
            job.desc.d = d;
            ZF_REQUIRE(cp.bn_scale && cp.bn_bias && cp.bn_mean && cp.bn_var, "op %d: BatchNorm leaf is NULL", i);
            job.bn_scale = cp.bn_scale; job.bn_bias = cp.bn_bias; job.bn_mean = cp.bn_mean; job.bn_var = cp.bn_var;
            int kin = job.desc.F;
            plan.act_rows = std::max(plan.act_rows, ru(kin, KC));
            for (int l = 0; l <= cp.n_hidden; ++l) {
                ZF_REQUIRE(cp.kernel[l] && cp.bias[l], "op %d: Dense_%d leaf is NULL", i, l);
                ZF_REQUIRE((reinterpret_cast<uintptr_t>(cp.kernel[l]) & 3) == 0, "op %d: Dense_%d kernel misaligned", i, l);
                const int n = (l < cp.n_hidden) ? cp.hidden[l] : d * P;
                ZF_REQUIRE(n >= 1, "op %d: layer width must be positive", i);
                if (l < cp.n_hidden) job.desc.hidden[l] = n;
                job.kernel[l] = cp.kernel[l];
                job.bias[l] = cp.bias[l];
                job.Kin[l] = kin;
                job.N[l] = n;
                if (l < cp.n_hidden) plan.act_rows = std::max(plan.act_rows, ru(n, KC));
                kin = n;
            }
            plan.act_rows = std::max(plan.act_rows, ru((P | 1), 4));
        } else {
            return fail(ZF_ERR_INVALID, "op %d: unknown kind %d", i, op.kind);
        }
        plan.jobs.push_back(job);
    }
    plan.rot_total = rot;
    // constant-block layout: see choose_chain_kernel
    plan.w0img = plan.umma_ok && plan.n_couplings > 0 && (for_vjp || !plan.all_d1) && plan.Fmax <= 16;

    // workspace layout: StepDesc array, then per-step blocks (all multiples of 4 floats)
    size_t off = (sizeof(StepDesc) * std::max<size_t>(plan.jobs.size(), 1) + 15) / 16 * 4;
    auto take = [&](size_t n) { size_t o = off; off += (n + 3) / 4 * 4; return (int)o; };
    for (size_t si = 0; si < plan.jobs.size(); ++si) {
        PackJob& job = plan.jobs[si];
        job.step_index = (int)si;
        StepDesc& s = job.desc;
        if (s.kind == kStepKindShiftBounds) {
            s.off_sb = take((size_t)D * kSbStride);
        } else {
            const int F_p = ru(s.F, KC);
            s.off_bn = take((size_t)3 * F_p);
            for (int l = 0; l < s.n_hidden; ++l) {
                const int Kin_p = ru(job.Kin[l], KC), N_p = ru(job.N[l], KC);
                s.off_W[l] = take((size_t)Kin_p * N_p);
                s.off_b[l] = take((size_t)N_p);
            }
            const int L = s.n_hidden;
            const int Kin_p = ru(job.Kin[L], KC), Pp = ru(3 * s.K - 1, 4);
            s.off_W[L] = take((size_t)s.d * Kin_p * Pp);
            s.off_b[L] = take((size_t)s.d * Pp);
            if (s.umma_ok) {
                const int NL = ru(3 * s.K - 1, 16);
                off = (off + 31) / 32 * 32;  // images are fetched by 16-byte-aligned bulk copies
                for (int l = 1; l < L; ++l) s.off_U[l] = take((size_t)128 * 128);
                s.off_U[L] = take((size_t)s.d * NL * 128);
                job.cst = ucst_layout(plan.Fmax, plan.Hmax, plan.BLmax, plan.w0img);
                s.off_C = take((size_t)job.cst.total);
            }
        }
        if (off > (size_t)0x7fffffff) return fail(ZF_ERR_UNSUPPORTED, "packed parameters exceed 2^31 floats");
    }
    plan.ws_floats = off;
    return ZF_OK;
}

static LatentConst make_latent(int kind, float peakness) {
    LatentConst lc{};
    lc.kind = kind;
    lc.p1 = (float)((double)peakness - 1.0);
    lc.betaln = (float)(2.0 * lgamma((double)peakness) - lgamma(2.0 * (double)peakness));
    lc.lognorm = (float)log(2.0 * M_PI * 0.1 * 0.1);
    lc.logmass = (float)log(0.5 * (erf(5.0 / sqrt(2.0)) - erf(-5.0 / sqrt(2.0))));
    return lc;
}

enum PackMode : int { kPackAndRun = 0, kPackOnly = 1, kRunPacked = 2 };

ImplSwitch& impl_switch() {
    static ImplSwitch sw = [] {
        ImplSwitch v{};
        const char* e = getenv("ZF_CHAIN_IMPL");
        if (e) strncpy(v.chain, e, sizeof(v.chain) - 1);
        e = getenv("ZF_GEMM_IMPL");
        if (e) strncpy(v.gemm, e, sizeof(v.gemm) - 1);
        return v;
    }();
    return sw;
}
enum class ChainKernel { kNone, kFfma, kUmma, kUmmaPP, kUmmaVjp };
struct ChainLaunch {
    ChainKernel kernel;
    size_t smem;   // dynamic shared memory, bytes
};

// Which kernel runs a planned chain on this device, and the dynamic shared memory it needs.  impl is the chain
// developer switch (impl_switch().chain).  With
//   tc       = every coupling fits the tensor-core kernels (Plan::umma_ok), there is at least one, and impl != simt
//   fits(k)  = k's shared memory is within the device's opt-in limit
// an eval pass (forward, inverse, log_prob, sample) takes the first row that applies:
//   tc, fits(single-tile), all_d1, n_steps <= USTEPS, impl != umma8, fits(two-tile)  chain_umma_pp_kernel
//   tc, fits(single-tile)                                                            chain_umma_kernel
//   !tc, impl == umma                                                                ZF_ERR_UNSUPPORTED
//   fits(FFMA tile)        (a tc chain beyond the single-tile kernel's memory too)   chain_kernel
//   otherwise                                                                        ZF_ERR_UNSUPPORTED
// and the VJP of one coupling (vjp, the plan of vjp_plan), of its forward or of its inverse (the same plan, packing and
// shared memory; only the spline row differs):
//   tc, fits(single-tile VJP)   chain_umma_kernel<false, true> (forward) / <true, true> (inverse);
//   otherwise                   kNone (the unfused path of coupling_backward: spline_bwd_kernel<K, false | true>)
// The constant blocks are laid out by build_plan, before the device is known: for tc couplings with Fmax <= 16 they carry
// the first Dense's operand image (Plan::w0img: first Dense on the tensor cores), except in the eval passes of flows
// whose couplings all transform one dim.  Those take the two-tile kernel, whose first Dense is FFMA, and keep the FFMA
// first Dense when they fall back to the single-tile kernel (umma8, n_steps > USTEPS, two-tile memory).
static int choose_chain_kernel(const Plan& plan, const DeviceInfo& di, bool vjp, const char* impl, ChainLaunch* out) {
    const size_t limit = (size_t)di.max_smem_optin;
    const bool tc = plan.umma_ok && plan.n_couplings > 0 && impl[0] != 's';
    const size_t usmem = umma_smem_floats(plan.D, plan.C, plan.Fmax, plan.Hmax, plan.BLmax, vjp, plan.w0img) * sizeof(float);
    if (vjp) {
        *out = (tc && usmem <= limit) ? ChainLaunch{ChainKernel::kUmmaVjp, usmem} : ChainLaunch{ChainKernel::kNone, 0};
        return ZF_OK;
    }
    if (!tc && strcmp(impl, "umma") == 0)
        return fail(ZF_ERR_UNSUPPORTED, "ZF_CHAIN_IMPL=umma but this chain does not fit the tensor-core kernel");
    if (tc && usmem <= limit) {
        const size_t psmem = umma_pp_smem_floats(plan.D, plan.C, plan.Fmax, plan.Hmax, plan.BLmax) * sizeof(float);
        if (plan.all_d1 && (int)plan.jobs.size() <= USTEPS && strcmp(impl, "umma8") != 0 && psmem <= limit)
            *out = {ChainKernel::kUmmaPP, psmem};
        else
            *out = {ChainKernel::kUmma, usmem};
        return ZF_OK;
    }
    const size_t smem = ((size_t)(plan.D + plan.C) * TM + 2 * (size_t)plan.act_rows * TM + 2 * KC * NCOL) * sizeof(float);
    if (smem > limit)
        return fail(ZF_ERR_UNSUPPORTED, "chain tile needs %zu bytes of shared memory (limit %d): layers too wide", smem,
                    di.max_smem_optin);
    *out = {ChainKernel::kFfma, smem};
    return ZF_OK;
}

static int run_chain(cudaStream_t stream, const zf_chain* chain, int mode, int latent_kind, float peakness,
                     const float* x, const float* c, long long M, float* y, float* log_det, float* lp,
                     void* workspace, size_t workspace_bytes, int acc_log_det = 0, int sample = 0,
                     unsigned long long seed = 0, int* idx_out = nullptr, int pack_mode = kPackAndRun) {
    Plan plan;
    if (int rc = build_plan(chain, plan)) return rc;
    ZF_REQUIRE(M >= 0, "M must be >= 0");
    if (M == 0 && pack_mode != kPackOnly) return ZF_OK;
    if (pack_mode != kPackOnly) {
        ZF_REQUIRE(x != nullptr || sample, "input tensor is NULL");
        ZF_REQUIRE(chain->cdim == 0 || c != nullptr, "chain has cdim=%d but c is NULL", chain->cdim);
        if (sample) {
            ZF_REQUIRE(latent_kind >= 0 && latent_kind <= 3, "unknown latent kind %d", latent_kind);
            ZF_REQUIRE(latent_kind != ZF_LATENT_BETA || peakness >= 1.f, "peakness must be at least 1 (distributions.py:96-97)");
        }
        if (mode == kModeLogProb) {
            ZF_REQUIRE(lp != nullptr, "log_prob output is NULL");
            ZF_REQUIRE(latent_kind >= 0 && latent_kind <= 3, "unknown latent kind %d", latent_kind);
            ZF_REQUIRE(latent_kind != ZF_LATENT_BETA || peakness >= 1.f, "peakness must be at least 1 (distributions.py:96-97)");
        }
    }
    const size_t need = plan.ws_floats * sizeof(float);
    if (workspace_bytes < need || (need && !workspace))
        return fail(ZF_ERR_WORKSPACE, "workspace too small: need %zu bytes, got %zu", need, workspace_bytes);
    ZF_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 15) == 0, "workspace must be 16-byte aligned");
    DeviceInfo di;
    if (int rc = get_device_info(&di)) return rc;

    float* ws = static_cast<float*>(workspace);
    if (pack_mode != kRunPacked) {
        // latency-bound re-layout of ~50k parameters per coupling: one thin wave over all SMs per step, all steps of
        // the chain (up to kPackBatch) in one launch.  The 25 KB parameter block lives in a per-thread buffer.
        static thread_local PackBatch batch;
        for (size_t j0 = 0; j0 < plan.jobs.size(); j0 += kPackBatch) {
            const size_t nb = std::min<size_t>(kPackBatch, plan.jobs.size() - j0);
            for (size_t j = 0; j < nb; ++j) batch.jobs[j] = plan.jobs[j0 + j];
            pack_step_kernel<<<dim3((unsigned)di.sm_count, (unsigned)nb), 256, 0, stream>>>(batch, ws);
            count_launch();
        }
        ZF_CUDA_CHECK(cudaGetLastError());
        if (pack_mode == kPackOnly) return ZF_OK;
    }

    ChainArgs a{};
    a.x = x; a.c = c; a.y = y; a.log_det = log_det; a.lp = lp;
    a.ws = ws; a.M = M; a.D = chain->dim; a.C = chain->cdim;
    a.n_steps = (int)plan.jobs.size();
    a.rot_total = plan.rot_total;
    a.act_rows = plan.act_rows;
    a.mode = mode;
    a.acc_log_det = acc_log_det;
    a.sample = sample;
    a.seed = seed;
    a.peakness = peakness;
    a.lc = make_latent(latent_kind, peakness);
    a.idx_out = idx_out;
    a.n_couplings = plan.n_couplings;
    a.u_fmax = plan.Fmax;
    a.u_hmax = plan.Hmax;
    a.u_blmax = plan.BLmax;
    a.u_w0img = plan.w0img ? 1 : 0;

    ChainLaunch k;
    if (int rc = choose_chain_kernel(plan, di, false, impl_switch().chain, &k)) return rc;
    auto launch = [&](auto kern, long long blocks, unsigned threads) -> int {
        if (int rc = smem_optin((const void*)kern, k.smem)) return rc;
        kern<<<(unsigned)blocks, threads, k.smem, stream>>>(a);
        count_launch();
        ZF_CUDA_CHECK(cudaGetLastError());
        return ZF_OK;
    };
    const bool inv = mode == kModeInverse;
    const long long utiles = (M + UM - 1) / UM;
    switch (k.kernel) {
        case ChainKernel::kUmmaPP: {   // two tiles in flight per CTA
            const long long blocks = std::min<long long>((utiles + 1) / 2, di.sm_count);
            return inv ? launch(chain_umma_pp_kernel<true>, blocks, PP_THREADS) : launch(chain_umma_pp_kernel<false>, blocks, PP_THREADS);
        }
        case ChainKernel::kUmma: {
            const long long blocks = std::min<long long>(utiles, di.sm_count);
            return inv ? launch(chain_umma_kernel<true>, blocks, 320) : launch(chain_umma_kernel<false>, blocks, 320);
        }
        default: {   // kFfma (an eval pass is never kNone or kUmmaVjp)
            const int bps = (2 * (k.smem + 1024) <= (size_t)di.max_smem_optin) ? 2 : 1;
            const long long blocks = std::min<long long>((M + TM - 1) / TM, (long long)di.sm_count * bps);
            return inv ? launch(chain_kernel<true>, blocks, kChainThreads) : launch(chain_kernel<false>, blocks, kChainThreads);
        }
    }
}

// ---- fused conditioner recompute + spline VJP of ONE coupling (tensor-core path of zf_coupling_backward) ---------
// The coupling is planned and packed as a chain of one op; the kernel is chain_umma_kernel<false, true>, or
// chain_umma_kernel<true, true> for the VJP of the coupling's inverse (x_in is then the inverse's input, glp unused).
static int vjp_plan(const zf_coupling* cp, int D, int C, Plan& plan, zf_op& op, zf_chain& chain) {
    op = zf_op{};
    op.kind = ZF_OP_COUPLING;
    op.coupling = cp;
    chain = zf_chain{D, C, 1, &op};
    return build_plan(&chain, plan, true);
}

size_t coupling_vjp_ws_floats(const zf_coupling* cp, int D, int C) {
    Plan plan;
    zf_op op;
    zf_chain chain;
    DeviceInfo di;
    ChainLaunch k;
    if (vjp_plan(cp, D, C, plan, op, chain) != ZF_OK || get_device_info(&di) != ZF_OK ||
        choose_chain_kernel(plan, di, true, impl_switch().chain, &k) != ZF_OK || k.kernel != ChainKernel::kUmmaVjp)
        return 0;
    return plan.ws_floats;
}

int coupling_vjp_pack(cudaStream_t stream, const zf_coupling* cp, int D, int C, float* ws) {
    Plan plan;
    zf_op op;
    zf_chain chain;
    if (int rc = vjp_plan(cp, D, C, plan, op, chain)) return rc;
    DeviceInfo di;
    if (int rc = get_device_info(&di)) return rc;
    static thread_local PackBatch batch;
    batch.jobs[0] = plan.jobs[0];
    pack_step_kernel<<<dim3((unsigned)di.sm_count, 1u), 256, 0, stream>>>(batch, ws);
    count_launch();
    ZF_CUDA_CHECK(cudaGetLastError());
    return ZF_OK;
}

int coupling_vjp_run(cudaStream_t stream, const zf_coupling* cp, int D, int C, const float* ws, const float* x_in, const float* c,
                     const float* gy, int gy_rot, const float* glp, long long M, float* gx, void* img_h0, int wh0, void* const* img_act,
                     float* const* act_g, void* img_dtheta, bool inverse) {
    Plan plan;
    zf_op op;
    zf_chain chain;
    if (int rc = vjp_plan(cp, D, C, plan, op, chain)) return rc;
    DeviceInfo di;
    if (int rc = get_device_info(&di)) return rc;
    ChainArgs a{};
    a.x = x_in; a.c = c; a.ws = ws; a.M = M; a.D = D; a.C = C;
    a.n_steps = 1;
    a.rot_total = 0;
    a.act_rows = plan.act_rows;
    a.mode = kModeVjp;
    a.n_couplings = 1;
    a.u_fmax = plan.Fmax; a.u_hmax = plan.Hmax; a.u_blmax = plan.BLmax; a.u_w0img = plan.w0img ? 1 : 0;
    a.gy = gy; a.glp = glp; a.gx = gx;
    a.img_h0 = static_cast<char*>(img_h0); a.wh0 = wh0; a.img_dtheta = static_cast<char*>(img_dtheta);
    a.gy_rot = ((gy_rot % D) + D) % D;
    ZF_REQUIRE((reinterpret_cast<uintptr_t>(img_h0) & 15) == 0 && (reinterpret_cast<uintptr_t>(img_dtheta) & 15) == 0 && wh0 % 16 == 0,
               "coupling_vjp: images must be 16-byte aligned");
    for (int l = 0; l < cp->n_hidden; ++l) {
        a.img_act[l] = static_cast<char*>(img_act[l]);
        a.act_g[l] = act_g[l];
        ZF_REQUIRE(((reinterpret_cast<uintptr_t>(img_act[l]) | reinterpret_cast<uintptr_t>(act_g[l])) & 15) == 0,
                   "coupling_vjp: images must be 16-byte aligned");
    }
    ChainLaunch k;
    if (int rc = choose_chain_kernel(plan, di, true, impl_switch().chain, &k)) return rc;
    ZF_REQUIRE(k.kernel == ChainKernel::kUmmaVjp, "coupling_vjp: the coupling does not take the fused kernel (coupling_vjp_ws_floats is 0)");
    auto kern = inverse ? chain_umma_kernel<true, true> : chain_umma_kernel<false, true>;
    if (int rc = smem_optin((const void*)kern, k.smem)) return rc;
    const long long tiles = (M + UM - 1) / UM;
    if (tiles == 0) return ZF_OK;
    kern<<<(unsigned)std::min<long long>(tiles, (long long)di.sm_count), 320, k.smem, stream>>>(a);
    count_launch();
    ZF_CUDA_CHECK(cudaGetLastError());
    return ZF_OK;
}

}  // namespace zf

extern "C" size_t zf_chain_workspace_bytes(const zf_chain* chain, int64_t M) {
    (void)M;
    zf::Plan plan;
    if (zf::build_plan(chain, plan) != ZF_OK) return 0;
    return plan.ws_floats * sizeof(float);
}

extern "C" int zf_chain_forward(void* stream, const zf_chain* chain, const float* x, const float* c, int64_t M,
                                float* y, float* log_det, void* workspace, size_t workspace_bytes) {
    return zf::run_chain((cudaStream_t)stream, chain, zf::kModeForward, 0, 0.f, x, c, (long long)M, y, log_det,
                         nullptr, workspace, workspace_bytes);
}

extern "C" int zf_chain_forward_acc(void* stream, const zf_chain* chain, const float* x, const float* c, int64_t M,
                                    float* y, float* log_det, void* workspace, size_t workspace_bytes) {
    return zf::run_chain((cudaStream_t)stream, chain, zf::kModeForward, 0, 0.f, x, c, (long long)M, y, log_det,
                         nullptr, workspace, workspace_bytes, 1);
}

extern "C" int zf_chain_bin_indices(void* stream, const zf_chain* chain, const float* x, const float* c, int64_t M,
                                    int32_t* idx, void* workspace, size_t workspace_bytes) {
    ZF_REQUIRE(idx != nullptr || M == 0, "bin_indices: output tensor is NULL");
    return zf::run_chain((cudaStream_t)stream, chain, zf::kModeForward, 0, 0.f, x, c, (long long)M, nullptr, nullptr,
                         nullptr, workspace, workspace_bytes, 0, 0, 0, idx);
}

extern "C" int zf_chain_inverse(void* stream, const zf_chain* chain, const float* z, const float* c, int64_t M,
                                float* x, void* workspace, size_t workspace_bytes) {
    ZF_REQUIRE(x != nullptr || M == 0, "output tensor is NULL");
    return zf::run_chain((cudaStream_t)stream, chain, zf::kModeInverse, 0, 0.f, z, c, (long long)M, x, nullptr,
                         nullptr, workspace, workspace_bytes);
}

extern "C" int zf_flow_sample(void* stream, const zf_chain* chain, int32_t latent_kind, float peakness, uint64_t seed,
                              const float* c, int64_t M, float* x, void* workspace, size_t workspace_bytes) {
    ZF_REQUIRE(x != nullptr || M == 0, "output tensor is NULL");
    return zf::run_chain((cudaStream_t)stream, chain, zf::kModeInverse, latent_kind, peakness, nullptr, c, (long long)M, x,
                         nullptr, nullptr, workspace, workspace_bytes, 0, 1, (unsigned long long)seed);
}

extern "C" int zf_flow_log_prob(void* stream, const zf_chain* chain, int32_t latent_kind, float peakness,
                                const float* x, const float* c, int64_t M, float* log_prob, void* workspace,
                                size_t workspace_bytes) {
    return zf::run_chain((cudaStream_t)stream, chain, zf::kModeLogProb, latent_kind, peakness, x, c, (long long)M,
                         nullptr, nullptr, log_prob, workspace, workspace_bytes);
}

extern "C" int zf_debug_set_impl(const char* chain_impl, const char* gemm_impl) {
    zf::ImplSwitch& sw = zf::impl_switch();
    memset(sw.chain, 0, sizeof(sw.chain));
    memset(sw.gemm, 0, sizeof(sw.gemm));
    if (chain_impl) strncpy(sw.chain, chain_impl, sizeof(sw.chain) - 1);
    if (gemm_impl) strncpy(sw.gemm, gemm_impl, sizeof(sw.gemm) - 1);
    return ZF_OK;
}

// ---- the same passes with the parameter re-layout hoisted out (pack once per parameter update, run many times) ----
extern "C" int zf_chain_pack(void* stream, const zf_chain* chain, void* workspace, size_t workspace_bytes) {
    return zf::run_chain((cudaStream_t)stream, chain, zf::kModeForward, 0, 0.f, nullptr, nullptr, 0, nullptr, nullptr, nullptr,
                         workspace, workspace_bytes, 0, 0, 0, nullptr, zf::kPackOnly);
}

extern "C" int zf_chain_forward_packed(void* stream, const zf_chain* chain, const float* x, const float* c, int64_t M,
                                       float* y, float* log_det, void* workspace, size_t workspace_bytes) {
    return zf::run_chain((cudaStream_t)stream, chain, zf::kModeForward, 0, 0.f, x, c, (long long)M, y, log_det, nullptr,
                         workspace, workspace_bytes, 0, 0, 0, nullptr, zf::kRunPacked);
}

extern "C" int zf_chain_inverse_packed(void* stream, const zf_chain* chain, const float* z, const float* c, int64_t M,
                                       float* x, void* workspace, size_t workspace_bytes) {
    ZF_REQUIRE(x != nullptr || M == 0, "output tensor is NULL");
    return zf::run_chain((cudaStream_t)stream, chain, zf::kModeInverse, 0, 0.f, z, c, (long long)M, x, nullptr, nullptr,
                         workspace, workspace_bytes, 0, 0, 0, nullptr, zf::kRunPacked);
}

extern "C" int zf_flow_log_prob_packed(void* stream, const zf_chain* chain, int32_t latent_kind, float peakness,
                                       const float* x, const float* c, int64_t M, float* log_prob, void* workspace,
                                       size_t workspace_bytes) {
    return zf::run_chain((cudaStream_t)stream, chain, zf::kModeLogProb, latent_kind, peakness, x, c, (long long)M, nullptr,
                         nullptr, log_prob, workspace, workspace_bytes, 0, 0, 0, nullptr, zf::kRunPacked);
}

extern "C" int zf_flow_sample_packed(void* stream, const zf_chain* chain, int32_t latent_kind, float peakness,
                                     uint64_t seed, const float* c, int64_t M, float* x, void* workspace,
                                     size_t workspace_bytes) {
    ZF_REQUIRE(x != nullptr || M == 0, "output tensor is NULL");
    return zf::run_chain((cudaStream_t)stream, chain, zf::kModeInverse, latent_kind, peakness, nullptr, c, (long long)M, x,
                         nullptr, nullptr, workspace, workspace_bytes, 0, 1, (unsigned long long)seed, nullptr,
                         zf::kRunPacked);
}

#ifdef ZF_TRACE
extern "C" int zf_debug_trace_read(long long* out) {   // read and clear
    int rc = (int)cudaMemcpyFromSymbol(out, zf::g_zf_trace, sizeof(long long) * 4 * 64);
    static long long zeros[4 * 64];
    if (rc == 0) rc = (int)cudaMemcpyToSymbol(zf::g_zf_trace, zeros, sizeof(zeros));
    return rc;
}
#endif
