// The train step's fp32 GEMM family: every Dense layer of a coupling backward that the fused VJP kernel does not take
// (the unfused path of zf_coupling_backward) and every Dense layer of the Deep-Set Phi (zf_phi.cu).  fp32 in / fp32 out:
//   mode 0 (NN): C[m][n]  = sum_k opA(A[m][k]) * B[k][n] + bias[n]                      (Dense forward)
//   mode 1 (NT): C[m][k]  = (sum_n A[m][n] * B[k][n]) * act'(Z[m][k])      (Z optional) (grad wrt Dense input)
//   mode 2 (TN): C[k][n] += sum_m opA(A[m][k]) * B[m][n];  colsum[n] += sum_m B[m][n]   (grad wrt kernel, bias)
// opA = the activation when a_swish (stored pre-activations are re-activated on load).  Three kernels; launch_gemm, at the
// end of this file, chooses one:
//   umma_gemm_tma_kernel<MODE,TN>  tcgen05, operands fed by the copy engine
//   umma_gemm_kernel<MODE,TN>      tcgen05, register-path loaders (operands a tensor map cannot describe)
//   gemm_kernel<MODE>              fp32 FFMA, 64 x 64 x 16 tiles, 4 x 4 per thread (any activation)
//
// The tcgen05 kernels compute 3xTF32 split products (fp32-class accuracy) with swish as the activation.  One CTA computes a
// 128 x TN output tile.  The loaders apply opA, split x = hi + lo (tf32) and write K-major core-matrix images (zf_umma.cuh)
// of one reduction chunk into a shared-memory ring; warp 8 issues tcgen05.mma.kind::tf32 with both operands from shared
// memory; the main products accumulate in TMEM columns [0,TN), the two cross products in [TN,2TN) (the tensor core's
// accumulator truncates per step, see zf_chain.cu); the 8 loader warps then turn into the epilogue (TMEM -> registers ->
// global, bias / swish' / atomics).  The two kernels differ only in how the images are fed: 8 loader warps reading global
// memory through registers (umma_gemm_kernel), or a producer warp driving the copy engine and 8 converter warps
// (umma_gemm_tma_kernel).
#include "zf_umma.cuh"
#include "zf_math.cuh"

#include <cuda.h>

#include <algorithm>
#include <stdlib.h>

namespace zf {

// Reduction rows [rbeg, rend) of this CTA: all R of them, or in mode 2 slab blockIdx.z of g.r_slab rows.
template <int MODE>
__device__ __forceinline__ void gemm_rows(const GemmArgs& g, long long& rbeg, long long& rend) {
    rbeg = 0;
    rend = g.R;
    if (MODE == 2) {
        rbeg = (long long)blockIdx.z * g.r_slab;
        rend = (rbeg + g.r_slab < g.R) ? rbeg + g.r_slab : g.R;
    }
}

// =============================================================================================
// fp32 FFMA kernel
// =============================================================================================
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
    long long rbeg, rend;
    gemm_rows<MODE>(g, rbeg, rend);
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

// =============================================================================================
// What the two tcgen05 kernels share
// =============================================================================================
__device__ __forceinline__ float ug_swish(float x) { return __fdividef(x, 1.0f + __expf(-x)); }
__device__ __forceinline__ float ug_swish_grad(float z) {
    const float s = __fdividef(1.0f, 1.0f + __expf(-z));
    return s * (1.0f + z * (1.0f - s));
}

__device__ __forceinline__ void mma_tf32_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, bool accumulate) {
    uint32_t acc = accumulate ? 1u : 0u, z = 0u;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, {%5, %6, %7, %8}, p;\n\t"
        "}\n" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(acc), "r"(z), "r"(z), "r"(z), "r"(z)
        : "memory");
}

// Thread 0 initialises the barriers (init_bars), warp 8 allocates the 2 x TN accumulator columns of tensor memory; both
// are visible to the whole CTA on return.  Returns the tensor-memory base.
template <int TN, class InitBars>
__device__ __forceinline__ uint32_t ug_setup(uint32_t* tmem_slot, int tid, int warp, InitBars init_bars) {
    if (tid == 0) {
        init_bars();
        mbar_fence_init();
    }
    if (warp == 8) umma::tmem_alloc(tmem_slot, 2 * TN);
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    return *tmem_slot;
}
template <int TN>
__device__ __forceinline__ void ug_teardown(uint32_t tb, int warp) {
    umma::fence_before_sync();
    __syncthreads();
    if (warp == 8) umma::tmem_dealloc(tb, 2 * TN);
}

// The MMA warp.  Stage s of the image ring at `img` holds one KC-deep reduction chunk: the hi and lo images of A (128 x KC)
// then those of B (TN x KC).  Per chunk it waits on full[s], issues three kind::tf32 products per 8-deep k-step (the cross
// products lo*hi + hi*lo into columns [TN,2TN), the main product hi*hi into [0,TN)) and commits them to empty[s]; `done`
// fires when the last chunk's products have landed.
template <int TN, int KC, int STAGES>
__device__ __forceinline__ void ug_mma_warp(const float* img, uint64_t* full, uint64_t* empty, uint64_t* done, uint32_t tb,
                                            int n_chunks, int lane) {
    constexpr int A_FLOATS = 128 * KC, B_FLOATS = TN * KC, STAGE_FLOATS = 2 * A_FLOATS + 2 * B_FLOATS;
    const uint32_t idesc = umma::instr_desc_tf32(TN);
    const uint32_t lbo_a = 16u * 128u, lbo_b = (uint32_t)(TN / 8) * 128u;
    uint32_t stage = 0, phase = 0;
    for (int c = 0; c < n_chunks; ++c) {
        mbar_wait(&full[stage], phase);
        umma::fence_after_sync();
        if (umma::elect_one()) {
            const uint32_t base = smem_u32(img + (size_t)stage * STAGE_FLOATS);
            const uint32_t a_hi = base, a_lo = base + A_FLOATS * 4u;
            const uint32_t b_hi = base + 2u * A_FLOATS * 4u, b_lo = b_hi + B_FLOATS * 4u;
#pragma unroll
            for (int ks = 0; ks < KC / 8; ++ks) {
                const uint64_t dah = umma::smem_desc_kmajor(a_hi + ks * 2 * lbo_a, lbo_a, 128u);
                const uint64_t dal = umma::smem_desc_kmajor(a_lo + ks * 2 * lbo_a, lbo_a, 128u);
                const uint64_t dbh = umma::smem_desc_kmajor(b_hi + ks * 2 * lbo_b, lbo_b, 128u);
                const uint64_t dbl = umma::smem_desc_kmajor(b_lo + ks * 2 * lbo_b, lbo_b, 128u);
                const bool first = (c | ks) == 0;
                mma_tf32_ss(tb + TN, dal, dbh, idesc, !first);
                mma_tf32_ss(tb + TN, dah, dbl, idesc, true);
                mma_tf32_ss(tb, dah, dbh, idesc, !first);
            }
            umma::commit(&empty[stage]);
            if (c == n_chunks - 1) umma::commit(done);
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1u; }
    }
    if (n_chunks == 0 && lane == 0) umma::mbar_arrive(done);  // nothing to accumulate (never launched that way)
}

// Mode 2: the first row of CTAs adds the column sums of B.  Both kernels convert the transposed B so that a thread always
// serves image row (column of B) tid % TN; with TN = 128 two threads share a column and both add their part.
template <int MODE, int TN>
__device__ __forceinline__ void ug_colsum_flush(const GemmArgs& g, long long j0, int tid, float csum) {
    if (MODE == 2 && g.colsum && blockIdx.x == 0) {
        const int col = (TN == 256) ? tid : (tid & 127);
        if (j0 + col < g.J) atomicAdd(&g.colsum[j0 + col], csum);
    }
}

// Epilogue of the 8 loader warps, once the last MMA has landed: warp w takes TMEM lanes (w % 4) * 32.. (output rows) and
// half w / 4 of the TN columns, adds the main and cross accumulators and writes bias (mode 0) / * swish'(Z) (mode 1) /
// atomics (mode 2), 16 bytes at a time where the row and the operands allow.
template <int MODE, int TN>
__device__ __forceinline__ void ug_epilogue(const GemmArgs& g, uint32_t tb, uint64_t* done, long long i0, long long j0, int warp,
                                            int lane) {
    mbar_wait(done, 0);
    umma::fence_after_sync();
    const int q = warp & 3, half = warp >> 2;
    const long long i = i0 + q * 32 + lane;
    constexpr int HALF_COLS = TN / 2;
#pragma unroll 1
    for (int n0 = half * HALF_COLS; n0 < (half + 1) * HALF_COLS; n0 += 16) {
        float v[16], w[16];
        umma::ld16(umma::taddr(tb, q * 32, n0), v);
        umma::ld16(umma::taddr(tb, q * 32, TN + n0), w);
        umma::wait_ld();
        if (i < g.I) {
            float x[16];
#pragma unroll
            for (int t = 0; t < 16; ++t) x[t] = v[t] + w[t];
            const long long jb = j0 + n0;
            const bool full16 = jb + 15 < g.J, ldc4 = (g.ldc & 3) == 0;
            if (MODE != 2 && full16 && ldc4 && (reinterpret_cast<uintptr_t>(g.C) & 15) == 0 &&
                (MODE != 0 || !g.bias || (reinterpret_cast<uintptr_t>(g.bias) & 15) == 0) &&
                (MODE == 0 || !g.Z || ((g.ldz & 3) == 0 && (reinterpret_cast<uintptr_t>(g.Z) & 15) == 0))) {
                float4* dst = reinterpret_cast<float4*>(g.C + i * g.ldc + jb);
#pragma unroll
                for (int t4 = 0; t4 < 4; ++t4) {
                    float4 o = make_float4(x[t4 * 4], x[t4 * 4 + 1], x[t4 * 4 + 2], x[t4 * 4 + 3]);
                    if (MODE == 0) {
                        if (g.bias) {
                            const float4 bv = __ldg(reinterpret_cast<const float4*>(g.bias + jb) + t4);  // bias + jb is 16B aligned when jb % 4 == 0
                            o.x += bv.x; o.y += bv.y; o.z += bv.z; o.w += bv.w;
                        }
                    } else if (g.Z) {
                        const float4 zv = *(reinterpret_cast<const float4*>(g.Z + i * g.ldz + jb) + t4);
                        o.x *= ug_swish_grad(zv.x); o.y *= ug_swish_grad(zv.y);
                        o.z *= ug_swish_grad(zv.z); o.w *= ug_swish_grad(zv.w);
                    }
                    dst[t4] = o;
                }
            } else {
#pragma unroll
                for (int t = 0; t < 16; ++t) {
                    const long long j = jb + t;
                    if (j >= g.J) continue;
                    float xv = x[t];
                    if (MODE == 0) {
                        if (g.bias) xv += g.bias[j];
                        g.C[i * g.ldc + j] = xv;
                    } else if (MODE == 1) {
                        if (g.Z) xv *= ug_swish_grad(g.Z[i * g.ldz + j]);
                        g.C[i * g.ldc + j] = xv;
                    } else {
                        atomicAdd(&g.C[i * g.ldc + j], xv);
                    }
                }
            }
        }
    }
}

// =============================================================================================
// tcgen05 kernel with register-path loaders: 8 loader warps read the fp32 operands from global memory, apply opA, split
// and store the images of a KC-deep chunk; the next chunk is fetched into registers while the current one is stored.
// =============================================================================================
constexpr int UG_THREADS = 288;  // 8 loader/epilogue warps + 1 MMA warp
template <int TN> struct UgCfg {
    static constexpr int KC = (TN == 256) ? 32 : 16;
    static constexpr int STAGES = (TN == 256) ? 2 : 3;
    static constexpr size_t SMEM = ((size_t)STAGES * (2 * 128 * KC + 2 * TN * KC)) * sizeof(float) + 8 * 8 + 16;
};

// One 16-byte unit (4 consecutive reduction indices r4*4..+3 of image row `row`) of an operand image.
//   RCONTIG: X[(row0+row)*ld + r0 + r]      (reduction index contiguous in memory)
//   else   : X[(r0+r)*ld + row0 + row]      (transposed on load)
template <bool RCONTIG>
__device__ __forceinline__ float4 ug_load_unit(const float* __restrict__ X, long long ld, long long row, long long row_max,
                                               long long r, long long r_max, bool vec_ok) {
    float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
    if (row < row_max) {
        if (RCONTIG && vec_ok && r + 3 < r_max) {
            o = __ldg(reinterpret_cast<const float4*>(X + row * ld + r));
        } else {
            float v[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                if (r + i < r_max) v[i] = RCONTIG ? __ldg(X + row * ld + r + i) : __ldg(X + (r + i) * ld + row);
            }
            o = make_float4(v[0], v[1], v[2], v[3]);
        }
    }
    return o;
}

// Which 16-byte unit (image row, k-quad r4) thread `tid` handles in round q of a chunk of ROWS x R4 units.
//   transposed operands (reduction index strided in memory): lanes vary the row, so the four scalar loads of a
//     unit are coalesced along the row index and 8 lanes fill one 128-byte core matrix of the image;
//   reduction-contiguous operands: a quarter-warp takes 8 rows of one k-quad (conflict-free image stores) and the
//     four quarter-warps take 4 consecutive k-quads, so a warp load reads 64 contiguous bytes from each of 8 rows
//     (full sectors, 8 cache lines) instead of 16 bytes from each of 32 rows.
template <bool RCONTIG, int ROWS, int R4>
__device__ __forceinline__ void ug_unit(int tid, int q, int& row, int& r4) {
    const int u = tid + q * 256;
    if (!RCONTIG || R4 < 4) {
        row = u % ROWS;
        r4 = u / ROWS;
    } else {
        const int lane = u & 31, w = u >> 5;            // w: warp-sized group index in [0, ROWS * R4 / 32)
        constexpr int GROUPS_PER_ROWBLOCK = R4 / 4;      // groups that share the same 8 rows
        row = (w / GROUPS_PER_ROWBLOCK) * 8 + (lane & 7);
        r4 = (w % GROUPS_PER_ROWBLOCK) * 4 + (lane >> 3);
    }
}

template <int MODE, int TN>
__global__ void __launch_bounds__(UG_THREADS, (TN == 256) ? 1 : 2) umma_gemm_kernel(const __grid_constant__ GemmArgs g) {
    constexpr int UG_KC = UgCfg<TN>::KC;       // reduction depth per ring stage
    constexpr int A_FLOATS = 128 * UG_KC;      // one image (hi or lo) of the A chunk
    constexpr int B_FLOATS = TN * UG_KC;
    constexpr int STAGE_FLOATS = 2 * A_FLOATS + 2 * B_FLOATS;
    constexpr int STAGES = UgCfg<TN>::STAGES;
    constexpr bool A_RCONTIG = (MODE != 2);    // NN, NT: A[m][r]; TN: A[r][i]
    constexpr bool B_RCONTIG = (MODE == 1);    // NT: B[k][n] = [j][r]; NN, TN: B[r][j]

    extern __shared__ __align__(128) float smem[];
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)STAGES * STAGE_FLOATS);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 8);
    uint64_t* full = bars;            // [STAGES] count 256
    uint64_t* empty = bars + 3;       // [STAGES] count 1 (tcgen05.commit)
    uint64_t* done = bars + 6;        // count 1

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const long long i0 = (long long)blockIdx.x * 128, j0 = (long long)blockIdx.y * TN;
    long long rbeg, rend;
    gemm_rows<MODE>(g, rbeg, rend);
    const int n_chunks = (int)((rend - rbeg + UG_KC - 1) / UG_KC);

    const uint32_t tb = ug_setup<TN>(tmem_slot, tid, warp, [&] {
        for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 256); mbar_init(&empty[s], 1); }
        mbar_init(done, 1);
    });

    if (warp < 8) {
        // ------------------------------------------------------------------ loaders
        float csum = 0.f;  // mode 2: column sum of B for this thread's fixed column
        constexpr int R4 = UG_KC / 4;                               // 16-byte units per image row per chunk
        constexpr int UA = 128 * R4 / 256, UB = TN * R4 / 256;      // units per thread per chunk
        const bool vecA = ((g.lda & 3) == 0) && ((reinterpret_cast<uintptr_t>(g.A) & 15) == 0) && ((rbeg & 3) == 0);
        const bool vecB = ((g.ldb & 3) == 0) && ((reinterpret_cast<uintptr_t>(g.B) & 15) == 0) && ((rbeg & 3) == 0);
        // the whole next chunk is fetched into registers while the current one is converted and stored
        auto fetch = [&](int c, float4 (&ra)[UA], float4 (&rb)[UB]) {
            const long long r0 = rbeg + (long long)c * UG_KC;
#pragma unroll
            for (int q = 0; q < UA; ++q) {
                int row, r4;
                ug_unit<A_RCONTIG, 128, R4>(tid, q, row, r4);
                ra[q] = ug_load_unit<A_RCONTIG>(g.A, g.lda, i0 + row, g.I, r0 + r4 * 4, rend, vecA);
            }
#pragma unroll
            for (int q = 0; q < UB; ++q) {
                int row, r4;
                ug_unit<B_RCONTIG, TN, R4>(tid, q, row, r4);
                rb[q] = ug_load_unit<B_RCONTIG>(g.B, g.ldb, j0 + row, g.J, r0 + r4 * 4, rend, vecB);
            }
        };
        auto store = [&](float* st, const float4 (&ra)[UA], const float4 (&rb)[UB]) {
#pragma unroll
            for (int q = 0; q < UA; ++q) {
                int row, r4;
                ug_unit<A_RCONTIG, 128, R4>(tid, q, row, r4);
                float4 v = ra[q];
                if (g.a_swish) { v.x = ug_swish(v.x); v.y = ug_swish(v.y); v.z = ug_swish(v.z); v.w = ug_swish(v.w); }
                float4 hi, lo;
                umma::split_tf32(v.x, hi.x, lo.x); umma::split_tf32(v.y, hi.y, lo.y);
                umma::split_tf32(v.z, hi.z, lo.z); umma::split_tf32(v.w, hi.w, lo.w);
                const int off = (r4 * 16 + (row >> 3)) * 32 + (row & 7) * 4;
                *reinterpret_cast<float4*>(st + off) = hi;
                *reinterpret_cast<float4*>(st + A_FLOATS + off) = lo;
            }
#pragma unroll
            for (int q = 0; q < UB; ++q) {
                int row, r4;
                ug_unit<B_RCONTIG, TN, R4>(tid, q, row, r4);
                const float4 v = rb[q];
                if (MODE == 2) csum += (v.x + v.y) + (v.z + v.w);
                float4 hi, lo;
                umma::split_tf32(v.x, hi.x, lo.x); umma::split_tf32(v.y, hi.y, lo.y);
                umma::split_tf32(v.z, hi.z, lo.z); umma::split_tf32(v.w, hi.w, lo.w);
                const int off = (r4 * (TN / 8) + (row >> 3)) * 32 + (row & 7) * 4;
                *reinterpret_cast<float4*>(st + 2 * A_FLOATS + off) = hi;
                *reinterpret_cast<float4*>(st + 2 * A_FLOATS + B_FLOATS + off) = lo;
            }
        };
        float4 ra0[UA], rb0[UB], ra1[UA], rb1[UB];
        uint32_t stage = 0, phase = 0;
        if (n_chunks > 0) fetch(0, ra0, rb0);
        for (int c = 0; c < n_chunks; c += 2) {
            if (c + 1 < n_chunks) fetch(c + 1, ra1, rb1);
            mbar_wait(&empty[stage], phase ^ 1u);
            store(smem + (size_t)stage * STAGE_FLOATS, ra0, rb0);
            fence_proxy_async_smem();  // generic-proxy stores -> visible to the tensor core's async proxy
            umma::mbar_arrive(&full[stage]);
            if (++stage == STAGES) { stage = 0; phase ^= 1u; }
            if (c + 1 < n_chunks) {
                if (c + 2 < n_chunks) fetch(c + 2, ra0, rb0);
                mbar_wait(&empty[stage], phase ^ 1u);
                store(smem + (size_t)stage * STAGE_FLOATS, ra1, rb1);
                fence_proxy_async_smem();
                umma::mbar_arrive(&full[stage]);
                if (++stage == STAGES) { stage = 0; phase ^= 1u; }
            }
        }
        ug_colsum_flush<MODE, TN>(g, j0, tid, csum);
        ug_epilogue<MODE, TN>(g, tb, done, i0, j0, warp, lane);
    } else {
        ug_mma_warp<TN, UG_KC, STAGES>(smem, full, empty, done, tb, n_chunks, lane);
    }
    ug_teardown<TN>(tb, warp);
}

// =============================================================================================
// tcgen05 kernel fed by the copy engine (the default whenever the operands are 16-byte aligned with row strides that are
// multiples of 4).
//
// The register-path kernel converts its operands on the way from global memory to the shared-memory images through
// registers; with one CTA per SM that leaves ~32 KB in flight per SM and the loaders wait on every load
// (ncu: long-scoreboard stalls 2.5-5 per issue, 1.0-1.9 TB/s of operand traffic, tensor pipe 6-30 % active).
// Here the copy engine does the global reads: a producer thread issues 2-D tensor copies (cp.async.bulk.tensor,
// out-of-bounds rows / columns zero-filled by the hardware: no edge code) of raw fp32 boxes into a 3-stage staging
// ring; 8 converter warps turn a staged box into the tf32 hi / lo K-major images (shared -> registers -> shared,
// no global latency on their path) in a 2-stage image ring; the MMA warp consumes the images.  Reduction chunks
// are 16 deep (two MMA k-steps).  Reduction-contiguous boxes are staged with the 64-byte swizzle so that both the
// conversion reads and the image writes are bank-conflict free.
// =============================================================================================
constexpr int TG_THREADS = 320;   // 8 converter / epilogue warps + MMA warp + producer warp
constexpr int TG_KC = 16;
constexpr int TG_ISTAGES = 2;
template <int TN> struct TgStages { static constexpr int S = (TN == 256) ? 4 : 2; };   // staging stages (TN = 128: 2 CTAs per SM)

struct TGemmArgs {
    GemmArgs g;
    CUtensorMap mapA, mapB;
};

__device__ __forceinline__ void tma_load_2d(void* dst_smem, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::
            "r"(smem_u32(dst_smem)),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(smem_u32(bar))
        : "memory");
}

template <int TN> struct TgCfg {
    static constexpr int A_STAGE = 128 * TG_KC;                 // floats of one staged A box
    static constexpr int B_STAGE = TN * TG_KC;
    static constexpr int STAGE = A_STAGE + B_STAGE;
    static constexpr int IMG = 2 * STAGE;                       // hi | lo images of A and B
    static constexpr int SSTAGES = TgStages<TN>::S;
    static constexpr size_t SMEM = (size_t)(SSTAGES * STAGE + TG_ISTAGES * IMG) * 4 + 512 /* alignment */ + 256;
};

// Convert one staged operand box into its hi / lo images.  ROWS image rows (the MMA's M or N index), 16 reduction
// indices.  RCONTIG: staged as [ROWS][16] floats with the 64-byte swizzle; else staged as [16][ROWS].
template <bool RCONTIG, int ROWS, bool CSUM>
__device__ __forceinline__ void tg_convert(const float* __restrict__ stg, float* __restrict__ img_hi, float* __restrict__ img_lo,
                                           bool act, int tid, float& csum) {
    constexpr int UNITS = ROWS * 4 / 256;   // 16-byte image units per thread
#pragma unroll
    for (int q = 0; q < UNITS; ++q) {
        int row, r4;
        float4 v;
        if (RCONTIG) {
            const int u = tid + q * 256, lane = u & 31, w = u >> 5;
            row = w * 8 + (lane & 7);
            r4 = lane >> 3;
            const int chunk = r4 ^ ((row >> 1) & 3);   // CU_TENSOR_MAP_SWIZZLE_64B
            v = *reinterpret_cast<const float4*>(stg + row * TG_KC + chunk * 4);
        } else {
            const int u = tid + q * 256;
            row = u % ROWS;
            r4 = u / ROWS;
            v.x = stg[(r4 * 4 + 0) * ROWS + row];
            v.y = stg[(r4 * 4 + 1) * ROWS + row];
            v.z = stg[(r4 * 4 + 2) * ROWS + row];
            v.w = stg[(r4 * 4 + 3) * ROWS + row];
        }
        if (act) { v.x = ug_swish(v.x); v.y = ug_swish(v.y); v.z = ug_swish(v.z); v.w = ug_swish(v.w); }
        if (CSUM) csum += (v.x + v.y) + (v.z + v.w);
        float4 hi, lo;
        umma::split_tf32(v.x, hi.x, lo.x); umma::split_tf32(v.y, hi.y, lo.y);
        umma::split_tf32(v.z, hi.z, lo.z); umma::split_tf32(v.w, hi.w, lo.w);
        const int off = (r4 * (ROWS / 8) + (row >> 3)) * 32 + (row & 7) * 4;
        *reinterpret_cast<float4*>(img_hi + off) = hi;
        *reinterpret_cast<float4*>(img_lo + off) = lo;
    }
}

template <int MODE, int TN>
__global__ void __launch_bounds__(TG_THREADS, (TN == 256) ? 1 : 2) umma_gemm_tma_kernel(const __grid_constant__ TGemmArgs ta) {
    using Cfg = TgCfg<TN>;
    const GemmArgs& g = ta.g;
    constexpr bool A_RCONTIG = (MODE != 2);
    constexpr bool B_RCONTIG = (MODE == 1);

    extern __shared__ __align__(128) float smem_raw[];
    // staging stages must sit on 512-byte boundaries for the 64-byte swizzle pattern to start at row 0
    float* smem = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(smem_raw) + 511) & ~(uintptr_t)511);
    float* stage_base = smem;
    constexpr int TG_SSTAGES = Cfg::SSTAGES;
    float* img_base = smem + TG_SSTAGES * Cfg::STAGE;
    uint64_t* bars = reinterpret_cast<uint64_t*>(img_base + TG_ISTAGES * Cfg::IMG);
    uint64_t* s_full = bars;             // [<=4] TMA complete_tx
    uint64_t* s_empty = bars + 4;        // [<=4] 8 converter warps
    uint64_t* i_full = bars + 8;         // [2] 8 converter warps
    uint64_t* i_empty = bars + 10;       // [2] tcgen05.commit
    uint64_t* done = bars + 12;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 14);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const long long i0 = (long long)blockIdx.x * 128, j0 = (long long)blockIdx.y * TN;
    long long rbeg, rend;
    gemm_rows<MODE>(g, rbeg, rend);
    const int n_chunks = (int)((rend - rbeg + TG_KC - 1) / TG_KC);

    const uint32_t tb = ug_setup<TN>(tmem_slot, tid, warp, [&] {
        for (int s = 0; s < TG_SSTAGES; ++s) { mbar_init(&s_full[s], 1); mbar_init(&s_empty[s], 8); }
        for (int s = 0; s < TG_ISTAGES; ++s) { mbar_init(&i_full[s], 8); mbar_init(&i_empty[s], 1); }
        mbar_init(done, 1);
    });

    if (warp == 9) {
        // ------------------------------------------------------------------ producer (copy engine driver)
        if (lane == 0) {
            uint32_t stage = 0, phase = 0;
            for (int c = 0; c < n_chunks; ++c) {
                const int r0 = (int)(rbeg + (long long)c * TG_KC);
                mbar_wait(&s_empty[stage], phase ^ 1u);
                float* sa = stage_base + (size_t)stage * Cfg::STAGE;
                float* sb = sa + Cfg::A_STAGE;
                mbar_arrive_expect_tx(&s_full[stage], (uint32_t)Cfg::STAGE * 4u);
                // coordinates are (innermost, outermost); a slab's last chunk may reach into the next slab's rows:
                // those rows are part of the matrix, so the copy engine does not zero them - the converters do
                if (A_RCONTIG) tma_load_2d(sa, &ta.mapA, r0, (int)i0, &s_full[stage]);
                else tma_load_2d(sa, &ta.mapA, (int)i0, r0, &s_full[stage]);
                if (B_RCONTIG) tma_load_2d(sb, &ta.mapB, r0, (int)j0, &s_full[stage]);
                else tma_load_2d(sb, &ta.mapB, (int)j0, r0, &s_full[stage]);
                if (++stage == TG_SSTAGES) { stage = 0; phase ^= 1u; }
            }
        }
        __syncwarp();
    } else if (warp == 8) {
        ug_mma_warp<TN, TG_KC, TG_ISTAGES>(img_base, i_full, i_empty, done, tb, n_chunks, lane);
    } else {
        // ------------------------------------------------------------------ converters, then epilogue
        float csum = 0.f;
        uint32_t ss = 0, sp = 0, is = 0, ip = 0;
        for (int c = 0; c < n_chunks; ++c) {
            mbar_wait(&s_full[ss], sp);
            mbar_wait(&i_empty[is], ip ^ 1u);
            float* sa = stage_base + (size_t)ss * Cfg::STAGE;
            float* sb = sa + Cfg::A_STAGE;
            float* im = img_base + (size_t)is * Cfg::IMG;
            // reduction rows at or beyond this CTA's range (a slab's ragged last chunk) contribute nothing
            const long long r0 = rbeg + (long long)c * TG_KC;
            const int valid = (int)((rend - r0 < TG_KC) ? (rend - r0) : TG_KC);
            if (valid < TG_KC) {
                // zero the staged reduction indices >= valid (rare: once per CTA at most)
                for (int e = tid; e < 128 * TG_KC; e += 256) {
                    const int rr = A_RCONTIG ? (((e & 15) >> 2 ^ (((e >> 4) >> 1) & 3)) * 4 + (e & 3)) : (e / 128);
                    if (rr >= valid) sa[e] = 0.f;
                }
                for (int e = tid; e < TN * TG_KC; e += 256) {
                    const int rr = B_RCONTIG ? (((e & 15) >> 2 ^ (((e >> 4) >> 1) & 3)) * 4 + (e & 3)) : (e / TN);
                    if (rr >= valid) sb[e] = 0.f;
                }
                asm volatile("bar.sync 1, 256;" ::: "memory");
            }
            float dummy = 0.f;
            tg_convert<A_RCONTIG, 128, false>(sa, im, im + Cfg::A_STAGE, g.a_swish != 0, tid, dummy);
            tg_convert<B_RCONTIG, TN, MODE == 2>(sb, im + 2 * Cfg::A_STAGE, im + 2 * Cfg::A_STAGE + Cfg::B_STAGE, false, tid, csum);
            fence_proxy_async_smem();   // generic-proxy stores -> visible to the tensor core's async proxy
            __syncwarp();
            if (lane == 0) {
                umma::mbar_arrive(&i_full[is]);
                umma::mbar_arrive(&s_empty[ss]);
            }
            if (++ss == TG_SSTAGES) { ss = 0; sp ^= 1u; }
            if (++is == TG_ISTAGES) { is = 0; ip ^= 1u; }
        }
        ug_colsum_flush<MODE, TN>(g, j0, tid, csum);
        ug_epilogue<MODE, TN>(g, tb, done, i0, j0, warp, lane);
    }
    ug_teardown<TN>(tb, warp);
}

// ---- tensor maps (driver API reached through the runtime: the library keeps linking against cudart only) ----
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            p = nullptr;
        return reinterpret_cast<EncodeTiledFn>(p);
    }();
    return fn;
}

// 2-D fp32 row-major matrix [rows][cols] with row stride ld; box = box_rows x box_cols (cols innermost)
static bool make_map(CUtensorMap* m, const float* base, long long rows, long long cols, long long ld, int box_rows,
                     int box_cols, bool swizzle64) {
    EncodeTiledFn fn = encode_tiled_fn();
    if (!fn) return false;
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * 4};
    cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    return fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr,
              CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_NONE,
              CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// The arguments of the copy-engine-fed kernel: g and the tensor maps of A and B.  False when the operands do not fit a
// tensor map (16-byte aligned base, row stride a multiple of 4 floats, sizes below 2^31) or the driver has no encoder.
static bool make_tma_args(int mode, int TN, const GemmArgs& g, TGemmArgs* ta) {
    // A: NN/NT [I][R], TN [R][I];  B: NT [J][R], NN/TN [R][J]
    const bool a_rcontig = (mode != 2), b_rcontig = (mode == 1);
    auto ok = [](const float* p, long long ld) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0 && (ld & 3) == 0; };
    if (!ok(g.A, g.lda) || !ok(g.B, g.ldb)) return false;
    if (g.I > 0x7fffffffLL || g.J > 0x7fffffffLL || g.R > 0x7fffffffLL) return false;
    ta->g = g;
    const bool ma = a_rcontig ? make_map(&ta->mapA, g.A, g.I, g.R, g.lda, 128, TG_KC, true)
                              : make_map(&ta->mapA, g.A, g.R, g.I, g.lda, TG_KC, 128, false);
    const bool mb = b_rcontig ? make_map(&ta->mapB, g.B, g.J, g.R, g.ldb, TN, TG_KC, true)
                              : make_map(&ta->mapB, g.B, g.R, g.J, g.ldb, TG_KC, TN, false);
    return ma && mb;
}

// Grid of a tcgen05 GEMM: 128 x TN output tiles.  Mode 2 (grad-weight: a tiny output, a long reduction over samples)
// splits the reduction into gridDim.z slabs of g.r_slab rows, so that at least ~3 waves of CTAs are in flight; each CTA
// adds its partial tile with atomics.
static dim3 umma_grid(int mode, int TN, GemmArgs& g) {
    dim3 grid((unsigned)((g.I + 127) / 128), (unsigned)((g.J + TN - 1) / TN), 1);
    if (mode == 2) {
        const long long tiles = ((g.I + 127) / 128) * ((g.J + TN - 1) / TN);
        const long long slabs = std::max<long long>(1, (3 * 148 + tiles - 1) / tiles);
        const long long rs = (g.R + slabs - 1) / slabs;
        g.r_slab = std::max<long long>(256, (rs + 31) / 32 * 32);
        grid.z = (unsigned)((g.R + g.r_slab - 1) / g.r_slab);
    }
    return grid;
}

template <class Args>
static int launch_umma_kernel(void (*kernel)(Args), dim3 grid, int threads, size_t smem, cudaStream_t st, const Args& args) {
    if (int rc = smem_optin((const void*)kernel, smem)) return rc;
    kernel<<<grid, threads, smem, st>>>(args);
    count_launch();
    ZF_CUDA_CHECK(cudaGetLastError());
    return ZF_OK;
}

// The tcgen05 kernel of one mode and tile width: fed by the copy engine when ta is given, else register-path loaders.
template <int MODE, int TN>
static int launch_umma(cudaStream_t st, dim3 grid, const GemmArgs& g, const TGemmArgs* ta) {
    if (ta) return launch_umma_kernel(umma_gemm_tma_kernel<MODE, TN>, grid, TG_THREADS, TgCfg<TN>::SMEM, st, *ta);
    return launch_umma_kernel(umma_gemm_kernel<MODE, TN>, grid, UG_THREADS, UgCfg<TN>::SMEM, st, g);
}

// Which GEMM computes a product, and its launch.  impl is the GEMM developer switch (impl_switch().gemm); the first row
// that applies:
//   impl == simt, or act != swish                                          gemm_kernel<mode>           (FFMA)
//   impl != legacy, A and B 16-byte aligned, lda and ldb multiples of 4,
//     I, J, R < 2^31, tensor-map encoder found                             umma_gemm_tma_kernel<mode, TN>
//   otherwise                                                              umma_gemm_kernel<mode, TN>
// with TN = 256 when J > 128, else 128.  Mode 2 splits the reduction into gridDim.z slabs: g.r_slab rows each for the FFMA
// kernel; for the tcgen05 kernels r_slab = max(256, round_up32(ceil(R / slabs))) with slabs = max(1, ceil(444 / tiles))
// and tiles = the number of 128 x TN output tiles (umma_grid).
int launch_gemm(cudaStream_t st, int mode, const GemmArgs& g) {
    const char* impl = impl_switch().gemm;
    if (impl[0] == 's' || g.act != ZF_ACT_SWISH) {
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
    const bool wide = g.J > 128;
    GemmArgs u = g;
    const dim3 grid = umma_grid(mode, wide ? 256 : 128, u);
    if (grid.x == 0 || grid.y == 0 || u.R <= 0) return ZF_OK;
    TGemmArgs ta;
    const TGemmArgs* tma = (impl[0] != 'l' && make_tma_args(mode, wide ? 256 : 128, u, &ta)) ? &ta : nullptr;
    if (mode == 0) return wide ? launch_umma<0, 256>(st, grid, u, tma) : launch_umma<0, 128>(st, grid, u, tma);
    if (mode == 1) return wide ? launch_umma<1, 256>(st, grid, u, tma) : launch_umma<1, 128>(st, grid, u, tma);
    return wide ? launch_umma<2, 256>(st, grid, u, tma) : launch_umma<2, 128>(st, grid, u, tma);
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
