// Single-CTA self-test of the tcgen05 building blocks: out[128][N] = A[128][K] * B[N][K]^T with
// 3xTF32 split products, A staged registers -> TMEM, B as a shared-memory image, D in TMEM.
#include "zf_umma.cuh"

namespace zf {

__global__ void __launch_bounds__(160) umma_selftest_kernel(const float* __restrict__ A, const float* __restrict__ B,
                                                            int N, int K, float* __restrict__ out, int mask_mode) {
    extern __shared__ __align__(128) float sB[];  // hi image then lo image, N*K floats each
    __shared__ uint32_t tmem_base_s;
    __shared__ __align__(8) uint64_t bar;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (warp == 4) umma::tmem_alloc(&tmem_base_s, 512);
    if (tid == 0) { mbar_init(&bar, 1); mbar_fence_init(); }
    for (int e = tid; e < N * K; e += blockDim.x) {
        const int n = e / K, k = e - n * K;
        float hi, lo;
        umma::split_tf32(B[e], hi, lo);
        sB[umma::b_image_index(n, k, N)] = hi;
        sB[N * K + umma::b_image_index(n, k, N)] = lo;
    }
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tb = tmem_base_s;
    const uint32_t colAhi = 0, colAlo = 128, colD = 256;
    if (warp < 4) {  // one thread per row m: split and store A into tensor memory
        const int m = warp * 32 + lane;
        for (int k0 = 0; k0 < K; k0 += 8) {
            float hi[8], lo[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) umma::split_tf32(A[m * K + k0 + i], hi[i], lo[i]);
            umma::st8(umma::taddr(tb, warp * 32, colAhi + k0), hi);
            umma::st8(umma::taddr(tb, warp * 32, colAlo + k0), lo);
        }
        if (mask_mode) {  // sentinel in D: masked lanes must keep it
            float sv[8] = {777.f, 777.f, 777.f, 777.f, 777.f, 777.f, 777.f, 777.f};
            for (int n0 = 0; n0 < N; n0 += 8) umma::st8(umma::taddr(tb, warp * 32, colD + n0), sv);
        }
        umma::wait_st();
    }
    fence_proxy_async_smem();  // B images were written through the generic proxy
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    if (warp == 4) {
        if (umma::elect_one()) {
            const uint32_t idesc = umma::instr_desc_tf32(N);
            const uint32_t lbo = (uint32_t)(N >> 3) * 128u, sbo = 128u;
            const uint32_t bhi = smem_u32(sB), blo = smem_u32(sB + N * K);
            for (int ks = 0; ks < K / 8; ++ks) {
                const uint64_t dhi = umma::smem_desc_kmajor(bhi + ks * 2 * lbo, lbo, sbo);
                const uint64_t dlo = umma::smem_desc_kmajor(blo + ks * 2 * lbo, lbo, sbo);
                const uint32_t lo_m = mask_mode == 2 ? 0xffffffffu : 0u, hi_m = mask_mode == 1 ? 0xffffffffu : 0u;
                umma::mma_tf32_ts_masked(tb + colD, tb + colAlo + ks * 8, dhi, idesc, ks > 0, lo_m, lo_m, hi_m, hi_m);
                umma::mma_tf32_ts_masked(tb + colD, tb + colAhi + ks * 8, dlo, idesc, true, lo_m, lo_m, hi_m, hi_m);
                umma::mma_tf32_ts_masked(tb + colD, tb + colAhi + ks * 8, dhi, idesc, true, lo_m, lo_m, hi_m, hi_m);
            }
            umma::commit(&bar);
        }
        __syncwarp();
    }
    if (warp < 4) {
        mbar_wait(&bar, 0);
        umma::fence_after_sync();
        const int m = warp * 32 + lane;
        for (int n0 = 0; n0 < N; n0 += 8) {
            float v[8];
            umma::ld8(umma::taddr(tb, warp * 32, colD + n0), v);
            umma::wait_ld();
#pragma unroll
            for (int i = 0; i < 8; ++i) out[m * N + n0 + i] = v[i];
        }
    }
    umma::fence_before_sync();
    __syncthreads();
    if (warp == 4) umma::tmem_dealloc(tb, 512);
}
}  // namespace zf

// The same product with the 3xFP16 split (kind::f16): A as fp16 pairs in tensor memory (K / 2 columns per part),
// B as fp16 K-major images, main and cross accumulators.  variant bit 0: swap the two halves of every A word
// (layout probe); bit 1: skip the cross products (plain fp16).
namespace zf {
__global__ void __launch_bounds__(160) umma_selftest_f16_kernel(const float* __restrict__ A, const float* __restrict__ B,
                                                                int N, int K, float* __restrict__ out, int variant) {
    extern __shared__ __align__(128) float sBf[];  // hi image then lo image, N*K halves each
    __half* sB = reinterpret_cast<__half*>(sBf);
    __shared__ uint32_t tmem_base_s;
    __shared__ __align__(8) uint64_t bar;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (warp == 4) umma::tmem_alloc(&tmem_base_s, 512);
    if (tid == 0) { mbar_init(&bar, 1); mbar_fence_init(); }
    for (int e = tid; e < N * K; e += blockDim.x) {
        const int n = e / K, k = e - n * K;
        const float x = B[e];
        const __half h = __float2half_rn(x);
        const __half l = __float2half_rn((x - __half2float(h)) * umma::kF16LoScale);
        sB[umma::b_image_index_f16(n, k, N)] = h;
        sB[N * K + umma::b_image_index_f16(n, k, N)] = l;
    }
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tb = tmem_base_s;
    const uint32_t colAhi = 0, colAlo = 64, colD = 128, colX = 256;
    if (warp < 4) {
        const int m = warp * 32 + lane;
        for (int k0 = 0; k0 < K; k0 += 16) {
            uint32_t hi[8], lo[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const float x0 = A[m * K + k0 + 2 * i], x1 = A[m * K + k0 + 2 * i + 1];
                if (variant & 1) umma::split_f16x2(x1, x0, hi[i], lo[i]);
                else umma::split_f16x2(x0, x1, hi[i], lo[i]);
            }
            umma::st8u(umma::taddr(tb, warp * 32, colAhi + k0 / 2), hi);
            umma::st8u(umma::taddr(tb, warp * 32, colAlo + k0 / 2), lo);
        }
        umma::wait_st();
    }
    fence_proxy_async_smem();
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    if (warp == 4) {
        if (umma::elect_one()) {
            const uint32_t idesc = umma::instr_desc_f16(N);
            const uint32_t lbo = (uint32_t)(N >> 3) * 128u, sbo = 128u;
            const uint32_t bhi = smem_u32(sB), blo = smem_u32(sB + N * K);
            for (int ks = 0; ks < K / 16; ++ks) {
                const uint64_t dhi = umma::smem_desc_kmajor(bhi + ks * 2 * lbo, lbo, sbo);
                const uint64_t dlo = umma::smem_desc_kmajor(blo + ks * 2 * lbo, lbo, sbo);
                if (!(variant & 2)) {
                    umma::mma_f16_ts(tb + colX, tb + colAlo + ks * 8, dhi, idesc, ks > 0);
                    umma::mma_f16_ts(tb + colX, tb + colAhi + ks * 8, dlo, idesc, true);
                }
                umma::mma_f16_ts(tb + colD, tb + colAhi + ks * 8, dhi, idesc, ks > 0);
            }
            umma::commit(&bar);
        }
        __syncwarp();
    }
    if (warp < 4) {
        mbar_wait(&bar, 0);
        umma::fence_after_sync();
        const int m = warp * 32 + lane;
        for (int n0 = 0; n0 < N; n0 += 8) {
            float v[8], w[8];
            umma::ld8(umma::taddr(tb, warp * 32, colD + n0), v);
            umma::ld8(umma::taddr(tb, warp * 32, colX + n0), w);
            umma::wait_ld();
#pragma unroll
            for (int i = 0; i < 8; ++i) out[m * N + n0 + i] = (variant & 2) ? v[i] : fmaf(w[i], umma::kF16LoUnscale, v[i]);
        }
    }
    umma::fence_before_sync();
    __syncthreads();
    if (warp == 4) umma::tmem_dealloc(tb, 512);
}
}  // namespace zf

// out[128][N] = A[128][K] * B[N][K]^T with the bf16 x 2 split, BOTH operands from shared memory, each either as a
// K-major image ([k/8][r/8][r%8][k%8]) or as an MN-major one ([r/8][k/8][k%8][r%8]).  flags bit 0 / 1: A / B MN-major;
// bit 2: descriptor probe - swap which of LBO / SBO carries the MN-direction stride of an MN-major operand.
namespace zf {
__global__ void __launch_bounds__(160) umma_selftest_bf16_kernel(const float* __restrict__ A, const float* __restrict__ B,
                                                                 int N, int K, float* __restrict__ out, int flags) {
    extern __shared__ __align__(128) float sraw[];
    uint16_t* sA = reinterpret_cast<uint16_t*>(sraw);          // hi image then lo image, 128*K half-words each
    uint16_t* sB = sA + 2 * 128 * K;                            // hi image then lo image, N*K each
    __shared__ uint32_t tmem_base_s;
    __shared__ __align__(8) uint64_t bar;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const bool a_mn = flags & 1, b_mn = flags & 2, swap = flags & 4;
    if (warp == 4) umma::tmem_alloc(&tmem_base_s, 128);
    if (tid == 0) { mbar_init(&bar, 1); mbar_fence_init(); }
    auto put = [&](uint16_t* img, int R, bool mn, int r, int k, float x) {
        uint32_t hi, lo;
        umma::split_bf16x2(x, 0.f, hi, lo);
        const int ii = mn ? umma::mn_image_index_bf16(r, k, K) : umma::b_image_index_f16(r, k, R);
        img[ii] = (uint16_t)(hi & 0xffffu);
        img[R * K + ii] = (uint16_t)(lo & 0xffffu);
    };
    for (int e = tid; e < 128 * K; e += blockDim.x) put(sA, 128, a_mn, e / K, e % K, A[e]);
    for (int e = tid; e < N * K; e += blockDim.x) put(sB, N, b_mn, e / K, e % K, B[e]);
    fence_proxy_async_smem();
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tb = tmem_base_s;
    if (warp == 4) {
        if (umma::elect_one()) {
            const uint32_t idesc = umma::instr_desc_bf16(N, a_mn, b_mn);
            // operand of R rows: byte strides between core matrices along K and along MN, and the step of one MMA (K = 16)
            auto desc = [&](uint32_t base, int R, bool mn, int ks) {
                const uint32_t k_stride = mn ? 128u : (uint32_t)(R >> 3) * 128u;
                const uint32_t mn_stride = mn ? (uint32_t)(K >> 3) * 128u : 128u;
                const uint32_t lbo = (mn && swap) ? mn_stride : k_stride, sbo = (mn && swap) ? k_stride : mn_stride;
                return umma::smem_desc_kmajor(base + (uint32_t)ks * 2u * k_stride, lbo, sbo);
            };
            const uint32_t ahi = smem_u32(sA), alo = smem_u32(sA + 128 * K), bhi = smem_u32(sB), blo = smem_u32(sB + N * K);
            for (int ks = 0; ks < K / 16; ++ks) {
                umma::mma_f16_ss(tb, desc(alo, 128, a_mn, ks), desc(bhi, N, b_mn, ks), idesc, ks > 0);
                umma::mma_f16_ss(tb, desc(ahi, 128, a_mn, ks), desc(blo, N, b_mn, ks), idesc, true);
                umma::mma_f16_ss(tb, desc(ahi, 128, a_mn, ks), desc(bhi, N, b_mn, ks), idesc, true);
            }
            umma::commit(&bar);
        }
        __syncwarp();
    }
    if (warp < 4) {
        mbar_wait(&bar, 0);
        umma::fence_after_sync();
        const int m = warp * 32 + lane;
        for (int n0 = 0; n0 < N; n0 += 8) {
            float v[8];
            umma::ld8(umma::taddr(tb, warp * 32, n0), v);
            umma::wait_ld();
#pragma unroll
            for (int i = 0; i < 8; ++i) out[m * N + n0 + i] = v[i];
        }
    }
    umma::fence_before_sync();
    __syncthreads();
    if (warp == 4) umma::tmem_dealloc(tb, 128);
}
}  // namespace zf

extern "C" int zf_selftest_umma_bf16(void* stream, const float* A, const float* B, int32_t N, int32_t K, float* out,
                                     int32_t flags) {
    ZF_REQUIRE(A && B && out, "selftest_umma_bf16: null argument");
    ZF_REQUIRE(N >= 16 && N <= 128 && N % 16 == 0 && K >= 16 && K <= 128 && K % 16 == 0, "selftest_umma_bf16: bad N/K");
    const size_t smem = (size_t)2 * (128 + N) * K * sizeof(uint16_t);
    if (int rc = zf::smem_optin((const void*)zf::umma_selftest_bf16_kernel, smem)) return rc;
    zf::umma_selftest_bf16_kernel<<<1, 160, smem, (cudaStream_t)stream>>>(A, B, N, K, out, flags);
    zf::count_launch();
    ZF_CUDA_CHECK(cudaGetLastError());
    return ZF_OK;
}

extern "C" int zf_selftest_umma_f16(void* stream, const float* A, const float* B, int32_t N, int32_t K, float* out,
                                    int32_t variant) {
    ZF_REQUIRE(A && B && out, "selftest_umma_f16: null argument");
    ZF_REQUIRE(N >= 16 && N <= 128 && N % 16 == 0 && K >= 16 && K <= 128 && K % 16 == 0, "selftest_umma_f16: bad N/K");
    const size_t smem = (size_t)2 * N * K * sizeof(__half);
    if (int rc = zf::smem_optin((const void*)zf::umma_selftest_f16_kernel, smem)) return rc;
    zf::umma_selftest_f16_kernel<<<1, 160, smem, (cudaStream_t)stream>>>(A, B, N, K, out, variant);
    zf::count_launch();
    ZF_CUDA_CHECK(cudaGetLastError());
    return ZF_OK;
}

extern "C" int zf_selftest_umma(void* stream, const float* A, const float* B, int32_t N, int32_t K, float* out,
                                int32_t mask_mode) {
    ZF_REQUIRE(A && B && out, "selftest_umma: null argument");
    ZF_REQUIRE(N >= 16 && N <= 128 && N % 16 == 0 && K >= 8 && K <= 128 && K % 8 == 0, "selftest_umma: bad N/K");
    const size_t smem = (size_t)2 * N * K * sizeof(float);
    if (int rc = zf::smem_optin((const void*)zf::umma_selftest_kernel, smem)) return rc;
    zf::umma_selftest_kernel<<<1, 160, smem, (cudaStream_t)stream>>>(A, B, N, K, out, mask_mode);
    zf::count_launch();
    ZF_CUDA_CHECK(cudaGetLastError());
    return ZF_OK;
}

#ifdef ZF_TRACE
// Developer microbenchmark (scripts/umma_rate.py, -DZF_TRACE builds only): cycles per tcgen05.mma for the shapes the
// chain kernel issues.  mode 0: every product into one accumulator; 1: cross products into a second accumulator;
// bit 2 (mode | 4): four more warps keep reading the accumulator with tcgen05.ld while the MMAs run.
namespace zf {
__global__ void __launch_bounds__(192) umma_rate_kernel(int N, int reps, int mode, long long* out) {
    extern __shared__ __align__(128) float sB[];
    __shared__ uint32_t tmem_base_s;
    __shared__ __align__(8) uint64_t bar;
    __shared__ volatile int stop;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (warp == 4) umma::tmem_alloc(&tmem_base_s, 512);
    if (tid == 0) { mbar_init(&bar, 1); mbar_fence_init(); stop = 0; }
    for (int e = tid; e < 2 * N * 32; e += blockDim.x) sB[e] = 0.f;
    fence_proxy_async_smem();
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tb = tmem_base_s;
    if (warp < 4) {
        float z[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        for (int c = 0; c < 512; c += 8) umma::st8(umma::taddr(tb, warp * 32, c), z);
        umma::wait_st();
    }
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    if (warp == 4) {
        if (umma::elect_one()) {
            const uint32_t idesc = umma::instr_desc_tf32(N);
            const uint32_t lbo = (uint32_t)(N >> 3) * 128u;
            const uint32_t bhi = smem_u32(sB), blo = bhi + (uint32_t)N * 128u;
            const uint32_t dmain = tb + 256u, dcross = (mode & 1) ? tb + 384u : dmain;
            const long long t0 = clock64();
            for (int r = 0; r < reps; ++r) {
#pragma unroll
                for (int c = 0; c < 4; ++c) {
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks) {
                        const uint64_t dhi = umma::smem_desc_kmajor(bhi + ks * 2 * lbo, lbo, 128u);
                        const uint64_t dlo = umma::smem_desc_kmajor(blo + ks * 2 * lbo, lbo, 128u);
                        const uint32_t acol = (uint32_t)(c * 32 + ks * 8);
                        if (mode & 2) {   // one product only (plain TF32)
                            umma::mma_tf32_ts(dmain, tb + acol, dhi, idesc, true);
                        } else {
                            umma::mma_tf32_ts(dcross, tb + 128u + acol, dhi, idesc, true);
                            umma::mma_tf32_ts(dcross, tb + acol, dlo, idesc, true);
                            umma::mma_tf32_ts(dmain, tb + acol, dhi, idesc, true);
                        }
                    }
                }
            }
            const long long t1 = clock64();
            umma::commit(&bar);
            mbar_wait(&bar, 0);
            const long long t2 = clock64();
            out[0] = t1 - t0;   // issue
            out[1] = t2 - t0;   // issue + drain
            stop = 1;
        }
        __syncwarp();
    } else if (warp < 4 && (mode & 4)) {
        float v[16];
        float acc = 0.f;
        while (!stop) {
            umma::ld16(umma::taddr(tb, warp * 32, 256 + (lane & 1) * 16), v);
            umma::wait_ld();
            acc += v[0];
        }
        if (acc == 123.f) out[2] = 1;
    }
    umma::fence_before_sync();
    __syncthreads();
    if (warp == 4) umma::tmem_dealloc(tb, 512);
}
}  // namespace zf

extern "C" int zf_debug_umma_rate(int32_t N, int32_t reps, int32_t mode, int32_t ctas, long long* host_out) {
    const size_t smem = (size_t)2 * N * 32 * sizeof(float);
    if (zf::smem_optin((const void*)zf::umma_rate_kernel, smem)) return 1;
    long long* d = nullptr;
    if (cudaMalloc(&d, 4 * sizeof(long long)) != cudaSuccess) return 1;
    cudaMemset(d, 0, 4 * sizeof(long long));
    zf::umma_rate_kernel<<<ctas, 192, smem>>>(N, reps, mode, d);
    const int rc = (int)cudaDeviceSynchronize();
    cudaMemcpy(host_out, d, 4 * sizeof(long long), cudaMemcpyDeviceToHost);
    cudaFree(d);
    return rc;
}
#endif
