// tcgen05 GEMMs of the train step's Dense VJPs (bijectors.py:343-347 under jax.grad, train.py:82) on EVENT-ROW IMAGES.
//
// An event-major matrix X (M events x W features) travels between the kernels of the backward pass as a bf16 x 2
// split (hi = bf16(x), lo = bf16(x - hi): 16 significant bits, fp32's exponent range) laid out in tensor-core core
// matrices, written once by the kernel that produces it:
//     tile t = events [128 t, 128 t + 128):  [part hi | lo][w / 8][e / 8][e % 8][w % 8]   (W x 256 bytes per part)
// The same bytes are a K-major operand for a reduction over FEATURES (grad-input GEMMs: 8 event rows x 16 bytes of
// features per core matrix) and an MN-major operand for a reduction over EVENTS (grad-weight GEMMs: 8 event rows x
// 16 bytes of features is then 8 K rows x 8 MN elements), so no operand is ever converted or transposed: every
// stage of both kernels is bulk copies (copy engine) -> tcgen05.mma, both operands from shared memory.
// Rows of the last tile beyond M are ZERO in every image (producers write them), so reductions over events need no
// masking.  Products: hi*hi + hi*lo + lo*hi in one fp32 accumulator (gradient tolerance, 1e-4 of the leaf maximum).
//
//   img_nt_kernel  out[e][n] = (sum_k X[e][k] W[n][k]) * G[e][n]      grad wrt a Dense input (times swish')
//   img_tn_kernel  C[a][b]  += sum_e A[e][a] B[e][b];  colsum[b] += sum_e B[e][b]    grad wrt kernel and bias
#include "zf_umma.cuh"

#include <algorithm>

namespace zf {

constexpr int IG_THREADS = 192;   // warps 0-3: epilogue (one thread per accumulator lane), warp 4: producer, warp 5: MMA issuer

__device__ __forceinline__ uint64_t ig_desc(uint32_t addr, uint32_t lbo, uint32_t sbo) { return umma::smem_desc_kmajor(addr, lbo, sbo); }

// ---------------------------------------------------------------------------------------------------------------------
// grad-input: one 128-event tile per accumulator, reduction over the KW features of X in chunks of <= 64
// ---------------------------------------------------------------------------------------------------------------------
struct ImgNtArgs {
    const char* X; int KW;      // event-row image, KW % 16 == 0
    const char* W; int N;       // [part][k / 8][n / 8][n % 8][k % 8] bf16 x 2, N rows (16 .. 128, % 16 == 0)
    const float* G; int ldg;    // optional fp32: the product is multiplied by it (swish' of the pre-activations); (M, ldg >= N) row-major,
                                // or ldg < 0: tile image [tile][n / 4][event % 128][n % 4] of width 128 (coalesced on both sides)
    char* out_img;              // optional event-row image of width N
    float* out_f32; int ldo, n_valid;   // optional fp32 (M, ldo), the first n_valid columns
    long long M;
};
constexpr int NT_STAGES = 3, NT_KC = 64;
constexpr int NT_STAGE_BYTES = 2 * NT_KC * 256 + 2 * NT_KC * 128 * 2;   // A: 2 parts x 64 features x 256 B; B: 2 parts x 64 k x 128 n x 2 B

__global__ void __launch_bounds__(IG_THREADS, 1) img_nt_kernel(const __grid_constant__ ImgNtArgs g) {
    extern __shared__ __align__(128) char smem[];
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + NT_STAGES * NT_STAGE_BYTES);
    uint64_t *full = bars, *empty = bars + NT_STAGES, *dfull = bars + 2 * NT_STAGES, *dempty = dfull + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(dempty + 2);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const long long n_tiles = (g.M + 127) / 128;
    const int N = g.N, KW = g.KW;
    if (tid == 0) {
        for (int s = 0; s < NT_STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(&dfull[b], 1); mbar_init(&dempty[b], 128); }
        mbar_fence_init();
    }
    if (warp == 5) umma::tmem_alloc(tmem_slot, 256);
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tb = *tmem_slot;
    const int n_chunks = (KW + NT_KC - 1) / NT_KC;

    if (warp == 4) {
        if (lane == 0) {
            uint32_t stage = 0, phase = 0;
            for (long long t = blockIdx.x; t < n_tiles; t += gridDim.x) {
                const char* xt = g.X + (size_t)t * 2 * KW * 256;
                for (int c = 0; c < n_chunks; ++c) {
                    const int k0 = c * NT_KC, kc = min(NT_KC, KW - k0);   // features of this chunk (multiple of 16)
                    const uint32_t abytes = (uint32_t)kc * 256u, bbytes = (uint32_t)kc * (uint32_t)N * 2u;
                    char* sa = smem + stage * NT_STAGE_BYTES;
                    char* sb = sa + 2 * NT_KC * 256;
                    mbar_wait(&empty[stage], phase ^ 1u);
                    mbar_arrive_expect_tx(&full[stage], 2u * (abytes + bbytes));
                    for (int p = 0; p < 2; ++p) {
                        bulk_copy_g2s(sa + p * NT_KC * 256, xt + (size_t)p * KW * 256 + (size_t)k0 * 256, abytes, &full[stage]);
                        bulk_copy_g2s(sb + p * NT_KC * 128 * 2, g.W + (size_t)p * KW * N * 2 + (size_t)k0 * N * 2, bbytes, &full[stage]);
                    }
                    if (++stage == NT_STAGES) { stage = 0; phase ^= 1u; }
                }
            }
        }
        __syncwarp();
    } else if (warp == 5) {
        uint32_t stage = 0, phase = 0, it = 0;
        const uint32_t idesc = umma::instr_desc_bf16(N, false, false);
        const uint32_t b_kstride = (uint32_t)N * 16u;   // bytes between k groups of the weight image
        for (long long t = blockIdx.x; t < n_tiles; t += gridDim.x, ++it) {
            const uint32_t buf = it & 1u;
            mbar_wait(&dempty[buf], ((it >> 1) & 1u) ^ 1u);
            umma::fence_after_sync();
            const uint32_t d = tb + buf * 128u;
            for (int c = 0; c < n_chunks; ++c) {
                const int kc = min(NT_KC, KW - c * NT_KC);
                mbar_wait(&full[stage], phase);
                umma::fence_after_sync();
                if (umma::elect_one()) {
                    const uint32_t sa = smem_u32(smem + stage * NT_STAGE_BYTES), sb = sa + 2 * NT_KC * 256;
                    for (int ks = 0; ks < kc / 16; ++ks) {
                        const uint64_t ahi = ig_desc(sa + ks * 4096u, 2048u, 128u), alo = ig_desc(sa + NT_KC * 256 + ks * 4096u, 2048u, 128u);
                        const uint64_t bhi = ig_desc(sb + ks * 2u * b_kstride, b_kstride, 128u);
                        const uint64_t blo = ig_desc(sb + NT_KC * 128 * 2 + ks * 2u * b_kstride, b_kstride, 128u);
                        umma::mma_f16_ss(d, alo, bhi, idesc, (c | ks) != 0);
                        umma::mma_f16_ss(d, ahi, blo, idesc, true);
                        umma::mma_f16_ss(d, ahi, bhi, idesc, true);
                    }
                    umma::commit(&empty[stage]);
                    if (c == n_chunks - 1) umma::commit(&dfull[buf]);
                }
                __syncwarp();
                if (++stage == NT_STAGES) { stage = 0; phase ^= 1u; }
            }
        }
    } else {
        const int m = warp * 32 + lane;
        uint32_t it = 0;
        for (long long t = blockIdx.x; t < n_tiles; t += gridDim.x, ++it) {
            const uint32_t buf = it & 1u;
            const long long e = t * 128 + m;
            const bool valid = e < g.M;
            // The multiplier's whole row of this tile (N <= 128 columns: 32 float4 registers) is requested BEFORE the
            // accumulator is awaited: one exposed memory latency per tile instead of one per 16-column chunk (the four
            // epilogue warps are alone on their schedulers, nothing else would hide it).
            const bool tiled = g.ldg < 0;
            const int gq = tiled ? 128 : 1;   // float4 units between consecutive 4-column groups
            const bool use_g = g.G != nullptr && valid;
            float4 gall[32];
            if (use_g) {
                const float4* gp = tiled ? reinterpret_cast<const float4*>(g.G + (size_t)t * (128 * 128) + (size_t)m * 4)
                                         : reinterpret_cast<const float4*>(g.G + e * g.ldg);
#pragma unroll
                for (int q = 0; q < 32; ++q)
                    if (4 * q < N) gall[q] = gp[q * gq];
            }
            mbar_wait(&dfull[buf], (it >> 1) & 1u);
            umma::fence_after_sync();
            char* ot = g.out_img ? g.out_img + (size_t)t * 2 * N * 256 + (size_t)(m >> 3) * 128 + (size_t)(m & 7) * 16 : nullptr;
#pragma unroll
            for (int ci = 0; ci < 8; ++ci) {
                const int c0 = ci * 16;
                if (c0 >= N) break;
                float v[16];
                umma::ld16(umma::taddr(tb, warp * 32, buf * 128u + c0), v);
                umma::wait_ld();
                if (use_g) {
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const float4 gv = gall[4 * ci + q];
                        v[4 * q] *= gv.x; v[4 * q + 1] *= gv.y; v[4 * q + 2] *= gv.z; v[4 * q + 3] *= gv.w;
                    }
                }
                if (!valid) {
#pragma unroll
                    for (int j = 0; j < 16; ++j) v[j] = 0.f;
                }
                if (g.out_f32 && valid) {
#pragma unroll
                    for (int j = 0; j < 16; ++j)
                        if (c0 + j < g.n_valid) g.out_f32[e * g.ldo + c0 + j] = v[j];
                }
                if (ot) {
#pragma unroll
                    for (int u = 0; u < 2; ++u) {
                        uint32_t hi[4], lo[4];
#pragma unroll
                        for (int q = 0; q < 4; ++q) umma::split_bf16x2(v[8 * u + 2 * q], v[8 * u + 2 * q + 1], hi[q], lo[q]);
                        char* dst = ot + (size_t)((c0 >> 3) + u) * 2048;
                        *reinterpret_cast<uint4*>(dst) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                        *reinterpret_cast<uint4*>(dst + (size_t)N * 256) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
                    }
                }
            }
            umma::fence_before_sync();
            umma::mbar_arrive(&dempty[buf]);
        }
    }
    umma::fence_before_sync();
    __syncthreads();
    if (warp == 5) umma::tmem_dealloc(tb, 256);
}

// ---------------------------------------------------------------------------------------------------------------------
// grad-weight: each CTA owns a slab of NS output columns and a range of event tiles; the accumulator lives in tensor
// memory for the whole range and is added to C with atomics at the end
// ---------------------------------------------------------------------------------------------------------------------
struct ImgTnArgs {
    const char* A;              // event-row image of width 128: its features are the output rows a
    const char* B; int WB;      // event-row image: its features are the output columns b
    float* C; long long ldca, ldcb; int a_valid, b_valid;   // C[a ldca + b ldcb] += sum_e A[e][a] B[e][b]
    float* colsum;              // optional (b_valid): += sum_e B[e][b]
    float* arow_sum; int arow_col;   // optional: column b == arow_col of the product goes to arow_sum[a] instead of C
    long long n_tiles;
    int NS;                     // columns per CTA (<= 128, % 16 == 0); gridDim.y slabs
};
// Shared memory is a ring of 32 KB slots; a 128-event tile takes four of them, each ONE bulk copy (a whole part of a
// tile is contiguous in the image: the A part always, the B part for a slab of consecutive feature groups).  Six slots =
// one and a half tiles in flight.  The products run pass by pass in the order A lo B hi, A hi B hi, A hi B lo and the
// parts are fetched in the order A lo, B hi, A hi, B lo: slots are then handed back in exactly the order they were
// filled (A lo after pass 1, B hi after pass 2, A hi and B lo after pass 3), so the ring never waits for the END of a
// tile before it can fetch the next tile's first operands (with the passes ordered lo-hi, hi-lo, hi-hi the B parts of
// tile t+1 sat behind tile t's A hi slot, released last: one exposed load latency per tile).
constexpr int TN_SLOTS = 6, TN_SLOT_BYTES = 32768, TN_NS = 128;

__global__ void __launch_bounds__(IG_THREADS, 1) img_tn_kernel(const __grid_constant__ ImgTnArgs g) {
    extern __shared__ __align__(128) char smem[];
    char* ones = smem + TN_SLOTS * TN_SLOT_BYTES;    // K-major 128 x 16 image of 1.0 (bf16): the column sums as an MMA
    uint64_t* bars = reinterpret_cast<uint64_t*>(ones + 4096);
    uint64_t *full = bars, *empty = bars + TN_SLOTS, *done = bars + 2 * TN_SLOTS;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done + 1);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int NS = g.NS, n0 = blockIdx.y * NS, ns = min(NS, g.WB - n0);   // this CTA's columns [n0, n0 + ns), ns % 16 == 0
    const long long t0 = (long long)blockIdx.x * g.n_tiles / gridDim.x, t1 = (long long)(blockIdx.x + 1) * g.n_tiles / gridDim.x;
    if (tid == 0) {
        for (int s = 0; s < TN_SLOTS; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        mbar_init(done, 1);
        mbar_fence_init();
    }
    for (int i = tid; i < 2048; i += IG_THREADS) reinterpret_cast<uint16_t*>(ones)[i] = 0x3f80;   // bf16 1.0
    fence_proxy_async_smem();
    if (warp == 5) umma::tmem_alloc(tmem_slot, 256);
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tb = *tmem_slot;
    const uint32_t bbytes = (uint32_t)ns * 256u;

    if (warp == 4) {
        if (lane == 0) {
            uint32_t slot = 0, phase = 0;
            auto put = [&](const char* src, uint32_t bytes) {
                mbar_wait(&empty[slot], phase ^ 1u);
                mbar_arrive_expect_tx(&full[slot], bytes);
                bulk_copy_g2s(smem + slot * TN_SLOT_BYTES, src, bytes, &full[slot]);
                if (++slot == TN_SLOTS) { slot = 0; phase ^= 1u; }
            };
            for (long long t = t0; t < t1; ++t) {
                const char* at = g.A + (size_t)t * 2 * 128 * 256;
                const char* bt = g.B + (size_t)t * 2 * g.WB * 256 + (size_t)(n0 >> 3) * 2048;
                put(at + 32768, 32768u);                 // A lo
                put(bt, bbytes);                         // B hi
                put(at, 32768u);                         // A hi
                put(bt + (size_t)g.WB * 256, bbytes);    // B lo
            }
        }
        __syncwarp();
    } else if (warp == 5) {
        uint32_t slot = 0, phase = 0;
        const uint32_t idesc = umma::instr_desc_bf16(ns, true, true), idesc1 = umma::instr_desc_bf16(ns, false, true);
        const uint64_t one_d = ig_desc(smem_u32(ones), 2048u, 128u);
        bool first = true;
        for (long long t = t0; t < t1; ++t) {
            uint32_t sl[4], ph[4];
            for (int i = 0; i < 4; ++i) {
                sl[i] = slot; ph[i] = phase;
                if (++slot == TN_SLOTS) { slot = 0; phase ^= 1u; }
            }
            for (int i = 0; i < 2; ++i) mbar_wait(&full[sl[i]], ph[i]);   // pass 1's operands; the others are awaited by the issuer
            umma::fence_after_sync();
            if (umma::elect_one()) {
                const uint32_t alo = smem_u32(smem + sl[0] * TN_SLOT_BYTES), bhi = smem_u32(smem + sl[1] * TN_SLOT_BYTES);
                const uint32_t ahi = smem_u32(smem + sl[2] * TN_SLOT_BYTES), blo = smem_u32(smem + sl[3] * TN_SLOT_BYTES);
                // MN-major operands: K (events) direction stride 128 B = LBO, MN (features) direction 2048 B = SBO;
                // one MMA = 16 events = 256 bytes along K
#pragma unroll
                for (int ks = 0; ks < 8; ++ks) {
                    umma::mma_f16_ss(tb, ig_desc(alo + ks * 256u, 128u, 2048u), ig_desc(bhi + ks * 256u, 128u, 2048u), idesc, !(first && ks == 0));
                }
                umma::commit(&empty[sl[0]]);
                mbar_wait(&full[sl[2]], ph[2]);
                umma::fence_after_sync();
#pragma unroll
                for (int ks = 0; ks < 8; ++ks) {
                    umma::mma_f16_ss(tb, ig_desc(ahi + ks * 256u, 128u, 2048u), ig_desc(bhi + ks * 256u, 128u, 2048u), idesc, true);
                    if (g.colsum) umma::mma_f16_ss(tb + 128u, one_d, ig_desc(bhi + ks * 256u, 128u, 2048u), idesc1, !(first && ks == 0));
                }
                umma::commit(&empty[sl[1]]);
                mbar_wait(&full[sl[3]], ph[3]);
                umma::fence_after_sync();
#pragma unroll
                for (int ks = 0; ks < 8; ++ks) {
                    umma::mma_f16_ss(tb, ig_desc(ahi + ks * 256u, 128u, 2048u), ig_desc(blo + ks * 256u, 128u, 2048u), idesc, true);
                    if (g.colsum) umma::mma_f16_ss(tb + 128u, one_d, ig_desc(blo + ks * 256u, 128u, 2048u), idesc1, true);
                }
                umma::commit(&empty[sl[2]]);
                umma::commit(&empty[sl[3]]);
            }
            __syncwarp();
            first = false;
        }
        if (umma::elect_one()) umma::commit(done);
        __syncwarp();
    } else if (t1 > t0) {
        const int a = warp * 32 + lane;
        mbar_wait(done, 0);
        umma::fence_after_sync();
#pragma unroll 1
        for (int c0 = 0; c0 < ns; c0 += 16) {
            float v[16];
            umma::ld16(umma::taddr(tb, warp * 32, c0), v);
            umma::wait_ld();
            if (a < g.a_valid) {
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const int b = n0 + c0 + j;
                    if (g.arow_sum && b == g.arow_col) atomicAdd(g.arow_sum + a, v[j]);
                    else if (b < g.b_valid) atomicAdd(g.C + a * g.ldca + b * g.ldcb, v[j]);
                }
            }
            if (g.colsum) {
                umma::ld16(umma::taddr(tb, warp * 32, 128 + c0), v);
                umma::wait_ld();
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const int b = n0 + c0 + j;
                    if (c0 + j == a && b < g.b_valid) atomicAdd(g.colsum + b, v[j]);   // every lane holds the same sums
                }
            }
        }
    }
    umma::fence_before_sync();
    __syncthreads();
    if (warp == 5) umma::tmem_dealloc(tb, 256);
}

// ---------------------------------------------------------------------------------------------------------------------
// weight image for img_nt_kernel: Wimg(n, k) = W[n * ldw + (k / NL) * P + k % NL] for n < n_valid and k % NL < P, else 0
// (Dense kernel leaf (in, out) read as [n = in][k = out]; the last layer's columns padded per transformed dim)
// ---------------------------------------------------------------------------------------------------------------------
constexpr int kMaxPackW = ZF_MAX_LAYERS + 1;
struct PackWBatch { PackWJob job[kMaxPackW]; int n; };

// all weight images of a coupling in one launch: block b works on the job whose [block0, block0 + blocks) holds it
__global__ void __launch_bounds__(256) pack_w_images_kernel(const __grid_constant__ PackWBatch b) {
    int i = 0;
    while (i + 1 < b.n && (int)blockIdx.x >= b.job[i + 1].block0) ++i;
    const PackWJob& j = b.job[i];
    const float* __restrict__ W = j.W;
    uint16_t* __restrict__ img = static_cast<uint16_t*>(j.img);
    const int N = j.N, KW = j.KW, NL = j.NL, P = j.P;
    const int total = N * KW;
    for (int e = ((int)blockIdx.x - j.block0) * 256 + threadIdx.x; e < total; e += j.blocks * 256) {
        const int k = e / N, n = e - k * N;
        const int jj = k / NL, p = k - jj * NL;
        const float x = (n < j.n_valid && p < P) ? W[(size_t)n * j.ldw + jj * P + p] : 0.f;
        uint32_t hi, lo;
        umma::split_bf16x2(x, 0.f, hi, lo);
        const int ii = umma::b_image_index_f16(n, k, N);
        img[ii] = (uint16_t)(hi & 0xffffu);
        img[(size_t)N * KW + ii] = (uint16_t)(lo & 0xffffu);
    }
}

size_t img_bytes(long long M, int W) { return (size_t)((M + 127) / 128) * 2 * W * 256; }
size_t w_image_bytes(int N, int KW) { return (size_t)2 * N * KW * 2; }

int pack_w_images(cudaStream_t st, const PackWJob* jobs, int n) {
    ZF_REQUIRE(jobs && n >= 1 && n <= kMaxPackW, "pack_w_images: bad job list");
    PackWBatch b{};
    b.n = n;
    int grid = 0;
    for (int i = 0; i < n; ++i) {
        b.job[i] = jobs[i];
        b.job[i].block0 = grid;
        b.job[i].blocks = std::max(1, std::min(148, (jobs[i].N * jobs[i].KW + 255) / 256));
        grid += b.job[i].blocks;
    }
    pack_w_images_kernel<<<grid, 256, 0, st>>>(b);
    count_launch();
    ZF_CUDA_CHECK(cudaGetLastError());
    return ZF_OK;
}


int launch_img_nt(cudaStream_t st, const void* X, int KW, const void* Wimg, int N, const float* G, int ldg, void* out_img,
                  float* out_f32, int ldo, int n_valid, long long M) {
    ZF_REQUIRE(KW % 16 == 0 && N % 16 == 0 && N >= 16 && N <= 128, "img_nt: bad shape");
    DeviceInfo di;
    if (int rc = get_device_info(&di)) return rc;
    const size_t smem = (size_t)NT_STAGES * NT_STAGE_BYTES + 256;
    if (int rc = smem_optin((const void*)img_nt_kernel, smem)) return rc;
    ImgNtArgs a{static_cast<const char*>(X), KW, static_cast<const char*>(Wimg), N, G, ldg, static_cast<char*>(out_img), out_f32, ldo, n_valid, M};
    const long long tiles = (M + 127) / 128;
    if (tiles == 0) return ZF_OK;
    img_nt_kernel<<<(unsigned)std::min<long long>(tiles, di.sm_count), IG_THREADS, smem, st>>>(a);
    count_launch();
    ZF_CUDA_CHECK(cudaGetLastError());
    return ZF_OK;
}

int launch_img_tn(cudaStream_t st, const void* A, const void* B, int WB, float* C, long long ldca, long long ldcb, int a_valid,
                  int b_valid, float* colsum, float* arow_sum, int arow_col, long long M) {
    ZF_REQUIRE(WB % 16 == 0 && WB >= 16, "img_tn: bad shape");
    DeviceInfo di;
    if (int rc = get_device_info(&di)) return rc;
    const size_t smem = (size_t)TN_SLOTS * TN_SLOT_BYTES + 4096 + 256;
    if (int rc = smem_optin((const void*)img_tn_kernel, smem)) return rc;
    const long long tiles = (M + 127) / 128;
    if (tiles == 0) return ZF_OK;
    const int NS = std::min(TN_NS, WB);
    const int slabs = (WB + NS - 1) / NS;
    const unsigned gx = (unsigned)std::max<long long>(1, std::min<long long>(tiles, di.sm_count / slabs));
    ImgTnArgs a{static_cast<const char*>(A), static_cast<const char*>(B), WB, C, ldca, ldcb, a_valid, b_valid, colsum, arow_sum, arow_col, tiles, NS};
    img_tn_kernel<<<dim3(gx, (unsigned)slabs), IG_THREADS, smem, st>>>(a);
    count_launch();
    ZF_CUDA_CHECK(cudaGetLastError());
    return ZF_OK;
}

}  // namespace zf
