// Standalone spline stage: raw conditioner output theta (M, d, 3K-1) streamed once from HBM.
//
//   zf_rqs_forward  <- utils.py:37-62 normalize_spline_params + :65-141 rqs forward
//   zf_rqs_inverse  <- utils.py:144-202 rqs inverse
//
// HBM-bound by design (algorithmic bytes per sample: 4*(d*(3K-1) + 2d + 1) forward): theta
// tiles of R rows are pulled into a shared-memory ring with 1-D bulk async copies (TMA
// engine, mbarrier completion) while the previous tile is being evaluated, one thread per
// (sample, dim) row.  The row stride 3K-1 is odd for even K, so row-per-thread shared
// memory reads are bank-conflict free without padding.
#include "zf_common.cuh"
#include "zf_math.cuh"

namespace zf {

struct StageArgs {
    const float* theta;
    const float* v;
    float* out;
    float* log_det;
    int32_t* idx;
    long long n_rows;   // M*d
    int d, K, P;
    int R;              // rows per tile (multiple of 4 and of d)
    long long n_tiles;
    int stages;
    int use_bulk;
    KnotNorm kn;
};

constexpr int kStageThreads = 256;   // at most; 128 when that lets two blocks share an SM (see launch_stage)

template <int KT, bool INVERSE>
__global__ void __launch_bounds__(kStageThreads)
rqs_stage_kernel(const __grid_constant__ StageArgs a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int tid = threadIdx.x, nthr = blockDim.x;
    const int P = a.P, R = a.R, S = a.stages, d = a.d;
    const int tile_floats = R * P;  // R % 4 == 0 -> 16-byte multiple
    float* bufs = reinterpret_cast<float*>(smem_raw);
    // K = 16 / 32: per-thread scratch columns of the lean row ([K / 4][threads] float4)
    float4* scratch = reinterpret_cast<float4*>(bufs + (size_t)S * tile_floats);
    float* ldrow = reinterpret_cast<float*>(scratch + (KT > 0 ? (KT / 4) * nthr : 0));
    uint64_t* bars = reinterpret_cast<uint64_t*>(ldrow + ((R + 3) & ~3));

    if (tid == 0) {
        for (int s = 0; s < S; ++s) mbar_init(&bars[s], 1);
        mbar_fence_init();
    }
    __syncthreads();

    auto issue = [&](long long tile, int stage) {
        const long long row0 = tile * R;
        const long long rem = a.n_rows - row0;
        const int rows = rem < R ? (int)rem : R;
        const uint32_t bytes = (uint32_t)rows * P * 4u;
        if (a.use_bulk && (bytes & 15u) == 0u) {
            mbar_arrive_expect_tx(&bars[stage], bytes);
            bulk_copy_g2s(bufs + (size_t)stage * tile_floats, a.theta + row0 * P, bytes, &bars[stage]);
        }
    };

    if (tid == 0) {
        for (int s = 0; s < S; ++s) {
            long long t = (long long)blockIdx.x + (long long)s * gridDim.x;
            if (t < a.n_tiles) issue(t, s);
        }
    }

    int it = 0;
    for (long long tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x, ++it) {
        const int stage = it % S;
        const uint32_t parity = (uint32_t)(it / S) & 1u;
        const long long row0 = tile * R;
        const long long rem = a.n_rows - row0;
        const int rows = rem < R ? (int)rem : R;
        const uint32_t bytes = (uint32_t)rows * P * 4u;
        float* buf = bufs + (size_t)stage * tile_floats;

        // the element this thread transforms first (issued before waiting on the tile)
        float v0 = (tid < rows) ? a.v[row0 + tid] : 0.f;

        if (a.use_bulk && (bytes & 15u) == 0u) {
            mbar_wait(&bars[stage], parity);
        } else {  // ragged last tile or unaligned theta: cooperative coalesced load
            const float* src = a.theta + row0 * P;
            for (int i = tid; i < rows * P; i += nthr) buf[i] = ld_stream(src + i);
            __syncthreads();
        }

        // d a power of two up to 32: the d rows of a sample sit in d consecutive lanes (tiles and passes start at
        // multiples of d), their log-dets are summed with shuffles; otherwise through shared memory below
        const bool shfl_sum = !INVERSE && d > 1 && d <= 32 && (d & (d - 1)) == 0;
        for (int r0 = 0; r0 < rows; r0 += nthr) {
            const int r = r0 + tid;
            const bool active = r < rows;
            float ld = 0.f;
            if (active) {
                const float v = (r == tid) ? v0 : a.v[row0 + r];
                RqsBin b;
                if constexpr (KT > 0) rqs_locate_lean<KT>(buf + (size_t)r * P, !INVERSE, v, a.kn, b, scratch + tid, nthr);
                else rqs_locate<KT>(buf + (size_t)r * P, a.K, !INVERSE, v, a.kn, b);
                if (!INVERSE) {
                    float y;
                    rqs_eval_forward(v, b, y, ld);
                    a.out[row0 + r] = y;
                    if (d == 1) a.log_det[row0 + r] = ld;
                    else if (!shfl_sum) ldrow[r] = ld;
                } else {
                    a.out[row0 + r] = rqs_eval_inverse(v, b);
                }
                if (a.idx) a.idx[row0 + r] = b.idx;
            }
            if (shfl_sum) {
                for (int o = d >> 1; o > 0; o >>= 1) ld += __shfl_xor_sync(0xffffffffu, ld, o);
                if (active && (r & (d - 1)) == 0) a.log_det[(row0 + r) / d] = ld;
            }
        }

        if (!INVERSE && d > 1 && !shfl_sum) {  // log_det.sum(axis=1), utils.py:139
            __syncthreads();
            const int ns = rows / d;
            for (int s = tid; s < ns; s += nthr) {
                float acc = ldrow[s * d];
                for (int j = 1; j < d; ++j) acc += ldrow[s * d + j];
                a.log_det[row0 / d + s] = acc;
            }
        }

        fence_proxy_async_smem();
        __syncthreads();  // everyone is done with this stage's buffer (and with ldrow)
        if (tid == 0) {
            long long next = tile + (long long)S * gridDim.x;
            if (next < a.n_tiles) issue(next, stage);
        }
    }
}

template <bool INVERSE>
static int launch_stage(cudaStream_t stream, const float* theta, const float* v, long long M, int d,
                        int K, float* out, float* log_det, int32_t* idx) {
    if (M == 0) return ZF_OK;
    ZF_REQUIRE(M > 0 && d >= 1 && K >= 1, "rqs: need M >= 0, d >= 1, K >= 1 (M=%lld d=%d K=%d)", M, d, K);
    ZF_REQUIRE(theta && v && out, "rqs: null tensor pointer");
    ZF_REQUIRE(INVERSE || log_det, "rqs_forward: log_det must not be NULL");
    DeviceInfo di;
    if (int rc = get_device_info(&di)) return rc;

    StageArgs a{};
    a.theta = theta; a.v = v; a.out = out; a.log_det = log_det; a.idx = idx;
    a.d = d; a.K = K; a.P = 3 * K - 1;
    a.n_rows = M * d;
    a.kn = make_knot_norm(K);
    a.use_bulk = ((reinterpret_cast<uintptr_t>(theta) & 15u) == 0) ? 1 : 0;

    // tile: TS samples (multiple of 4 so that every full tile is a 16-byte multiple), about
    // one row per thread, at most ~96 KB so that two stages always fit.
    const size_t row_bytes = (size_t)a.P * 4;
    const size_t budget = (size_t)di.max_smem_optin;
    int threads = kStageThreads, blocks_per_sm = 1, stages = 1;
    size_t tile_bytes = 0, misc = 0;
    auto config = [&](int T) -> bool {   // false: not even one tile fits
        int TS = (T / d) & ~3;
        if (TS < 4) TS = 4;
        while (TS > 4 && (size_t)TS * d * row_bytes > 96 * 1024) TS -= 4;
        a.R = TS * d;
        threads = T;
        tile_bytes = (size_t)a.R * row_bytes;
        const size_t lean_scratch = (K == 16 || K == 32) ? (size_t)(K / 4) * T * 16 : 0;
        misc = (size_t)((a.R + 3) & ~3) * 4 + 8 * 8 + 128 + lean_scratch;
        if (tile_bytes + misc > budget) return false;
        // two resident blocks of two stages when tiles are small, else one block with up to 4 stages
        if (2 * (2 * tile_bytes + misc) + 2048 <= budget) { blocks_per_sm = 2; stages = 2; }
        else {
            blocks_per_sm = 1;
            stages = (int)((budget - misc) / tile_bytes);
            if (stages > 4) stages = 4;
            if (stages < 1) stages = 1;
        }
        return true;
    };
    if (!config(kStageThreads))
        return fail(ZF_ERR_UNSUPPORTED, "rqs: one tile of %d rows x %d params does not fit shared memory", a.R, a.P);
    // big rows (d = 8, K = 32: 97 KB tiles): two blocks of 128 threads keep four copies in flight per SM instead of two
    // and decouple the tiles' barriers
    if (blocks_per_sm == 1 && d <= kStageThreads / 2 / 4) {
        const int R0 = a.R, st0 = stages;
        const size_t tb0 = tile_bytes, misc0 = misc;
        if (!(config(kStageThreads / 2) && blocks_per_sm == 2)) { a.R = R0; threads = kStageThreads; blocks_per_sm = 1; stages = st0; tile_bytes = tb0; misc = misc0; }
    }
    a.stages = stages;
    a.n_tiles = (a.n_rows + a.R - 1) / a.R;
    const size_t smem = (size_t)stages * tile_bytes + misc;

    long long grid = (long long)di.sm_count * blocks_per_sm;
    if (grid > a.n_tiles) grid = a.n_tiles;

    auto run = [&](auto kernel) -> int {
        if (int rc = smem_optin((const void*)kernel, smem)) return rc;
        kernel<<<(unsigned)grid, threads, smem, stream>>>(a);
        count_launch();
        ZF_CUDA_CHECK(cudaGetLastError());
        return ZF_OK;
    };
    switch (K) {
        case 16: return run(rqs_stage_kernel<16, INVERSE>);
        case 32: return run(rqs_stage_kernel<32, INVERSE>);
        default: return run(rqs_stage_kernel<0, INVERSE>);
    }
}

}  // namespace zf

extern "C" int zf_rqs_forward(void* stream, const float* theta, const float* x, int64_t M, int32_t d,
                              int32_t K, float* y, float* log_det, int32_t* idx) {
    return zf::launch_stage<false>((cudaStream_t)stream, theta, x, (long long)M, d, K, y, log_det, idx);
}

extern "C" int zf_rqs_inverse(void* stream, const float* theta, const float* y, int64_t M, int32_t d,
                              int32_t K, float* x, int32_t* idx) {
    return zf::launch_stage<true>((cudaStream_t)stream, theta, y, (long long)M, d, K, x, nullptr, idx);
}

// ---- self-test of the exact-arithmetic fast paths -------------------------------------------
namespace zf {
__global__ void selftest_exact_math_kernel(unsigned long long* bad) {
    const unsigned long long gtid = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x;
    const unsigned long long gsz = (unsigned long long)gridDim.x * blockDim.x;
    unsigned long long bad_sqrt = 0, bad_div = 0, bad_sp = 0;
    // every float in [2^-100, 2^100]: sqrt_rn_normal == sqrt.rn
    for (unsigned long long b = 0x0d800000ull + gtid; b <= 0x71800000ull; b += gsz) {
        float a = __uint_as_float((unsigned)b);
        if (__float_as_uint(sqrt_rn_normal(a)) != __float_as_uint(__fsqrt_rn(a))) ++bad_sqrt;
    }
    // squareplus_fast == squareplus_rn on every float with |x| < 2^40 (both signs)
    for (unsigned long long b = gtid; b < 0x53800000ull; b += gsz) {
        float x = __uint_as_float((unsigned)b);
        if (__float_as_uint(squareplus_fast(x)) != __float_as_uint(squareplus_rn(x))) ++bad_sp;
        if (__float_as_uint(squareplus_fast(-x)) != __float_as_uint(squareplus_rn(-x))) ++bad_sp;
    }
    // Markstein division vs div.rn on pseudo-random (a <= b) pairs and the knot constants
    unsigned long long s = 0x9E3779B97F4A7C15ull * (gtid + 1);
    for (int it = 0; it < 4096; ++it) {
        s ^= s << 13; s ^= s >> 7; s ^= s << 17;
        unsigned mb = (unsigned)s & 0x7fffffu, eb = 110u + (unsigned)((s >> 23) % 40u);
        unsigned ma = (unsigned)(s >> 32) & 0x7fffffu, ea = eb - (unsigned)((s >> 56) % 60u);
        if ((it & 15) == 0) mb = 0x7fffffu - (it & 3u);
        float b = __uint_as_float((eb << 23) | mb), a = __uint_as_float((ea << 23) | ma);
        if (a > b) a = b;
        float q = div_rn_recip(a, b, __frcp_rn(b));
        if (fabsf(__fmul_rn(a, __frcp_rn(b))) > 7.9e-31f && __float_as_uint(q) != __float_as_uint(__fdiv_rn(a, b))) ++bad_div;
        KnotNorm kn = make_knot_norm(1 + (it & 63));
        float t = __uint_as_float(((117u + (unsigned)(s % 11u)) << 23) | ma);
        if (__float_as_uint(div_rn_recip(t, kn.den, kn.rden)) != __float_as_uint(__fdiv_rn(t, kn.den))) ++bad_div;
    }
    if (bad_sqrt) atomicAdd(&bad[0], bad_sqrt);
    if (bad_sp) atomicAdd(&bad[1], bad_sp);
    if (bad_div) atomicAdd(&bad[2], bad_div);
}
}  // namespace zf

extern "C" int zf_selftest_exact_math(void* stream, uint64_t* mismatches) {
    ZF_REQUIRE(mismatches != nullptr, "mismatches is NULL");
    ZF_CUDA_CHECK(cudaMemsetAsync(mismatches, 0, 3 * sizeof(uint64_t), (cudaStream_t)stream));
    zf::selftest_exact_math_kernel<<<148 * 8, 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<unsigned long long*>(mismatches));
    zf::count_launch();
    ZF_CUDA_CHECK(cudaGetLastError());
    return ZF_OK;
}
