// Shared host/device helpers: error reporting across the C ABI, mbarrier / bulk-async-copy
// PTX wrappers (sm_100a), device properties cache.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>

#include "../../include/zenflow_b200.h"

namespace zf {

// ---- error plumbing (never throw across the ABI; include/zenflow_b200.h) -------------
void set_error(const char* fmt, ...);
int fail(int code, const char* fmt, ...);

#define ZF_CUDA_CHECK(expr)                                                              \
    do {                                                                                 \
        cudaError_t _e = (expr);                                                         \
        if (_e != cudaSuccess)                                                           \
            return zf::fail(ZF_ERR_CUDA, "%s failed: %s (%s:%d)", #expr,                 \
                            cudaGetErrorString(_e), __FILE__, __LINE__);                 \
    } while (0)

#define ZF_REQUIRE(cond, ...)                                       \
    do {                                                            \
        if (!(cond)) return zf::fail(ZF_ERR_INVALID, __VA_ARGS__);  \
    } while (0)

struct DeviceInfo {
    int device;
    int sm_count;
    int max_smem_optin;
    int cc_major, cc_minor;
};
// Cached per device (once-per-device init is the only global mutable state).
int get_device_info(DeviceInfo* out);

// Opt kernel `fn` in to `bytes` of dynamic shared memory on the current device.  The attribute is per device, so the
// largest value set is remembered per (function, device) and only a larger request calls the runtime again.
int smem_optin(const void* fn, size_t bytes);

// Adds one to the launch counter of zf_launch_count.
void count_launch();

// Developer switches, for tests and measurements that compare implementations (zf_chain.cu):
//   chain  "" automatic | "simt" FFMA chain_kernel | "umma" tensor-core kernel or an error | "umma8" single-tile
//          tensor-core kernel for single-dim flows too (choose_chain_kernel)
//   gemm   "" automatic | "simt" FFMA gemm_kernel | "legacy" tcgen05 GEMM with register-path loaders, for every train
//          GEMM: the unfused coupling backward and the Deep-Set Phi (launch_gemm)
// The environment (ZF_CHAIN_IMPL, ZF_GEMM_IMPL) is read once per process; zf_debug_set_impl overrides it afterwards.
struct ImplSwitch {
    char chain[16];
    char gemm[16];
};
ImplSwitch& impl_switch();

// ---- entry points shared between translation units -------------------------------------

// One product of the train step's fp32 GEMM family (zf_gemm.cu; the modes are described there).
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
    long long r_slab;    // mode 2, FFMA kernel only: reduction rows per CTA; the tcgen05 kernels choose their own slabs
};
// Runs one product; the only place that chooses between the three GEMM kernels (the table is at its definition).
int launch_gemm(cudaStream_t st, int mode, const GemmArgs& g);

// Fused conditioner recompute + spline VJP of one coupling (zf_chain.cu), of its forward or (inverse) of its inverse.
// ws_floats is 0 when the coupling or the device does not take the fused kernel.
size_t coupling_vjp_ws_floats(const zf_coupling* cp, int D, int C);
int coupling_vjp_pack(cudaStream_t stream, const zf_coupling* cp, int D, int C, float* ws);
int coupling_vjp_run(cudaStream_t stream, const zf_coupling* cp, int D, int C, const float* ws, const float* x_in, const float* c,
                     const float* gy, int gy_rot, const float* glp, long long M, float* gx, void* img_h0, int wh0, void* const* img_act,
                     float* const* act_g, void* img_dtheta, bool inverse);

// zf_coupling_backward (zf_train.cu) for either direction.  inverse = false: the VJP of the coupling's forward, as the
// public entry.  inverse = true: the VJP of NeuralSplineCoupling.inverse (bijectors.py:367-371) with x_in its input (the
// forward's output), gy the cotangent of its output read at column (j + gy_rot) % D, glp the cotangent of the inverse's
// log|dx/dy| per event or NULL (Flow.sample_and_log_prob's VJP passes one, Flow.inverse's does not); gx is the
// cotangent of x_in.  The BatchNorm running statistics are constants either way (the inverse is always eval-mode).
int coupling_backward(cudaStream_t st, const zf_coupling* cp, const zf_coupling_grads* gr, int D, int C, const float* x_in,
                      const float* c, const float* gy, int gy_rot, const float* glp, long long M, float* gx, float* gh0,
                      double* bn_sums, void* workspace, size_t workspace_bytes, long long micro_batch, bool inverse);

// One weight image of pack_w_images (zf_img_gemm.cu): Wimg(n, k) = W[n * ldw + (k / NL) * P + k % NL] for n < n_valid and
// k % NL < P, else 0, as the bf16x2 hi | lo operand image of img_nt_kernel.  block0 / blocks are filled by the launcher.
struct PackWJob {
    const float* W;
    void* img;
    int ldw, n_valid, N, KW, P, NL;
    int block0, blocks;
};

// Dense VJPs on event-row images (zf_img_gemm.cu).
size_t img_bytes(long long M, int W);
size_t w_image_bytes(int N, int KW);
int pack_w_images(cudaStream_t st, const PackWJob* jobs, int n);
int launch_img_nt(cudaStream_t st, const void* X, int KW, const void* Wimg, int N, const float* G, int ldg, void* out_img,
                  float* out_f32, int ldo, int n_valid, long long M);
int launch_img_tn(cudaStream_t st, const void* A, const void* B, int WB, float* C, long long ldca, long long ldcb, int a_valid,
                  int b_valid, float* colsum, float* arow_sum, int arow_col, long long M);

// In-place all-reduce over the data-parallel ranks of `comm` (zf_dp.cu); op 0 = sum, 1 = min.  A null comm is a no-op.
int dp_allreduce(cudaStream_t st, void* comm, void* buf, long long n, int is_f64, int op);

// Eval-mode pieces of the step loop (zf_train.cu, sequenced by zf_step.cu).
// zf_flow_loss_grad_ct; zero_dead = 1 also zeroes gz on rows whose cotangent is 0 (nan_to_num rows), where the latent's
// derivative may be infinite: eval batches may hold events outside the running ShiftBounds range.
int flow_loss_grad(cudaStream_t st, int latent_kind, float peakness, const float* z, const float* log_det, long long M, int D,
                   double global_count, const float* lp_cotangent, float* lp, float* gz, float* glp, double* lp_sum,
                   int zero_dead);
// Eval-mode BatchNorm VJP into its inputs (running statistics are constants): gx[:, D/2 + f] += dh_f,
// gc[:, f - (D - D/2)] += dh_f, dh = gh0 * scale * rstd(cp->bn_var).
int bn_backward_eval(cudaStream_t st, const zf_coupling* cp, int D, int C, const float* gh0, long long M, float* gx, float* gc);
// Eval-mode ShiftBounds VJP: gx (M, D) = d/dx of the ShiftBounds output (cotangent gz, column i read at (i + gz_rot) % D)
// and of its log-det (cotangent glp), with the running sb->xmin / sb->xmax.
int shift_bounds_backward(cudaStream_t st, const zf_shift_bounds* sb, int D, const float* x, const float* gz, int gz_rot,
                          const float* glp, long long M, float* gx);
// VJP of ShiftBounds.inverse (bijectors.py:210-240) with the running sb->xmin / sb->xmax: gz (M, D) = d/dz for the
// cotangent gx of its output x.  dx/dz is b - a (both bounds), xmax - xmin (running statistics), exp(t) (xmax - xmin)
// (lower bound) or -exp(t) (xmax - xmin) (upper bound), t = z xmax + (1 - z) xmin.  glp (or NULL) is the cotangent of
// the inverse's log-det (log(b - a), log(xmax - xmin), + t on one-sided columns).
int shift_bounds_inverse_backward(cudaStream_t st, const zf_shift_bounds* sb, int D, const float* z, const float* gx,
                                  const float* glp, long long M, float* gz);
// Flow.sample_and_log_prob's VJP (zf_train.cu).  glp = the cotangent of the chain's inverse log-det, -lp_cotangent, or 0 on
// rows whose lp (the nan_to_num'ed output) was not finite.  latent_score_acc: gz -= glp * d log p_latent / dz, the latent
// term of lp = sum_j log p(z_j) - log|det dx/dz| (rows with glp = 0 are left alone: the score may be infinite there).
int inverse_lp_cotangent(cudaStream_t st, const float* lp, const float* lp_cotangent, long long M, float* glp);
int latent_score_acc(cudaStream_t st, int latent_kind, float peakness, const float* z, const float* glp, long long M, int D,
                     float* gz);

// ---- PTX wrappers ----------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "ZF_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra ZF_DONE;\n"
        "bra ZF_WAIT;\n"
        "ZF_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// 1-D bulk async copy global -> shared (TMA engine, SASS UBLKCP); 16-byte aligned, size % 16 == 0.
__device__ __forceinline__ void bulk_copy_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes,
                                              uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::
            "r"(smem_u32(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}
// Order generic-proxy shared-memory accesses before later async-proxy (bulk copy) writes.
__device__ __forceinline__ void fence_proxy_async_smem() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

__device__ __forceinline__ void cp_async_16(void* dst_smem, const void* src_gmem) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst_smem)), "l"(src_gmem)
                 : "memory");
}
__device__ __forceinline__ void cp_async_4(void* dst_smem, const void* src_gmem) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(dst_smem)), "l"(src_gmem) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

__device__ __forceinline__ float ld_stream(const float* p) {
    float v;
    asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
    return v;
}

}  // namespace zf
