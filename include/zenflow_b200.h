/* zenflow_b200 — C ABI of the B200-native spline-coupling hot path.
 *
 * The reference (HDembinski/zenflow) is pure Python/JAX and has no FFI of its own; this
 * header is the boundary a `jax.ffi` / XLA custom-call adapter (or the ctypes host layer
 * in zenflow_b200/_lib.py) binds.  Every entry point names the reference function it
 * replaces (paths relative to the reference's src/zenflow/).
 *
 * Conventions
 *  - plain C: pointers, sizes and small POD structs; no C++/torch/XLA types;
 *  - `stream` is a cudaStream_t passed as void*; work is only enqueued on it, the
 *    library never synchronises, allocates, frees or retains device pointers;
 *  - all tensors are DEVICE pointers, fp32 row-major unless stated; descriptor structs
 *    (zf_chain, zf_op, zf_coupling, zf_shift_bounds) live in HOST memory and hold
 *    device pointers to the unmodified FLAX variable leaves;
 *  - scratch is supplied by the caller (`workspace`), sized by zf_*_workspace_bytes;
 *  - return value: ZF_OK (0) or a zf_status error; zf_last_error() returns a
 *    thread-local message.  Nothing throws across the ABI;
 *  - entry points are re-entrant; the only global state is a per-device cache of
 *    device attributes and cudaFuncSetAttribute calls.
 */
#ifndef ZENFLOW_B200_H
#define ZENFLOW_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ZF_ABI_VERSION 3
#define ZF_MAX_LAYERS 8   /* hidden layers per conditioner */
#define ZF_MAX_DIM 64     /* columns of x */

typedef enum zf_status {
    ZF_OK = 0,
    ZF_ERR_INVALID = 1,      /* bad argument (shape, null pointer, alignment)            */
    ZF_ERR_UNSUPPORTED = 2,  /* valid but outside what the kernels are built for         */
    ZF_ERR_CUDA = 3,         /* a CUDA runtime call failed; message has the CUDA error   */
    ZF_ERR_WORKSPACE = 4     /* workspace too small                                       */
} zf_status;

typedef enum zf_op_kind { ZF_OP_SHIFT_BOUNDS = 0, ZF_OP_ROLL = 1, ZF_OP_COUPLING = 2 } zf_op_kind;

/* distributions.py:50-126 */
typedef enum zf_latent_kind {
    ZF_LATENT_BETA = 0,       /* Beta(peakness, peakness), distributions.py:81-116 */
    ZF_LATENT_NORMAL = 1,     /* Normal(0.5, 0.1),         distributions.py:50-62  */
    ZF_LATENT_TRUNCNORMAL = 2,/* truncnorm(-5,5,0.5,0.1),  distributions.py:65-78  */
    ZF_LATENT_UNIFORM = 3     /* Uniform(0,1),             distributions.py:119-126 */
} zf_latent_kind;

/* ShiftBounds column treatment, bijectors.py:183-205 */
typedef enum zf_bound_kind {
    ZF_BOUND_NONE = 0,   /* unit-interval map from running min/max            */
    ZF_BOUND_BOTH = 1,   /* (x-a)/(b-a)                                         */
    ZF_BOUND_LOWER = 2,  /* t = log(x-a+tiny), then unit-interval map of t     */
    ZF_BOUND_UPPER = 3   /* t = log(b-x+tiny), then unit-interval map of t     */
} zf_bound_kind;

/* bijectors.py:132-273 ShiftBounds.  xmin/xmax: DEVICE arrays of `dim` floats packing the
 * batch_stats leaves xmin_i/xmax_i (entries of ZF_BOUND_BOTH columns are ignored). */
typedef struct zf_shift_bounds {
    int32_t kind[ZF_MAX_DIM];
    double lo[ZF_MAX_DIM];   /* a (Python double in the reference, bijectors.py:185-192) */
    double hi[ZF_MAX_DIM];   /* b */
    double margin;
    float* xmin;
    float* xmax;
} zf_shift_bounds;

/* bijectors.py:319 NeuralSplineCoupling.act: the conditioner's activation (jax.nn definitions; gelu is the tanh
 * form, jax's default).  ZF_ACT_SWISH (the reference default, = 0 so a zeroed struct keeps it) runs on the
 * tensor-core kernels; the others take the fp32 FFMA kernels (eval and train). */
typedef enum zf_act_kind {
    ZF_ACT_SWISH = 0,
    ZF_ACT_RELU = 1,
    ZF_ACT_TANH = 2,
    ZF_ACT_SIGMOID = 3,
    ZF_ACT_GELU = 4,
    ZF_ACT_ELU = 5,
    ZF_ACT_SOFTPLUS = 6,
    ZF_ACT_LEAKY_RELU = 7
} zf_act_kind;

/* bijectors.py:300-371 NeuralSplineCoupling.  Leaves exactly as FLAX stores them:
 * BatchNorm_0 scale/bias (params), mean/var (batch_stats), all (F,), F = dim - dim/2 + cdim;
 * Dense_j kernel (in,out) row-major and bias (out,), j = 0..n_hidden (the last one has
 * out = (dim/2)*(3*knots-1), column index = j_dim*(3*knots-1) + p, bijectors.py:346-347). */
typedef struct zf_coupling {
    int32_t knots;
    int32_t n_hidden;
    int32_t hidden[ZF_MAX_LAYERS];
    const float* bn_scale;
    const float* bn_bias;
    float* bn_mean;
    float* bn_var;
    const float* kernel[ZF_MAX_LAYERS + 1];
    const float* bias[ZF_MAX_LAYERS + 1];
    int32_t act;   /* zf_act_kind, bijectors.py:319,345 */
} zf_coupling;

typedef struct zf_op {
    int32_t kind;   /* zf_op_kind */
    int32_t shift;  /* ZF_OP_ROLL: jnp.roll shift, bijectors.py:286-297 */
    const zf_shift_bounds* shift_bounds;
    const zf_coupling* coupling;
} zf_op;

/* bijectors.py:90-124 Chain (a single bijector is a chain of one op). */
typedef struct zf_chain {
    int32_t dim;    /* D, columns of x                      */
    int32_t cdim;   /* C, columns of c (0: unconditional)   */
    int32_t n_ops;
    const zf_op* ops;
} zf_chain;

int32_t zf_abi_version(void);
const char* zf_last_error(void);
/* Number of kernels this library has launched on the calling thread (bench bookkeeping). */
int64_t zf_launch_count(void);
/* A host that replays a captured CUDA graph of calls into this library adds the graph's kernel count here. */
void zf_launch_count_add(int64_t n);

/* ---- spline stage on raw conditioner output --------------------------------------------
 * theta (M, d, 3K-1): raw widths | heights | slopes per transformed dim (bijectors.py:347-355).
 * Replaces utils.py:37-62 normalize_spline_params + :65-141 rational_quadratic_spline_forward
 * (+ :205-250 _compute_rqs_input/_knots/_index).  x, y (M, d); log_det (M,);
 * idx (M, d) int32 bin indices in [0, K] (may be NULL). */
int zf_rqs_forward(void* stream, const float* theta, const float* x, int64_t M, int32_t d,
                   int32_t K, float* y, float* log_det, int32_t* idx);
/* utils.py:144-202 rational_quadratic_spline_inverse on raw theta (bins searched in yk). */
int zf_rqs_inverse(void* stream, const float* theta, const float* y, int64_t M, int32_t d,
                   int32_t K, float* x, int32_t* idx);

/* ---- the reference's L0 functions on NORMALISED parameters (zenflow/utils.py public surface) ----------------
 * The hot path fuses the normalisation into the spline kernels (zf_rqs_forward above); these are the drop-ins for
 * code written against zenflow.utils.  dx, dy (M, d, K) bin widths / heights, slope (M, d, K-1) knot derivatives. */
/* utils.py:18-20 squareplus, elementwise. */
int zf_squareplus(void* stream, const float* x, int64_t n, float* y);
/* utils.py:37-62 normalize_spline_params on rows of raw theta (rows, 3K-1) = widths | heights | slopes. */
int zf_normalize_spline_params(void* stream, const float* theta, int64_t rows, int32_t K, float* dx, float* dy,
                               float* slope);
/* utils.py:65-141 rational_quadratic_spline_forward: y (M, d), log_det (M,) (may be NULL), idx (M, d) (may be NULL). */
int zf_rqs_forward_normalized(void* stream, const float* x, const float* dx, const float* dy, const float* slope,
                              int64_t M, int32_t d, int32_t K, float* y, float* log_det, int32_t* idx);
/* utils.py:144-202 rational_quadratic_spline_inverse (bins searched in the y knots). */
int zf_rqs_inverse_normalized(void* stream, const float* y, const float* dx, const float* dy, const float* slope,
                              int64_t M, int32_t d, int32_t K, float* x, int32_t* idx);

/* Developer switch (parity tests): force a chain kernel ("simt", "umma", "umma8"; NULL / "" = automatic) and a train
 * GEMM ("simt" = the fp32 FFMA GEMM; "legacy" = the tcgen05 GEMM with register-path loaders for every shape; NULL / "" =
 * tcgen05, fed by the copy engine where the operands allow tensor maps).  The GEMM switch applies to every Dense layer
 * the fused VJP kernel does not take, and to the Deep-Set Phi's.  The ZF_CHAIN_IMPL / ZF_GEMM_IMPL environment
 * variables give the initial values and are read once per process. */
int zf_debug_set_impl(const char* chain_impl, const char* gemm_impl);

/* Exhaustive device self-test of the exact-arithmetic fast paths the bin search relies on
 * (zf_math.cuh): mismatches[0] = sqrt fast path vs sqrt.rn over every float in [2^-100, 2^100],
 * [1] = squareplus fast vs IEEE over |x| < 2^40, [2] = reciprocal-form division vs div.rn.
 * mismatches: DEVICE array of 3 uint64; all must be 0. */
int zf_selftest_exact_math(void* stream, uint64_t* mismatches);

/* Self-test of the tcgen05 building blocks (3xTF32 split GEMM, A in tensor memory, B image in
 * shared memory): out (128, N) = A (128, K) * B (N, K)^T, N % 16 == 0 <= 128, K % 8 == 0 <= 128. */
int zf_selftest_umma(void* stream, const float* A, const float* B, int32_t N, int32_t K, float* out,
                     int32_t mask_mode /* 0: all lanes; 1: lanes 64-127 keep a 777 sentinel; 2: lanes 0-63 do */);

/* The same product with the 3xFP16 split on kind::f16 (A as fp16 pairs in tensor memory, separate cross accumulator
 * at scale 2^11), N % 16 == 0 <= 128, K % 16 == 0 <= 128.  variant 0 is the product layout; bit 0 swaps the halves of
 * every A word (layout probe), bit 1 drops the cross products (plain fp16). */
int zf_selftest_umma_f16(void* stream, const float* A, const float* B, int32_t N, int32_t K, float* out, int32_t variant);
/* the same product with the bf16 x 2 split and both operands in shared memory (the train step's image GEMMs,
 * csrc/zf_img_gemm.cu); flags bit 0 / 1: A / B stored MN-major, bit 2: descriptor-field probe (developer) */
int zf_selftest_umma_bf16(void* stream, const float* A, const float* B, int32_t N, int32_t K, float* out, int32_t flags);

/* Self-test of the train step's GEMM family through the train step's own dispatcher (activation swish), fp32 in/out;
 * the GEMM switch of zf_debug_set_impl selects which of the three GEMMs runs:
 * mode 0: C[I][J] = opA(A[I][R]) B[R][J] + bias; mode 1: C[I][J] = (A[I][R] B[J][R]^T) * swish'(Z[I][J]);
 * mode 2: C[I][J] += opA(A[R][I])^T B[R][J], colsum[J] += column sums of B (r_slab rows per CTA of the FFMA GEMM;
 * the tcgen05 GEMM sizes its own slabs). */
int zf_selftest_umma_gemm(void* stream, int32_t mode, const float* A, int64_t lda, const float* B, int64_t ldb,
                          float* C, int64_t ldc, const float* bias, float* colsum, const float* Z, int64_t ldz,
                          int32_t a_swish, int64_t I, int64_t J, int64_t R, int64_t r_slab);

/* ---- whole-chain eval passes -------------------------------------------------------------
 * One fused pass per call: ShiftBounds, conditioner MLP (eval-mode BatchNorm), spline,
 * Roll (as column renaming) and, for log_prob, the latent log-pdf + nan_to_num. */
size_t zf_chain_workspace_bytes(const zf_chain* chain, int64_t M);

/* Chain.__call__(x, c, train=False), bijectors.py:104-111.  y (M,D) and/or log_det (M,)
 * may be NULL.  c is (M,C) or NULL when cdim == 0. */
int zf_chain_forward(void* stream, const zf_chain* chain, const float* x, const float* c, int64_t M,
                     float* y, float* log_det, void* workspace, size_t workspace_bytes);
/* Parity evidence (SURVEY.md H3): the bin index (utils.py:244-250 _index, in [0, K]) of every spline evaluation of
 * Chain.__call__(x, c): idx (M, n_couplings, D/2) int32, coupling-major in op order.  Same kernels, same
 * arithmetic as zf_chain_forward; nothing else is written. */
int zf_chain_bin_indices(void* stream, const zf_chain* chain, const float* x, const float* c, int64_t M,
                         int32_t* idx, void* workspace, size_t workspace_bytes);
/* Chain.inverse(z, c), bijectors.py:113-116. */
int zf_chain_inverse(void* stream, const zf_chain* chain, const float* z, const float* c, int64_t M,
                     float* x, void* workspace, size_t workspace_bytes);
/* Flow.__call__(x, c, train=False), flow.py:22-48: latent.log_prob(bijector(x)) + log_det,
 * nan_to_num(nan=-inf). */
int zf_flow_log_prob(void* stream, const zf_chain* chain, int32_t latent_kind, float peakness,
                     const float* x, const float* c, int64_t M, float* log_prob, void* workspace,
                     size_t workspace_bytes);

/* Flow.sample(size | conditions, seed), flow.py:50-78: the latent draw (distributions.py samplers;
 * counter-based Philox streams keyed by (seed, event, column), see zf_rng.cuh) happens inside the
 * inverse chain kernel's tile load, then bijector.inverse.  x (M,D) out; c (M,C) or NULL. */
int zf_flow_sample(void* stream, const zf_chain* chain, int32_t latent_kind, float peakness, uint64_t seed,
                   const float* c, int64_t M, float* x, void* workspace, size_t workspace_bytes);

/* Flow.sample_and_log_prob / Flow.inverse_and_log_prob: a draw and its log-density in ONE inverse pass.
 *   x  = Chain.inverse(z, c), bit-identical to zf_chain_inverse (z given) / zf_flow_sample (z NULL: drawn in-kernel
 *        from (latent_kind, peakness, seed) exactly as zf_flow_sample draws it)
 *   lp = nan_to_num(sum_j log p_latent(z_j) - log|det dx/dz|), nan_to_num as zf_flow_log_prob's
 * log|det dx/dz| is the exact change of variables of the inverse as bijectors.py / utils.py write it: per transformed
 * element, log|dx/dy| of the analytic quadratic-root inverse (utils.py:191-201: no EPS, no clip) in the bin the inverse
 * searched; ShiftBounds.inverse adds log(b - a) (two-sided column), log(xmax - xmin) (unbounded) or
 * u + log(xmax - xmin) (one-sided: x = a + e^u or b - e^u); Roll and elements outside [0, 1) add 0.  This is the
 * density of the map that produced x, not zf_flow_log_prob(x): that one differs by the forward's EPS terms and clip
 * and by bin flips near knots.  The idx == K corner gives NaN x (as zf_chain_inverse) and lp = -FLT_MAX.
 *   x (M,D)     optional output (NULL: lp only); log_prob (M,) required; same workspace as zf_chain_inverse */
int zf_flow_sample_log_prob(void* stream, const zf_chain* chain, int32_t latent_kind, float peakness, uint64_t seed,
                            const float* z, const float* c, int64_t M, float* x, float* log_prob, void* workspace,
                            size_t workspace_bytes);

/* The same passes with the per-call parameter re-layout hoisted out: zf_chain_pack writes the packed parameter
 * blocks of `chain` into `workspace` once (after every parameter / statistics update); the *_packed calls then
 * only launch the fused kernel.  `chain` must describe the same ops and the same workspace must be passed. */
int zf_chain_pack(void* stream, const zf_chain* chain, void* workspace, size_t workspace_bytes);
int zf_chain_forward_packed(void* stream, const zf_chain* chain, const float* x, const float* c, int64_t M,
                            float* y, float* log_det, void* workspace, size_t workspace_bytes);
int zf_chain_inverse_packed(void* stream, const zf_chain* chain, const float* z, const float* c, int64_t M,
                            float* x, void* workspace, size_t workspace_bytes);
int zf_flow_log_prob_packed(void* stream, const zf_chain* chain, int32_t latent_kind, float peakness,
                            const float* x, const float* c, int64_t M, float* log_prob, void* workspace,
                            size_t workspace_bytes);
int zf_flow_sample_packed(void* stream, const zf_chain* chain, int32_t latent_kind, float peakness, uint64_t seed,
                          const float* c, int64_t M, float* x, void* workspace, size_t workspace_bytes);

/* Same as zf_chain_forward but log_det[m] += (this chain's log-det): Chain's running sum
 * (bijectors.py:107-110) when the train step applies the bijectors one phase at a time. */
int zf_chain_forward_acc(void* stream, const zf_chain* chain, const float* x, const float* c, int64_t M,
                         float* y, float* log_det, void* workspace, size_t workspace_bytes);

/* ---- train step phases (train.py:64-86: loss_fn, jax.grad, optimizer.update) -------------------
 * Train mode couples the samples of a batch (ShiftBounds batch min/max, BatchNorm batch moments),
 * so the step is a sequence of phases; a data-parallel host all-reduces the small statistics
 * between phases (SURVEY.md 8e).  Gradient buffers are ACCUMULATED into (+=): zero them first. */

/* Device pointers to the cotangents of a coupling's params, same shapes as in zf_coupling. */
typedef struct zf_coupling_grads {
    float* bn_scale;
    float* bn_bias;
    float* kernel[ZF_MAX_LAYERS + 1];
    float* bias[ZF_MAX_LAYERS + 1];
} zf_coupling_grads;

/* bijectors.py:250-252: per-column min and max of the (log-transformed, for one-sided bounds)
 * column over this rank's batch.  minmax: 2*D floats (min[D] then max[D]); scratch: 2*D uint32. */
int zf_shift_bounds_minmax(void* stream, const zf_shift_bounds* sb, const float* x, int64_t M, int32_t D,
                           float* minmax, void* scratch);
/* bijectors.py:253-260: widen by margin, merge into the running sb->xmin/xmax (in place). */
int zf_shift_bounds_update(void* stream, const zf_shift_bounds* sb, int32_t D, const float* minmax);

/* flax BatchNorm(use_running_average=False) (bijectors.py:342): sums[0..F) = sum of h,
 * sums[F..2F) = sum of h^2 over this rank's batch, h = hstack(x[:, D/2:], c), F = D - D/2 + C. */
int zf_bn_moments(void* stream, const float* x, const float* c, int64_t M, int32_t D, int32_t C, double* sums);
/* mean / biased variance (E[x^2]-E[x]^2, clipped at 0) from (all-reduced) sums and the global
 * count; running stats updated with `momentum` (flax default 0.99) when not NULL. */
int zf_bn_finalize(void* stream, const double* sums, double count, int32_t F, float momentum,
                   float* batch_mean, float* batch_var, float* ra_mean, float* ra_var);

/* flow.py:46-47 + train.py:73: lp = nan_to_num(latent.log_prob(z) + log_det); adds sum(lp) to
 * *lp_sum; cotangents of loss = -sum(lp)/global_count: glp (M,) for the log-dets and
 * gz (M,D) = glp * d latent/dz.  lp (M,) may be NULL. */
int zf_flow_loss_grad(void* stream, int32_t latent_kind, float peakness, const float* z, const float* log_det,
                      int64_t M, int32_t D, double global_count, float* lp, float* gz, float* glp, double* lp_sum);
/* The same with a caller-supplied cotangent of lp (M,), e.g. from a jax.custom_vjp backward rule; NULL = the
 * -1/global_count of loss = -mean(lp). */
int zf_flow_loss_grad_ct(void* stream, int32_t latent_kind, float peakness, const float* z, const float* log_det,
                         int64_t M, int32_t D, double global_count, const float* lp_cotangent, float* lp, float* gz,
                         float* glp, double* lp_sum);

/* VJP of NeuralSplineCoupling.__call__(train=True) (bijectors.py:329-365) except the BatchNorm
 * input path: recomputes the conditioner in micro-batches, then
 *   gx (M,D)   = d/dx_in through the spline (transformed columns) and the pass-through columns,
 *   gh0 (M,F)  = d/d(BatchNorm output),
 *   grads      += d/d(Dense kernels and biases)   (NULL: skipped, only the products toward the inputs run),
 *   bn_sums[0..F) = sum gh0, [F..2F) = sum gh0*xhat  (for BatchNorm's own VJP; NULL: skipped).
 * cp->bn_mean/bn_var must hold the statistics used in the forward (the BATCH statistics in train
 * mode, the running ones in eval mode).  gy is the cotangent of the coupling output; its column j
 * is read at (j + gy_rot) % D (folds the following Rolls). */
size_t zf_coupling_backward_workspace_bytes(const zf_coupling* cp, int32_t D, int32_t C, int64_t micro_batch);
int zf_coupling_backward(void* stream, const zf_coupling* cp, const zf_coupling_grads* grads, int32_t D, int32_t C,
                         const float* x_in, const float* c, const float* gy, int32_t gy_rot, const float* glp,
                         int64_t M, float* gx, float* gh0, double* bn_sums, void* workspace, size_t workspace_bytes,
                         int64_t micro_batch);
/* d/d(BatchNorm scale, bias) += (sum gh0*xhat, sum gh0) from this rank's bn_sums. */
int zf_bn_param_grads(void* stream, const double* bn_sums, int32_t F, float* g_scale, float* g_bias);
/* Train-mode BatchNorm VJP into its inputs with (all-reduced) bn_sums and the global count:
 * gx[:, D/2 + f] += dh_f for the x columns, gc[:, f - (D - D/2)] += dh_f for the conditions. */
int zf_bn_backward_apply(void* stream, const zf_coupling* cp, int32_t D, int32_t C, const float* x_in,
                         const float* c, const float* gh0, const double* bn_sums, double global_count, int64_t M,
                         float* gx, float* gc);

/* optax.nadamw / adamw (train.py:12-15,84-85) on flat buffers: scale_by_adam(b1,b2,eps,nesterov)
 * -> add_decayed_weights(weight_decay) -> scale(-lr).  count = number of updates done so far. */
int zf_nadamw_update(void* stream, int64_t n, float* params, const float* grads, float* mu, float* nu,
                     int64_t count, float lr, float b1, float b2, float eps, float weight_decay, int32_t nesterov);

/* The same update with the step counter in DEVICE memory: count_dev[0] = updates done so far, read for the bias
 * corrections and then incremented on the stream; bias_scratch: 3 device floats.  No argument changes from step to
 * step, so a CUDA graph captured around a whole train step (zf_flow_value_and_grad + this) can be replayed. */
int zf_nadamw_update_dev(void* stream, int64_t n, float* params, const float* grads, float* mu, float* nu,
                         int64_t* count_dev, float* bias_scratch, float lr, float b1, float b2, float eps,
                         float weight_decay, int32_t nesterov);

/* ---- train() epoch loop helpers (train.py:101-121) ----------------------------------------------
 * X_perm = X_train[perm] (train.py:104-108): out (N,D) = rows of x (N,D) in a pseudo-random order that
 * is a permutation of [0,N) fully determined by `seed` (fold the epoch into it); call with the same
 * seed for x and c to keep rows paired.  Out of place. */
int zf_permute_rows(void* stream, const float* x, int64_t N, int32_t D, uint64_t seed, float* out);
/* *out = -sum(lp[0..M)) in double (metric_fn / loss: divide by M, train.py:73,78). */
int zf_neg_sum(void* stream, const float* lp, int64_t M, double* out);

/* ---- data-parallel helpers (SURVEY.md 8e; the reference has no distributed code) ------------------------
 * The collectives between the train-step phases, issued with NCCL on the caller's stream.  `comm` is an
 * ncclComm_t (as void*); NULL means single device and every call is a no-op.  libnccl.so.2 is resolved at run
 * time (the copy already loaded into the process wins; ZF_NCCL_LIBRARY overrides). */
#define ZF_DP_UNIQUE_ID_BYTES 128
/* ncclGetUniqueId: id_out = ZF_DP_UNIQUE_ID_BYTES host bytes, to be broadcast to the other ranks by the host. */
int zf_dp_unique_id(void* id_out);
/* ncclCommInitRank on the calling thread's current device; *comm_out is the ncclComm_t. */
int zf_dp_comm_create(const void* id, int32_t rank, int32_t world, void** comm_out);
int zf_dp_comm_destroy(void* comm);
int zf_dp_comm_size(void* comm, int32_t* world_out);
/* In-place all-reduce(sum) of DEVICE buffers: BatchNorm moment sums (double) and gradients (float). */
int zf_dp_allreduce_sum_f32(void* stream, void* comm, float* buf, int64_t n);
int zf_dp_allreduce_sum_f64(void* stream, void* comm, double* buf, int64_t n);
/* ShiftBounds batch statistics (bijectors.py:250-252): minmax = min[D] | max[D]; ONE all-reduce(min) over
 * [min | -max]. */
int zf_dp_allreduce_minmax_f32(void* stream, void* comm, float* minmax, int32_t D);

/* ---- value and gradient of the train loss in one call (train.py:64-86: loss_fn + jax.grad) ---------------
 * loss = -sum(lp) / global_count over Flow.__call__(x, c, train=True) (or, with lp_cotangent, the VJP of lp for
 * a caller-supplied cotangent: the backward rule of a jax.custom_vjp around the flow).  Runs every phase of
 * the step on `stream`: per bijector the batch statistics (all-reduced over dp_comm when given), the fused
 * forward, then the loss cotangents and the backward of every coupling.
 *   chain        ops as for zf_chain_forward; the coupling's bn_mean / bn_var and the ShiftBounds' xmin / xmax are
 *                the RUNNING statistics ("batch_stats" collection) and are UPDATED IN PLACE (mutable=["batch_stats"],
 *                train.py:66-72).  Layout accepted: [ShiftBounds]? (NeuralSplineCoupling Roll*)+ (bijectors.py:418-423).
 *   grads        one zf_coupling_grads per coupling op, in op order; accumulated into (+=).  NULL: forward only
 *                (lp, lp_sum and the statistics updates: Flow.__call__(train=True), the fwd rule of a custom_vjp)
 *   lp (M,)      optional output; lp_sum: DEVICE double, += sum of lp over this rank's rows
 *   gc (M,C)     optional output: d loss / d c (the cotangent a Deep-Set conditioner upstream needs,
 *                examples/deep_set.ipynb:320-323); overwritten
 *   dp_comm      ncclComm_t or NULL.  With it the statistics are global and, when grad_flat is given, the
 *                gradient buckets grad_flat[bucket_off[k] .. bucket_off[k+1]) (coupling k in op order) are
 *                all-reduced as soon as coupling k's backward is queued: on aux_stream through dp_grad_comm when
 *                both are given (overlapping the next coupling's backward; `stream` waits for them before
 *                returning), else on `stream` through dp_comm. */
size_t zf_flow_value_and_grad_workspace_bytes(const zf_chain* chain, int64_t M, int64_t micro_batch);
int zf_flow_value_and_grad(void* stream, void* aux_stream, const zf_chain* chain, const zf_coupling_grads* grads,
                           int32_t latent_kind, float peakness, const float* x, const float* c, int64_t M,
                           double global_count, const float* lp_cotangent, float* lp, double* lp_sum, float* gc,
                           void* dp_comm, void* dp_grad_comm, float* grad_flat, const int64_t* bucket_off,
                           void* workspace, size_t workspace_bytes, int64_t micro_batch);

/* ---- VJP of the eval-mode log-density (flow.py:22-48: jax.grad of Flow.__call__(x, c, train=False)) -----------
 * The running statistics (the couplings' bn_mean / bn_var, the ShiftBounds' xmin / xmax) are read, never written.
 * Same plan and loop as zf_flow_value_and_grad without the statistics phases: the BatchNorm input VJP is the
 * diagonal one of fixed statistics, and the backward continues through a leading ShiftBounds into gx.
 *   chain         layout as for zf_flow_value_and_grad; a chain with no coupling ([ShiftBounds] Roll*) is accepted too
 *   grads         one zf_coupling_grads per coupling op, in op order; accumulated into (+=).  NULL: input cotangents
 *                 only (no grad-weight products, no BatchNorm parameter sums)
 *   lp_cotangent  (M,) required: the cotangent of lp (ones = per-event gradients of log p, the events being
 *                 independent in eval mode); events whose lp is not finite (nan_to_num) get zero gradients
 *   lp (M,)       optional output: the log-density as recomputed by this call
 *   gx (M,D), gc (M,C)  optional outputs, overwritten: d/dx and d/dc */
size_t zf_flow_log_prob_vjp_workspace_bytes(const zf_chain* chain, int64_t M, int64_t micro_batch);
int zf_flow_log_prob_vjp(void* stream, const zf_chain* chain, const zf_coupling_grads* grads, int32_t latent_kind,
                         float peakness, const float* x, const float* c, int64_t M, const float* lp_cotangent,
                         float* lp, float* gx, float* gc, void* workspace, size_t workspace_bytes, int64_t micro_batch);

/* ---- VJP of Chain.inverse (bijectors.py:113-116) and of Flow.sample's inverse pass (flow.py:76-77) --------------
 * What jax.grad through flow.apply(v, u, c, method="inverse") or method="sample" gives: the inverse is always eval-mode,
 * so the running statistics are read, never written.  Same plan and loop as zf_flow_log_prob_vjp in inverse mode: the
 * groups' inverses are recomputed last to first (one zf_chain_inverse per Roll run and per group), then the VJPs run first
 * to last; the spline's is that of the analytic inverse as written (utils.py:191-201: no EPS, no clip).
 *   chain         layout as for zf_flow_log_prob_vjp ([ShiftBounds]? (Coupling Roll*)*)
 *   z (M,D)       the inverse's input; NULL: sample it from (latent_kind, peakness, seed) exactly as zf_flow_sample does
 *   grads         as for zf_flow_log_prob_vjp (+=; NULL = input cotangents only)
 *   x_cotangent   (M,D) required: the cotangent of the inverse's output x
 *   x (M,D)       optional output: the inverse as recomputed by this call
 *   gz (M,D)      optional output, overwritten: d/dz; must be NULL when z is NULL (the latent draw is a constant)
 *   gc (M,C)      optional output, overwritten: d/dc */
size_t zf_chain_inverse_vjp_workspace_bytes(const zf_chain* chain, int64_t M, int64_t micro_batch);
int zf_chain_inverse_vjp(void* stream, const zf_chain* chain, const zf_coupling_grads* grads, const float* z,
                         int32_t latent_kind, float peakness, uint64_t seed, const float* c, int64_t M,
                         const float* x_cotangent, float* x, float* gz, float* gc,
                         void* workspace, size_t workspace_bytes, int64_t micro_batch);

/* ---- VJP of zf_flow_sample_log_prob: (x, lp) jointly ------------------------------------------------------------
 * zf_chain_inverse_vjp's plan and loop plus the log-density: every group's inverse log-det takes the per-event
 * cotangent -lp_cotangent, gz also takes lp_cotangent d log p_latent / dz, and events whose lp is not finite
 * (nan_to_num) take a zero lp cotangent (their x cotangent flows as in zf_chain_inverse_vjp).  Running statistics are
 * constants.  Validation and layout as zf_chain_inverse_vjp, except:
 *   x_cotangent (M,D) or NULL, lp_cotangent (M,) or NULL; not both NULL.  With lp_cotangent NULL the outputs are
 *                 bit-identical to zf_chain_inverse_vjp's
 *   lp (M,)       optional output: the log-density as zf_flow_sample_log_prob computes it
 *   workspace     zf_flow_sample_log_prob_vjp_workspace_bytes (the plan's, with room for the whole chain's pass) */
size_t zf_flow_sample_log_prob_vjp_workspace_bytes(const zf_chain* chain, int64_t M, int64_t micro_batch);
int zf_flow_sample_log_prob_vjp(void* stream, const zf_chain* chain, const zf_coupling_grads* grads, const float* z,
                                int32_t latent_kind, float peakness, uint64_t seed, const float* c, int64_t M,
                                const float* x_cotangent, const float* lp_cotangent, float* x, float* lp, float* gz,
                                float* gc, void* workspace, size_t workspace_bytes, int64_t micro_batch);

/* ---- Deep-Set conditioner Phi (examples/deep_set.ipynb:138-160; SURVEY.md 8f-4) ---------------------------
 * The FLAX module on the other side of the flow's conditions in the deep_set config:
 *   BatchNorm_0 -> NNBlock_0 = (Dense_l + swish) x n_hidden, Dense_{n_hidden} (out_dim) -> Dropout(rate) -> sum_matrix @ .
 * Leaves exactly as FLAX stores them (kernels (in, out) row-major); bn_mean / bn_var are the running statistics and
 * are updated in place by a train-mode forward.  The notebook's BCOO sum matrix of ones (deep_set.ipynb:60-74) is
 * passed as its COO index list: entry e adds row row_idx[e] of the embeddings to set set_idx[e]. */
typedef struct zf_phi {
    int32_t in_dim;    /* columns of x */
    int32_t out_dim;   /* columns of c */
    int32_t n_hidden;
    int32_t hidden[ZF_MAX_LAYERS];
    const float* bn_scale;
    const float* bn_bias;
    float* bn_mean;
    float* bn_var;
    const float* kernel[ZF_MAX_LAYERS + 1];
    const float* bias[ZF_MAX_LAYERS + 1];
} zf_phi;

size_t zf_phi_workspace_bytes(const zf_phi* phi, int64_t N);
/* Phi.__call__(x, sum_matrix, train): x (N, in_dim) -> c (S, out_dim).  train != 0: batch-moment BatchNorm (over all
 * N rows, padding included, as in the notebook), running statistics updated, dropout active; the layer
 * pre-activations stay in `workspace` for zf_phi_backward.  dropout_mask: optional (N, out_dim) multipliers
 * (0 or 1/(1-rate)); NULL draws the keep-mask from Philox keyed by (dropout_seed, row, column). */
int zf_phi_forward(void* stream, const zf_phi* phi, const float* x, int64_t N, const int32_t* set_idx,
                   const int32_t* row_idx, int64_t nnz, int64_t S, int32_t train, float dropout_rate,
                   uint64_t dropout_seed, const float* dropout_mask, float* c_out, void* workspace, size_t workspace_bytes);
/* VJP of the train-mode forward above wrt the parameters: grads (+=, same struct as a coupling's: BatchNorm scale /
 * bias, Dense kernels / biases) from gc (S, out_dim) = d loss / d c, e.g. zf_flow_value_and_grad's gc.  Must follow
 * the matching zf_phi_forward(train = 1) on the same workspace, with the same dropout arguments. */
int zf_phi_backward(void* stream, const zf_phi* phi, const zf_coupling_grads* grads, const float* x, int64_t N,
                    const int32_t* set_idx, const int32_t* row_idx, int64_t nnz, int64_t S, float dropout_rate,
                    uint64_t dropout_seed, const float* dropout_mask, const float* gc, void* workspace,
                    size_t workspace_bytes);

#ifdef __cplusplus
}
#endif
#endif /* ZENFLOW_B200_H */
