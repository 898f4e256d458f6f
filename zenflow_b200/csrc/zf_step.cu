// zf_flow_value_and_grad: the whole `loss_fn` + `jax.grad` of train.py:64-86 as ONE C-ABI call, and
// zf_flow_log_prob_vjp: the VJP of Flow.__call__(x, c, train=False), flow.py:22-48 (what jax.grad of the eval-mode
// log-density gives: the score d/dx, d/dc and the parameter gradients with the running statistics held fixed).
//
// Train mode couples the events of a batch (ShiftBounds batch min/max, bijectors.py:250-260; BatchNorm batch
// moments, bijectors.py:342), so the step is a sequence of phases, each a kernel (or a few) of zf_train.cu /
// zf_chain.cu; here they are sequenced from C++ on the caller's stream, with the data-parallel exchanges
// (zf_dp.cu) in between, so that a host framework issues one call per step instead of ~170.
//   forward   per bijector group (a ShiftBounds or a coupling, plus the Rolls behind it):
//             statistics -> [all-reduce] -> finalize -> fused forward of the group into states[g]
//   loss      lp = nan_to_num(latent.log_prob(z) + log_det), cotangents of z and of the log-dets
//   backward  per coupling in reverse: recompute + spline VJP + Dense VJPs -> [all-reduce BatchNorm sums] ->
//             BatchNorm VJP into x and c; the coupling's gradient bucket is all-reduced behind it
// Eval mode runs the same plan and the same loop (run_step) with three differences: no statistics phase (the
// couplings and the ShiftBounds read their running statistics), the diagonal BatchNorm VJP instead of the
// batch-coupled one, and the backward continues through a leading ShiftBounds into d/dx.
//
// zf_chain_inverse_vjp: the VJP of Chain.inverse (bijectors.py:113-116) and of Flow.sample's inverse pass (flow.py:76-77),
// the inverse mode of the same plan and loop.  Chain.inverse walks the groups last to first, a group's inverse being its
// Rolls' inverses and then the coupling's (or the ShiftBounds') inverse, always with the running statistics:
//   forward   per group, last to first: u_g = Roll^-1(input) (zf_chain_inverse on the Rolls; in sample mode the first
//             pass draws the latent, zf_flow_sample), then the group's own inverse from u_g; u_g is kept
//   backward  per group, first to last (the cotangent travels from x toward z): the ShiftBounds' inverse VJP, or the
//             coupling's (conditioner recompute + spline-inverse VJP + Dense VJPs) and the diagonal BatchNorm VJP;
//             the cotangent of u_g reaches the next group's output through its Rolls by index arithmetic.
#include "zf_common.cuh"

#include <algorithm>
#include <vector>

namespace zf {

struct StepGroup {
    int kind;                 // ZF_OP_SHIFT_BOUNDS or ZF_OP_COUPLING
    int op_index;
    int coupling_index;       // ordinal among the couplings (for grads / buckets)
    int rot;                  // sum of the Roll shifts behind it
    std::vector<zf_op> ops;   // the group's sub-chain
};

// train: value_and_grad; eval: log_prob_vjp; inverse: chain_inverse_vjp
enum StepMode { kStepTrain, kStepEval, kStepInverse };

struct StepPlan {
    std::vector<StepGroup> groups;
    int n_couplings = 0;
    int Fmax = 1;
    // workspace carve-up in bytes
    size_t off_states = 0, off_ld = 0, off_glp = 0, off_ga = 0, off_gb = 0, off_gh0 = 0, off_stats = 0, off_chain = 0,
           off_bwd = 0, off_lp_sum = 0, off_xtmp = 0, total = 0;
    size_t stats_stride = 0, chain_bytes = 0, bwd_bytes = 0;
};

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// Per-coupling statistics block: bmean[F] bvar[F] (float) | fwd sums 2F (double) | bwd sums 2F (double);
// the ShiftBounds group uses the same block for minmax[2D] (float) | scratch[2D] (uint32).
// Eval mode uses only the bwd sums (parameter gradients of the BatchNorm) and adds a slot for the lp sum the loss
// kernel keeps; it also accepts a chain with no coupling, whose only derivative is d/dx through the ShiftBounds.
// Inverse mode uses the states for u_g, the input of group g's own inverse, and adds one (M, D) buffer for the outputs
// that are not states (x_g when group g-1 has Rolls, and x when the caller does not ask for it).
static int build_step_plan(const zf_chain* chain, long long M, long long micro_batch, StepMode mode, StepPlan& p) {
    const bool train = mode == kStepTrain;
    const char* who = train ? "value_and_grad" : mode == kStepEval ? "log_prob_vjp" : "chain_inverse_vjp";
    ZF_REQUIRE(chain && chain->n_ops >= 1 && chain->ops, "%s: empty chain", who);
    const int D = chain->dim, C = chain->cdim;
    ZF_REQUIRE(D >= (train ? 2 : 1) && D <= ZF_MAX_DIM, "%s: dim must be in [%d, %d]", who, train ? 2 : 1, ZF_MAX_DIM);
    ZF_REQUIRE(M >= 1 && micro_batch >= 1, "%s: bad batch", who);
    for (int i = 0; i < chain->n_ops; ++i) {
        const zf_op& op = chain->ops[i];
        if (op.kind == ZF_OP_ROLL) {
            if (p.groups.empty())
                return fail(ZF_ERR_UNSUPPORTED, "%s: a chain that starts with Roll is not supported", who);
            p.groups.back().ops.push_back(op);
            p.groups.back().rot += op.shift;
        } else if (op.kind == ZF_OP_SHIFT_BOUNDS) {
            if (!p.groups.empty())
                return fail(ZF_ERR_UNSUPPORTED, "%s: ShiftBounds after another bijector is not supported", who);
            ZF_REQUIRE(op.shift_bounds, "%s: op %d: shift_bounds is NULL", who, i);
            p.groups.push_back(StepGroup{ZF_OP_SHIFT_BOUNDS, i, -1, 0, {op}});
        } else if (op.kind == ZF_OP_COUPLING) {
            ZF_REQUIRE(op.coupling, "%s: op %d: coupling is NULL", who, i);
            p.groups.push_back(StepGroup{ZF_OP_COUPLING, i, p.n_couplings++, 0, {op}});
        } else {
            return fail(ZF_ERR_INVALID, "%s: op %d: unknown kind %d", who, i, op.kind);
        }
    }
    ZF_REQUIRE(!train || p.n_couplings >= 1, "value_and_grad: the chain has no coupling (nothing to differentiate)");
    const int F = D - D / 2 + C;
    p.Fmax = F;
    ZF_REQUIRE(F <= 256, "%s: at most 256 conditioner inputs", who);
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
    p.off_states = take(p.groups.size() * (size_t)M * D * 4);
    p.off_ld = take((size_t)M * 4);
    p.off_glp = take((size_t)M * 4);
    p.off_ga = take((size_t)M * D * 4);
    p.off_gb = take((size_t)M * D * 4);
    p.off_gh0 = take((size_t)M * F * 4);
    p.stats_stride = align_up(std::max<size_t>((size_t)2 * F * 4 + (size_t)4 * F * 8, (size_t)4 * D * 4), 256);
    p.off_stats = take(p.groups.size() * p.stats_stride);
    const long long mb = std::min<long long>(micro_batch, M);
    for (const StepGroup& g : p.groups) {
        zf_chain sub{D, C, (int32_t)g.ops.size(), g.ops.data()};
        const size_t cb = zf_chain_workspace_bytes(&sub, M);
        if (cb == 0) return ZF_ERR_INVALID;   // message set by the plan builder
        p.chain_bytes = std::max(p.chain_bytes, cb);
        if (g.kind == ZF_OP_COUPLING)
            p.bwd_bytes = std::max(p.bwd_bytes, zf_coupling_backward_workspace_bytes(g.ops[0].coupling, D, C, mb));
    }
    p.off_chain = take(p.chain_bytes);
    p.off_bwd = take(p.bwd_bytes);
    if (mode == kStepEval) p.off_lp_sum = take(sizeof(double));
    if (mode == kStepInverse) p.off_xtmp = take((size_t)M * D * 4);
    p.total = off;
    return ZF_OK;
}

struct AuxEvents {
    cudaEvent_t main_done = nullptr, aux_done = nullptr;
    int device = -1;
};
static int aux_events(AuxEvents** out) {
    static thread_local AuxEvents ev;
    int dev = 0;
    ZF_CUDA_CHECK(cudaGetDevice(&dev));
    if (ev.device != dev) {
        ZF_CUDA_CHECK(cudaEventCreateWithFlags(&ev.main_done, cudaEventDisableTiming));
        ZF_CUDA_CHECK(cudaEventCreateWithFlags(&ev.aux_done, cudaEventDisableTiming));
        ev.device = dev;
    }
    *out = &ev;
    return ZF_OK;
}

// The arguments of the three entry points.  Train-only fields (global_count, lp_sum, the communicators and buckets) are
// unused in eval mode; gx (d/dx) is eval-only.  Inverse mode reads x as z (NULL: sample with latent_kind, peakness, seed),
// x_ct as the cotangent of its output, writes x_out (optional) and gz (optional), and uses none of the loss fields.
struct StepCall {
    StepMode mode;
    cudaStream_t st, aux;
    const zf_chain* chain;
    const zf_coupling_grads* grads;
    int latent_kind;
    float peakness;
    const float* x;
    const float* c;
    long long M;
    double global_count;
    const float* lp_cotangent;
    float* lp;
    double* lp_sum;
    float* gx;
    float* gc;
    void* dp_comm;
    void* dp_grad_comm;
    float* grad_flat;
    const int64_t* bucket_off;
    char* ws;
    long long micro_batch;
    const float* x_ct;
    float* x_out;
    float* gz;
    unsigned long long seed;
};

static int pmod_rot(int r, int D) { return ((r % D) + D) % D; }

// One plan, one loop: the forward per group, the loss cotangents, the backward per group in reverse.  In inverse mode the
// forward visits the groups last to first, there is no loss, and the backward visits them first to last.
static int run_step(StepPlan& p, const StepCall& a) {
    const bool train = a.mode == kStepTrain, inv = a.mode == kStepInverse;
    const size_t G = p.groups.size();
    const int D = a.chain->dim, C = a.chain->cdim, F = D - D / 2 + C;
    cudaStream_t st = a.st;
    char* ws = a.ws;
    const long long M = a.M;
    const float* x = a.x;
    const float* c = a.c;
    float* ld = reinterpret_cast<float*>(ws + p.off_ld);
    float* glp = reinterpret_cast<float*>(ws + p.off_glp);
    float* gy = reinterpret_cast<float*>(ws + p.off_ga);
    float* gx = reinterpret_cast<float*>(ws + p.off_gb);
    float* gh0 = reinterpret_cast<float*>(ws + p.off_gh0);
    void* chain_ws = ws + p.off_chain;
    void* bwd_ws = ws + p.off_bwd;
    const long long mb = std::min<long long>(a.micro_batch, M);
    auto state = [&](size_t g) { return reinterpret_cast<float*>(ws + p.off_states + g * (size_t)M * D * 4); };
    auto stats = [&](size_t g) { return ws + p.off_stats + g * p.stats_stride; };

    if (!inv) ZF_CUDA_CHECK(cudaMemsetAsync(ld, 0, (size_t)M * 4, st));
    if (a.gc && C) ZF_CUDA_CHECK(cudaMemsetAsync(a.gc, 0, (size_t)M * C * 4, st));

    // ---- forward, one bijector group at a time (in train mode the batch statistics couple the events)
    std::vector<zf_coupling> batch_cp(G);    // couplings reading the BATCH statistics (train mode)
    std::vector<const float*> u_in(G);       // inverse mode: the input of each group's own inverse
    float* xtmp = reinterpret_cast<float*>(ws + p.off_xtmp);
    const float* cur = x;
    for (size_t k = 0; k < G; ++k) {
        const size_t gi = inv ? G - 1 - k : k;
        StepGroup& g = p.groups[gi];
        float* nxt = state(gi);
        if (inv) {
            // Roll^-1 of the group's input (the latent draw for the first pass when sampling) into u_g, then the group's
            // own inverse into the next state (x_g is u_{g-1} when group g-1 has no Rolls) or into the output buffer
            zf_chain rolls{D, 0, (int32_t)g.ops.size() - 1, g.ops.data() + 1};
            if (!x && k == 0) {
                if (int rc = zf_flow_sample(st, &rolls, a.latent_kind, a.peakness, a.seed, nullptr, M, nxt, chain_ws, p.chain_bytes))
                    return rc;
                u_in[gi] = nxt;
            } else if (pmod_rot(g.rot, D) != 0) {
                if (int rc = zf_chain_inverse(st, &rolls, cur, nullptr, M, nxt, chain_ws, p.chain_bytes)) return rc;
                u_in[gi] = nxt;
            } else {
                u_in[gi] = cur;
            }
            float* out = gi == 0 ? (a.x_out ? a.x_out : xtmp) : pmod_rot(p.groups[gi - 1].rot, D) != 0 ? xtmp : state(gi - 1);
            zf_chain own{D, C, 1, g.ops.data()};
            if (int rc = zf_chain_inverse(st, &own, u_in[gi], c, M, out, chain_ws, p.chain_bytes)) return rc;
            cur = out;
            continue;
        }
        if (!train) {
            // the chain's own ShiftBounds and couplings: running statistics, read only
        } else if (g.kind == ZF_OP_SHIFT_BOUNDS) {
            const zf_shift_bounds* sb = g.ops[0].shift_bounds;
            float* mm = reinterpret_cast<float*>(stats(gi));
            void* scratch = mm + 2 * D;
            if (int rc = zf_shift_bounds_minmax(st, sb, cur, M, D, mm, scratch)) return rc;
            if (int rc = zf_dp_allreduce_minmax_f32(st, a.dp_comm, mm, D)) return rc;
            if (int rc = zf_shift_bounds_update(st, sb, D, mm)) return rc;
        } else {
            const zf_coupling* cp = g.ops[0].coupling;
            float* bmean = reinterpret_cast<float*>(stats(gi));
            float* bvar = bmean + F;
            double* sums = reinterpret_cast<double*>(stats(gi) + align_up((size_t)2 * F * 4, 8));
            if (int rc = zf_bn_moments(st, cur, c, M, D, C, sums)) return rc;
            if (int rc = dp_allreduce(st, a.dp_comm, sums, 2 * F, 1, 0)) return rc;
            if (int rc = zf_bn_finalize(st, sums, a.global_count, F, 0.99f /* flax BatchNorm momentum */, bmean, bvar,
                                        cp->bn_mean, cp->bn_var))
                return rc;
            batch_cp[gi] = *cp;
            batch_cp[gi].bn_mean = bmean;
            batch_cp[gi].bn_var = bvar;
            g.ops[0].coupling = &batch_cp[gi];
        }
        zf_chain sub{D, C, (int32_t)g.ops.size(), g.ops.data()};
        if (int rc = zf_chain_forward_acc(st, &sub, cur, c, M, nxt, ld, chain_ws, p.chain_bytes)) return rc;
        cur = nxt;
    }

    // ---- loss and the cotangents of z and of the log-dets (flow.py:46-47, train.py:73)
    if (!inv) {
        double* lp_sum = train ? a.lp_sum : reinterpret_cast<double*>(ws + p.off_lp_sum);
        if (int rc = flow_loss_grad(st, a.latent_kind, a.peakness, cur, ld, M, D, a.global_count, a.lp_cotangent, a.lp, gy, glp,
                                    lp_sum, train ? 0 : 1))
            return rc;
        if (train && !a.grads) return ZF_OK;
    }

    // ---- backward
    const bool bucketed = a.dp_comm && a.grad_flat;
    const bool overlap = bucketed && a.aux && a.dp_grad_comm;
    AuxEvents* ev = nullptr;
    if (overlap)
        if (int rc = aux_events(&ev)) return rc;
    const float* g_in = a.x_ct;   // inverse mode: the cotangent of the current group's output, read at (j + g_rot) % D
    int g_rot = 0;
    for (size_t k = 0; k < G; ++k) {
        const size_t gi = inv ? k : G - 1 - k;
        StepGroup& g = p.groups[gi];
        if (inv) {
            // the cotangent of u_g; the last group's goes straight to gz when its Rolls are the identity
            const bool last = gi + 1 == G;
            float* dst = (last && a.gz && pmod_rot(g.rot, D) == 0) ? a.gz : gy;
            if (g.kind == ZF_OP_SHIFT_BOUNDS) {
                if (int rc = shift_bounds_inverse_backward(st, g.ops[0].shift_bounds, D, u_in[gi], g_in, M, dst)) return rc;
            } else {
                const zf_coupling* cp = g.ops[0].coupling;
                const zf_coupling_grads* gr = a.grads ? &a.grads[g.coupling_index] : nullptr;
                double* bsums = gr ? reinterpret_cast<double*>(stats(gi) + align_up((size_t)2 * F * 4, 8)) + 2 * F : nullptr;
                if (int rc = coupling_backward(st, cp, gr, D, C, u_in[gi], c, g_in, g_rot, nullptr, M, dst, gh0, bsums, bwd_ws,
                                               p.bwd_bytes, mb, true))
                    return rc;
                if (gr)
                    if (int rc = zf_bn_param_grads(st, bsums, F, gr->bn_scale, gr->bn_bias)) return rc;
                if (int rc = bn_backward_eval(st, cp, D, C, gh0, M, dst, a.gc)) return rc;
            }
            // the group's output u_g is rolled into the next group's input: its cotangent is read back through the Rolls
            if (last && a.gz && dst != a.gz) {
                zf_chain rolls{D, 0, (int32_t)g.ops.size() - 1, g.ops.data() + 1};
                if (int rc = zf_chain_forward(st, &rolls, dst, nullptr, M, a.gz, nullptr, chain_ws, p.chain_bytes)) return rc;
            }
            g_in = dst;
            g_rot = pmod_rot(-g.rot, D);
            std::swap(gy, gx);
            continue;
        }
        const float* x_in = gi == 0 ? x : state(gi - 1);
        float* dst = (gi == 0 && a.gx) ? a.gx : gx;   // the cotangent of x goes straight to the caller's buffer
        if (g.kind != ZF_OP_COUPLING) {
            // a leading ShiftBounds has no parameters: in train mode x needs no cotangent
            if (train || !a.gx) break;
            if (int rc = shift_bounds_backward(st, g.ops[0].shift_bounds, D, x, gy, g.rot, glp, M, a.gx)) return rc;
            break;
        }
        const zf_coupling* cp = train ? &batch_cp[gi] : g.ops[0].coupling;
        const zf_coupling_grads* gr = a.grads ? &a.grads[g.coupling_index] : nullptr;
        // sum gh0 and sum gh0 xhat: the BatchNorm's parameter gradients, and in train mode also its input VJP
        double* bsums = gr ? reinterpret_cast<double*>(stats(gi) + align_up((size_t)2 * F * 4, 8)) + 2 * F : nullptr;
        if (int rc = coupling_backward(st, cp, gr, D, C, x_in, c, gy, g.rot, glp, M, dst, gh0, bsums, bwd_ws, p.bwd_bytes, mb, false))
            return rc;
        if (gr)
            if (int rc = zf_bn_param_grads(st, bsums, F, gr->bn_scale, gr->bn_bias)) return rc;
        if (!train) {
            if (int rc = bn_backward_eval(st, cp, D, C, gh0, M, dst, a.gc)) return rc;
            std::swap(gy, gx);
            continue;
        }
        if (bucketed) {   // this coupling's parameter gradients are complete: reduce them behind the next backward
            float* b0 = a.grad_flat + a.bucket_off[g.coupling_index];
            const long long bn = a.bucket_off[g.coupling_index + 1] - a.bucket_off[g.coupling_index];
            if (overlap) {
                ZF_CUDA_CHECK(cudaEventRecord(ev->main_done, st));
                ZF_CUDA_CHECK(cudaStreamWaitEvent(a.aux, ev->main_done, 0));
                if (int rc = dp_allreduce(a.aux, a.dp_grad_comm, b0, bn, 0, 0)) return rc;
            } else {
                if (int rc = dp_allreduce(st, a.dp_comm, b0, bn, 0, 0)) return rc;
            }
        }
        if (int rc = dp_allreduce(st, a.dp_comm, bsums, 2 * F, 1, 0)) return rc;
        if (int rc = zf_bn_backward_apply(st, cp, D, C, x_in, c, gh0, bsums, a.global_count, M, dst, a.gc)) return rc;
        std::swap(gy, gx);
    }
    if (overlap) {
        ZF_CUDA_CHECK(cudaEventRecord(ev->aux_done, a.aux));
        ZF_CUDA_CHECK(cudaStreamWaitEvent(st, ev->aux_done, 0));
    }
    return ZF_OK;
}

}  // namespace zf

using namespace zf;

extern "C" size_t zf_flow_value_and_grad_workspace_bytes(const zf_chain* chain, int64_t M, int64_t micro_batch) {
    StepPlan p;
    if (build_step_plan(chain, M, micro_batch, kStepTrain, p) != ZF_OK) return 0;
    return p.total;
}

extern "C" int zf_flow_value_and_grad(void* stream, void* aux_stream, const zf_chain* chain, const zf_coupling_grads* grads,
                                      int32_t latent_kind, float peakness, const float* x, const float* c, int64_t M,
                                      double global_count, const float* lp_cotangent, float* lp, double* lp_sum, float* gc,
                                      void* dp_comm, void* dp_grad_comm, float* grad_flat, const int64_t* bucket_off,
                                      void* workspace, size_t workspace_bytes, int64_t micro_batch) {
    StepPlan p;
    if (int rc = build_step_plan(chain, M, micro_batch, kStepTrain, p)) return rc;
    ZF_REQUIRE(x && lp_sum && workspace, "value_and_grad: null argument");
    ZF_REQUIRE(chain->cdim == 0 || c, "value_and_grad: chain has cdim=%d but c is NULL", chain->cdim);
    ZF_REQUIRE(global_count >= 1, "value_and_grad: global_count must be >= 1");
    ZF_REQUIRE(!grad_flat || bucket_off, "value_and_grad: grad_flat needs bucket_off");
    ZF_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "value_and_grad: workspace must be 256-byte aligned");
    if (workspace_bytes < p.total)
        return fail(ZF_ERR_WORKSPACE, "value_and_grad: workspace too small: need %zu bytes, got %zu", p.total, workspace_bytes);
    StepCall a{kStepTrain, (cudaStream_t)stream, (cudaStream_t)aux_stream, chain, grads, latent_kind, peakness, x, c, M,
               global_count, lp_cotangent, lp, lp_sum, nullptr, gc, dp_comm, dp_grad_comm, grad_flat, bucket_off,
               static_cast<char*>(workspace), micro_batch};
    return run_step(p, a);
}

extern "C" size_t zf_flow_log_prob_vjp_workspace_bytes(const zf_chain* chain, int64_t M, int64_t micro_batch) {
    StepPlan p;
    if (build_step_plan(chain, M, micro_batch, kStepEval, p) != ZF_OK) return 0;
    return p.total;
}

extern "C" int zf_flow_log_prob_vjp(void* stream, const zf_chain* chain, const zf_coupling_grads* grads, int32_t latent_kind,
                                    float peakness, const float* x, const float* c, int64_t M, const float* lp_cotangent,
                                    float* lp, float* gx, float* gc, void* workspace, size_t workspace_bytes,
                                    int64_t micro_batch) {
    StepPlan p;
    if (int rc = build_step_plan(chain, M, micro_batch, kStepEval, p)) return rc;
    ZF_REQUIRE(x && lp_cotangent && workspace, "log_prob_vjp: null argument");
    ZF_REQUIRE(chain->cdim == 0 || c, "log_prob_vjp: chain has cdim=%d but c is NULL", chain->cdim);
    ZF_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "log_prob_vjp: workspace must be 256-byte aligned");
    if (workspace_bytes < p.total)
        return fail(ZF_ERR_WORKSPACE, "log_prob_vjp: workspace too small: need %zu bytes, got %zu", p.total, workspace_bytes);
    // the cotangent is given, so the count that scales the train loss plays no part
    StepCall a{kStepEval, (cudaStream_t)stream, nullptr, chain, grads, latent_kind, peakness, x, c, M, 1.0, lp_cotangent, lp,
               nullptr, gx, gc, nullptr, nullptr, nullptr, nullptr, static_cast<char*>(workspace), micro_batch};
    return run_step(p, a);
}

extern "C" size_t zf_chain_inverse_vjp_workspace_bytes(const zf_chain* chain, int64_t M, int64_t micro_batch) {
    StepPlan p;
    if (build_step_plan(chain, M, micro_batch, kStepInverse, p) != ZF_OK) return 0;
    return p.total;
}

extern "C" int zf_chain_inverse_vjp(void* stream, const zf_chain* chain, const zf_coupling_grads* grads, const float* z,
                                    int32_t latent_kind, float peakness, uint64_t seed, const float* c, int64_t M,
                                    const float* x_cotangent, float* x, float* gz, float* gc, void* workspace,
                                    size_t workspace_bytes, int64_t micro_batch) {
    StepPlan p;
    if (int rc = build_step_plan(chain, M, micro_batch, kStepInverse, p)) return rc;
    ZF_REQUIRE(x_cotangent && workspace, "chain_inverse_vjp: null argument");
    ZF_REQUIRE(chain->cdim == 0 || c, "chain_inverse_vjp: chain has cdim=%d but c is NULL", chain->cdim);
    ZF_REQUIRE(z || !gz, "chain_inverse_vjp: gz must be NULL when sampling (z is NULL): the latent draw is a constant");
    if (!z) {
        ZF_REQUIRE(latent_kind >= 0 && latent_kind <= 3, "chain_inverse_vjp: unknown latent kind %d", latent_kind);
        ZF_REQUIRE(latent_kind != ZF_LATENT_BETA || peakness >= 1.f, "chain_inverse_vjp: peakness must be at least 1");
    }
    ZF_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "chain_inverse_vjp: workspace must be 256-byte aligned");
    if (workspace_bytes < p.total)
        return fail(ZF_ERR_WORKSPACE, "chain_inverse_vjp: workspace too small: need %zu bytes, got %zu", p.total, workspace_bytes);
    StepCall a{kStepInverse, (cudaStream_t)stream, nullptr, chain, grads, latent_kind, peakness, z, c, M, 1.0, nullptr, nullptr,
               nullptr, nullptr, gc, nullptr, nullptr, nullptr, nullptr, static_cast<char*>(workspace), micro_batch,
               x_cotangent, x, gz, (unsigned long long)seed};
    return run_step(p, a);
}
