// zf_flow_value_and_grad: the whole `loss_fn` + `jax.grad` of train.py:64-86 as ONE C-ABI call.
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

struct StepPlan {
    std::vector<StepGroup> groups;
    int n_couplings = 0;
    int Fmax = 1;
    // workspace carve-up in bytes
    size_t off_states = 0, off_ld = 0, off_glp = 0, off_ga = 0, off_gb = 0, off_gh0 = 0, off_stats = 0, off_chain = 0,
           off_bwd = 0, total = 0;
    size_t stats_stride = 0, chain_bytes = 0, bwd_bytes = 0;
};

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// Per-coupling statistics block: bmean[F] bvar[F] (float) | fwd sums 2F (double) | bwd sums 2F (double);
// the ShiftBounds group uses the same block for minmax[2D] (float) | scratch[2D] (uint32).
static int build_step_plan(const zf_chain* chain, long long M, long long micro_batch, StepPlan& p) {
    ZF_REQUIRE(chain && chain->n_ops >= 1 && chain->ops, "value_and_grad: empty chain");
    const int D = chain->dim, C = chain->cdim;
    ZF_REQUIRE(D >= 2 && D <= ZF_MAX_DIM, "value_and_grad: dim must be in [2, %d]", ZF_MAX_DIM);
    ZF_REQUIRE(M >= 1 && micro_batch >= 1, "value_and_grad: bad batch");
    for (int i = 0; i < chain->n_ops; ++i) {
        const zf_op& op = chain->ops[i];
        if (op.kind == ZF_OP_ROLL) {
            if (p.groups.empty())
                return fail(ZF_ERR_UNSUPPORTED, "value_and_grad: a chain that starts with Roll is not supported");
            p.groups.back().ops.push_back(op);
            p.groups.back().rot += op.shift;
        } else if (op.kind == ZF_OP_SHIFT_BOUNDS) {
            if (!p.groups.empty())
                return fail(ZF_ERR_UNSUPPORTED, "value_and_grad: ShiftBounds after another bijector is not supported");
            ZF_REQUIRE(op.shift_bounds, "value_and_grad: op %d: shift_bounds is NULL", i);
            p.groups.push_back(StepGroup{ZF_OP_SHIFT_BOUNDS, i, -1, 0, {op}});
        } else if (op.kind == ZF_OP_COUPLING) {
            ZF_REQUIRE(op.coupling, "value_and_grad: op %d: coupling is NULL", i);
            p.groups.push_back(StepGroup{ZF_OP_COUPLING, i, p.n_couplings++, 0, {op}});
        } else {
            return fail(ZF_ERR_INVALID, "value_and_grad: op %d: unknown kind %d", i, op.kind);
        }
    }
    ZF_REQUIRE(p.n_couplings >= 1, "value_and_grad: the chain has no coupling (nothing to differentiate)");
    const int F = D - D / 2 + C;
    p.Fmax = F;
    ZF_REQUIRE(F <= 256, "value_and_grad: at most 256 conditioner inputs");
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

}  // namespace zf

using namespace zf;

extern "C" size_t zf_flow_value_and_grad_workspace_bytes(const zf_chain* chain, int64_t M, int64_t micro_batch) {
    StepPlan p;
    if (build_step_plan(chain, M, micro_batch, p) != ZF_OK) return 0;
    return p.total;
}

extern "C" int zf_flow_value_and_grad(void* stream, void* aux_stream, const zf_chain* chain, const zf_coupling_grads* grads,
                                      int32_t latent_kind, float peakness, const float* x, const float* c, int64_t M,
                                      double global_count, const float* lp_cotangent, float* lp, double* lp_sum, float* gc,
                                      void* dp_comm, void* dp_grad_comm, float* grad_flat, const int64_t* bucket_off,
                                      void* workspace, size_t workspace_bytes, int64_t micro_batch) {
    StepPlan p;
    if (int rc = build_step_plan(chain, M, micro_batch, p)) return rc;
    ZF_REQUIRE(x && lp_sum && workspace, "value_and_grad: null argument");
    const bool fwd_only = (grads == nullptr);   // train-mode forward only: lp, lp_sum and the statistics updates
    ZF_REQUIRE(chain->cdim == 0 || c, "value_and_grad: chain has cdim=%d but c is NULL", chain->cdim);
    ZF_REQUIRE(global_count >= 1, "value_and_grad: global_count must be >= 1");
    ZF_REQUIRE(!grad_flat || bucket_off, "value_and_grad: grad_flat needs bucket_off");
    ZF_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "value_and_grad: workspace must be 256-byte aligned");
    if (workspace_bytes < p.total)
        return fail(ZF_ERR_WORKSPACE, "value_and_grad: workspace too small: need %zu bytes, got %zu", p.total, workspace_bytes);
    const int D = chain->dim, C = chain->cdim, F = D - D / 2 + C;
    cudaStream_t st = (cudaStream_t)stream, aux = (cudaStream_t)aux_stream;
    char* ws = static_cast<char*>(workspace);
    float* ld = reinterpret_cast<float*>(ws + p.off_ld);
    float* glp = reinterpret_cast<float*>(ws + p.off_glp);
    float* gy = reinterpret_cast<float*>(ws + p.off_ga);
    float* gx = reinterpret_cast<float*>(ws + p.off_gb);
    float* gh0 = reinterpret_cast<float*>(ws + p.off_gh0);
    void* chain_ws = ws + p.off_chain;
    void* bwd_ws = ws + p.off_bwd;
    const long long mb = std::min<long long>(micro_batch, M);
    auto state = [&](size_t g) { return reinterpret_cast<float*>(ws + p.off_states + g * (size_t)M * D * 4); };
    auto stats = [&](size_t g) { return ws + p.off_stats + g * p.stats_stride; };

    ZF_CUDA_CHECK(cudaMemsetAsync(ld, 0, (size_t)M * 4, st));
    if (gc && C) ZF_CUDA_CHECK(cudaMemsetAsync(gc, 0, (size_t)M * C * 4, st));

    // ---- forward, one bijector group at a time (the batch statistics couple the events)
    std::vector<zf_coupling> batch_cp(p.groups.size());   // couplings reading the BATCH statistics
    const float* cur = x;
    for (size_t gi = 0; gi < p.groups.size(); ++gi) {
        StepGroup& g = p.groups[gi];
        float* nxt = state(gi);
        if (g.kind == ZF_OP_SHIFT_BOUNDS) {
            const zf_shift_bounds* sb = g.ops[0].shift_bounds;
            float* mm = reinterpret_cast<float*>(stats(gi));
            void* scratch = mm + 2 * D;
            if (int rc = zf_shift_bounds_minmax(st, sb, cur, M, D, mm, scratch)) return rc;
            if (int rc = zf_dp_allreduce_minmax_f32(st, dp_comm, mm, D)) return rc;
            if (int rc = zf_shift_bounds_update(st, sb, D, mm)) return rc;
        } else {
            const zf_coupling* cp = g.ops[0].coupling;
            float* bmean = reinterpret_cast<float*>(stats(gi));
            float* bvar = bmean + F;
            double* sums = reinterpret_cast<double*>(stats(gi) + align_up((size_t)2 * F * 4, 8));
            if (int rc = zf_bn_moments(st, cur, c, M, D, C, sums)) return rc;
            if (int rc = dp_allreduce(st, dp_comm, sums, 2 * F, 1, 0)) return rc;
            if (int rc = zf_bn_finalize(st, sums, global_count, F, 0.99f /* flax BatchNorm momentum */, bmean, bvar,
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
    if (int rc = zf_flow_loss_grad_ct(st, latent_kind, peakness, cur, ld, M, D, global_count, lp_cotangent, lp, gy, glp, lp_sum))
        return rc;
    if (fwd_only) return ZF_OK;

    // ---- backward
    const bool bucketed = dp_comm && grad_flat;
    const bool overlap = bucketed && aux && dp_grad_comm;
    AuxEvents* ev = nullptr;
    if (overlap)
        if (int rc = aux_events(&ev)) return rc;
    for (size_t gi = p.groups.size(); gi-- > 0;) {
        StepGroup& g = p.groups[gi];
        if (g.kind != ZF_OP_COUPLING) break;   // a leading ShiftBounds has no parameters; x needs no cotangent
        const zf_coupling* cp = &batch_cp[gi];
        const zf_coupling_grads* gr = &grads[g.coupling_index];
        const float* x_in = gi == 0 ? x : state(gi - 1);
        double* bsums = reinterpret_cast<double*>(stats(gi) + align_up((size_t)2 * F * 4, 8)) + 2 * F;
        if (int rc = zf_coupling_backward(st, cp, gr, D, C, x_in, c, gy, g.rot, glp, M, gx, gh0, bsums, bwd_ws, p.bwd_bytes, mb))
            return rc;
        if (int rc = zf_bn_param_grads(st, bsums, F, gr->bn_scale, gr->bn_bias)) return rc;
        if (bucketed) {   // this coupling's parameter gradients are complete: reduce them behind the next backward
            float* b0 = grad_flat + bucket_off[g.coupling_index];
            const long long bn = bucket_off[g.coupling_index + 1] - bucket_off[g.coupling_index];
            if (overlap) {
                ZF_CUDA_CHECK(cudaEventRecord(ev->main_done, st));
                ZF_CUDA_CHECK(cudaStreamWaitEvent(aux, ev->main_done, 0));
                if (int rc = dp_allreduce(aux, dp_grad_comm, b0, bn, 0, 0)) return rc;
            } else {
                if (int rc = dp_allreduce(st, dp_comm, b0, bn, 0, 0)) return rc;
            }
        }
        if (int rc = dp_allreduce(st, dp_comm, bsums, 2 * F, 1, 0)) return rc;
        if (int rc = zf_bn_backward_apply(st, cp, D, C, x_in, c, gh0, bsums, global_count, M, gx, gc)) return rc;
        std::swap(gy, gx);
    }
    if (overlap) {
        ZF_CUDA_CHECK(cudaEventRecord(ev->aux_done, aux));
        ZF_CUDA_CHECK(cudaStreamWaitEvent(st, ev->aux_done, 0));
    }
    return ZF_OK;
}
