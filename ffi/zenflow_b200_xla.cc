// XLA FFI adapter over the C ABI of include/zenflow_b200.h: what lets the reference keep jax.Arrays, jax.jit and
// its FLAX modules while the hot path runs in libzenflow_b200.so (north_star; SURVEY.md 8b).
//
// Build (only where JAX is installed - it is NOT in the image this repository is developed in, see ffi/build.py):
//   python ffi/build.py      (g++ -shared -fPIC -I<jax.ffi.include_dir()> -Iinclude ffi/zenflow_b200_xla.cc
//                             -Lzenflow_b200/_native -lzenflow_b200 -lcudart -o ffi/libzenflow_b200_xla.so)
// tests/test_ffi_sources.py compiles this file against a minimal stand-in of xla/ffi/api/ffi.h (tests/stubs/) so
// that at least its C++ and its use of the C ABI are checked in the development image.
//
// Calling convention shared by every handler (ffi/zenflow_jax.py builds it from the FLAX modules):
//   attribute "program" (int32[]): the chain, one record per bijector
//       ShiftBounds        : 0, D kinds (zf_bound_kind)                      + attribute "bounds" (f64[2 D], lo then hi),
//                                                                              attribute "margin" (f64)
//       Roll               : 1, shift
//       NeuralSplineCoupling: 2, knots | act << 16, n_hidden, hidden widths...   (act: zf_act_kind, 0 = nn.swish)
//   operands: x (M, D) [, c (M, C) when cdim > 0], then the FLAX leaves in op order:
//       ShiftBounds        : xmin (D,), xmax (D,)            (the batch_stats xmin_i / xmax_i packed)
//       coupling           : BatchNorm scale, bias, mean, var, then kernel_0, bias_0, ..., kernel_L, bias_L
#include <cstdint>
#include <cstring>
#include <string>
#include <vector>

#include "xla/ffi/api/ffi.h"
#include "zenflow_b200.h"

namespace ffi = xla::ffi;
using F32 = ffi::Buffer<ffi::F32>;

namespace {

// Everything a zf_chain points to, kept alive for the duration of one handler call.
struct ChainStorage {
    zf_chain chain{};
    std::vector<zf_op> ops;
    std::vector<zf_coupling> couplings;
    std::vector<zf_shift_bounds> bounds;
    std::vector<zf_coupling_grads> grads;   // filled by BindGradients
    int n_leaves = 0;                       // operands consumed from `leaves`
    int n_param_leaves = 0;                 // trainable leaves (BatchNorm scale/bias, kernels, biases), op order
};

ffi::Error Invalid(const std::string& msg) { return ffi::Error(ffi::ErrorCode::kInvalidArgument, "zenflow_b200: " + msg); }
ffi::Error FromStatus(int rc) {
    return rc == ZF_OK ? ffi::Error::Success() : ffi::Error(ffi::ErrorCode::kInternal, std::string("zenflow_b200: ") + zf_last_error());
}

// Build the native chain from the program attribute and the leaf operands (see the header comment).  `mutable_stats`:
// the statistics leaves are taken from `stats_out` (result buffers pre-filled with the input values by the caller's
// input_output_aliases), because a train-mode call updates them in place.
ffi::Error BuildChainFromLeaves(ffi::Span<const int32_t> program, ffi::Span<const double> bounds, double margin, int D, int C,
                                ffi::RemainingArgs leaves, int first_leaf, ChainStorage* cs) {
    size_t n_couplings = 0, n_bounds = 0;
    for (size_t i = 0; i < program.size();) {   // first pass: counts (the vectors must not reallocate afterwards)
        const int kind = program[i];
        if (kind == ZF_OP_SHIFT_BOUNDS) { ++n_bounds; i += 1 + D; }
        else if (kind == ZF_OP_ROLL) { i += 2; }
        else if (kind == ZF_OP_COUPLING) { if (i + 2 >= program.size()) return Invalid("truncated program"); ++n_couplings; i += 3 + program[i + 2]; }
        else return Invalid("unknown bijector kind in program");
    }
    cs->couplings.reserve(n_couplings);
    cs->bounds.reserve(n_bounds);
    int leaf = first_leaf;
    auto next = [&](float** out) -> bool {
        if (leaf >= (int)leaves.size()) return false;
        auto b = leaves.get<F32>(leaf++);
        if (!b.has_value()) return false;
        *out = b.value().typed_data();
        return true;
    };
    for (size_t i = 0; i < program.size();) {
        zf_op op{};
        op.kind = program[i];
        if (op.kind == ZF_OP_SHIFT_BOUNDS) {
            if (bounds.size() != (size_t)2 * D) return Invalid("bounds must hold 2*D doubles");
            zf_shift_bounds sb{};
            for (int j = 0; j < D; ++j) {
                sb.kind[j] = program[i + 1 + j];
                sb.lo[j] = bounds[j];
                sb.hi[j] = bounds[D + j];
            }
            sb.margin = margin;
            if (!next(&sb.xmin) || !next(&sb.xmax)) return Invalid("missing ShiftBounds statistics operands");
            cs->bounds.push_back(sb);
            op.shift_bounds = &cs->bounds.back();
            i += 1 + D;
        } else if (op.kind == ZF_OP_ROLL) {
            op.shift = program[i + 1];
            i += 2;
        } else {
            zf_coupling cp{};
            cp.knots = program[i + 1] & 0xffff;
            cp.act = (program[i + 1] >> 16) & 0xff;   // bijectors.py:319
            cp.n_hidden = program[i + 2];
            if (cp.n_hidden < 0 || cp.n_hidden > ZF_MAX_LAYERS) return Invalid("too many hidden layers");
            for (int l = 0; l < cp.n_hidden; ++l) cp.hidden[l] = program[i + 3 + l];
            float *scale, *bias;
            if (!next(&scale) || !next(&bias) || !next(&cp.bn_mean) || !next(&cp.bn_var)) return Invalid("missing BatchNorm operands");
            cp.bn_scale = scale;
            cp.bn_bias = bias;
            for (int l = 0; l <= cp.n_hidden; ++l) {
                float *k, *b;
                if (!next(&k) || !next(&b)) return Invalid("missing Dense operands");
                cp.kernel[l] = k;
                cp.bias[l] = b;
            }
            cs->n_param_leaves += 2 + 2 * (cp.n_hidden + 1);
            cs->couplings.push_back(cp);
            op.coupling = &cs->couplings.back();
            i += 3 + cp.n_hidden;
        }
        cs->ops.push_back(op);
    }
    cs->n_leaves = leaf - first_leaf;
    cs->chain.dim = D;
    cs->chain.cdim = C;
    cs->chain.n_ops = (int32_t)cs->ops.size();
    cs->chain.ops = cs->ops.data();
    return ffi::Error::Success();
}

// Result buffers for the parameter cotangents, one per trainable leaf in op order -> zf_coupling_grads[]
ffi::Error BindGradients(ffi::RemainingRets rets, int first_ret, ChainStorage* cs) {
    int r = first_ret;
    auto next = [&](float** out) -> bool {
        if (r >= (int)rets.size()) return false;
        auto b = rets.get<F32>(r++);
        if (!b.has_value()) return false;
        *out = b.value()->typed_data();
        return true;
    };
    for (const zf_coupling& cp : cs->couplings) {
        zf_coupling_grads g{};
        if (!next(&g.bn_scale) || !next(&g.bn_bias)) return Invalid("missing BatchNorm gradient results");
        for (int l = 0; l <= cp.n_hidden; ++l)
            if (!next(&g.kernel[l]) || !next(&g.bias[l])) return Invalid("missing Dense gradient results");
        cs->grads.push_back(g);
    }
    return ffi::Error::Success();
}

// The entries accumulate into the gradient buffers: start them from zero.
void ZeroGradients(const ChainStorage& cs, int D, int C, cudaStream_t stream) {
    const int F = D - D / 2 + C, d = D / 2;
    for (size_t k = 0; k < cs.grads.size(); ++k) {
        const zf_coupling& cp = cs.couplings[k];
        cudaMemsetAsync(cs.grads[k].bn_scale, 0, sizeof(float) * F, stream);
        cudaMemsetAsync(cs.grads[k].bn_bias, 0, sizeof(float) * F, stream);
        int fan_in = F;
        for (int l = 0; l <= cp.n_hidden; ++l) {
            const int out = l < cp.n_hidden ? cp.hidden[l] : d * (3 * cp.knots - 1);
            cudaMemsetAsync(cs.grads[k].kernel[l], 0, sizeof(float) * (size_t)fan_in * out, stream);
            cudaMemsetAsync(cs.grads[k].bias[l], 0, sizeof(float) * out, stream);
            fan_in = out;
        }
    }
}

struct Shapes { int64_t M; int D, C; };
ffi::Error ReadShapes(const F32& x, int32_t cdim, ffi::RemainingArgs leaves, Shapes* s, const float** c) {
    if (x.dimensions().size() != 2) return Invalid("x must be (M, D)");
    s->M = x.dimensions()[0];
    s->D = (int)x.dimensions()[1];
    s->C = cdim;
    *c = nullptr;
    if (cdim > 0) {
        auto cb = leaves.get<F32>(0);
        if (!cb.has_value()) return Invalid("conditional flow: c operand missing");
        *c = cb.value().typed_data();
    }
    return ffi::Error::Success();
}

// ---- Flow.__call__(x, c, train=False), flow.py:22-48 ------------------------------------------------------
ffi::Error LogProbImpl(cudaStream_t stream, ffi::ScratchAllocator scratch, F32 x, ffi::RemainingArgs rest,
                       ffi::Result<F32> lp, ffi::Span<const int32_t> program, ffi::Span<const double> bounds, double margin,
                       int32_t cdim, int32_t latent, float peakness) {
    Shapes s;
    const float* c;
    if (auto e = ReadShapes(x, cdim, rest, &s, &c); e.failure()) return e;
    ChainStorage cs;
    if (auto e = BuildChainFromLeaves(program, bounds, margin, s.D, s.C, rest, cdim > 0 ? 1 : 0, &cs); e.failure()) return e;
    const size_t bytes = zf_chain_workspace_bytes(&cs.chain, s.M);
    auto ws = scratch.Allocate(bytes, 256);
    if (!ws.has_value()) return ffi::Error(ffi::ErrorCode::kResourceExhausted, "zenflow_b200: scratch allocation failed");
    return FromStatus(zf_flow_log_prob(stream, &cs.chain, latent, peakness, x.typed_data(), c, s.M, lp->typed_data(), *ws, bytes));
}

// ---- Chain.inverse(z, c), bijectors.py:113-116 (Flow.sample with the latent drawn by jax.random: parity mode) ----
ffi::Error InverseImpl(cudaStream_t stream, ffi::ScratchAllocator scratch, F32 z, ffi::RemainingArgs rest, ffi::Result<F32> x,
                       ffi::Span<const int32_t> program, ffi::Span<const double> bounds, double margin, int32_t cdim) {
    Shapes s;
    const float* c;
    if (auto e = ReadShapes(z, cdim, rest, &s, &c); e.failure()) return e;
    ChainStorage cs;
    if (auto e = BuildChainFromLeaves(program, bounds, margin, s.D, s.C, rest, cdim > 0 ? 1 : 0, &cs); e.failure()) return e;
    const size_t bytes = zf_chain_workspace_bytes(&cs.chain, s.M);
    auto ws = scratch.Allocate(bytes, 256);
    if (!ws.has_value()) return ffi::Error(ffi::ErrorCode::kResourceExhausted, "zenflow_b200: scratch allocation failed");
    return FromStatus(zf_chain_inverse(stream, &cs.chain, z.typed_data(), c, s.M, x->typed_data(), *ws, bytes));
}

// ---- Flow.sample throughput mode, flow.py:50-78: Philox latent draw fused into the inverse chain ----------------
// operand 0 is a dummy (M, D) shape carrier (XLA needs an operand to size the call; its values are not read)
ffi::Error SampleImpl(cudaStream_t stream, ffi::ScratchAllocator scratch, F32 like, ffi::RemainingArgs rest, ffi::Result<F32> x,
                      ffi::Span<const int32_t> program, ffi::Span<const double> bounds, double margin, int32_t cdim,
                      int32_t latent, float peakness, int64_t seed) {
    Shapes s;
    const float* c;
    if (auto e = ReadShapes(like, cdim, rest, &s, &c); e.failure()) return e;
    ChainStorage cs;
    if (auto e = BuildChainFromLeaves(program, bounds, margin, s.D, s.C, rest, cdim > 0 ? 1 : 0, &cs); e.failure()) return e;
    const size_t bytes = zf_chain_workspace_bytes(&cs.chain, s.M);
    auto ws = scratch.Allocate(bytes, 256);
    if (!ws.has_value()) return ffi::Error(ffi::ErrorCode::kResourceExhausted, "zenflow_b200: scratch allocation failed");
    return FromStatus(zf_flow_sample(stream, &cs.chain, latent, peakness, (uint64_t)seed, c, s.M, x->typed_data(), *ws, bytes));
}

// ---- train mode: Flow.__call__(train=True, mutable=["batch_stats"]) and its VJP (train.py:64-86) ----------------
// Results: lp (M,), lp_sum (1,) f64 [, parameter cotangents (one per trainable leaf, op order), gc (M, C)].
// The statistics leaves among the operands are aliased to results by the caller (input_output_aliases) and are
// updated in place.  with_grads = 0 is the forward rule of the custom_vjp, with_grads = 1 its backward rule, which
// takes the cotangent of lp as the operand right after x [, c].
ffi::Error TrainImpl(cudaStream_t stream, ffi::ScratchAllocator scratch, F32 x, ffi::RemainingArgs rest, ffi::RemainingRets rets,
                     ffi::Span<const int32_t> program, ffi::Span<const double> bounds, double margin, int32_t cdim,
                     int32_t latent, float peakness, double global_count, int32_t with_grads, int64_t micro_batch) {
    Shapes s;
    const float* c;
    if (auto e = ReadShapes(x, cdim, rest, &s, &c); e.failure()) return e;
    int first = cdim > 0 ? 1 : 0;
    const float* ct = nullptr;
    if (with_grads) {
        auto b = rest.get<F32>(first++);
        if (!b.has_value()) return Invalid("backward rule: cotangent of lp missing");
        ct = b.value().typed_data();
    }
    ChainStorage cs;
    if (auto e = BuildChainFromLeaves(program, bounds, margin, s.D, s.C, rest, first, &cs); e.failure()) return e;
    auto lp = rets.get<F32>(0);
    auto lp_sum = rets.get<ffi::Buffer<ffi::F64>>(1);
    if (!lp.has_value() || !lp_sum.has_value()) return Invalid("results lp / lp_sum missing");
    float* gc = nullptr;
    if (with_grads) {
        if (auto e = BindGradients(rets, 2, &cs); e.failure()) return e;
        if (cdim > 0) {
            auto g = rets.get<F32>(2 + cs.n_param_leaves);
            if (!g.has_value()) return Invalid("result gc missing");
            gc = g.value()->typed_data();
        }
        ZeroGradients(cs, s.D, s.C, stream);
    }
    cudaMemsetAsync(lp_sum.value()->typed_data(), 0, sizeof(double), stream);
    const size_t bytes = zf_flow_value_and_grad_workspace_bytes(&cs.chain, s.M, micro_batch);
    if (bytes == 0) return FromStatus(ZF_ERR_INVALID);
    auto ws = scratch.Allocate(bytes, 256);
    if (!ws.has_value()) return ffi::Error(ffi::ErrorCode::kResourceExhausted, "zenflow_b200: scratch allocation failed");
    // single device here; under shard_map the statistics / gradient exchanges are the zf_dp_* entries with the
    // ncclComm_t of the mesh (or lax.psum on the phase-level entries), see INTEGRATION.md
    return FromStatus(zf_flow_value_and_grad(stream, nullptr, &cs.chain, with_grads ? cs.grads.data() : nullptr, latent, peakness,
                                             x.typed_data(), c, s.M, global_count, ct, lp.value()->typed_data(),
                                             lp_sum.value()->typed_data(), gc, nullptr, nullptr, nullptr, nullptr, *ws, bytes,
                                             micro_batch));
}

// ---- jax.grad of Flow.__call__(x, c, train=False), flow.py:22-48: the backward rule of flow_log_prob ------------
// Operands: x [, c], the cotangent of lp (M,), the leaves.  Results: gx (M, D) [, gc (M, C)], then one cotangent per
// trainable leaf in op order.  The running statistics are read, never written (they get zero cotangents on the
// Python side).
ffi::Error LogProbVjpImpl(cudaStream_t stream, ffi::ScratchAllocator scratch, F32 x, ffi::RemainingArgs rest,
                          ffi::RemainingRets rets, ffi::Span<const int32_t> program, ffi::Span<const double> bounds,
                          double margin, int32_t cdim, int32_t latent, float peakness, int64_t micro_batch) {
    Shapes s;
    const float* c;
    if (auto e = ReadShapes(x, cdim, rest, &s, &c); e.failure()) return e;
    int first = cdim > 0 ? 1 : 0;
    auto ctb = rest.get<F32>(first++);
    if (!ctb.has_value()) return Invalid("log_prob_vjp: cotangent of lp missing");
    ChainStorage cs;
    if (auto e = BuildChainFromLeaves(program, bounds, margin, s.D, s.C, rest, first, &cs); e.failure()) return e;
    auto gx = rets.get<F32>(0);
    if (!gx.has_value()) return Invalid("result gx missing");
    float* gc = nullptr;
    if (cdim > 0) {
        auto g = rets.get<F32>(1);
        if (!g.has_value()) return Invalid("result gc missing");
        gc = g.value()->typed_data();
    }
    if (auto e = BindGradients(rets, cdim > 0 ? 2 : 1, &cs); e.failure()) return e;
    ZeroGradients(cs, s.D, s.C, stream);
    const size_t bytes = zf_flow_log_prob_vjp_workspace_bytes(&cs.chain, s.M, micro_batch);
    if (bytes == 0) return FromStatus(ZF_ERR_INVALID);
    auto ws = scratch.Allocate(bytes, 256);
    if (!ws.has_value()) return ffi::Error(ffi::ErrorCode::kResourceExhausted, "zenflow_b200: scratch allocation failed");
    return FromStatus(zf_flow_log_prob_vjp(stream, &cs.chain, cs.grads.empty() ? nullptr : cs.grads.data(), latent, peakness,
                                           x.typed_data(), c, s.M, ctb.value().typed_data(), nullptr,
                                           gx.value()->typed_data(), gc, *ws, bytes, micro_batch));
}

// ---- jax.grad of Chain.inverse(z, c) (bijectors.py:113-116) or of Flow.sample's inverse pass (flow.py:76-77) -------
// The backward rule of chain_inverse (sample = 0) and flow_sample (sample = 1).  Operands: z (M, D) (sample: a shape
// carrier whose values are not read) [, c], the cotangent of x (M, D), the leaves.  Results: gz (M, D) (not when
// sampling: the draw is a constant) [, gc (M, C)], then one cotangent per trainable leaf in op order.  The running
// statistics are read, never written.
ffi::Error InverseVjpImpl(cudaStream_t stream, ffi::ScratchAllocator scratch, F32 z, ffi::RemainingArgs rest,
                          ffi::RemainingRets rets, ffi::Span<const int32_t> program, ffi::Span<const double> bounds,
                          double margin, int32_t cdim, int32_t latent, float peakness, int64_t seed, int32_t sample,
                          int64_t micro_batch) {
    Shapes s;
    const float* c;
    if (auto e = ReadShapes(z, cdim, rest, &s, &c); e.failure()) return e;
    int first = cdim > 0 ? 1 : 0;
    auto ctb = rest.get<F32>(first++);
    if (!ctb.has_value()) return Invalid("inverse_vjp: cotangent of x missing");
    ChainStorage cs;
    if (auto e = BuildChainFromLeaves(program, bounds, margin, s.D, s.C, rest, first, &cs); e.failure()) return e;
    int r = 0;
    float* gz = nullptr;
    if (!sample) {
        auto g = rets.get<F32>(r++);
        if (!g.has_value()) return Invalid("result gz missing");
        gz = g.value()->typed_data();
    }
    float* gc = nullptr;
    if (cdim > 0) {
        auto g = rets.get<F32>(r++);
        if (!g.has_value()) return Invalid("result gc missing");
        gc = g.value()->typed_data();
    }
    if (auto e = BindGradients(rets, r, &cs); e.failure()) return e;
    ZeroGradients(cs, s.D, s.C, stream);
    const size_t bytes = zf_chain_inverse_vjp_workspace_bytes(&cs.chain, s.M, micro_batch);
    if (bytes == 0) return FromStatus(ZF_ERR_INVALID);
    auto ws = scratch.Allocate(bytes, 256);
    if (!ws.has_value()) return ffi::Error(ffi::ErrorCode::kResourceExhausted, "zenflow_b200: scratch allocation failed");
    return FromStatus(zf_chain_inverse_vjp(stream, &cs.chain, cs.grads.empty() ? nullptr : cs.grads.data(),
                                           sample ? nullptr : z.typed_data(), latent, peakness, (uint64_t)seed, c, s.M,
                                           ctb.value().typed_data(), nullptr, gz, gc, *ws, bytes, micro_batch));
}

// ---- optimizer.update + optax.apply_updates on the flattened pytree, train.py:84-85 ------------------------------
// params / mu / nu are aliased to the results (updated in place).
ffi::Error NadamwImpl(cudaStream_t stream, F32 params, F32 grads, F32 mu, F32 nu, ffi::Result<F32> params_out, ffi::Result<F32> mu_out,
                      ffi::Result<F32> nu_out, int64_t count, float lr, float b1, float b2, float eps, float weight_decay,
                      int32_t nesterov) {
    if (params_out->typed_data() != params.typed_data() || mu_out->typed_data() != mu.typed_data() || nu_out->typed_data() != nu.typed_data())
        return Invalid("nadamw: params / mu / nu must be aliased to the results (input_output_aliases)");
    return FromStatus(zf_nadamw_update(stream, (int64_t)params.element_count(), params_out->typed_data(), grads.typed_data(),
                                       mu_out->typed_data(), nu_out->typed_data(), count, lr, b1, b2, eps, weight_decay, nesterov));
}

}  // namespace

#define ZF_CHAIN_ATTRS()                                                                                      \
    .Attr<ffi::Span<const int32_t>>("program").Attr<ffi::Span<const double>>("bounds").Attr<double>("margin") \
        .Attr<int32_t>("cdim")

XLA_FFI_DEFINE_HANDLER_SYMBOL(ZfFlowLogProb, LogProbImpl,
                              ffi::Ffi::Bind()
                                  .Ctx<ffi::PlatformStream<cudaStream_t>>()
                                  .Ctx<ffi::ScratchAllocator>()
                                  .Arg<F32>()
                                  .RemainingArgs()
                                  .Ret<F32>() ZF_CHAIN_ATTRS()
                                  .Attr<int32_t>("latent")
                                  .Attr<float>("peakness"));

XLA_FFI_DEFINE_HANDLER_SYMBOL(ZfChainInverse, InverseImpl,
                              ffi::Ffi::Bind()
                                  .Ctx<ffi::PlatformStream<cudaStream_t>>()
                                  .Ctx<ffi::ScratchAllocator>()
                                  .Arg<F32>()
                                  .RemainingArgs()
                                  .Ret<F32>() ZF_CHAIN_ATTRS());

XLA_FFI_DEFINE_HANDLER_SYMBOL(ZfFlowSample, SampleImpl,
                              ffi::Ffi::Bind()
                                  .Ctx<ffi::PlatformStream<cudaStream_t>>()
                                  .Ctx<ffi::ScratchAllocator>()
                                  .Arg<F32>()
                                  .RemainingArgs()
                                  .Ret<F32>() ZF_CHAIN_ATTRS()
                                  .Attr<int32_t>("latent")
                                  .Attr<float>("peakness")
                                  .Attr<int64_t>("seed"));

XLA_FFI_DEFINE_HANDLER_SYMBOL(ZfFlowTrain, TrainImpl,
                              ffi::Ffi::Bind()
                                  .Ctx<ffi::PlatformStream<cudaStream_t>>()
                                  .Ctx<ffi::ScratchAllocator>()
                                  .Arg<F32>()
                                  .RemainingArgs()
                                  .RemainingRets() ZF_CHAIN_ATTRS()
                                  .Attr<int32_t>("latent")
                                  .Attr<float>("peakness")
                                  .Attr<double>("global_count")
                                  .Attr<int32_t>("with_grads")
                                  .Attr<int64_t>("micro_batch"));

XLA_FFI_DEFINE_HANDLER_SYMBOL(ZfFlowLogProbVjp, LogProbVjpImpl,
                              ffi::Ffi::Bind()
                                  .Ctx<ffi::PlatformStream<cudaStream_t>>()
                                  .Ctx<ffi::ScratchAllocator>()
                                  .Arg<F32>()
                                  .RemainingArgs()
                                  .RemainingRets() ZF_CHAIN_ATTRS()
                                  .Attr<int32_t>("latent")
                                  .Attr<float>("peakness")
                                  .Attr<int64_t>("micro_batch"));

XLA_FFI_DEFINE_HANDLER_SYMBOL(ZfChainInverseVjp, InverseVjpImpl,
                              ffi::Ffi::Bind()
                                  .Ctx<ffi::PlatformStream<cudaStream_t>>()
                                  .Ctx<ffi::ScratchAllocator>()
                                  .Arg<F32>()
                                  .RemainingArgs()
                                  .RemainingRets() ZF_CHAIN_ATTRS()
                                  .Attr<int32_t>("latent")
                                  .Attr<float>("peakness")
                                  .Attr<int64_t>("seed")
                                  .Attr<int32_t>("sample")
                                  .Attr<int64_t>("micro_batch"));

XLA_FFI_DEFINE_HANDLER_SYMBOL(ZfNadamwUpdate, NadamwImpl,
                              ffi::Ffi::Bind()
                                  .Ctx<ffi::PlatformStream<cudaStream_t>>()
                                  .Arg<F32>()
                                  .Arg<F32>()
                                  .Arg<F32>()
                                  .Arg<F32>()
                                  .Ret<F32>()
                                  .Ret<F32>()
                                  .Ret<F32>()
                                  .Attr<int64_t>("count")
                                  .Attr<float>("lr")
                                  .Attr<float>("b1")
                                  .Attr<float>("b2")
                                  .Attr<float>("eps")
                                  .Attr<float>("weight_decay")
                                  .Attr<int32_t>("nesterov"));
