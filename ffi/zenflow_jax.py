"""Reference-side wiring of libzenflow_b200_xla.so: what a maintainer of HDembinski/zenflow adds next to
``zenflow/flow.py`` so that Flow keeps jax.Arrays, jax.jit and its FLAX modules while the hot path runs in CUDA.

NOT importable in the image this repository is developed in (no jax / flax): ``encode_program`` and
``leaf_order`` are pure Python and are unit-tested here (tests/test_ffi_sources.py) against duck-typed stand-ins
of the reference's modules; everything that touches jax is imported lazily inside the functions that need it.

Calling convention = the header comment of ffi/zenflow_b200_xla.cc.

reference call site                                   -> handler
  Flow.__call__(x, c, train=False)   flow.py:45-47    -> ZfFlowLogProb      (flow_log_prob, a jax.custom_vjp)
  jax.grad of it (wrt x, c, params)                   -> ZfFlowLogProbVjp   (its backward rule)
  Chain.inverse(z, c)         bijectors.py:113-116    -> ZfChainInverse     (chain_inverse, a jax.custom_vjp)
  Flow.sample                        flow.py:50-78    -> ZfFlowSample       (flow_sample, a jax.custom_vjp; Philox mode)
                                                         or latent.sample (jax.random) + chain_inverse (parity mode)
  jax.grad of either (wrt z, c, params)               -> ZfChainInverseVjp  (their backward rule)
  Flow.sample_and_log_prob / inverse_and_log_prob     -> ZfFlowSampleLogProb (flow_sample_and_log_prob,
                                                         inverse_and_log_prob: jax.custom_vjps with two outputs)
  jax.grad of either (wrt z, c, params)               -> ZfFlowSampleLogProbVjp (their backward rule)
  Flow.__call__(train=True, mutable=["batch_stats"]) + jax.grad(loss_fn)   train.py:64-86
                                                      -> ZfFlowTrain        (flow_log_prob_train, a jax.custom_vjp)
  optimizer.update + apply_updates  train.py:84-85    -> ZfNadamwUpdate     (nadamw_update)
"""
from __future__ import annotations

import ctypes
import os
from typing import Any, Dict, List, Sequence, Tuple

# zf_op_kind / zf_bound_kind / zf_latent_kind of include/zenflow_b200.h
OP_SHIFT_BOUNDS, OP_ROLL, OP_COUPLING = 0, 1, 2
BOUND_NONE, BOUND_BOTH, BOUND_LOWER, BOUND_UPPER = 0, 1, 2, 3
# zf_act_kind by the name of the jax.nn function (silu is jax's alias of swish)
ACT_KINDS = {"swish": 0, "silu": 0, "relu": 1, "tanh": 2, "sigmoid": 3, "gelu": 4, "elu": 5, "softplus": 6, "leaky_relu": 7}
LATENT = {"Beta": 0, "Normal": 1, "TruncatedNormal": 2, "Uniform": 3}

_TARGETS = {
    "zf_flow_log_prob": "ZfFlowLogProb",
    "zf_flow_log_prob_vjp": "ZfFlowLogProbVjp",
    "zf_chain_inverse": "ZfChainInverse",
    "zf_flow_sample": "ZfFlowSample",
    "zf_chain_inverse_vjp": "ZfChainInverseVjp",
    "zf_flow_sample_log_prob": "ZfFlowSampleLogProb",
    "zf_flow_sample_log_prob_vjp": "ZfFlowSampleLogProbVjp",
    "zf_flow_train": "ZfFlowTrain",
    "zf_nadamw_update": "ZfNadamwUpdate",
}
_registered = False


def register(path: str | None = None) -> None:
    """jax.ffi.register_ffi_target for every handler of libzenflow_b200_xla.so (idempotent)."""
    global _registered
    if _registered:
        return
    import jax

    path = path or os.path.join(os.path.dirname(os.path.abspath(__file__)), "libzenflow_b200_xla.so")
    lib = ctypes.CDLL(path)  # raises when the adapter has not been built: there is no fallback
    for target, symbol in _TARGETS.items():
        jax.ffi.register_ffi_target(target, jax.ffi.pycapsule(getattr(lib, symbol)), platform="CUDA")
    _registered = True


# ---------------------------------------------------------------------------------------------------------------
# program / leaves: pure Python (tested here)
# ---------------------------------------------------------------------------------------------------------------
def _is_set(v) -> bool:  # bijectors.py:24-25
    return v is not None


def _flatten(bijector) -> List[Any]:
    """Chain (bijectors.py:90-129) -> flat list of leaf bijectors, in application order."""
    subs = getattr(bijector, "bijectors", None)
    if subs is None:
        return [bijector]
    out: List[Any] = []
    for b in subs:
        out += _flatten(b)
    return out


def encode_program(bijector, dim: int) -> Tuple[List[int], List[float], float]:
    """The ``program`` / ``bounds`` / ``margin`` attributes the handlers take.

    One record per bijector: ShiftBounds ``0, kind_0..kind_{D-1}``; Roll ``1, shift``; NeuralSplineCoupling
    ``2, knots | act << 16, n_hidden, widths...`` (act: zf_act_kind, 0 = nn.swish).  ``bounds`` = D lower then D upper limits (0 where unset).
    """
    program: List[int] = []
    lo, hi, margin = [0.0] * dim, [0.0] * dim, 0.0
    n_sb = 0
    for b in _flatten(bijector):
        name = type(b).__name__
        if name == "ShiftBounds":
            n_sb += 1
            if n_sb > 1:
                raise ValueError("one ShiftBounds per chain (the bounds attribute holds one set of limits)")
            kinds = [BOUND_NONE] * dim
            for i, a, bb in b.bounds:  # bijectors.py:176,183-201
                if i >= dim:
                    raise ValueError(f"index {i} is out of bounds")
                if _is_set(a) and _is_set(bb):
                    if bb < a:
                        raise ValueError("upper bound must be larger than lower bound")
                    kinds[i], lo[i], hi[i] = BOUND_BOTH, float(a), float(bb)
                elif _is_set(a):
                    kinds[i], lo[i] = BOUND_LOWER, float(a)
                elif _is_set(bb):
                    kinds[i], hi[i] = BOUND_UPPER, float(bb)
            margin = float(b.margin)
            program += [OP_SHIFT_BOUNDS] + kinds
        elif name == "Roll":
            program += [OP_ROLL, int(b.shift)]
        elif name == "NeuralSplineCoupling":
            act = ACT_KINDS.get(getattr(b.act, "__name__", ""))  # bijectors.py:319; matched by the jax.nn function's name
            if act is None:
                raise NotImplementedError(f"the CUDA conditioner implements act in {sorted(ACT_KINDS)} (jax.nn functions "
                                          "with their default arguments); nn.swish is the reference default")
            if not 1 <= int(b.knots) < 1 << 16:
                raise ValueError("knots must be in [1, 65535]")
            program += [OP_COUPLING, int(b.knots) | act << 16, len(b.layers)] + [int(w) for w in b.layers]
        else:
            raise NotImplementedError(f"bijector {name} has no CUDA implementation")
    return program, lo + hi, margin


def leaf_order(bijector, variables: Dict[str, Any], dim: int, stack=None):
    """Operands after x [, c]: the FLAX leaves in the order BuildChainFromLeaves consumes them.

    Returns ``(leaves, is_stat, paths)``: ``is_stat[i]`` marks batch_stats leaves (ShiftBounds xmin/xmax packed to
    (D,), BatchNorm mean/var) which a train-mode call updates in place; ``paths[i]`` is ``(collection, module
    path..., name)`` so the results can be put back into the variable tree.  Module naming follows FLAX's
    auto-naming inside Chain (bijectors.py:104-111: ``bijectors_{i}``) and NeuralSplineCoupling
    (bijectors.py:342-347: ``BatchNorm_0``, ``Dense_{j}``).  ``stack(list_of_(1,)_arrays) -> (D,)`` packs the
    per-column ShiftBounds statistics (jnp.concatenate under jax; list under test).
    """
    stack = stack or (lambda xs: xs)
    leaves, is_stat, paths = [], [], []
    flat = _flatten(bijector)
    is_chain = getattr(bijector, "bijectors", None) is not None

    def scope(coll: str, i: int):
        tree = variables.get(coll, {})
        return tree.get(f"bijectors_{i}", {}) if is_chain else tree

    for i, b in enumerate(flat):
        name = type(b).__name__
        if name == "ShiftBounds":
            st = scope("batch_stats", i)
            kinds = encode_program(b, dim)[0][1:]
            for which, fill in (("xmin", 0.0), ("xmax", 1.0)):
                cols = [st[f"{which}_{j}"] if kinds[j] != BOUND_BOTH else None for j in range(dim)]
                leaves.append(stack([c if c is not None else fill for c in cols]))
                is_stat.append(True)
                paths.append(("batch_stats", i, which))
        elif name == "NeuralSplineCoupling":
            p, st = scope("params", i), scope("batch_stats", i)
            for coll, tree, key, stat in (("params", p, "scale", False), ("params", p, "bias", False),
                                          ("batch_stats", st, "mean", True), ("batch_stats", st, "var", True)):
                leaves.append(tree["BatchNorm_0"][key])
                is_stat.append(stat)
                paths.append((coll, i, "BatchNorm_0", key))
            for j in range(len(b.layers) + 1):
                for key in ("kernel", "bias"):
                    leaves.append(p[f"Dense_{j}"][key])
                    is_stat.append(False)
                    paths.append(("params", i, f"Dense_{j}", key))
    return leaves, is_stat, paths


# ---------------------------------------------------------------------------------------------------------------
# jax side
# ---------------------------------------------------------------------------------------------------------------
def _attrs(program, bounds, margin, cdim):
    import numpy as np

    return dict(program=np.asarray(program, np.int32), bounds=np.asarray(bounds, np.float64), margin=np.float64(margin),
                cdim=np.int32(cdim))


def _stack(xs):
    import jax.numpy as jnp

    return jnp.concatenate([jnp.reshape(jnp.asarray(v, jnp.float32), (1,)) for v in xs])


def _operands(flow, variables, x, c):
    dim = x.shape[1]
    program, bounds, margin = encode_program(flow.bijector, dim)
    sub = {k: v.get("bijector", v) for k, v in variables.items()}  # Flow holds the chain as field `bijector`
    leaves, is_stat, paths = leaf_order(flow.bijector, sub, dim, stack=_stack)
    cdim = 0 if c is None else c.shape[1]
    head = [x] if c is None else [x, c]
    return head, leaves, is_stat, paths, _attrs(program, bounds, margin, cdim)


def _latent(flow):
    import numpy as np

    lat = flow.latent
    return dict(latent=np.int32(LATENT[type(lat).__name__]), peakness=np.float32(getattr(lat, "peakness", 12.0)))


def flow_log_prob(flow, variables, x, c=None, *, micro_batch: int = 1 << 18):
    """Flow.__call__(x, c, train=False), flow.py:45-47: one fused launch (chain + latent + nan_to_num).

    A jax.custom_vjp: jax.grad wrt x, c and the params leaves runs ZfFlowLogProbVjp (one zf_flow_log_prob_vjp call,
    the conditioner recomputed in micro-batches of ``micro_batch`` events) with the running statistics held fixed;
    the statistics leaves get zero cotangents, as in make_flow_log_prob_train."""
    import jax
    import jax.numpy as jnp
    import numpy as np

    register()
    _, leaves, is_stat, _, attrs = _operands(flow, variables, x, c)
    latent = _latent(flow)

    def _head(x, c):
        return [x] if c is None else [x, c]

    @jax.custom_vjp
    def f(x, c, leaves):
        call = jax.ffi.ffi_call("zf_flow_log_prob", jax.ShapeDtypeStruct((x.shape[0],), jnp.float32))
        return call(*_head(x, c), *leaves, **attrs, **latent)

    def f_fwd(x, c, leaves):
        return f(x, c, leaves), (x, c, leaves)

    def f_bwd(saved, ct_lp):
        x, c, leaves = saved
        outs = [jax.ShapeDtypeStruct(v.shape, jnp.float32) for v in _head(x, c)]
        outs += [jax.ShapeDtypeStruct(v.shape, jnp.float32) for v, s in zip(leaves, is_stat) if not s]
        call = jax.ffi.ffi_call("zf_flow_log_prob_vjp", outs)
        res = call(*_head(x, c), ct_lp, *leaves, **attrs, **latent, micro_batch=np.int64(micro_batch))
        n_in = len(_head(x, c))
        gp = iter(res[n_in:])
        gl = [jnp.zeros_like(v) if s else next(gp) for v, s in zip(leaves, is_stat)]
        return res[0], (res[1] if c is not None else None), gl

    f.defvjp(f_fwd, f_bwd)
    return f(x, c, list(leaves))


def _inverse_custom_vjp(target, z_or_like, c, leaves, is_stat, attrs, extra, sample, micro_batch):
    """The forward ffi call ``target`` wrapped in a jax.custom_vjp whose backward runs ZfChainInverseVjp (one
    zf_chain_inverse_vjp call) with the running statistics held fixed; the statistics leaves get zero cotangents, and
    z gets none when sampling (the draw is a constant)."""
    import jax
    import jax.numpy as jnp
    import numpy as np

    def _head(z, c):
        return [z] if c is None else [z, c]

    @jax.custom_vjp
    def f(z, c, leaves):
        call = jax.ffi.ffi_call(target, jax.ShapeDtypeStruct(z.shape, jnp.float32))
        return call(*_head(z, c), *leaves, **attrs, **extra)

    def f_fwd(z, c, leaves):
        return f(z, c, leaves), (z, c, leaves)

    def f_bwd(saved, ct_x):
        z, c, leaves = saved
        outs = [] if sample else [jax.ShapeDtypeStruct(z.shape, jnp.float32)]
        outs += [] if c is None else [jax.ShapeDtypeStruct(c.shape, jnp.float32)]
        outs += [jax.ShapeDtypeStruct(v.shape, jnp.float32) for v, s in zip(leaves, is_stat) if not s]
        call = jax.ffi.ffi_call("zf_chain_inverse_vjp", outs)
        lat = dict(latent=np.int32(0), peakness=np.float32(1.0), seed=np.int64(0))
        lat.update(extra)
        res = call(*_head(z, c), ct_x, *leaves, **attrs, **lat, sample=np.int32(1 if sample else 0),
                   micro_batch=np.int64(micro_batch))
        res = iter(res)
        gz = jnp.zeros_like(z) if sample else next(res)
        gc = None if c is None else next(res)
        gp = res
        gl = [jnp.zeros_like(v) if s else next(gp) for v, s in zip(leaves, is_stat)]
        return gz, gc, gl

    f.defvjp(f_fwd, f_bwd)
    return f(z_or_like, c, list(leaves))


def chain_inverse(flow, variables, z, c=None, *, micro_batch: int = 1 << 18):
    """Chain.inverse(z, c), bijectors.py:113-116 (Flow.sample after latent.sample: bit-parity mode).

    A jax.custom_vjp: jax.grad wrt z, c and the params leaves runs ZfChainInverseVjp (one zf_chain_inverse_vjp call)."""
    register()
    _, leaves, is_stat, _, attrs = _operands(flow, variables, z, c)
    return _inverse_custom_vjp("zf_chain_inverse", z, c, leaves, is_stat, attrs, {}, False, micro_batch)


def flow_sample(flow, variables, conditions_or_size, dim: int, *, seed: int = 0, micro_batch: int = 1 << 18):
    """Flow.sample, flow.py:50-78, with the latent drawn inside the kernel (Philox4x32-10; same distribution, not
    the jax.random stream).  A jax.custom_vjp: jax.grad wrt c and the params leaves (reparameterised samples) runs
    ZfChainInverseVjp, which redraws the same latent."""
    import jax.numpy as jnp
    import numpy as np

    register()
    if isinstance(conditions_or_size, int):
        c, n = None, conditions_or_size
    else:
        c = jnp.asarray(conditions_or_size, jnp.float32)
        c = c.reshape(-1, 1) if c.ndim == 1 else c  # flow.py:100-108 _normalize_c
        n = c.shape[0]
    like = jnp.zeros((n, dim), jnp.float32)  # shape carrier (values unread)
    _, leaves, is_stat, _, attrs = _operands(flow, variables, like, c)
    extra = dict(_latent(flow), seed=np.int64(seed))
    return _inverse_custom_vjp("zf_flow_sample", like, c, leaves, is_stat, attrs, extra, True, micro_batch)


def _sample_log_prob_custom_vjp(z_or_like, c, leaves, is_stat, attrs, extra, sample, micro_batch):
    """ZfFlowSampleLogProb wrapped in a jax.custom_vjp with two outputs (x, lp) whose backward runs
    ZfFlowSampleLogProbVjp (one zf_flow_sample_log_prob_vjp call) with the running statistics held fixed; the statistics
    leaves get zero cotangents, and z gets none when sampling (the draw is a constant)."""
    import jax
    import jax.numpy as jnp
    import numpy as np

    def _head(z, c):
        return [z] if c is None else [z, c]

    flags = dict(extra, sample=np.int32(1 if sample else 0))

    @jax.custom_vjp
    def f(z, c, leaves):
        outs = (jax.ShapeDtypeStruct(z.shape, jnp.float32), jax.ShapeDtypeStruct(z.shape[:1], jnp.float32))
        call = jax.ffi.ffi_call("zf_flow_sample_log_prob", outs)
        return tuple(call(*_head(z, c), *leaves, **attrs, **flags))

    def f_fwd(z, c, leaves):
        return f(z, c, leaves), (z, c, leaves)

    def f_bwd(saved, cts):
        z, c, leaves = saved
        ct_x, ct_lp = cts
        outs = [] if sample else [jax.ShapeDtypeStruct(z.shape, jnp.float32)]
        outs += [] if c is None else [jax.ShapeDtypeStruct(c.shape, jnp.float32)]
        outs += [jax.ShapeDtypeStruct(v.shape, jnp.float32) for v, s in zip(leaves, is_stat) if not s]
        call = jax.ffi.ffi_call("zf_flow_sample_log_prob_vjp", outs)
        res = iter(call(*_head(z, c), ct_x, ct_lp, *leaves, **attrs, **flags, micro_batch=np.int64(micro_batch)))
        gz = jnp.zeros_like(z) if sample else next(res)
        gc = None if c is None else next(res)
        gl = [jnp.zeros_like(v) if s else next(res) for v, s in zip(leaves, is_stat)]
        return gz, gc, gl

    f.defvjp(f_fwd, f_bwd)
    return f(z_or_like, c, list(leaves))


def inverse_and_log_prob(flow, variables, z, c=None, *, micro_batch: int = 1 << 18):
    """(Chain.inverse(z, c), its log-density) in one fused pass: lp = nan_to_num(latent.log_prob(z) - log|det dx/dz|),
    the density of the map that produced x (include/zenflow_b200.h, zf_flow_sample_log_prob).  A jax.custom_vjp with two
    outputs: jax.grad wrt z, c and the params leaves runs ZfFlowSampleLogProbVjp."""
    import numpy as np

    register()
    _, leaves, is_stat, _, attrs = _operands(flow, variables, z, c)
    extra = dict(_latent(flow), seed=np.int64(0))
    return _sample_log_prob_custom_vjp(z, c, leaves, is_stat, attrs, extra, False, micro_batch)


def flow_sample_and_log_prob(flow, variables, conditions_or_size, dim: int, *, seed: int = 0, micro_batch: int = 1 << 18):
    """Flow.sample (Philox draw in-kernel, as flow_sample) and the samples' log-density in one fused pass.  A
    jax.custom_vjp with two outputs: jax.grad wrt c and the params leaves runs ZfFlowSampleLogProbVjp, which redraws
    the same latent."""
    import jax.numpy as jnp
    import numpy as np

    register()
    if isinstance(conditions_or_size, int):
        c, n = None, conditions_or_size
    else:
        c = jnp.asarray(conditions_or_size, jnp.float32)
        c = c.reshape(-1, 1) if c.ndim == 1 else c  # flow.py:100-108 _normalize_c
        n = c.shape[0]
    like = jnp.zeros((n, dim), jnp.float32)  # shape carrier (values unread)
    _, leaves, is_stat, _, attrs = _operands(flow, variables, like, c)
    extra = dict(_latent(flow), seed=np.int64(seed))
    return _sample_log_prob_custom_vjp(like, c, leaves, is_stat, attrs, extra, True, micro_batch)


def make_flow_log_prob_train(flow, dim: int, cdim: int, *, global_count=None, micro_batch: int = 0):
    """``f(params_leaves, stat_leaves, x, c) -> (lp, new_stat_leaves)`` with a custom VJP wrt params_leaves and c:
    Flow.apply(variables, x, c, train=True, mutable=["batch_stats"]) under jax.grad (train.py:64-73,82).

    fwd = ZfFlowTrain(with_grads=0): lp + updated statistics.  bwd = ZfFlowTrain(with_grads=1) on the ORIGINAL
    statistics (the step recomputes its forward with the batch statistics, SURVEY.md H5) with the cotangent of lp:
    parameter cotangents in leaf order and d/dc.  The statistics carry no gradient (FLAX treats batch_stats as
    non-differentiable state).
    """
    import jax
    import jax.numpy as jnp
    import numpy as np

    register()
    program, bounds, margin = encode_program(flow.bijector, dim)
    attrs = dict(_attrs(program, bounds, margin, cdim), **_latent(flow))
    # which operand positions are statistics, from a structure-only walk
    class _Any(dict):
        def __missing__(self, k):
            return _Any()
    _, is_stat, _ = leaf_order(flow.bijector, _Any(), dim, stack=lambda xs: 0)
    stat_pos = [i for i, s in enumerate(is_stat) if s]
    par_pos = [i for i, s in enumerate(is_stat) if not s]

    def _merge(params, stats):
        leaves = [None] * len(is_stat)
        for p, i in zip(params, par_pos):
            leaves[i] = p
        for s, i in zip(stats, stat_pos):
            leaves[i] = s
        return leaves

    def _call(with_grads, params, stats, x, c, ct=None):
        M = x.shape[0]
        head = [x] + ([c] if cdim else []) + ([ct] if with_grads else [])
        leaves = _merge(params, stats)
        outs = [jax.ShapeDtypeStruct((M,), jnp.float32), jax.ShapeDtypeStruct((1,), jnp.float64)]
        n_fixed = len(outs)
        if with_grads:
            outs += [jax.ShapeDtypeStruct(p.shape, jnp.float32) for p in params]
            if cdim:
                outs.append(jax.ShapeDtypeStruct(c.shape, jnp.float32))
        # statistics operands are updated in place: alias each to an extra result
        aliases = {}
        for k, i in enumerate(stat_pos):
            aliases[len(head) + i] = len(outs) + k
        outs_all = outs + [jax.ShapeDtypeStruct(s.shape, jnp.float32) for s in stats]
        call = jax.ffi.ffi_call("zf_flow_train", outs_all, input_output_aliases=aliases)
        res = call(*head, *leaves, **attrs, global_count=np.float64(global_count or M), with_grads=np.int32(with_grads),
                   micro_batch=np.int64(micro_batch))
        return res[:n_fixed], res[n_fixed:len(outs)], res[len(outs):]

    @jax.custom_vjp
    def f(params, stats, x, c):
        (lp, _), _, new_stats = _call(0, params, stats, x, c)
        return lp, tuple(new_stats)

    def f_fwd(params, stats, x, c):
        (lp, _), _, new_stats = _call(0, params, stats, x, c)
        return (lp, tuple(new_stats)), (params, stats, x, c)

    def f_bwd(saved, cts):
        params, stats, x, c = saved
        ct_lp, _ = cts
        _, grads, _ = _call(1, params, stats, x, c, ct_lp)
        gp = tuple(grads[:len(params)])
        gc = grads[len(params)] if cdim else None
        zeros = tuple(jnp.zeros_like(s) for s in stats)
        return gp, zeros, jnp.zeros_like(x), gc

    f.defvjp(f_fwd, f_bwd)
    return f


def nadamw_update(params_flat, grads_flat, mu, nu, count: int, *, lr=1e-3, b1=0.9, b2=0.999, eps=1e-8,
                  weight_decay=1e-4, nesterov=True):
    """optax.nadamw(lr).update + optax.apply_updates on the raveled pytree (train.py:84-85)."""
    import jax
    import jax.numpy as jnp
    import numpy as np

    register()
    shp = jax.ShapeDtypeStruct(params_flat.shape, jnp.float32)
    call = jax.ffi.ffi_call("zf_nadamw_update", (shp, shp, shp), input_output_aliases={0: 0, 2: 1, 3: 2})
    return call(params_flat, grads_flat, mu, nu, count=np.int64(count), lr=np.float32(lr), b1=np.float32(b1),
                b2=np.float32(b2), eps=np.float32(eps), weight_decay=np.float32(weight_decay),
                nesterov=np.int32(bool(nesterov)))
