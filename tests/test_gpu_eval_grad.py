"""GPU parity of the eval-mode log-density VJP (zf_flow_log_prob_vjp; Flow.__call__(train=False) under torch autograd)
against float64 autograd of the eval forward (tests/eval_oracle.py, the role jax.grad plays for the reference's
Flow.__call__(x, c, train=False)).  Every backward path is covered: single-dim couplings, the fused VJP kernel behind a
ShiftBounds with all four column kinds, more than 16 conditioner inputs, the unfused GEMM path, a non-swish activation,
several micro-batches with a ragged last one, and a chain with no coupling."""
import numpy as np
import pytest
import torch

from oracle import zenflow_oracle as zo
from tests import eval_oracle as eo
from tests.helpers import product_chain, to64, trained_variables

pytestmark = pytest.mark.gpu

GRAD_RTOL = 1e-4   # of the largest entry of the float64 reference (per leaf)

# D, C, K, layers, n_couplings, roll, M, bounds, act, micro_batch
CASES = [
    (2, 1, 16, (128, 128), None, 1, 700, (), "swish", 128),             # two_moons_conditional: single-dim couplings
    (16, 0, 32, (128, 128), 3, 2, 300,                                  # fused VJP kernel, every ShiftBounds column kind
     ((1, -1.0, 4.0), (2, -2.0, None), (3, None, 5.0), (6, -3.0, 6.0)), "swish", 1 << 18),
    (24, 8, 16, (128, 128), 2, 3, 300, (), "swish", 100),               # 20 conditioner inputs
    (4, 2, 8, (16, 16), None, 1, 515, (), "swish", 128),                # widths != 128, K = 8: the unfused GEMM path
    (4, 1, 16, (128, 128), 2, 1, 400, (), "gelu", 96),                  # non-swish act: the FFMA kernels
]
IDS = ["two_moons", "dim16_bounds", "F20", "gemm_path", "gelu"]


def _flow_vars(v):
    return {"params": {"bijector": v["params"]}, "batch_stats": {"bijector": v["batch_stats"]}}


def _inputs(rng, D, C, M, bounds):
    x = rng.normal(0.3, 1.0, (M, D))
    for i, a, b in bounds:   # inside the declared bounds, away from them
        lo = a + 0.3 if a is not None else (b - 6.0)
        hi = b - 0.3 if b is not None else (a + 6.0)
        x[:, i] = rng.uniform(lo, hi, M)
    c = rng.uniform(0, 1, (M, C)).astype(np.float32) if C else None
    return x.astype(np.float32), c


def _setup(case, seed=0):
    D, C, K, layers, ncoup, roll, M, bounds, act, mb = case
    rng = np.random.default_rng(M + seed)
    ops = zo.make_chain(D, K, layers, bounds=bounds, n_couplings=ncoup, roll_shift=roll)
    for op in ops:
        if op["kind"] == "coupling":
            op["act"] = act
    x, c = _inputs(rng, D, C, M, bounds)
    v = trained_variables(ops, x, c, seed=2, weight_scale=1.5 if D < 16 else 1.0)
    from zenflow_b200 import Flow

    flow = Flow(product_chain(ops))
    flow.latent._latch_dim(D)
    return ops, x, c, v, flow, rng


def _direct(flow, fv, x, c, ct, **kw):
    """One zf_flow_log_prob_vjp call through the ChainSpec the Flow emits."""
    from zenflow_b200._chain import ChainSpec

    def run(self, x, c):
        spec = ChainSpec(x.shape[1], 0 if c is None else c.shape[1])
        self.bijector._emit(spec, self.scope.child("bijector"))
        kind, peak = self.latent._native()
        return spec.log_prob_vjp(x, c, kind, peak, ct, **kw)

    return flow.apply(fv, x, c, method=run)


def _coupling_names(ops):
    return [f"bijectors_{i}" for i, op in enumerate(ops) if op["kind"] == "coupling"]


def _leaf_keys(ops, name):
    i = int(name.split("_")[1])
    n = len(ops[i]["layers"]) + 1
    keys = [("BatchNorm_0", "scale"), ("BatchNorm_0", "bias")]
    for j in range(n):
        keys += [(f"Dense_{j}", "kernel"), (f"Dense_{j}", "bias")]
    return keys


def _rel(got, ref):
    got = np.asarray(got, np.float64)
    return np.abs(got - ref).max() / (np.abs(ref).max() + 1e-30)


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_eval_vjp_matches_float64_autograd(case):
    ops, x, c, v, flow, rng = _setup(case)
    D, C, M, act, mb = case[0], case[1], case[6], case[8], case[9]
    fv = _flow_vars(v)
    x64, c64 = x.astype(np.float64), None if c is None else c.astype(np.float64)
    worst = 0.0
    for ct, micro in ((rng.normal(size=M).astype(np.float32), mb), (np.ones(M, np.float32), 1 << 18)):
        gx, gc, gp, lp = _direct(flow, fv, x, c, ct, micro_batch=micro, want_lp=True)
        lp64, gx64, gc64, gp64 = eo.log_prob_vjp(ops, to64(v), x64, c64, ct.astype(np.float64))
        assert np.isfinite(lp64).all()
        np.testing.assert_allclose(lp.cpu().numpy(), lp64, rtol=0, atol=1e-4 * np.abs(lp64).max())
        e = _rel(gx.cpu().numpy(), gx64)
        assert e <= GRAD_RTOL, f"gx: rel err {e:.2e}"
        if C:
            e = _rel(gc.cpu().numpy(), gc64)
            assert e <= GRAD_RTOL, f"gc: rel err {e:.2e}"
        for k, name in enumerate(_coupling_names(ops)):
            for j, (mname, lname) in enumerate(_leaf_keys(ops, name)):
                e = _rel(gp[k][j].cpu().numpy(), gp64[name][mname][lname])
                worst = max(worst, e)
                assert e <= GRAD_RTOL, f"{name}/{mname}/{lname}: rel err {e:.2e} (micro_batch {micro})"
    print(f"\n{act} D={D}: worst parameter-gradient rel err {worst:.2e}")


@pytest.mark.parametrize("case", [CASES[0], CASES[1], CASES[3]], ids=["two_moons", "dim16_bounds", "gemm_path"])
def test_autograd_through_flow_call_matches_the_c_abi(case):
    """torch.autograd.grad of Flow.__call__(train=False) is one zf_flow_log_prob_vjp with ones: gx and gc bit for bit,
    parameter gradients to rel 1e-6 (atomic sums); lp is the non-grad call's output bit for bit; the running
    statistics the kernels read are not written."""
    ops, x, c, v, flow, rng = _setup(case, seed=1)
    C, M = case[1], case[6]
    fv = _flow_vars(v)
    cuda = lambda t: {k: cuda(a) for k, a in t.items()} if isinstance(t, dict) else torch.tensor(np.asarray(t), device="cuda")
    tv = cuda(fv)
    names = _coupling_names(ops)
    leaves = [tv["params"]["bijector"][n][m][l].requires_grad_(True) for n in names for m, l in _leaf_keys(ops, n)]
    stats = [tv["batch_stats"]["bijector"][n]["BatchNorm_0"][k] for n in names for k in ("mean", "var")]
    before = [s.clone() for s in stats]
    xt = torch.tensor(x, device="cuda", requires_grad=True)
    ctt = torch.tensor(c, device="cuda", requires_grad=True) if C else None

    lp = flow.apply(tv, xt, ctt)
    assert lp.grad_fn is not None and lp.is_cuda
    plain = flow.apply(fv, x, c)                                  # numpy in, numpy out, no autograd
    assert np.array_equal(lp.detach().cpu().numpy(), plain, equal_nan=True)
    with torch.no_grad():
        assert flow.apply(tv, xt, ctt).grad_fn is None
    nograd = flow.apply(cuda(fv), xt.detach(), None if ctt is None else ctt.detach())   # nothing requires grad
    assert nograd.grad_fn is None and torch.equal(nograd, lp.detach())

    wrt = [xt] + ([ctt] if C else []) + leaves
    got = torch.autograd.grad(lp.sum(), wrt)
    for s, b in zip(stats, before):
        assert torch.equal(s, b)
    gx, gc, gp, _ = _direct(flow, fv, x, c, np.ones(M, np.float32))
    assert torch.equal(got[0], gx)
    if C:
        assert got[1].shape == ctt.shape and torch.equal(got[1], gc)
    flat = [g for per in gp for g in per]
    for g, ref, leaf in zip(got[1 + (1 if C else 0):], flat, leaves):
        assert g.shape == leaf.shape and g.dtype == leaf.dtype
        assert _rel(g.cpu().numpy(), ref.double().cpu().numpy()) <= 1e-6


def test_autograd_returns_gradients_in_the_leaf_device_and_dtype():
    """CPU float64 inputs and parameters requiring grad get CPU float64 gradients of their own shape; c given as (N,)
    gets an (N,) gradient."""
    ops, x, c, v, flow, rng = _setup(CASES[0], seed=2)
    fv = _flow_vars(v)
    cpu = lambda t: {k: cpu(a) for k, a in t.items()} if isinstance(t, dict) else torch.tensor(np.asarray(t, np.float64))
    tv = cpu(fv)
    k0 = tv["params"]["bijector"]["bijectors_1"]["Dense_0"]["kernel"].requires_grad_(True)
    xt = torch.tensor(x, dtype=torch.float64, requires_grad=True)
    c1 = torch.tensor(c[:, 0], dtype=torch.float64, requires_grad=True)
    gx, gc, gk = torch.autograd.grad(flow.apply(tv, xt, c1).sum(), [xt, c1, k0])
    for g, t in ((gx, xt), (gc, c1), (gk, k0)):
        assert g.device.type == "cpu" and g.dtype == torch.float64 and g.shape == t.shape
        assert torch.isfinite(g).all() and g.abs().max() > 0


def test_event_outside_the_running_range_gets_zero_gradients():
    """A row pushed outside the running ShiftBounds range maps to the edge of the latent's support: its lp is
    nan_to_num'ed, and its gradients are zero, not NaN (nor do they poison the parameter sums)."""
    ops, x, c, v, flow, rng = _setup(CASES[0], seed=3)
    x = x.copy()
    x[5, 0] = float(v["batch_stats"]["bijectors_0"]["xmax_0"][0]) + 10.0
    x[9, 1] = float(v["batch_stats"]["bijectors_0"]["xmin_1"][0]) - 10.0
    M = x.shape[0]
    gx, gc, gp, lp = _direct(flow, _flow_vars(v), x, c, np.ones(M, np.float32), micro_batch=128, want_lp=True)
    gx, gc = gx.cpu().numpy(), gc.cpu().numpy()
    assert np.isfinite(lp.cpu().numpy()).all()
    assert np.isfinite(gx).all() and np.isfinite(gc).all()
    # row 5 sits at z = 1 through the whole chain (the spline passes x >= 1 unchanged): log p = -inf, all gradients 0;
    # row 9's clipped column has no derivative, its other column still has one
    assert (gx[5] == 0).all() and (gc[5] == 0).all() and gx[9, 1] == 0
    assert all(bool(torch.isfinite(g).all()) for per in gp for g in per)
    # the other rows are what they are without the two outliers
    keep = np.setdiff1d(np.arange(M), [5, 9])
    gx2, _, _, _ = _direct(flow, _flow_vars(v), x[keep], c[keep], np.ones(len(keep), np.float32), micro_batch=128)
    np.testing.assert_allclose(gx[keep], gx2.cpu().numpy(), rtol=1e-6, atol=1e-6 * np.abs(gx).max())


def test_chain_without_coupling():
    """Flow(Chain([ShiftBounds(...)])): the VJP wrt x of the ShiftBounds alone, every column kind."""
    rng = np.random.default_rng(7)
    D, M = 4, 333
    bounds = ((1, -1.0, 4.0), (2, -2.0, None), (3, None, 5.0))
    ops = [{"kind": "shift_bounds", "margin": 0.1, "bounds": bounds}]
    x, _ = _inputs(rng, D, 0, M, bounds)
    v = trained_variables(ops, x, None, seed=0)
    from zenflow_b200 import Flow

    flow = Flow(product_chain(ops))
    flow.latent._latch_dim(D)
    ct = rng.normal(size=M).astype(np.float32)
    gx, gc, gp, lp = _direct(flow, _flow_vars(v), x, None, ct, want_lp=True)
    assert gc is None and gp is None
    lp64, gx64, _, _ = eo.log_prob_vjp(ops, to64(v), x.astype(np.float64), None, ct.astype(np.float64))
    assert _rel(gx.cpu().numpy(), gx64) <= GRAD_RTOL
    xt = torch.tensor(x, device="cuda", requires_grad=True)
    (g,) = torch.autograd.grad(flow.apply(_flow_vars(v), xt).sum(), [xt])
    gx1, _, _, _ = _direct(flow, _flow_vars(v), x, None, np.ones(M, np.float32))
    assert torch.equal(g, gx1)


def test_inputs_only_vjp_matches_the_full_one():
    """grads = NULL (no parameter leaf requires grad) skips the grad-weight products; gx and gc do not change."""
    for case in (CASES[1], CASES[3]):
        ops, x, c, v, flow, rng = _setup(case, seed=4)
        M = case[6]
        ct = rng.normal(size=M).astype(np.float32)
        full = _direct(flow, _flow_vars(v), x, c, ct, micro_batch=case[9])
        lean = _direct(flow, _flow_vars(v), x, c, ct, micro_batch=case[9], want_params=False)
        assert lean[2] is None
        assert torch.equal(full[0], lean[0])
        if c is not None:
            assert torch.equal(full[1], lean[1])
