"""GPU parity of the inverse-chain VJP (zf_chain_inverse_vjp; Flow.inverse and Flow.sample under torch autograd) against
float64 autograd of the inverse chain (tests/inverse_oracle.py, the role jax.grad plays for the reference's
flow.apply(v, u, c, method="inverse") and method="sample").  The cases are those of the eval VJP: single-dim couplings,
the fused <true, true> VJP kernel behind a ShiftBounds with all four column kinds (and the same case on the unfused path),
more than 16 conditioner inputs, the unfused GEMM path, a non-swish activation, each with a ragged last micro-batch."""
import numpy as np
import pytest
import torch

from oracle import zenflow_oracle as zo
from tests import inverse_oracle as io
from tests.helpers import product_chain, to64, trained_variables

pytestmark = pytest.mark.gpu

GRAD_RTOL = 1e-4   # of the largest entry of the float64 reference (per leaf)

# D, C, K, layers, n_couplings, roll, M, bounds, act, micro_batch
CASES = [
    (2, 1, 16, (128, 128), None, 1, 700, (), "swish", 128),             # two_moons_conditional: single-dim couplings
    (16, 0, 32, (128, 128), 3, 2, 300,                                  # fused VJP kernel, every ShiftBounds column kind
     ((1, -1.0, 4.0), (2, -2.0, None), (3, None, 5.0), (6, -3.0, 6.0)), "swish", 128),
    (24, 8, 16, (128, 128), 2, 3, 300, (), "swish", 100),               # 20 conditioner inputs
    (4, 2, 8, (16, 16), None, 1, 515, (), "swish", 128),                # widths != 128, K = 8: the unfused GEMM path
    (4, 1, 16, (128, 128), 2, 1, 400, (), "gelu", 96),                  # non-swish act: the FFMA kernels
]
IDS = ["two_moons", "dim16_bounds", "F20", "gemm_path", "gelu"]


def _flow_vars(v):
    return {"params": {"bijector": v["params"]}, "batch_stats": {"bijector": v["batch_stats"]}}


def _setup(case, seed=0):
    D, C, K, layers, ncoup, roll, M, bounds, act, mb = case
    rng = np.random.default_rng(M + seed)
    ops = zo.make_chain(D, K, layers, bounds=bounds, n_couplings=ncoup, roll_shift=roll)
    for op in ops:
        if op["kind"] == "coupling":
            op["act"] = act
    x = rng.normal(0.3, 1.0, (M, D))
    for i, a, b in bounds:
        x[:, i] = rng.uniform(a + 0.3 if a is not None else b - 6.0, b - 0.3 if b is not None else a + 6.0, M)
    x = x.astype(np.float32)
    c = rng.uniform(0, 1, (M, C)).astype(np.float32) if C else None
    v = trained_variables(ops, x, c, seed=2, weight_scale=1.5 if D < 16 else 1.0)
    z = rng.beta(12, 12, (M, D)).astype(np.float32)
    from zenflow_b200 import Flow

    flow = Flow(product_chain(ops))
    flow.latent._latch_dim(D)
    return ops, z, c, v, flow, rng


def _direct(flow, fv, z, c, ct, **kw):
    """One zf_chain_inverse_vjp call through the ChainSpec the Flow emits."""
    from zenflow_b200._chain import ChainSpec

    def run(self, z, c):
        spec = ChainSpec(self.latent.dim, 0 if c is None else c.shape[1])
        self.bijector._emit(spec, self.scope.child("bijector"))
        return spec.inverse_vjp(z, c, ct, **kw)

    return flow.apply(fv, z, c, method=run)


def _coupling_names(ops):
    return [f"bijectors_{i}" for i, op in enumerate(ops) if op["kind"] == "coupling"]


def _leaf_keys(ops, name):
    n = len(ops[int(name.split("_")[1])]["layers"]) + 1
    keys = [("BatchNorm_0", "scale"), ("BatchNorm_0", "bias")]
    for j in range(n):
        keys += [(f"Dense_{j}", "kernel"), (f"Dense_{j}", "bias")]
    return keys


def _rel(got, ref):
    got = np.asarray(got, np.float64)
    return np.abs(got - ref).max() / (np.abs(ref).max() + 1e-30)


def _cuda(t):
    return {k: _cuda(a) for k, a in t.items()} if isinstance(t, dict) else torch.tensor(np.asarray(t), device="cuda")


@pytest.mark.parametrize("impl", ["auto", "simt"])
@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_inverse_vjp_matches_float64_autograd(case, impl):
    if impl == "simt" and case is not CASES[1]:
        pytest.skip("the unfused path is checked on the 16-D case (the others do not take the fused kernel or run it)")
    from zenflow_b200 import _lib

    lib = _lib.load()
    ops, z, c, v, flow, rng = _setup(case)
    D, C, M, mb = case[0], case[1], case[6], case[9]
    z64, c64 = z.astype(np.float64), None if c is None else c.astype(np.float64)
    ct = rng.normal(size=(M, D)).astype(np.float32)
    if impl == "simt":
        lib.zf_debug_set_impl(b"simt", None)
    try:
        gz, gc, gp, x = _direct(flow, _flow_vars(v), z, c, ct, micro_batch=mb, want_x=True)
    finally:
        lib.zf_debug_set_impl(None, None)
    x64, gz64, gc64, gp64 = io.inverse_vjp(ops, to64(v), z64, c64, ct.astype(np.float64))
    assert np.isfinite(x64).all() and np.isfinite(gz64).all()
    assert _rel(x.cpu().numpy(), x64) <= 1e-4
    worst = 0.0
    for name_, got, ref in (("gz", gz, gz64), ("gc", gc, gc64)):
        if ref is not None:
            e = _rel(got.cpu().numpy(), ref)
            assert e <= GRAD_RTOL, f"{name_}: rel err {e:.2e}"
    for k, name in enumerate(_coupling_names(ops)):
        for j, (mname, lname) in enumerate(_leaf_keys(ops, name)):
            e = _rel(gp[k][j].cpu().numpy(), gp64[name][mname][lname])
            worst = max(worst, e)
            assert e <= GRAD_RTOL, f"{name}/{mname}/{lname}: rel err {e:.2e}"
    print(f"\n{impl} D={D}: worst parameter-gradient rel err {worst:.2e}")


@pytest.mark.parametrize("case", [CASES[0], CASES[1], CASES[3]], ids=["two_moons", "dim16_bounds", "gemm_path"])
def test_autograd_through_flow_inverse_matches_the_c_abi(case):
    """torch.autograd.grad of Flow.inverse is one zf_chain_inverse_vjp: gz and gc bit for bit, parameter gradients to
    rel 1e-6 (atomic sums); x is the non-grad call's output bit for bit; the running statistics are not written."""
    ops, z, c, v, flow, rng = _setup(case, seed=1)
    C, M, D = case[1], case[6], case[0]
    fv = _flow_vars(v)
    tv = _cuda(fv)
    names = _coupling_names(ops)
    leaves = [tv["params"]["bijector"][n][m][l].requires_grad_(True) for n in names for m, l in _leaf_keys(ops, n)]
    stats = [t for n in tv["batch_stats"]["bijector"].values() for t in
             (n["BatchNorm_0"].values() if "BatchNorm_0" in n else n.values())]
    before = [s.clone() for s in stats]
    zt = torch.tensor(z, device="cuda", requires_grad=True)
    ctt = torch.tensor(c, device="cuda", requires_grad=True) if C else None

    x = flow.apply(tv, zt, ctt, method="inverse")
    assert x.grad_fn is not None and x.is_cuda
    plain = flow.apply(fv, z, c, method="inverse")                 # numpy in, numpy out, no autograd
    assert np.array_equal(x.detach().cpu().numpy(), plain, equal_nan=True)
    with torch.no_grad():
        assert flow.apply(tv, zt, ctt, method="inverse").grad_fn is None

    ct = rng.normal(size=(M, D)).astype(np.float32)
    wrt = [zt] + ([ctt] if C else []) + leaves
    got = torch.autograd.grad(x, wrt, grad_outputs=torch.tensor(ct, device="cuda"))
    for s, b in zip(stats, before):
        assert torch.equal(s, b)
    gz, gc, gp, xr = _direct(flow, fv, z, c, ct, want_x=True)
    assert torch.equal(got[0], gz)
    if C:
        assert got[1].shape == ctt.shape and torch.equal(got[1], gc)
    flat = [g for per in gp for g in per]
    for g, ref, leaf in zip(got[1 + (1 if C else 0):], flat, leaves):
        assert g.shape == leaf.shape and g.dtype == leaf.dtype
        assert _rel(g.cpu().numpy(), ref.double().cpu().numpy()) <= 1e-6
    # the VJP recomputes the inverse one group at a time: the same per-coupling arithmetic as the fused chain pass
    d = (xr - x.detach()).abs().max().item()
    print(f"\nrecomputed x vs Flow.inverse: max abs diff {d:.3e} ({'bit-identical' if d == 0 else 'not bit-identical'})")
    assert d <= 1e-5 * max(1.0, x.detach().abs().max().item())


def test_flow_sample_is_differentiable():
    """Flow.sample under grad: the value is the non-grad call's bit for bit; its VJP is the inverse VJP at
    z = flow.latent.sample(M, seed): gc bit for bit, parameter gradients to rel 1e-6 (they are accumulated with atomics,
    so their summation order varies from call to call); as_numpy=True stays a detached host array."""
    case = CASES[0]
    ops, z, c, v, flow, rng = _setup(case, seed=2)
    M, D = case[6], case[0]
    fv = _flow_vars(v)
    tv = _cuda(fv)
    names = _coupling_names(ops)
    leaves = [tv["params"]["bijector"][n][m][l].requires_grad_(True) for n in names for m, l in _leaf_keys(ops, n)]
    ctt = torch.tensor(c, device="cuda", requires_grad=True)
    xs = flow.apply(tv, ctt, method="sample", seed=11)
    assert xs.grad_fn is not None and xs.is_cuda
    plain = flow.apply(fv, c, method="sample", seed=11)
    assert np.array_equal(xs.detach().cpu().numpy(), plain, equal_nan=True)
    host = flow.apply(tv, ctt, method="sample", seed=11, as_numpy=True)
    assert isinstance(host, np.ndarray) and np.array_equal(host, plain, equal_nan=True)

    ct = torch.tensor(rng.normal(size=(M, D)).astype(np.float32), device="cuda")
    got = torch.autograd.grad(xs, [ctt] + leaves, grad_outputs=ct)
    zs = flow.apply(fv, M, method=lambda self, n: self.latent.sample(n, 11))
    zt = torch.tensor(zs.cpu().numpy(), device="cuda", requires_grad=True)
    ref = torch.autograd.grad(flow.apply(tv, zt, ctt, method="inverse"), [ctt] + leaves, grad_outputs=ct)
    assert torch.equal(got[0], ref[0])
    for g, r in zip(got[1:], ref[1:]):
        assert _rel(g.cpu().numpy(), r.double().cpu().numpy()) <= 1e-6


def test_rows_outside_the_unit_interval_pass_through():
    """A coupling input outside [0, 1) takes the identity branch: its cotangent passes through unchanged and it adds
    nothing to the parameter gradients."""
    ops = zo.make_chain(2, 16, (128, 128), n_couplings=1)[1:]   # one coupling, no ShiftBounds
    rng = np.random.default_rng(9)
    M = 300
    z = rng.uniform(0.05, 0.95, (M, 2)).astype(np.float32)
    out = np.arange(0, M, 7)
    z[out, 0] = rng.choice([-0.5, 1.0, 1.7], out.size).astype(np.float32)
    v = trained_variables(ops, z, None, seed=3, weight_scale=1.5)
    from zenflow_b200 import Flow

    flow = Flow(product_chain(ops))
    flow.latent._latch_dim(2)
    ct = np.zeros((M, 2), np.float32)
    ct[out, 0] = rng.normal(size=out.size)
    gz, _, gp, _ = _direct(flow, _flow_vars(v), z, None, ct)
    gz = gz.cpu().numpy()
    np.testing.assert_array_equal(gz[out, 0], ct[out, 0])
    assert (gz[:, 1] == 0).all() and all(bool((g == 0).all()) for per in gp for g in per)
    ct2 = rng.normal(size=(M, 2)).astype(np.float32)
    gz2, _, gp2, _ = _direct(flow, _flow_vars(v), z, None, ct2)
    _, gz64, _, gp64 = io.inverse_vjp(ops, to64(v), z.astype(np.float64), None, ct2.astype(np.float64))
    np.testing.assert_array_equal(gz2.cpu().numpy()[out, 0], ct2[out, 0])
    assert _rel(gz2.cpu().numpy(), gz64) <= GRAD_RTOL


def test_chain_without_coupling():
    """Flow(Chain([ShiftBounds(...)])).inverse: the VJP wrt z of ShiftBounds.inverse alone, every column kind."""
    rng = np.random.default_rng(7)
    D, M = 4, 333
    bounds = ((1, -1.0, 4.0), (2, -2.0, None), (3, None, 5.0))
    ops = [{"kind": "shift_bounds", "margin": 0.1, "bounds": bounds}]
    x = rng.uniform(0.0, 3.0, (M, D)).astype(np.float32)
    v = trained_variables(ops, x, None, seed=0)
    from zenflow_b200 import Flow

    flow = Flow(product_chain(ops))
    flow.latent._latch_dim(D)
    z = rng.uniform(0.05, 0.95, (M, D)).astype(np.float32)
    ct = rng.normal(size=(M, D)).astype(np.float32)
    gz, gc, gp, x = _direct(flow, _flow_vars(v), z, None, ct, want_x=True)
    assert gc is None and gp is None
    x64, gz64, _, _ = io.inverse_vjp(ops, to64(v), z.astype(np.float64), None, ct.astype(np.float64))
    assert _rel(gz.cpu().numpy(), gz64) <= GRAD_RTOL
    assert _rel(x.cpu().numpy(), x64) <= 1e-5
