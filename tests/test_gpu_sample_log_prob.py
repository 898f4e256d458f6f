"""GPU checks of Flow.sample_and_log_prob / Flow.inverse_and_log_prob (zf_flow_sample_log_prob and its VJP
zf_flow_sample_log_prob_vjp) against the float64 reference of tests/sample_log_prob_oracle.py.  The cases are those of
tests/test_gpu_inverse_grad.py: single-dim couplings (the two-tile kernel), the fused VJP kernel behind every ShiftBounds
column kind (and the same case forced onto the FFMA kernels and the unfused backward), more than 16 conditioner inputs,
the unfused GEMM path and a non-swish activation, each with a ragged last micro-batch; plus each latent kind, the
normalisation of the density over its box and a short reverse-KL fit."""
import math

import numpy as np
import pytest
import torch

from oracle import zenflow_oracle as zo
from tests import sample_log_prob_oracle as so
from tests.helpers import assert_fp32_parity, product_chain, to64, trained_variables
from tests.test_gpu_inverse_grad import CASES, GRAD_RTOL, IDS, _coupling_names, _cuda, _flow_vars, _leaf_keys, _rel, _setup

pytestmark = pytest.mark.gpu

LATENTS = {"beta": ("Beta", 12.0), "normal": ("Normal", 1.0), "truncnorm": ("TruncatedNormal", 1.0),
           "uniform": ("Uniform", 1.0)}


def _latent(name):
    from zenflow_b200 import distributions

    return getattr(distributions, LATENTS[name][0])()


def _flow(ops, D, latent="beta"):
    from zenflow_b200 import Flow

    flow = Flow(product_chain(ops), _latent(latent)) if latent != "beta" else Flow(product_chain(ops))
    flow.latent._latch_dim(D)
    return flow


def _spec_call(flow, fv, z, c, fn):
    """fn(spec, z, c) on the ChainSpec the Flow emits."""
    from zenflow_b200._chain import ChainSpec

    def run(self, z, c):
        spec = ChainSpec(self.latent.dim, 0 if c is None else c.shape[1])
        self.bijector._emit(spec, self.scope.child("bijector"))
        return fn(spec, z, c)

    return flow.apply(fv, z, c, method=run)


def _with_impl(impl, f):
    from zenflow_b200 import _lib

    lib = _lib.load()
    if impl != "auto":
        lib.zf_debug_set_impl(impl.encode(), None)
    try:
        return f()
    finally:
        lib.zf_debug_set_impl(None, None)


@pytest.mark.parametrize("impl", ["auto", "simt", "umma8"])
@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_values_match_float64_reference(case, impl):
    """x is Flow.inverse's bit for bit; lp is within fp32 parity of the float64 closed form; lp - Flow.__call__(x) is the
    float64 reference's own difference (EPS terms, clip) within fp32 tolerance."""
    if impl != "auto" and case not in (CASES[0], CASES[1]):
        pytest.skip("forced kernels are checked on the two-tile and the 16-D cases")
    ops, z, c, v, _, _ = _setup(case)
    D = case[0]
    flow = _flow(ops, D)
    fv = _flow_vars(v)
    x, lp = _with_impl(impl, lambda: flow.apply(fv, z, c, method="inverse_and_log_prob"))
    xi = _with_impl(impl, lambda: flow.apply(fv, z, c, method="inverse"))
    assert isinstance(x, np.ndarray) and np.array_equal(x, xi, equal_nan=True)
    x64, lp64 = so.sample_log_prob(ops, to64(v), z.astype(np.float64), None if c is None else c.astype(np.float64))
    _, lp32 = so.sample_log_prob(ops, v, z, c, dtype=torch.float32)
    assert np.isfinite(lp64).all()
    assert_fp32_parity(lp, lp64, lp32, f"lp [{impl}]", slack=4.0)
    # the difference to the forward density on the sample, against the reference's own
    fwd = _with_impl(impl, lambda: flow.apply(fv, x, c))
    fwd64, _ = zo.flow_log_prob(ops, to64(v), x64, None if c is None else c.astype(np.float64))
    fwd32, _ = zo.flow_log_prob(ops, v, x.astype(np.float32), c)
    d, d64, d32 = lp.astype(np.float64) - fwd, lp64 - fwd64, lp32.astype(np.float64) - fwd32
    ok = np.isfinite(d64) & (np.abs(fwd64) < 1e30)
    assert ok.mean() > 0.9
    err = np.abs(d - d64)[ok]
    tol = 4.0 * np.abs(d32 - d64)[ok].max() + 1e-4 * (1 + np.abs(lp64[ok]).max())
    print(f"\n{impl} D={D}: |lp - fwd| ref max {np.abs(d64[ok]).max():.2e}, err max {err.max():.2e} (tol {tol:.2e})")
    assert err.max() <= tol


@pytest.mark.parametrize("latent", list(LATENTS))
def test_sample_and_log_prob_each_latent(latent):
    """Drawn in-kernel: x is Flow.sample's bit for bit for the same seed, lp that of the reference at the draw."""
    case = CASES[0]
    ops, _, c, v, _, _ = _setup(case)
    D, M = case[0], case[6]
    flow = _flow(ops, D, latent)
    fv = _flow_vars(v)
    x, lp = flow.apply(fv, c, method="sample_and_log_prob", seed=5)
    assert isinstance(x, np.ndarray) and isinstance(lp, np.ndarray)
    assert np.array_equal(x, flow.apply(fv, c, method="sample", seed=5), equal_nan=True)
    zs = flow.apply(fv, M, method=lambda self, n: self.latent.sample(n, 5)).cpu().numpy()
    kind, peak = latent, LATENTS[latent][1]
    x64, lp64 = so.sample_log_prob(ops, to64(v), zs.astype(np.float64), c.astype(np.float64), latent=kind, peakness=peak)
    _, lp32 = so.sample_log_prob(ops, v, zs, c, latent=kind, peakness=peak, dtype=torch.float32)
    assert_fp32_parity(lp, lp64, lp32, f"lp [{latent}]", slack=4.0)
    xg, lpg = flow.apply(fv, zs, c, method="inverse_and_log_prob")
    assert np.array_equal(xg, x, equal_nan=True) and np.array_equal(lpg, lp, equal_nan=True)


def _vjp_ref_check(ops, v, z, c, gxc, glc, got, what, latent="beta", peak=12.0):
    gz, gc, gp = got
    _, _, gz64, gc64, gp64 = so.sample_log_prob_vjp(ops, to64(v), z.astype(np.float64),
                                                    None if c is None else c.astype(np.float64),
                                                    None if gxc is None else gxc.astype(np.float64),
                                                    None if glc is None else glc.astype(np.float64),
                                                    latent=latent, peakness=peak)
    for name_, g, ref in (("gz", gz, gz64), ("gc", gc, gc64)):
        if ref is not None and g is not None:
            e = _rel(g.cpu().numpy(), ref)
            assert e <= GRAD_RTOL, f"{what} {name_}: rel err {e:.2e}"
    worst = 0.0
    for k, name in enumerate(_coupling_names(ops)):
        for j, (mname, lname) in enumerate(_leaf_keys(ops, name)):
            e = _rel(gp[k][j].cpu().numpy(), gp64[name][mname][lname])
            worst = max(worst, e)
            assert e <= GRAD_RTOL, f"{what} {name}/{mname}/{lname}: rel err {e:.2e}"
    return worst


@pytest.mark.parametrize("impl", ["auto", "simt"])
@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_vjp_matches_float64_autograd(case, impl):
    """gz, gc and every params leaf within rel 1e-4 of float64 autograd for g_x only, g_lp only and both; with g_lp
    absent the outputs are zf_chain_inverse_vjp's (gz, gc, x bit for bit; parameter sums to rel 1e-6, atomics)."""
    if impl == "simt" and case is not CASES[1]:
        pytest.skip("the unfused path is checked on the 16-D case")
    ops, z, c, v, flow, rng = _setup(case)
    D, M, mb = case[0], case[6], case[9]
    fv = _flow_vars(v)
    gxc = rng.normal(size=(M, D)).astype(np.float32)
    glc = rng.normal(size=M).astype(np.float32)
    for what, a, b in (("g_x", gxc, None), ("g_lp", None, glc), ("both", gxc, glc)):
        out = _with_impl(impl, lambda: _spec_call(flow, fv, z, c, lambda s, z_, c_: s.sample_log_prob_vjp(
            z_, c_, 0, 12.0, a, b, micro_batch=mb, want_x=True, want_lp=True)))
        gz, gc, gp, x, lp = out
        worst = _vjp_ref_check(ops, v, z, c, a, b, (gz, gc, gp), f"[{impl}] {what}")
        print(f"\n{impl} D={D} {what}: worst parameter-gradient rel err {worst:.2e}")
        if b is None:
            ref = _with_impl(impl, lambda: _spec_call(flow, fv, z, c, lambda s, z_, c_: s.inverse_vjp(
                z_, c_, a, micro_batch=mb, want_x=True)))
            assert torch.equal(gz, ref[0]) and torch.equal(x, ref[3])
            if c is not None:
                assert torch.equal(gc, ref[1])
            for per, rper in zip(gp, ref[2]):
                for g, r in zip(per, rper):
                    assert _rel(g.cpu().numpy(), r.double().cpu().numpy()) <= 1e-6
        xs, lps = _with_impl(impl, lambda: flow.apply(fv, z, c, method="inverse_and_log_prob"))
        assert np.array_equal(x.cpu().numpy(), xs, equal_nan=True) and np.array_equal(lp.cpu().numpy(), lps)


@pytest.mark.parametrize("latent", list(LATENTS))
def test_vjp_each_latent_matches_float64_autograd(latent):
    """The latent term of gz (g_lp d log p / dz, latent_score_kernel) for every latent kind, with g_x and g_lp both given:
    gz, gc and every params leaf within rel 1e-4 of float64 autograd."""
    from zenflow_b200 import _lib

    case = CASES[0]
    ops, z, c, v, flow, rng = _setup(case)
    D, M, mb = case[0], case[6], case[9]
    kind, peak = _lib.LATENT_KINDS[latent], LATENTS[latent][1]
    gxc = rng.normal(size=(M, D)).astype(np.float32)
    glc = rng.normal(size=M).astype(np.float32)
    gz, gc, gp, _, _ = _spec_call(flow, _flow_vars(v), z, c, lambda s, z_, c_: s.sample_log_prob_vjp(
        z_, c_, kind, peak, gxc, glc, micro_batch=mb))
    worst = _vjp_ref_check(ops, v, z, c, gxc, glc, (gz, gc, gp), f"[{latent}]", latent=latent, peak=peak)
    print(f"\n{latent}: worst parameter-gradient rel err {worst:.2e}")


@pytest.mark.parametrize("case", [CASES[0], CASES[1], CASES[3]], ids=["two_moons", "dim16_bounds", "gemm_path"])
def test_autograd_matches_the_c_abi(case):
    """torch.autograd.grad through Flow.inverse_and_log_prob is one zf_flow_sample_log_prob_vjp: gz and gc bit for bit,
    parameter gradients to rel 1e-6 (atomic sums); the values are the non-grad call's; the statistics are not written."""
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
    x, lp = flow.apply(tv, zt, ctt, method="inverse_and_log_prob")
    assert x.grad_fn is not None and lp.grad_fn is not None
    px, plp = flow.apply(fv, z, c, method="inverse_and_log_prob")
    assert np.array_equal(x.detach().cpu().numpy(), px, equal_nan=True) and np.array_equal(lp.detach().cpu().numpy(), plp)
    gxc = rng.normal(size=(M, D)).astype(np.float32)
    glc = rng.normal(size=M).astype(np.float32)
    wrt = [zt] + ([ctt] if C else []) + leaves
    for which in ("both", "lp", "x"):
        outs, gos = [], []
        if which in ("both", "x"):
            outs.append(x); gos.append(torch.tensor(gxc, device="cuda"))
        if which in ("both", "lp"):
            outs.append(lp); gos.append(torch.tensor(glc, device="cuda"))
        got = torch.autograd.grad(outs, wrt, grad_outputs=gos, retain_graph=True)
        for s, b in zip(stats, before):
            assert torch.equal(s, b)
        gz, gc, gp, _, _ = _spec_call(flow, fv, z, c, lambda s, z_, c_: s.sample_log_prob_vjp(
            z_, c_, 0, 12.0, gxc if which != "lp" else None, glc if which != "x" else None))
        assert torch.equal(got[0], gz), which
        if C:
            assert got[1].shape == ctt.shape and torch.equal(got[1], gc)
        flat = [g for per in gp for g in per]
        for g, ref, leaf in zip(got[1 + (1 if C else 0):], flat, leaves):
            assert g.shape == leaf.shape and g.dtype == leaf.dtype
            assert _rel(g.cpu().numpy(), ref.double().cpu().numpy()) <= 1e-6


def test_flow_sample_and_log_prob_is_differentiable():
    """Drawn in-kernel under grad: values are the non-grad call's; the VJP is that of inverse_and_log_prob at the draw
    (gc bit for bit, parameters to rel 1e-6); as_numpy=True stays detached."""
    case = CASES[0]
    ops, z, c, v, flow, rng = _setup(case, seed=2)
    M, D = case[6], case[0]
    fv = _flow_vars(v)
    tv = _cuda(fv)
    names = _coupling_names(ops)
    leaves = [tv["params"]["bijector"][n][m][l].requires_grad_(True) for n in names for m, l in _leaf_keys(ops, n)]
    ctt = torch.tensor(c, device="cuda", requires_grad=True)
    xs, lps = flow.apply(tv, ctt, method="sample_and_log_prob", seed=11)
    assert xs.grad_fn is not None and lps.grad_fn is not None
    px, plp = flow.apply(fv, c, method="sample_and_log_prob", seed=11)
    assert np.array_equal(xs.detach().cpu().numpy(), px, equal_nan=True) and np.array_equal(lps.detach().cpu().numpy(), plp)
    hx, hlp = flow.apply(tv, ctt, method="sample_and_log_prob", seed=11, as_numpy=True)
    assert isinstance(hx, np.ndarray) and np.array_equal(hx, px, equal_nan=True) and np.array_equal(hlp, plp)
    gxc = torch.tensor(rng.normal(size=(M, D)).astype(np.float32), device="cuda")
    glc = torch.tensor(rng.normal(size=M).astype(np.float32), device="cuda")
    got = torch.autograd.grad([xs, lps], [ctt] + leaves, grad_outputs=[gxc, glc])
    zs = flow.apply(fv, M, method=lambda self, n: self.latent.sample(n, 11))
    zt = torch.tensor(zs.cpu().numpy(), device="cuda")
    xr, lpr = flow.apply(tv, zt, ctt, method="inverse_and_log_prob")
    ref = torch.autograd.grad([xr, lpr], [ctt] + leaves, grad_outputs=[gxc, glc])
    assert torch.equal(got[0], ref[0])
    for g, r in zip(got[1:], ref[1:]):
        assert _rel(g.cpu().numpy(), r.double().cpu().numpy()) <= 1e-6


def test_non_finite_rows_get_zero_lp_gradients():
    """Draws outside the Beta latent's support have lp = -inf -> nan_to_num: their lp cotangent is dropped, so the
    gradients equal those of the same call with that cotangent zeroed there."""
    case = CASES[0]
    ops, z, c, v, flow, rng = _setup(case, seed=3)
    M = case[6]
    fv = _flow_vars(v)
    dead = np.arange(0, M, 9)
    z = z.copy()
    z[dead, 1] = 1.25
    glc = rng.normal(size=M).astype(np.float32)
    glc0 = glc.copy()
    glc0[dead] = 0.0
    run = lambda g: _spec_call(flow, fv, z, c, lambda s, z_, c_: s.sample_log_prob_vjp(z_, c_, 0, 12.0, None, g, want_lp=True))
    gz, gc, gp, _, lp = run(glc)
    gz0, gc0, gp0, _, _ = run(glc0)
    lp = lp.cpu().numpy()
    assert (lp[dead] == -np.finfo(np.float32).max).all() and np.isfinite(np.delete(lp, dead)).all()
    assert torch.equal(gz, gz0) and torch.equal(gc, gc0)
    assert (gz.cpu().numpy()[dead] == 0).all()
    for per, per0 in zip(gp, gp0):
        for g, g0 in zip(per, per0):
            assert _rel(g.cpu().numpy(), g0.double().cpu().numpy()) <= 1e-6


def _box_flow(jitter):
    """3-D flow with a two-sided, a lower-bounded and an unbounded column, a Uniform latent, and its box volume."""
    D = 3
    ops = zo.make_chain(D, 16, (128, 128), bounds=((0, -1.0, 3.0), (1, -2.0, None)), n_couplings=2, roll_shift=1)
    rng = np.random.default_rng(21)
    x = np.stack([rng.uniform(-0.9, 2.9, 4096), rng.uniform(-1.9, 3.0, 4096), rng.normal(0, 2, 4096)], 1).astype(np.float32)
    v = trained_variables(ops, x, None, seed=4, weight_scale=1.0)
    if jitter:
        def jit(t):
            return {k: jit(a) for k, a in t.items()} if isinstance(t, dict) else \
                (np.asarray(t) + 0.1 * rng.normal(size=np.shape(t))).astype(np.float32)
        v["params"] = jit(v["params"])
    st = v["batch_stats"]["bijectors_0"]
    f = lambda k: float(np.asarray(st[k]).reshape(-1)[0])
    vol = 4.0 * (math.exp(f("xmax_1")) - math.exp(f("xmin_1"))) * (f("xmax_2") - f("xmin_2"))
    return _flow(ops, D, "uniform"), _flow_vars(v), vol


@pytest.mark.parametrize("jitter", [False, True], ids=["random_init", "jittered"])
def test_density_normalises_over_the_box(jitter):
    """With a Uniform latent x covers the ShiftBounds box exactly and 1/q is bounded: E_q[exp(-lp)] is the box volume.
    4M samples; within 4 standard errors estimated from the same samples."""
    flow, fv, vol = _box_flow(jitter)
    n = 1 << 22
    _, lp = flow.apply(fv, n, method="sample_and_log_prob", seed=17)
    # a draw within one float32 ulp of 1 can pass the last knot's rounded cumsum: the reference's NaN corner, lp = -FLT_MAX
    corner = lp == -torch.finfo(torch.float32).max
    assert int(corner.sum()) <= 8
    w = torch.where(corner, torch.zeros_like(lp, dtype=torch.float64), torch.exp(-lp.double()))
    est, se = w.mean().item(), (w.std() / math.sqrt(n)).item()
    print(f"\n{'jittered' if jitter else 'random-init'}: E[1/q] = {est:.5f} +- {se:.5f}, box volume {vol:.5f}")
    assert abs(est - vol) <= 4 * se + 1e-6 * vol


def test_reverse_kl_fit():
    """A short reverse-KL fit of a 2-D flow to a normalised target inside its box (a product of Beta(2, 2) densities on
    [-1, 3] x [-2, 2]) with torch Adam on the params leaves: the KL estimate stays >= -3 s.e. and falls."""
    D = 2
    ops = zo.make_chain(D, 16, (64, 64), bounds=((0, -1.0, 3.0), (1, -2.0, 2.0)), n_couplings=2, roll_shift=1)
    rng = np.random.default_rng(5)
    x0 = np.stack([rng.uniform(-1, 3, 1024), rng.uniform(-2, 2, 1024)], 1).astype(np.float32)
    v = trained_variables(ops, x0, None, seed=6, weight_scale=0.5)
    flow = _flow(ops, D)
    tv = _cuda(_flow_vars(v))
    names = _coupling_names(ops)
    leaves = [tv["params"]["bijector"][n][m][l].requires_grad_(True) for n in names for m, l in _leaf_keys(ops, n)]
    opt = torch.optim.Adam(leaves, lr=1e-2)
    lo = torch.tensor([-1.0, -2.0], device="cuda", dtype=torch.float64)
    width = torch.tensor([4.0, 4.0], device="cuda", dtype=torch.float64)

    def log_target(x):
        t = (x.double() - lo) / width
        return (math.log(6.0) + torch.log(t) + torch.log1p(-t) - torch.log(width)).sum(-1)

    kls = []
    for step in range(60):
        x, lp = flow.apply(tv, 1 << 16, method="sample_and_log_prob", seed=100 + step)
        r = lp.double() - log_target(x)
        kl, se = r.mean(), r.std() / math.sqrt(r.numel())
        assert kl.item() >= -3 * se.item(), (step, kl.item(), se.item())
        kls.append(kl.item())
        opt.zero_grad()
        kl.backward()
        opt.step()
    print(f"\nreverse KL: {kls[0]:.4f} -> {kls[-1]:.4f}")
    assert np.mean(kls[-5:]) < 0.8 * np.mean(kls[:5])
