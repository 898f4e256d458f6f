"""Host-only checks of the inverse-chain VJP (zf_chain_inverse_vjp): the float64 reference (tests/inverse_oracle.py)
against the numpy oracle, central differences and the forward chain, and the entry's argument validation and workspace
planning without a GPU."""
import ctypes

import numpy as np
import torch

from oracle import zenflow_oracle as zo
from tests import inverse_oracle as io
from tests.helpers import to64
from tests.test_eval_grad_host import _fake_chain


def _setup(rng, D=4, C=1, K=5, M=7, n_couplings=2):
    bounds = ((1, -1.0, 3.0), (2, -2.0, None), (3, None, 4.0))
    ops = zo.make_chain(D, K, (8,), bounds=bounds, n_couplings=n_couplings, roll_shift=1)
    x = rng.uniform(0.0, 2.0, (M, D))
    c = rng.uniform(0, 1, (M, C))
    v = to64(zo.init_variables(ops, D, C, 1, weight_scale=1.5, randomize_bn=True))
    _, _, st = zo.chain_forward(ops, v, x, c, train=True)
    v["batch_stats"]["bijectors_0"] = st["bijectors_0"]
    return ops, v, x, c


def test_inverse_oracle_matches_numpy_oracle_and_inverts_the_forward():
    """x of the torch reference equals zo.chain_inverse in float64, and inverse(forward(x)) recovers x (to the forward's
    EPS terms)."""
    rng = np.random.default_rng(0)
    ops, v, x, c = _setup(rng, M=64)
    z, _, _ = zo.chain_forward(ops, v, x, c, train=False)
    params = io.to.to_torch(v["params"])
    with torch.no_grad():
        xi = io.chain_inverse(ops, params, v["batch_stats"], torch.tensor(z), torch.tensor(c)).numpy()
    np.testing.assert_allclose(xi, zo.chain_inverse(ops, v, z, c), rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(xi, x, rtol=0, atol=1e-3)
    u = rng.uniform(0.05, 0.95, (64, 4))
    with torch.no_grad():
        xu = io.chain_inverse(ops, params, v["batch_stats"], torch.tensor(u), torch.tensor(c)).numpy()
    np.testing.assert_allclose(xu, zo.chain_inverse(ops, v, u, c), rtol=1e-12, atol=1e-12)


def test_inverse_oracle_matches_central_differences():
    """The float64 autograd reference against central differences of its own forward: every ShiftBounds column kind,
    two conditional couplings with a Roll, z, c and a sample of parameter entries."""
    rng = np.random.default_rng(3)
    ops, v, _, c = _setup(rng)
    M, D = c.shape[0], 4
    z = rng.uniform(0.05, 0.95, (M, D))
    ct = rng.normal(size=(M, D))
    x, gz, gc, gp = io.inverse_vjp(ops, v, z, c, ct)
    assert np.isfinite(x).all()
    params = io.to.to_torch(v["params"])

    def f(zv, cv, pv):
        with torch.no_grad():
            out = io.chain_inverse(ops, pv, v["batch_stats"], torch.tensor(zv), torch.tensor(cv))
        return float((out.numpy() * ct).sum())

    h = 1e-6
    for arr, g in ((z, gz), (c, gc)):
        num = np.zeros_like(arr)
        for idx in np.ndindex(arr.shape):
            a0 = arr[idx]
            arr[idx] = a0 + h; fp = f(z, c, params)
            arr[idx] = a0 - h; fm = f(z, c, params)
            arr[idx] = a0
            num[idx] = (fp - fm) / (2 * h)
        np.testing.assert_allclose(g, num, rtol=1e-5, atol=1e-5 * np.abs(num).max())
    for name, mod in params.items():
        for lname, leaves in mod.items():
            for leaf, t in leaves.items():
                flat = t.view(-1)
                for k in rng.choice(flat.numel(), size=min(3, flat.numel()), replace=False):
                    a0 = float(flat[k])
                    flat[k] = a0 + h; fp = f(z, c, params)
                    flat[k] = a0 - h; fm = f(z, c, params)
                    flat[k] = a0
                    got = gp[name][lname][leaf].reshape(-1)[k]
                    assert abs(got - (fp - fm) / (2 * h)) <= 1e-5 * max(1.0, abs(got)), (name, lname, leaf, k)


def test_inverse_oracle_identity_branch():
    """An element outside [0, 1) at a coupling passes through: cotangent 1 wrt itself, nothing to the parameters."""
    rng = np.random.default_rng(5)
    ops = zo.make_chain(2, 5, (8,), n_couplings=1)[1:]   # one coupling, no ShiftBounds
    v = to64(zo.init_variables(ops, 2, 0, 1, randomize_bn=True))
    z = np.array([[1.5, 0.3], [-0.2, 0.6]])
    ct = rng.normal(size=(2, 2))
    x, gz, _, gp = io.inverse_vjp(ops, v, z, None, ct)
    np.testing.assert_array_equal(x[:, 0], z[:, 0])
    np.testing.assert_array_equal(gz[:, 0], ct[:, 0])
    assert np.isfinite(gz).all()
    for lname in ("Dense_0", "Dense_1"):
        for g in gp["bijectors_0"][lname].values():
            assert np.isfinite(g).all() and (g == 0).all()


def test_inverse_vjp_workspace_planning_is_host_only():
    """The inverse VJP plans the eval VJP's layout without the lp-sum slot and with one more (M, D) buffer; like it, it
    takes a chain with no coupling."""
    from zenflow_b200 import _lib

    lib = _lib.load()
    for D, C, K, hidden, n in [(2, 1, 16, (128, 128), 2), (16, 0, 32, (128, 128), 8), (4, 2, 8, (16, 16), 3)]:
        ch, keep = _fake_chain(D, C, K, hidden, n)
        for M, mb in [(1000, 128), (1 << 20, 1 << 18)]:
            inv = lib.zf_chain_inverse_vjp_workspace_bytes(ctypes.byref(ch), M, mb)
            ev = lib.zf_flow_log_prob_vjp_workspace_bytes(ctypes.byref(ch), M, mb)
            assert ev > 0 and inv == ev - 256 + (M * D * 4 + 255) // 256 * 256, (D, M, inv, ev)
    sb_only, keep = _fake_chain(3, 0, 16, (), 0)
    n = lib.zf_chain_inverse_vjp_workspace_bytes(ctypes.byref(sb_only), 100, 100)
    assert n > 0 and n % 256 == 0


def test_inverse_vjp_argument_validation_without_gpu():
    """Bad arguments are refused with a status and a message before any CUDA call."""
    from zenflow_b200 import _lib

    lib = _lib.load()
    ws_fn = lib.zf_chain_inverse_vjp_workspace_bytes
    fake = 0x40000   # 256-byte aligned, never dereferenced on these paths
    rolled, keep = _fake_chain(4, 0, 16, (128,), 2, shift_bounds=False, lead_roll=True)
    assert ws_fn(ctypes.byref(rolled), 10, 10) == 0 and b"Roll" in lib.zf_last_error()
    assert lib.zf_chain_inverse_vjp(None, ctypes.byref(rolled), None, fake, 0, 12.0, 0, None, 10, fake, None, fake, None,
                                    fake, 1 << 20, 10) == 2   # ZF_ERR_UNSUPPORTED
    late, keep2 = _fake_chain(4, 0, 16, (128,), 1, sb_last=True)
    assert ws_fn(ctypes.byref(late), 10, 10) == 0 and b"ShiftBounds after" in lib.zf_last_error()

    ch, keep3 = _fake_chain(4, 2, 16, (128, 128), 2)
    need = ws_fn(ctypes.byref(ch), 100, 64)
    assert need > 0
    call = lambda **kw: lib.zf_chain_inverse_vjp(
        None, ctypes.byref(ch), None, kw.get("z", fake), kw.get("kind", 0), kw.get("peak", 12.0), 7, kw.get("c", fake),
        kw.get("M", 100), kw.get("ct", fake), None, kw.get("gz", fake), fake, kw.get("ws", fake), kw.get("nbytes", need),
        kw.get("mb", 64))
    assert call(ct=None) == 1 and b"null" in lib.zf_last_error()
    assert call(ws=None) == 1 and b"null" in lib.zf_last_error()
    assert call(c=None) == 1 and b"cdim" in lib.zf_last_error()
    assert call(z=None) == 1 and b"gz must be NULL" in lib.zf_last_error()
    assert call(z=None, gz=None, kind=7) == 1 and b"latent kind" in lib.zf_last_error()
    assert call(z=None, gz=None, peak=0.5) == 1 and b"peakness" in lib.zf_last_error()
    assert call(M=0) == 1 and b"batch" in lib.zf_last_error()
    assert call(mb=0) == 1 and b"batch" in lib.zf_last_error()
    assert call(ws=fake + 16) == 1 and b"aligned" in lib.zf_last_error()
    assert call(nbytes=need - 1) == 4 and b"too small" in lib.zf_last_error()
