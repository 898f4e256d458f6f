"""Host-only checks of Flow.sample_and_log_prob's reference and native entries (zf_flow_sample_log_prob,
zf_flow_sample_log_prob_vjp): the closed-form log-density of tests/sample_log_prob_oracle.py against the log-determinant
of the autograd Jacobian and against central differences of the numpy oracle's inverse, its gradients against central
differences, and the entries' argument validation and workspace planning without a GPU."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import zenflow_oracle as zo
from tests import sample_log_prob_oracle as so
from tests.test_eval_grad_host import _fake_chain
from tests.test_inverse_grad_host import _setup

LATENTS = [("beta", 12.0), ("normal", 1.0), ("truncnorm", 1.0), ("uniform", 1.0)]


@pytest.mark.parametrize("latent,peak", LATENTS)
def test_closed_form_matches_jacobian_log_det(latent, peak):
    """Every ShiftBounds column kind, two conditional couplings and a Roll: the per-element closed form equals
    latent - log|det J| with J the autograd Jacobian of the whole inverse chain, and x equals the numpy oracle's."""
    rng = np.random.default_rng(11)
    ops, v, _, c = _setup(rng, M=40)
    z = rng.uniform(0.3, 0.7, (40, 4))
    x, lp = so.sample_log_prob(ops, v, z, c, latent=latent, peakness=peak)
    np.testing.assert_allclose(x, zo.chain_inverse(ops, v, z, c), rtol=1e-12, atol=1e-12)
    lpj = so.jacobian_lp(ops, v, z, c, latent=latent, peakness=peak)
    assert np.isfinite(lp).all()
    np.testing.assert_allclose(lp, lpj, rtol=1e-10, atol=1e-9)


def test_log_det_matches_central_differences_of_the_numpy_inverse():
    """log|det dx/dz| from central differences of zo.chain_inverse, event by event."""
    rng = np.random.default_rng(4)
    ops, v, _, c = _setup(rng, M=12)
    M, D = 12, 4
    z = rng.uniform(0.1, 0.9, (M, D))
    _, lp = so.sample_log_prob(ops, v, z, c, latent="uniform", peakness=1.0)
    h = 1e-6
    J = np.zeros((M, D, D))
    for j in range(D):
        zp, zm = z.copy(), z.copy()
        zp[:, j] += h
        zm[:, j] -= h
        J[:, :, j] = (zo.chain_inverse(ops, v, zp, c) - zo.chain_inverse(ops, v, zm, c)) / (2 * h)
    np.testing.assert_allclose(lp, -np.linalg.slogdet(J)[1], rtol=1e-6, atol=1e-6)


def test_vjp_reference_matches_central_differences():
    """The gradient reference (autograd of the closed form) for g_x and g_lp together, wrt z and c."""
    rng = np.random.default_rng(6)
    ops, v, _, c = _setup(rng, M=6)
    M, D = 6, 4
    z = rng.uniform(0.2, 0.8, (M, D))
    gxc, glc = rng.normal(size=(M, D)), rng.normal(size=M)
    _, _, gz, gc, _ = so.sample_log_prob_vjp(ops, v, z, c, gxc, glc, latent="beta", peakness=12.0)

    def f(zv, cv):
        x, lp = so.sample_log_prob(ops, v, zv, cv, latent="beta", peakness=12.0)
        return float((x * gxc).sum() + (lp * glc).sum())

    h = 1e-6
    for arr, g in ((z, gz), (c, gc)):
        num = np.zeros_like(arr)
        for idx in np.ndindex(arr.shape):
            a0 = arr[idx]
            arr[idx] = a0 + h; fp = f(z, c)
            arr[idx] = a0 - h; fm = f(z, c)
            arr[idx] = a0
            num[idx] = (fp - fm) / (2 * h)
        np.testing.assert_allclose(g, num, rtol=1e-5, atol=1e-5 * np.abs(num).max())


def test_workspace_planning_is_host_only():
    """The VJP's workspace is the inverse VJP's plan, with the chain slot large enough for the whole chain's pass."""
    from zenflow_b200 import _lib

    lib = _lib.load()
    for D, C, K, hidden, n in [(2, 1, 16, (128, 128), 2), (16, 0, 32, (128, 128), 8), (4, 2, 8, (16, 16), 3)]:
        ch, keep = _fake_chain(D, C, K, hidden, n)
        for M, mb in [(1000, 128), (1 << 20, 1 << 18)]:
            inv = lib.zf_chain_inverse_vjp_workspace_bytes(ctypes.byref(ch), M, mb)
            slp = lib.zf_flow_sample_log_prob_vjp_workspace_bytes(ctypes.byref(ch), M, mb)
            whole = lib.zf_chain_workspace_bytes(ctypes.byref(ch), M)
            assert inv > 0 and whole > 0 and slp >= inv and slp % 256 == 0, (D, M, inv, slp)
            assert slp <= inv + (whole + 255) // 256 * 256
    sb_only, keep = _fake_chain(3, 0, 16, (), 0)
    assert lib.zf_flow_sample_log_prob_vjp_workspace_bytes(ctypes.byref(sb_only), 100, 100) > 0


def test_argument_validation_without_gpu():
    """Bad arguments are refused with a status and a message before any CUDA call."""
    from zenflow_b200 import _lib

    lib = _lib.load()
    ws_fn = lib.zf_flow_sample_log_prob_vjp_workspace_bytes
    fake = 0x40000   # 256-byte aligned, never dereferenced on these paths
    rolled, keep = _fake_chain(4, 0, 16, (128,), 2, shift_bounds=False, lead_roll=True)
    assert ws_fn(ctypes.byref(rolled), 10, 10) == 0 and b"Roll" in lib.zf_last_error()

    ch, keep3 = _fake_chain(4, 2, 16, (128, 128), 2)
    need = ws_fn(ctypes.byref(ch), 100, 64)
    assert need > 0
    call = lambda **kw: lib.zf_flow_sample_log_prob_vjp(
        None, ctypes.byref(ch), None, kw.get("z", fake), kw.get("kind", 0), kw.get("peak", 12.0), 7, kw.get("c", fake),
        kw.get("M", 100), kw.get("ct", fake), kw.get("lct", fake), None, None, kw.get("gz", fake), fake, kw.get("ws", fake),
        kw.get("nbytes", need), kw.get("mb", 64))
    assert call(ct=None, lct=None) == 1 and b"both NULL" in lib.zf_last_error()
    assert call(ws=None) == 1 and b"null" in lib.zf_last_error()
    assert call(c=None) == 1 and b"cdim" in lib.zf_last_error()
    assert call(z=None) == 1 and b"gz must be NULL" in lib.zf_last_error()
    assert call(kind=7) == 1 and b"latent kind" in lib.zf_last_error()
    assert call(peak=0.5) == 1 and b"peakness" in lib.zf_last_error()
    assert call(M=0) == 1 and b"batch" in lib.zf_last_error()
    assert call(mb=0) == 1 and b"batch" in lib.zf_last_error()
    assert call(ws=fake + 16) == 1 and b"aligned" in lib.zf_last_error()
    assert call(nbytes=need - 1) == 4 and b"too small" in lib.zf_last_error()
    # the forward entry: lp is required, the latent is checked
    fwd = lambda **kw: lib.zf_flow_sample_log_prob(None, ctypes.byref(ch), kw.get("kind", 0), kw.get("peak", 12.0), 7,
                                                   kw.get("z", fake), fake, 100, None, kw.get("lp", fake), fake, 1 << 30)
    assert fwd(lp=None) == 1 and b"log_prob" in lib.zf_last_error()
    assert fwd(kind=9) == 1 and b"latent kind" in lib.zf_last_error()
    assert fwd(z=None, peak=0.5) == 1 and b"peakness" in lib.zf_last_error()
