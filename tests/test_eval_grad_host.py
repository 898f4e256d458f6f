"""Host-only checks of the eval-mode log-density VJP (zf_flow_log_prob_vjp): argument validation and workspace planning
without a GPU, and the float64 reference (tests/eval_oracle.py) against central differences."""
import ctypes

import numpy as np
import torch

from oracle import zenflow_oracle as zo
from tests import eval_oracle as eo
from tests.helpers import to64


def _fake_chain(D, C, K, hidden, n_couplings, *, shift_bounds=True, lead_roll=False, sb_last=False):
    """A zf_chain with well-formed descriptors and fake (non-null, aligned) device pointers: enough for the host-side
    planning and argument checks, which never dereference them."""
    from zenflow_b200 import _lib

    keep, ops = [], []
    if lead_roll:
        r = _lib.ZfOp(); r.kind = _lib.OP_ROLL; r.shift = 1
        ops.append(r)
    if shift_bounds:
        sb = _lib.ZfShiftBounds()
        for i in range(D):
            sb.lo[i], sb.hi[i] = 0.0, 1.0
        sb.margin = 0.1
        sb.xmin = sb.xmax = 0x10000
        sb_op = _lib.ZfOp(); sb_op.kind = _lib.OP_SHIFT_BOUNDS; sb_op.shift_bounds = ctypes.pointer(sb)
        keep.append(sb)
        if not sb_last:
            ops.append(sb_op)
    for j in range(n_couplings):
        cp = _lib.ZfCoupling()
        cp.knots = K
        cp.n_hidden = len(hidden)
        for i, w in enumerate(hidden):
            cp.hidden[i] = w
        cp.bn_scale = cp.bn_bias = cp.bn_mean = cp.bn_var = 0x10000
        for i in range(len(hidden) + 1):
            cp.kernel[i] = 0x20000
            cp.bias[i] = 0x30000
        op = _lib.ZfOp(); op.kind = _lib.OP_COUPLING; op.coupling = ctypes.pointer(cp)
        ops.append(op); keep.append(cp)
        if j + 1 < n_couplings:
            r = _lib.ZfOp(); r.kind = _lib.OP_ROLL; r.shift = 1
            ops.append(r)
    if shift_bounds and sb_last:
        ops.append(sb_op)
    arr = (_lib.ZfOp * max(1, len(ops)))(*ops)
    ch = _lib.ZfChain()
    ch.dim, ch.cdim, ch.n_ops = D, C, len(ops)
    ch.ops = ctypes.cast(arr, ctypes.POINTER(_lib.ZfOp))
    keep += [arr, ops]
    return ch, keep


def test_vjp_workspace_planning_is_host_only():
    """The eval VJP plans the train step's layout plus one lp-sum slot; it also takes a chain with no coupling (d/dx
    through the ShiftBounds alone), which the train step refuses."""
    from zenflow_b200 import _lib

    lib = _lib.load()
    for D, C, K, hidden, n in [(2, 1, 16, (128, 128), 2), (16, 0, 32, (128, 128), 8), (4, 2, 8, (16, 16), 3)]:
        ch, keep = _fake_chain(D, C, K, hidden, n)
        for M, mb in [(1000, 128), (1 << 20, 1 << 18)]:
            ev = lib.zf_flow_log_prob_vjp_workspace_bytes(ctypes.byref(ch), M, mb)
            tr = lib.zf_flow_value_and_grad_workspace_bytes(ctypes.byref(ch), M, mb)
            assert tr > 0 and ev == tr + 256, (D, M, ev, tr)
    sb_only, keep = _fake_chain(3, 0, 16, (), 0)
    assert lib.zf_flow_value_and_grad_workspace_bytes(ctypes.byref(sb_only), 100, 100) == 0
    assert b"no coupling" in lib.zf_last_error()
    n = lib.zf_flow_log_prob_vjp_workspace_bytes(ctypes.byref(sb_only), 100, 100)
    assert n > 0 and n % 256 == 0
    one, keep = _fake_chain(1, 0, 16, (), 0)   # a one-column ShiftBounds flow has a VJP too
    assert lib.zf_flow_log_prob_vjp_workspace_bytes(ctypes.byref(one), 10, 10) > 0


def test_vjp_argument_validation_without_gpu():
    """Bad arguments are refused with a status and a message before any CUDA call."""
    from zenflow_b200 import _lib

    lib = _lib.load()
    ws_fn = lib.zf_flow_log_prob_vjp_workspace_bytes
    rolled, keep = _fake_chain(4, 0, 16, (128,), 2, shift_bounds=False, lead_roll=True)
    assert ws_fn(ctypes.byref(rolled), 10, 10) == 0
    assert b"Roll" in lib.zf_last_error()
    fake = 0x40000   # 256-byte aligned, never dereferenced on these paths
    assert lib.zf_flow_log_prob_vjp(None, ctypes.byref(rolled), None, 0, 12.0, fake, None, 10, fake, None, fake, None,
                                    fake, 1 << 20, 10) == 2   # ZF_ERR_UNSUPPORTED, as in train mode
    late, keep2 = _fake_chain(4, 0, 16, (128,), 1, sb_last=True)
    assert ws_fn(ctypes.byref(late), 10, 10) == 0 and b"ShiftBounds after" in lib.zf_last_error()

    ch, keep3 = _fake_chain(4, 2, 16, (128, 128), 2)
    need = ws_fn(ctypes.byref(ch), 100, 64)
    assert need > 0
    call = lambda **kw: lib.zf_flow_log_prob_vjp(
        None, ctypes.byref(ch), None, 0, 12.0, kw.get("x", fake), kw.get("c", fake), kw.get("M", 100), kw.get("ct", fake),
        None, fake, fake, kw.get("ws", fake), kw.get("nbytes", need), kw.get("mb", 64))
    assert call(x=None) == 1 and b"null" in lib.zf_last_error()
    assert call(ct=None) == 1 and b"null" in lib.zf_last_error()
    assert call(c=None) == 1 and b"cdim" in lib.zf_last_error()
    assert call(M=0) == 1 and b"batch" in lib.zf_last_error()
    assert call(mb=0) == 1 and b"batch" in lib.zf_last_error()
    assert call(ws=fake + 16) == 1 and b"aligned" in lib.zf_last_error()
    assert call(nbytes=need - 1) == 4 and b"too small" in lib.zf_last_error()
    assert call(ws=None) == 1


def test_eval_oracle_matches_central_differences():
    """The float64 autograd reference of the eval VJP against central differences of its own forward: every column
    kind of ShiftBounds (unbounded, both, lower-only, upper-only), two conditional couplings with a Roll, the
    conditions and a sample of parameter entries."""
    rng = np.random.default_rng(3)
    D, C, K, M = 4, 1, 5, 7
    bounds = ((1, -1.0, 3.0), (2, -2.0, None), (3, None, 4.0))
    ops = zo.make_chain(D, K, (8,), bounds=bounds, n_couplings=2)
    x = rng.uniform(0.0, 2.0, (M, D))
    c = rng.uniform(0, 1, (M, C))
    v = to64(zo.init_variables(ops, D, C, 1, weight_scale=1.5, randomize_bn=True))
    _, _, st = zo.chain_forward(ops, v, x, c, train=True)
    v["batch_stats"]["bijectors_0"] = st["bijectors_0"]
    ct = rng.normal(size=M)
    lp, gx, gc, gp = eo.log_prob_vjp(ops, v, x, c, ct)
    assert np.isfinite(lp).all()
    params = eo.to.to_torch(v["params"])

    def f(xv, cv, pv):
        with torch.no_grad():
            out = eo.eval_log_prob(ops, pv, v["batch_stats"], torch.tensor(xv), torch.tensor(cv))
        return float((out.numpy() * ct).sum())

    h = 1e-6
    for arr, g in ((x, gx), (c, gc)):
        num = np.zeros_like(arr)
        for idx in np.ndindex(arr.shape):
            a0 = arr[idx]
            arr[idx] = a0 + h; fp = f(x, c, params)
            arr[idx] = a0 - h; fm = f(x, c, params)
            arr[idx] = a0
            num[idx] = (fp - fm) / (2 * h)
        np.testing.assert_allclose(g, num, rtol=1e-5, atol=1e-5 * np.abs(num).max())
    for name, mod in params.items():
        for lname, leaves in mod.items():
            for leaf, t in leaves.items():
                flat = t.view(-1)
                for k in rng.choice(flat.numel(), size=min(3, flat.numel()), replace=False):
                    a0 = float(flat[k])
                    flat[k] = a0 + h; fp = f(x, c, params)
                    flat[k] = a0 - h; fm = f(x, c, params)
                    flat[k] = a0
                    got = gp[name][lname][leaf].reshape(-1)[k]
                    assert abs(got - (fp - fm) / (2 * h)) <= 1e-5 * max(1.0, abs(got)), (name, lname, leaf, k)
