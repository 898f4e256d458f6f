"""Float64 reference of Flow.sample_and_log_prob / Flow.inverse_and_log_prob.  TEST INFRASTRUCTURE ONLY.

x = Chain.inverse(z, c) and lp = nan_to_num(sum_j log p_latent(z_j) - log|det dx/dz|) with the running statistics fixed.
Two independent statements of lp:
  jacobian_lp      log|det J| of the autograd Jacobian (torch.func.jacrev + vmap) of tests/inverse_oracle.chain_inverse,
                   which shares no per-element log-det formula with the kernels
  sample_log_prob  the per-element closed form the kernels use (log|dx/dy| = 2 log(den) - 2 log(s) - log(num2) at the
                   quadratic root; ShiftBounds.inverse's log(b - a), log(xmax - xmin), + u on one-sided columns), in any
                   torch dtype: float64 for the gradient reference (autograd of it), float32 for the "fp32 oracle"
They are checked against each other and against central differences of the numpy oracle's inverse
(tests/test_sample_log_prob_host.py).  Same identity-branch convention as tests/inverse_oracle.py.
"""
from __future__ import annotations

import math

import numpy as np
import torch

from oracle import torch_oracle as to
from tests import inverse_oracle as io


def _latent(z, kind, peakness):
    """distributions.py log-pdfs summed over the columns (torch_oracle._latent, any dtype)."""
    return to._latent(z, kind, peakness)


def rqs_inverse_ld(y, theta, K):
    """utils.py:144-202 on raw theta (M, d, 3K-1) and log|dx/dy| per element (0 outside [0, 1))."""
    dx = to._softmax_thr(theta[..., :K])
    dy = to._softmax_thr(theta[..., K:2 * K])
    sl = to._squareplus(theta[..., 2 * K:])
    xk, yk = to._knots(dx), to._knots(dy)
    one = torch.ones_like(sl[..., :1])
    dk = torch.cat([one, sl, one], -1)
    sk = dy / dx
    oob = (y < 0) | (y >= 1)
    ys = torch.where(oob, torch.full_like(y, 0.5), y)
    idx = ((yk <= ys[..., None]).sum(-1, keepdim=True) - 1).clamp(0, K - 1)
    g = lambda a, i: torch.take_along_dim(a, i, -1)[..., 0]
    xkk, ykk, dxk, dyk, dkk, dkp1, skk = g(xk, idx), g(yk, idx), g(dx, idx), g(dy, idx), g(dk, idx), g(dk, idx + 1), g(sk, idx)
    beta = dkp1 + dkk - 2 * skk
    a = dyk * (skk - dkk) + (ys - ykk) * beta
    b = dyk * dkk - (ys - ykk) * beta
    c = -skk * (ys - ykk)
    z = 2 * c / (-b - torch.sqrt(b * b - 4 * a * c))
    az = 1 - z
    den = skk + beta * z * az
    num2 = z * (dkp1 * z + 2 * skk * az) + dkk * az * az
    ld = 2 * torch.log(den) - 2 * torch.log(skk) - torch.log(num2)
    return torch.where(oob, y, z * dxk + xkk), torch.where(oob, torch.zeros_like(ld), ld)


def _stat(stats, key, like):
    return torch.tensor(float(np.asarray(stats[key]).reshape(-1)[0]), dtype=like.dtype)


def shift_bounds_inverse_ld(z, op, stats):
    bmap = {i: (a, b) for (i, a, b) in op["bounds"]}
    isset = lambda v: v is not None and np.isfinite(v)
    cols, ld = [], torch.zeros_like(z[:, 0])
    for i in range(z.shape[1]):
        zi = z[:, i]
        a, b = bmap.get(i, (None, None))
        if isset(a) and isset(b):
            cols.append(zi * b + (1 - zi) * a)
            ld = ld + math.log(b - a)
            continue
        lo, hi = _stat(stats, f"xmin_{i}", z), _stat(stats, f"xmax_{i}", z)
        t = zi * hi + (1 - zi) * lo
        ld = ld + torch.log(hi - lo) + (t if (isset(a) or isset(b)) else 0)
        cols.append(torch.exp(t) + a if isset(a) else (b - torch.exp(t) if isset(b) else t))
    return torch.stack(cols, 1), ld


def coupling_inverse_ld(y, c, op, p, s):
    K = op["knots"]
    d = y.shape[1] // 2
    yt, yc = y[:, :d], y[:, d:]
    h = torch.cat([yc, c], 1) if c is not None else yc
    bn = p["BatchNorm_0"]
    t = lambda a: torch.tensor(np.asarray(a, np.float64), dtype=y.dtype)
    h = to._batchnorm_eval(h, bn["scale"], bn["bias"], t(s["BatchNorm_0"]["mean"]), t(s["BatchNorm_0"]["var"]))
    n_dense = sum(1 for k in p if k.startswith("Dense_"))
    for j in range(n_dense - 1):
        h = to._ACT[op.get("act", "swish")](h @ p[f"Dense_{j}"]["kernel"] + p[f"Dense_{j}"]["bias"])
    j = n_dense - 1
    theta = (h @ p[f"Dense_{j}"]["kernel"] + p[f"Dense_{j}"]["bias"]).reshape(y.shape[0], d, 3 * K - 1)
    xt, ld = rqs_inverse_ld(yt, theta, K)
    return torch.cat([xt, yc], 1), ld.sum(-1)


def chain_inverse_ld(ops, params_t, stats, z, c):
    """(Chain.inverse(z, c), log|det dx/dz|) from the per-element closed form, in the dtype of z."""
    x, ld = z, torch.zeros_like(z[:, 0])
    for i in reversed(range(len(ops))):
        op, name = ops[i], f"bijectors_{i}"
        if op["kind"] == "shift_bounds":
            x, l = shift_bounds_inverse_ld(x, op, stats[name])
            ld = ld + l
        elif op["kind"] == "roll":
            x = torch.roll(x, -op["shift"], -1)
        else:
            x, l = coupling_inverse_ld(x, c, op, params_t[name], stats[name])
            ld = ld + l
    return x, ld


def nan_to_num(lp):
    fi = torch.finfo(lp.dtype)
    lp = torch.where(torch.isnan(lp), torch.full_like(lp, -math.inf), lp)
    return torch.clamp(lp, fi.min, fi.max)


def _params(variables, dtype, requires_grad=False):
    p = to.to_torch(variables.get("params", {}), requires_grad=False)
    cast = lambda t: {k: cast(v) for k, v in t.items()} if isinstance(t, dict) else t.to(dtype).requires_grad_(requires_grad)
    return cast(p)


def sample_log_prob(ops, variables, z, c, *, latent="beta", peakness=12.0, dtype=torch.float64):
    """(x, lp) as numpy arrays of ``dtype``, from the closed form."""
    params_t = _params(variables, dtype)
    zt = torch.tensor(np.asarray(z), dtype=dtype)
    ct = None if c is None else torch.tensor(np.asarray(c), dtype=dtype)
    with torch.no_grad():
        x, ld = chain_inverse_ld(ops, params_t, variables["batch_stats"], zt, ct)
        lp = nan_to_num(_latent(zt, latent, peakness) - ld)
    return x.numpy(), lp.numpy()


def jacobian_lp(ops, variables, z, c, *, latent="beta", peakness=12.0):
    """lp in float64 from log|det| of the autograd Jacobian of tests/inverse_oracle.chain_inverse, one event at a time."""
    params_t = to.to_torch(variables.get("params", {}))
    stats = variables["batch_stats"]
    zt = torch.tensor(np.asarray(z, np.float64))
    ct = None if c is None else torch.tensor(np.asarray(c, np.float64))

    def one(zr, cr):
        return io.chain_inverse(ops, params_t, stats, zr[None], None if cr is None else cr[None])[0]

    if ct is None:
        J = torch.func.vmap(torch.func.jacrev(lambda zr: one(zr, None)))(zt)
    else:
        J = torch.func.vmap(torch.func.jacrev(one, argnums=0))(zt, ct)
    with torch.no_grad():
        lp = nan_to_num(_latent(zt, latent, peakness) - torch.linalg.slogdet(J)[1])
    return lp.numpy()


def sample_log_prob_vjp(ops, variables, z, c, x_ct, lp_ct, *, latent="beta", peakness=12.0):
    """float64 autograd of (x, lp) for the cotangents x_ct (M, D) and lp_ct (M,) (either may be None): (x, lp, gz, gc,
    param grads) as numpy float64.  Rows whose lp is not finite take a zero lp cotangent (nan_to_num's constants)."""
    params_t = to.to_torch(variables.get("params", {}), requires_grad=True)
    zt = torch.tensor(np.asarray(z, np.float64)).requires_grad_(True)
    ctt = None if c is None else torch.tensor(np.asarray(c, np.float64)).requires_grad_(True)
    x, ld = chain_inverse_ld(ops, params_t, variables["batch_stats"], zt, ctt)
    raw = _latent(zt, latent, peakness) - ld
    fin = torch.isfinite(raw).detach()
    loss = 0
    if x_ct is not None:
        loss = loss + (x * torch.tensor(np.asarray(x_ct, np.float64))).sum()
    if lp_ct is not None:
        w = torch.where(fin, torch.tensor(np.asarray(lp_ct, np.float64)), torch.zeros_like(raw))
        loss = loss + (torch.where(fin, raw, torch.zeros_like(raw)) * w).sum()
    loss.backward()
    gc = None if ctt is None else ctt.grad.numpy()
    return x.detach().numpy(), nan_to_num(raw.detach()).numpy(), zt.grad.numpy(), gc, to._grads_of(params_t)
