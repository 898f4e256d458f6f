"""Float64 reference of the eval-mode log-density and its VJP.  TEST INFRASTRUCTURE ONLY.

The reference differentiates ``Flow.__call__(x, c, train=False)`` (flow.py:22-48) with ``jax.grad``: the BatchNorm and
ShiftBounds running statistics are constants there.  This restates that forward with torch float64 ops, reusing the
pieces of oracle/torch_oracle.py (spline, eval BatchNorm, activations, latent), so that torch autograd plays the part of
``jax.grad``.  It is validated against central differences (tests/test_eval_grad_host.py).
"""
from __future__ import annotations

import math

import numpy as np
import torch

from oracle import torch_oracle as to


def _shift_bounds_eval(x, op, stats):
    """bijectors.py:164-208 with train=False: the running xmin_i / xmax_i, no update."""
    bmap = {i: (a, b) for (i, a, b) in op["bounds"]}
    isset = lambda v: v is not None and np.isfinite(v)
    tiny = torch.finfo(torch.float32).smallest_normal
    cols, ld = [], torch.zeros(x.shape[0], dtype=x.dtype)
    for i in range(x.shape[1]):
        xi = x[:, i]
        a, b = bmap.get(i, (None, None))
        if isset(a) and isset(b):
            mul = 1 / (b - a)
            cols.append((xi - a) * mul)
            ld = ld + math.log(mul)
            continue
        t = xi
        if isset(a):
            t = torch.log(xi - a + tiny)
        elif isset(b):
            t = torch.log(b - xi + tiny)
        xmin, xmax = float(np.asarray(stats[f"xmin_{i}"]).reshape(-1)[0]), float(np.asarray(stats[f"xmax_{i}"]).reshape(-1)[0])
        mul = 1 / (xmax - xmin)
        cols.append(((t - xmin) * mul).clamp(0, 1))
        ld = ld + (math.log(mul) - t if (isset(a) or isset(b)) else math.log(mul))
    return torch.stack(cols, 1), ld


def eval_log_prob(ops, params_t, stats, x, c, *, latent="beta", peakness=12.0):
    """Flow.__call__(x, c, train=False) in float64 torch ops (differentiable wrt x, c and params_t)."""
    ld_total = torch.zeros(x.shape[0], dtype=x.dtype)
    for i, op in enumerate(ops):
        name = f"bijectors_{i}"
        if op["kind"] == "shift_bounds":
            x, ld = _shift_bounds_eval(x, op, stats[name])
            ld_total = ld_total + ld
        elif op["kind"] == "roll":
            x = torch.roll(x, op["shift"], -1)
        else:
            p, s = params_t[name], stats[name]
            K = op["knots"]
            d = x.shape[1] // 2
            xt, xc = x[:, :d], x[:, d:]
            h = torch.cat([xc, c], 1) if c is not None else xc
            bn = p["BatchNorm_0"]
            h = to._batchnorm_eval(h, bn["scale"], bn["bias"], torch.tensor(np.asarray(s["BatchNorm_0"]["mean"], np.float64)),
                                   torch.tensor(np.asarray(s["BatchNorm_0"]["var"], np.float64)))
            n_dense = sum(1 for k in p if k.startswith("Dense_"))
            for j in range(n_dense - 1):
                h = to._ACT[op.get("act", "swish")](h @ p[f"Dense_{j}"]["kernel"] + p[f"Dense_{j}"]["bias"])
            j = n_dense - 1
            theta = (h @ p[f"Dense_{j}"]["kernel"] + p[f"Dense_{j}"]["bias"]).reshape(x.shape[0], d, 3 * K - 1)
            yt, ld = to.rqs_forward(xt, theta, K)
            x = torch.cat([yt, xc], 1)
            ld_total = ld_total + ld
    lp = to._latent(x, latent, peakness) + ld_total
    return torch.nan_to_num(lp, nan=-math.inf, posinf=torch.finfo(torch.float32).max, neginf=torch.finfo(torch.float32).min)


def log_prob_vjp(ops, variables, x, c, ct, *, latent="beta", peakness=12.0):
    """float64 autograd of eval lp for the cotangent ct: (lp, gx, gc, param grads) as numpy float64."""
    params_t = to.to_torch(variables.get("params", {}), requires_grad=True)
    xt = torch.tensor(np.asarray(x, np.float64)).requires_grad_(True)
    ctt = None if c is None else torch.tensor(np.asarray(c, np.float64)).requires_grad_(True)
    lp = eval_log_prob(ops, params_t, variables["batch_stats"], xt, ctt, latent=latent, peakness=peakness)
    (lp * torch.tensor(np.asarray(ct, np.float64))).sum().backward()
    gc = None if ctt is None else ctt.grad.numpy()
    return lp.detach().numpy(), xt.grad.numpy(), gc, to._grads_of(params_t)
