"""Float64 reference of the inverse chain and its VJP.  TEST INFRASTRUCTURE ONLY.

The reference differentiates ``Chain.inverse`` (bijectors.py:113-116; ``flow.apply(v, u, c, method="inverse")`` and the
inverse pass of ``method="sample"``) with ``jax.grad``.  The inverse is always eval-mode: the BatchNorm and ShiftBounds
running statistics are constants.  This restates it with torch float64 ops, reusing the spline normalisation, eval
BatchNorm and activations of oracle/torch_oracle.py, so that torch autograd plays the part of ``jax.grad``:
  rqs_inverse           utils.py:144-202 (bins searched in the height knots; no EPS, no clip)
  eval BatchNorm        bijectors.py:367-371 via torch_oracle._batchnorm_eval
  ShiftBounds.inverse   bijectors.py:210-240
  Roll.inverse          bijectors.py:295-297
It is validated against the numpy oracle and against central differences (tests/test_inverse_grad_host.py).

One convention differs from differentiating the reference's ``jnp.where`` literally: an element outside [0, 1) takes
the identity branch, and its discarded in-bin branch is evaluated at a safe point so that 0 * inf cannot leak NaN into
the gradients (the CUDA VJP gives such an element the pass-through cotangent and its parameters nothing).
"""
from __future__ import annotations

import numpy as np
import torch

from oracle import torch_oracle as to


def rqs_inverse(y, theta, K):
    """utils.py:144-202 on raw theta (M, d, 3K-1); in-range bins only (idx <= K-1)."""
    dx = to._softmax_thr(theta[..., :K])
    dy = to._softmax_thr(theta[..., K:2 * K])
    sl = to._squareplus(theta[..., 2 * K:])
    xk, yk = to._knots(dx), to._knots(dy)
    one = torch.ones_like(sl[..., :1])
    dk = torch.cat([one, sl, one], -1)
    sk = dy / dx
    oob = (y < 0) | (y >= 1)
    ys = torch.where(oob, torch.full_like(y, 0.5), y)   # the identity branch's discarded in-bin value, see above
    idx = ((yk <= ys[..., None]).sum(-1, keepdim=True) - 1).clamp(0, K - 1)
    g = lambda a, i: torch.take_along_dim(a, i, -1)[..., 0]
    xkk, ykk, dxk, dyk, dkk, dkp1, skk = g(xk, idx), g(yk, idx), g(dx, idx), g(dy, idx), g(dk, idx), g(dk, idx + 1), g(sk, idx)
    beta = dkp1 + dkk - 2 * skk
    a = dyk * (skk - dkk) + (ys - ykk) * beta
    b = dyk * dkk - (ys - ykk) * beta
    c = -skk * (ys - ykk)
    z = 2 * c / (-b - torch.sqrt(b * b - 4 * a * c))
    return torch.where(oob, y, z * dxk + xkk)


def _stat(stats, key):
    return float(np.asarray(stats[key]).reshape(-1)[0])


def shift_bounds_inverse(z, op, stats):
    """bijectors.py:210-240 with the running xmin_i / xmax_i."""
    bmap = {i: (a, b) for (i, a, b) in op["bounds"]}
    isset = lambda v: v is not None and np.isfinite(v)
    cols = []
    for i in range(z.shape[1]):
        zi = z[:, i]
        a, b = bmap.get(i, (None, None))
        if isset(a) and isset(b):
            cols.append(zi * b + (1 - zi) * a)
            continue
        t = zi * _stat(stats, f"xmax_{i}") + (1 - zi) * _stat(stats, f"xmin_{i}")
        cols.append(torch.exp(t) + a if isset(a) else (b - torch.exp(t) if isset(b) else t))
    return torch.stack(cols, 1)


def coupling_inverse(y, c, op, p, s):
    """bijectors.py:367-371: the conditioner reads the pass-through columns, which the inverse leaves as they are."""
    K = op["knots"]
    d = y.shape[1] // 2
    yt, yc = y[:, :d], y[:, d:]
    h = torch.cat([yc, c], 1) if c is not None else yc
    bn = p["BatchNorm_0"]
    h = to._batchnorm_eval(h, bn["scale"], bn["bias"], torch.tensor(np.asarray(s["BatchNorm_0"]["mean"], np.float64)),
                           torch.tensor(np.asarray(s["BatchNorm_0"]["var"], np.float64)))
    n_dense = sum(1 for k in p if k.startswith("Dense_"))
    for j in range(n_dense - 1):
        h = to._ACT[op.get("act", "swish")](h @ p[f"Dense_{j}"]["kernel"] + p[f"Dense_{j}"]["bias"])
    j = n_dense - 1
    theta = (h @ p[f"Dense_{j}"]["kernel"] + p[f"Dense_{j}"]["bias"]).reshape(y.shape[0], d, 3 * K - 1)
    return torch.cat([rqs_inverse(yt, theta, K), yc], 1)


def chain_inverse(ops, params_t, stats, z, c):
    """Chain.inverse(z, c) in float64 torch ops (differentiable wrt z, c and params_t)."""
    x = z
    for i in reversed(range(len(ops))):
        op, name = ops[i], f"bijectors_{i}"
        if op["kind"] == "shift_bounds":
            x = shift_bounds_inverse(x, op, stats[name])
        elif op["kind"] == "roll":
            x = torch.roll(x, -op["shift"], -1)
        else:
            x = coupling_inverse(x, c, op, params_t[name], stats[name])
    return x


def inverse_vjp(ops, variables, z, c, ct):
    """float64 autograd of Chain.inverse for the cotangent ct (M, D): (x, gz, gc, param grads) as numpy float64."""
    params_t = to.to_torch(variables.get("params", {}), requires_grad=True)
    zt = torch.tensor(np.asarray(z, np.float64)).requires_grad_(True)
    ctt = None if c is None else torch.tensor(np.asarray(c, np.float64)).requires_grad_(True)
    x = chain_inverse(ops, params_t, variables["batch_stats"], zt, ctt)
    (x * torch.tensor(np.asarray(ct, np.float64))).sum().backward()
    gc = None if ctt is None else ctt.grad.numpy()
    return x.detach().numpy(), zt.grad.numpy(), gc, to._grads_of(params_t)
