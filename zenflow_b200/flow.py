"""The Flow class — host-side mirror of zenflow/flow.py (a trainable conditional normalizing flow).

``Flow.__call__`` (eval) is a single fused kernel launch: ShiftBounds, every coupling's
conditioner MLP and spline, the Roll renamings, the latent log-pdf and nan_to_num
(zf_flow_log_prob).  When torch grad mode is on and x, c or a params leaf is a tensor that
requires grad, the result is differentiable: its backward is one zf_flow_log_prob_vjp call
(the running statistics stay fixed, as under jax.grad of the reference's eval call).  ``Flow.sample`` draws the latent
on the device and runs the fused inverse chain (zf_flow_sample); ``Flow.inverse`` runs it on a given draw
(zf_chain_inverse).  Both are differentiable in the same way, wrt c and the params leaves (and u for ``inverse``): the
backward is one zf_chain_inverse_vjp call.  ``Flow.sample_and_log_prob`` / ``Flow.inverse_and_log_prob`` return the
samples together with their log-density from one fused inverse pass (zf_flow_sample_log_prob), differentiable the
same way through one zf_flow_sample_log_prob_vjp call (reverse-KL fitting, importance weights, entropy estimates).
"""
from __future__ import annotations

from typing import Optional, Union

import numpy as np
import torch

from ._chain import (ChainSpec, _wants_grad, flow_inverse_differentiable, flow_inverse_log_prob_differentiable,
                     flow_log_prob_differentiable, flow_sample_differentiable, flow_sample_log_prob_differentiable)
from ._device import like_input
from .bijectors import Bijector, Chain, _cdim, _shape2
from .distributions import Beta, Distribution
from .module import Module

__all__ = ["Flow"]

_DEFAULT_LATENT = Beta()  # flow.py:20: the default instance is shared between Flow objects


def _normalize_c(c):
    """flow.py:98-101."""
    if c is not None and c.ndim == 1:
        c = c.reshape(-1, 1)
    return c


def _any_wants_grad(tree) -> bool:
    if isinstance(tree, dict):
        return any(_any_wants_grad(v) for v in tree.values())
    return _wants_grad(tree)


class Flow(Module):
    """A conditional normalizing flow (flow.py:16-95)."""

    def __init__(self, bijector: Bijector, latent: Distribution = _DEFAULT_LATENT):
        self.bijector = bijector
        self.latent = latent

    def __call__(self, x, c=None, *, train: bool = False):
        """Return log-likelihood of the samples: x (N, D), c (N, K) / (N,) / None -> (N,).

        With ``train=False``, torch grad mode on, and x, c or a ``params`` leaf a tensor that requires grad, the result
        is a CUDA tensor with a grad_fn (whatever the type of x): backward gives each of them its gradient in its own
        device, dtype and shape, with the running statistics held fixed (the reference's jax.grad of this call)."""
        c = _normalize_c(c)
        D = _shape2(x)[1]
        self.latent._latch_dim(D)  # distributions.py:31-32 via latent.log_prob
        child = self.scope.child("bijector")
        if self.is_initializing():
            with self.bijector._bound(child):
                self.bijector(x, c, train)
            return np.zeros(x.shape[0], np.float32)
        if not train:
            spec = ChainSpec(D, _cdim(c))
            kind, peak = self.latent._native()
            if torch.is_grad_enabled() and (_wants_grad(x) or _wants_grad(c) or _any_wants_grad(self.scope.subtree("params"))):
                # differentiable: a CUDA tensor with a grad_fn whatever the type of x
                with torch.no_grad():
                    self.bijector._emit(spec, child)
                return flow_log_prob_differentiable(spec, x, c, kind, peak)
            self.bijector._emit(spec, child)
            return like_input(spec.log_prob(x, c, kind, peak), x)
        from . import _train

        return _train.flow_train_log_prob(self, x, c)

    def sample(self, conditions_or_size: Union[int, "np.ndarray", "torch.Tensor"], *, seed: int = 0,
               as_numpy: Optional[bool] = None):
        """Return samples from the learned distribution (flow.py:50-78).

        Return type: like every entry point of the package the result mirrors the input - numpy conditions give a
        numpy array, torch conditions a CUDA tensor.  An int size has nothing to mirror: the samples stay on the
        device (CUDA ``torch.Tensor``), as for ``Distribution.sample``.  ``as_numpy=True`` / ``False`` overrides
        either way (``flow.apply(v, 1000, method="sample", as_numpy=True)`` for host-side plotting code).

        With torch grad mode on and c or a ``params`` leaf a tensor that requires grad, the samples are differentiable
        (reparameterised: x = T^-1(z; c, params) with the draw z a constant): the result is then a CUDA tensor with a
        grad_fn whatever the type of the conditions, unless ``as_numpy=True``, which still returns a detached host
        array."""
        if isinstance(conditions_or_size, (int, np.integer)):
            size = int(conditions_or_size)
            c = None
        else:
            size = conditions_or_size.shape[0]
            c = _normalize_c(conditions_or_size)
        if self.latent.dim is None:
            raise ValueError("latent.dim is not set yet: evaluate the flow (init/apply) once before sampling")
        from .distributions import _seed_of

        spec = ChainSpec(self.latent.dim, _cdim(c))
        kind, peak = self.latent._native()
        if as_numpy is not True and torch.is_grad_enabled() and (
                _wants_grad(c) or _any_wants_grad(self.scope.subtree("params"))):
            with torch.no_grad():
                self.bijector._emit(spec, self.scope.child("bijector"))
            return flow_sample_differentiable(spec, size, c, kind, peak, _seed_of(seed))
        self.bijector._emit(spec, self.scope.child("bijector"))
        # latent.sample(size, PRNGKey(seed)) and bijector.inverse in one fused pass (flow.py:76-77)
        x = spec.sample(size, c, kind, peak, _seed_of(seed))
        if as_numpy is None:
            as_numpy = not (c is None or isinstance(c, torch.Tensor))
        return x.cpu().numpy() if as_numpy else x

    def inverse(self, u, c=None):
        """bijector.inverse(u, c) with the latent draw given (flow.py:77); the parity-mode
        counterpart of ``sample`` since jax.random streams cannot be reproduced here.

        With torch grad mode on and u, c or a ``params`` leaf a tensor that requires grad, the result is a CUDA tensor
        with a grad_fn (whatever the type of u), differentiable wrt each of them with the running statistics fixed."""
        c = _normalize_c(c)
        spec = ChainSpec(_shape2(u)[1], _cdim(c))
        if torch.is_grad_enabled() and (_wants_grad(u) or _wants_grad(c) or _any_wants_grad(self.scope.subtree("params"))):
            with torch.no_grad():
                self.bijector._emit(spec, self.scope.child("bijector"))
            return flow_inverse_differentiable(spec, u, c)
        self.bijector._emit(spec, self.scope.child("bijector"))
        return like_input(spec.inverse(u, c), u)

    def sample_and_log_prob(self, conditions_or_size: Union[int, "np.ndarray", "torch.Tensor"], *, seed: int = 0,
                            as_numpy: Optional[bool] = None):
        """Return ``(x, lp)``: the samples ``sample`` returns for the same arguments (bit for bit) and their
        log-density, from one fused inverse pass.

        lp = nan_to_num(sum_j log p_latent(z_j) - log|det dx/dz|) is the exact density of the map that produced x: the
        change of variables of the inverse as the reference writes it (the analytic quadratic-root spline inverse, no EPS,
        no clip; ShiftBounds.inverse's scale).  It is not ``self(x, c)`` evaluated on the samples, which differs by the
        forward's EPS terms and clip and by bin flips near knots.  Return types and differentiability follow ``sample``:
        with grad mode on and c or a ``params`` leaf requiring grad, both outputs are CUDA tensors with grad_fns (the
        draw is a constant), unless ``as_numpy=True``."""
        if isinstance(conditions_or_size, (int, np.integer)):
            size = int(conditions_or_size)
            c = None
        else:
            size = conditions_or_size.shape[0]
            c = _normalize_c(conditions_or_size)
        if self.latent.dim is None:
            raise ValueError("latent.dim is not set yet: evaluate the flow (init/apply) once before sampling")
        from .distributions import _seed_of

        spec = ChainSpec(self.latent.dim, _cdim(c))
        kind, peak = self.latent._native()
        if as_numpy is not True and torch.is_grad_enabled() and (
                _wants_grad(c) or _any_wants_grad(self.scope.subtree("params"))):
            with torch.no_grad():
                self.bijector._emit(spec, self.scope.child("bijector"))
            return flow_sample_log_prob_differentiable(spec, size, c, kind, peak, _seed_of(seed))
        self.bijector._emit(spec, self.scope.child("bijector"))
        x, lp = spec.sample_log_prob(None, c, kind, peak, draw_seed=_seed_of(seed), n=size)
        if as_numpy is None:
            as_numpy = not (c is None or isinstance(c, torch.Tensor))
        return (x.cpu().numpy(), lp.cpu().numpy()) if as_numpy else (x, lp)

    def inverse_and_log_prob(self, u, c=None):
        """Return ``(x, lp)``: ``inverse(u, c)`` (bit for bit) and the log-density of x under the map that produced it
        from the latent draw u, as ``sample_and_log_prob`` defines it; the parity-mode counterpart of
        ``sample_and_log_prob``.  Differentiable wrt u, c and the params leaves as ``inverse`` is."""
        c = _normalize_c(c)
        D = _shape2(u)[1]
        self.latent._latch_dim(D)  # the log-density reads latent.log_prob(u)
        spec = ChainSpec(D, _cdim(c))
        kind, peak = self.latent._native()
        if torch.is_grad_enabled() and (_wants_grad(u) or _wants_grad(c) or _any_wants_grad(self.scope.subtree("params"))):
            with torch.no_grad():
                self.bijector._emit(spec, self.scope.child("bijector"))
            return flow_inverse_log_prob_differentiable(spec, u, c, kind, peak)
        self.bijector._emit(spec, self.scope.child("bijector"))
        x, lp = spec.sample_log_prob(u, c, kind, peak)
        return like_input(x, u), like_input(lp, u)

    def _steps(self, x, c=None, *, inverse: bool = False):
        """Per-bijector intermediate outputs (flow.py:80-95)."""
        if not isinstance(self.bijector, Chain):
            raise ValueError("only for Chain bijector")
        c = _normalize_c(c)
        results = []
        scope = self.scope.child("bijector")
        names = [f"bijectors_{i}" for i in range(len(self.bijector))]
        pairs = list(zip(names, self.bijector))
        if inverse:
            for name, b in pairs[::-1]:
                with b._bound(scope.child(name)):
                    x = b.inverse(x, c)
                results.append(x)
        else:
            for name, b in pairs:
                with b._bound(scope.child(name)):
                    x, _ = b(x, c, False)
                results.append(x)
        return results
