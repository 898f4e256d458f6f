"""Host-side assembly of the native chain description (zf_chain), the eval calls and the VJPs of the eval log-density,
of the inverse / sample pass and of the fused sample-and-log-density pass.

A ``ChainSpec`` is what the bijector modules emit: the op list of a Chain with device
pointers to the FLAX variable leaves.  It owns the torch tensors behind those pointers for
the duration of the call, and remembers which original leaf object each coupling's parameter
pointer came from (so gradients can be handed back to those objects).  No arithmetic happens here.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib
from ._device import ptr, require_cuda, stream_ptr, to_device_f32


class ChainSpec:
    def __init__(self, dim: int, cdim: int):
        if dim > _lib.ZF_MAX_DIM:
            raise ValueError(f"at most {_lib.ZF_MAX_DIM} columns are supported (got {dim})")
        self.dim = int(dim)
        self.cdim = int(cdim)
        self.device = require_cuda()
        self._ops: List[_lib.ZfOp] = []
        self._keep: list = []  # tensors and ctypes structs that must outlive the call
        # per coupling, in op order: the original params leaves (BatchNorm scale, bias, then kernel_j, bias_j per Dense)
        # and the float32 device tensors the zf_coupling points at, in zf_coupling_grads order
        self.coupling_params: List[Tuple[list, List[torch.Tensor]]] = []
        self.param_slots: List[Tuple[int, int]] = []   # (coupling, slot) of each torch leaf a differentiable call takes

    # -- emitters used by the bijectors -------------------------------------------------------
    def leaf(self, a) -> torch.Tensor:
        t = to_device_f32(a, self.device)
        self._keep.append(t)
        return t

    def add_roll(self, shift: int) -> None:
        op = _lib.ZfOp()
        op.kind = _lib.OP_ROLL
        op.shift = int(shift)
        self._ops.append(op)

    def add_shift_bounds(self, kinds: Sequence[int], lo: Sequence[float], hi: Sequence[float], margin: float,
                         xmin: Optional[torch.Tensor], xmax: Optional[torch.Tensor]) -> None:
        sb = _lib.ZfShiftBounds()
        for i in range(self.dim):
            sb.kind[i] = int(kinds[i])
            sb.lo[i] = float(lo[i])
            sb.hi[i] = float(hi[i])
        sb.margin = float(margin)
        sb.xmin = ptr(xmin)
        sb.xmax = ptr(xmax)
        self._keep += [sb, xmin, xmax]
        op = _lib.ZfOp()
        op.kind = _lib.OP_SHIFT_BOUNDS
        op.shift_bounds = C.pointer(sb)
        self._ops.append(op)

    def add_coupling(self, knots: int, hidden: Sequence[int], bn_scale, bn_bias, bn_mean, bn_var,
                     kernels: Sequence, biases: Sequence, act: int = 0) -> None:
        if len(hidden) > _lib.ZF_MAX_LAYERS:
            raise ValueError(f"at most {_lib.ZF_MAX_LAYERS} hidden layers are supported")
        cp = _lib.ZfCoupling()
        cp.knots = int(knots)
        cp.n_hidden = len(hidden)
        cp.act = int(act)
        for i, w in enumerate(hidden):
            cp.hidden[i] = int(w)
        scale_t, bias_t = self.leaf(bn_scale), self.leaf(bn_bias)
        cp.bn_scale = ptr(scale_t)
        cp.bn_bias = ptr(bias_t)
        src, dev = [bn_scale, bn_bias], [scale_t, bias_t]
        cp.bn_mean = ptr(self.leaf(bn_mean))
        cp.bn_var = ptr(self.leaf(bn_var))
        d = self.dim // 2
        fan_in = self.dim - d + self.cdim
        widths = list(hidden) + [d * (3 * knots - 1)]
        for i, (k, b) in enumerate(zip(kernels, biases)):
            kt, bt = self.leaf(k), self.leaf(b)
            if tuple(kt.shape) != (fan_in, widths[i]) or tuple(bt.shape) != (widths[i],):
                raise ValueError(f"Dense_{i}: kernel {tuple(kt.shape)} / bias {tuple(bt.shape)} do not match "
                                 f"the expected ({fan_in}, {widths[i]})")
            cp.kernel[i] = ptr(kt)
            cp.bias[i] = ptr(bt)
            src += [k, b]
            dev += [kt, bt]
            fan_in = widths[i]
        self._keep.append(cp)
        self.coupling_params.append((src, dev))
        op = _lib.ZfOp()
        op.kind = _lib.OP_COUPLING
        op.coupling = C.pointer(cp)
        self._ops.append(op)

    # -- native calls -------------------------------------------------------------------------
    def _chain(self) -> _lib.ZfChain:
        n = len(self._ops)
        arr = (_lib.ZfOp * max(n, 1))(*self._ops)
        ch = _lib.ZfChain()
        ch.dim, ch.cdim, ch.n_ops = self.dim, self.cdim, n
        ch.ops = C.cast(arr, C.POINTER(_lib.ZfOp))
        self._keep += [arr, ch]
        return ch

    def _inputs(self, x, c):
        xd = to_device_f32(x, self.device)
        if xd.ndim != 2 or xd.shape[1] != self.dim:
            raise ValueError(f"x must have shape (N, {self.dim}), got {tuple(xd.shape)}")
        cd = None
        if self.cdim:
            if c is None:
                raise ValueError("this chain is conditional: c is required")
            cd = to_device_f32(c, self.device)
            if cd.ndim == 1:
                cd = cd.reshape(-1, 1)
            if cd.shape != (xd.shape[0], self.cdim):
                raise ValueError(f"c must have shape ({xd.shape[0]}, {self.cdim}), got {tuple(cd.shape)}")
        return xd, cd

    def _workspace(self, lib, ch, M):
        nbytes = int(lib.zf_chain_workspace_bytes(C.byref(ch), M))
        ws = torch.empty(max(nbytes, 16), dtype=torch.uint8, device=self.device)
        return ws, nbytes

    def forward(self, x, c, want_y: bool = True, want_log_det: bool = True):
        lib = _lib.load()
        xd, cd = self._inputs(x, c)
        M = xd.shape[0]
        ch = self._chain()
        ws, nbytes = self._workspace(lib, ch, M)
        y = torch.empty_like(xd) if want_y else None
        ld = torch.empty(M, dtype=torch.float32, device=self.device) if want_log_det else None
        _lib.check(lib.zf_chain_forward(stream_ptr(), C.byref(ch), ptr(xd), ptr(cd), M, ptr(y), ptr(ld),
                                        ptr(ws), nbytes), "zf_chain_forward")
        return y, ld

    def bin_indices(self, x, c):
        """Bin index of every spline evaluation of the forward chain: (M, n_couplings, D//2) int32 in [0, K]
        (zf_chain_bin_indices; parity evidence, SURVEY.md H3)."""
        lib = _lib.load()
        xd, cd = self._inputs(x, c)
        M = xd.shape[0]
        ch = self._chain()
        ws, nbytes = self._workspace(lib, ch, M)
        n_c = sum(1 for op in self._ops if op.kind == _lib.OP_COUPLING)
        idx = torch.full((M, n_c, max(1, self.dim // 2)), -1, dtype=torch.int32, device=self.device)
        _lib.check(lib.zf_chain_bin_indices(stream_ptr(), C.byref(ch), ptr(xd), ptr(cd), M, ptr(idx), ptr(ws), nbytes),
                   "zf_chain_bin_indices")
        return idx

    def inverse(self, z, c):
        lib = _lib.load()
        zd, cd = self._inputs(z, c)
        M = zd.shape[0]
        ch = self._chain()
        ws, nbytes = self._workspace(lib, ch, M)
        x = torch.empty_like(zd)
        _lib.check(lib.zf_chain_inverse(stream_ptr(), C.byref(ch), ptr(zd), ptr(cd), M, ptr(x), ptr(ws), nbytes),
                   "zf_chain_inverse")
        return x

    def log_prob(self, x, c, latent_kind: int, peakness: float):
        lib = _lib.load()
        xd, cd = self._inputs(x, c)
        M = xd.shape[0]
        ch = self._chain()
        ws, nbytes = self._workspace(lib, ch, M)
        lp = torch.empty(M, dtype=torch.float32, device=self.device)
        _lib.check(lib.zf_flow_log_prob(stream_ptr(), C.byref(ch), int(latent_kind), float(peakness), ptr(xd),
                                        ptr(cd), M, ptr(lp), ptr(ws), nbytes), "zf_flow_log_prob")
        return lp

    def log_prob_vjp(self, x, c, latent_kind: int, peakness: float, lp_cotangent, *, want_gx: bool = True,
                     want_gc: bool = True, want_params: bool = True, micro_batch: int = 1 << 18, want_lp: bool = False):
        """VJP of the eval-mode log-density (zf_flow_log_prob_vjp) for the cotangent ``lp_cotangent`` (M,).

        Returns ``(gx, gc, param_grads, lp)``: float32 device tensors, None where not asked for;
        ``param_grads[k]`` lists coupling k's gradients in the order of ``coupling_params[k]``."""
        lib = _lib.load()
        xd, cd = self._inputs(x, c)
        M = xd.shape[0]
        ch = self._chain()
        ct = to_device_f32(lp_cotangent, self.device).reshape(-1)
        if ct.shape[0] != M:
            raise ValueError(f"lp_cotangent must have shape ({M},), got {tuple(ct.shape)}")
        nbytes = int(lib.zf_flow_log_prob_vjp_workspace_bytes(C.byref(ch), M, int(micro_batch)))
        if nbytes == 0:
            _lib.check(1, "zf_flow_log_prob_vjp_workspace_bytes")
        ws = torch.empty(nbytes + 256, dtype=torch.uint8, device=self.device)
        base = (ws.data_ptr() + 255) & ~255
        gx = torch.empty_like(xd) if want_gx else None
        gc = torch.empty_like(cd) if (want_gc and cd is not None) else None
        lp = torch.empty(M, dtype=torch.float32, device=self.device) if want_lp else None
        grads, arr = self._grads_array(want_params)
        _lib.check(lib.zf_flow_log_prob_vjp(stream_ptr(), C.byref(ch), arr, int(latent_kind), float(peakness), ptr(xd),
                                            ptr(cd), M, ptr(ct), ptr(lp), ptr(gx), ptr(gc), base,
                                            ws.numel() - (base - ws.data_ptr()), int(micro_batch)),
                   "zf_flow_log_prob_vjp")
        return gx, gc, grads, lp

    def _grads_array(self, want_params: bool):
        """Zeroed float32 gradient tensors of every coupling's parameters and the zf_coupling_grads array over them."""
        if not (want_params and self.coupling_params):
            return None, None
        grads = [[torch.zeros_like(t) for t in dev] for _, dev in self.coupling_params]
        arr = (_lib.ZfCouplingGrads * len(grads))()
        for k, gl in enumerate(grads):
            arr[k].bn_scale, arr[k].bn_bias = ptr(gl[0]), ptr(gl[1])
            for j in range((len(gl) - 2) // 2):
                arr[k].kernel[j] = ptr(gl[2 + 2 * j])
                arr[k].bias[j] = ptr(gl[3 + 2 * j])
        return grads, arr

    def inverse_vjp(self, z, c, x_cotangent, *, draw=None, want_gz: bool = True, want_gc: bool = True,
                    want_params: bool = True, micro_batch: int = 1 << 18, want_x: bool = False):
        """VJP of Chain.inverse(z, c) (zf_chain_inverse_vjp) for the cotangent ``x_cotangent`` (M, D) of its output.
        ``draw = (n, latent_kind, peakness, seed)`` differentiates Flow.sample's inverse pass instead: z is then the
        latent draw zf_flow_sample makes (pass z=None; there is no gz).

        Returns ``(gz, gc, param_grads, x)``: float32 device tensors, None where not asked for;
        ``param_grads[k]`` lists coupling k's gradients in the order of ``coupling_params[k]``."""
        lib = _lib.load()
        if draw is None:
            zd, cd = self._inputs(z, c)
            kind, peak, seed = 0, 1.0, 0
        else:
            n, kind, peak, seed = draw
            zd, cd = None, self._conditions(int(n), c)
            want_gz = False
        M = int(zd.shape[0]) if zd is not None else int(draw[0])
        ch = self._chain()
        ct = to_device_f32(x_cotangent, self.device)
        if tuple(ct.shape) != (M, self.dim):
            raise ValueError(f"x_cotangent must have shape ({M}, {self.dim}), got {tuple(ct.shape)}")
        nbytes = int(lib.zf_chain_inverse_vjp_workspace_bytes(C.byref(ch), M, int(micro_batch)))
        if nbytes == 0:
            _lib.check(1, "zf_chain_inverse_vjp_workspace_bytes")
        ws = torch.empty(nbytes + 256, dtype=torch.uint8, device=self.device)
        base = (ws.data_ptr() + 255) & ~255
        gz = torch.empty((M, self.dim), dtype=torch.float32, device=self.device) if want_gz else None
        gc = torch.empty_like(cd) if (want_gc and cd is not None) else None
        x = torch.empty((M, self.dim), dtype=torch.float32, device=self.device) if want_x else None
        grads, arr = self._grads_array(want_params)
        _lib.check(lib.zf_chain_inverse_vjp(stream_ptr(), C.byref(ch), arr, ptr(zd), int(kind), float(peak),
                                            int(seed) & 0xFFFFFFFFFFFFFFFF, ptr(cd), M, ptr(ct), ptr(x), ptr(gz), ptr(gc),
                                            base, ws.numel() - (base - ws.data_ptr()), int(micro_batch)),
                   "zf_chain_inverse_vjp")
        return gz, gc, grads, x

    def _draw_inputs(self, z, c, n):
        """(zd, cd, M): the float32 device tensors of a given draw z and its conditions, or (z None) zd = None and the
        conditions of ``n`` rows drawn in-kernel."""
        if z is not None:
            zd, cd = self._inputs(z, c)
            return zd, cd, int(zd.shape[0])
        return None, self._conditions(int(n), c), int(n)

    def sample_log_prob(self, z, c, latent_kind: int, peakness: float, *, draw_seed: Optional[int] = None,
                        n: Optional[int] = None, want_x: bool = True):
        """Flow.sample_and_log_prob / Flow.inverse_and_log_prob: x = Chain.inverse(z, c) and its log-density in one fused
        pass (zf_flow_sample_log_prob).  z None: draw ``n`` latent rows in-kernel with ``draw_seed`` as zf_flow_sample
        does.  Returns ``(x, lp)`` (x None when not asked for)."""
        lib = _lib.load()
        zd, cd, M = self._draw_inputs(z, c, n)
        ch = self._chain()
        ws, nbytes = self._workspace(lib, ch, M)
        x = torch.empty((M, self.dim), dtype=torch.float32, device=self.device) if want_x else None
        lp = torch.empty(M, dtype=torch.float32, device=self.device)
        seed = int(draw_seed or 0) if zd is None else 0
        _lib.check(lib.zf_flow_sample_log_prob(stream_ptr(), C.byref(ch), int(latent_kind), float(peakness),
                                               seed & 0xFFFFFFFFFFFFFFFF, ptr(zd), ptr(cd), M, ptr(x), ptr(lp), ptr(ws),
                                               nbytes), "zf_flow_sample_log_prob")
        return x, lp

    def sample_log_prob_vjp(self, z, c, latent_kind: int, peakness: float, x_cotangent=None, lp_cotangent=None, *,
                            draw_seed: Optional[int] = None, n: Optional[int] = None, want_gz: bool = True,
                            want_gc: bool = True, want_params: bool = True, micro_batch: int = 1 << 18,
                            want_x: bool = False, want_lp: bool = False):
        """Joint VJP of (x, lp) of sample_log_prob (zf_flow_sample_log_prob_vjp) for the cotangents ``x_cotangent``
        (M, D) and ``lp_cotangent`` (M,); either may be None, not both.  z None: the in-kernel draw (no gz).

        Returns ``(gz, gc, param_grads, x, lp)``: float32 device tensors, None where not asked for;
        ``param_grads[k]`` lists coupling k's gradients in the order of ``coupling_params[k]``."""
        lib = _lib.load()
        if x_cotangent is None and lp_cotangent is None:
            raise ValueError("sample_log_prob_vjp: pass x_cotangent, lp_cotangent or both")
        zd, cd, M = self._draw_inputs(z, c, n)
        if zd is None:
            want_gz = False
        ch = self._chain()
        gxc = None
        if x_cotangent is not None:
            gxc = to_device_f32(x_cotangent, self.device)
            if tuple(gxc.shape) != (M, self.dim):
                raise ValueError(f"x_cotangent must have shape ({M}, {self.dim}), got {tuple(gxc.shape)}")
        glc = None
        if lp_cotangent is not None:
            glc = to_device_f32(lp_cotangent, self.device).reshape(-1)
            if glc.shape[0] != M:
                raise ValueError(f"lp_cotangent must have shape ({M},), got {tuple(glc.shape)}")
        nbytes = int(lib.zf_flow_sample_log_prob_vjp_workspace_bytes(C.byref(ch), M, int(micro_batch)))
        if nbytes == 0:
            _lib.check(1, "zf_flow_sample_log_prob_vjp_workspace_bytes")
        ws = torch.empty(nbytes + 256, dtype=torch.uint8, device=self.device)
        base = (ws.data_ptr() + 255) & ~255
        gz = torch.empty((M, self.dim), dtype=torch.float32, device=self.device) if want_gz else None
        gc = torch.empty_like(cd) if (want_gc and cd is not None) else None
        x = torch.empty((M, self.dim), dtype=torch.float32, device=self.device) if want_x else None
        lp = torch.empty(M, dtype=torch.float32, device=self.device) if want_lp else None
        grads, arr = self._grads_array(want_params)
        seed = int(draw_seed or 0) if zd is None else 0
        _lib.check(lib.zf_flow_sample_log_prob_vjp(stream_ptr(), C.byref(ch), arr, ptr(zd), int(latent_kind),
                                                   float(peakness), seed & 0xFFFFFFFFFFFFFFFF, ptr(cd), M, ptr(gxc),
                                                   ptr(glc), ptr(x), ptr(lp), ptr(gz), ptr(gc), base,
                                                   ws.numel() - (base - ws.data_ptr()), int(micro_batch)),
                   "zf_flow_sample_log_prob_vjp")
        return gz, gc, grads, x, lp

    def _conditions(self, n: int, c):
        cd = None
        if self.cdim:
            if c is None:
                raise ValueError("this chain is conditional: pass one condition vector per sample")
            cd = to_device_f32(c, self.device)
            if cd.ndim == 1:
                cd = cd.reshape(-1, 1)
            if cd.shape != (n, self.cdim):
                raise ValueError(f"c must have shape ({n}, {self.cdim}), got {tuple(cd.shape)}")
        return cd

    def sample(self, n: int, c, latent_kind: int, peakness: float, seed: int):
        """Flow.sample: latent draw inside the inverse chain kernel (zf_flow_sample)."""
        lib = _lib.load()
        cd = self._conditions(n, c)
        ch = self._chain()
        ws, nbytes = self._workspace(lib, ch, n)
        x = torch.empty((n, self.dim), dtype=torch.float32, device=self.device)
        _lib.check(lib.zf_flow_sample(stream_ptr(), C.byref(ch), int(latent_kind), float(peakness),
                                      int(seed) & 0xFFFFFFFFFFFFFFFF, ptr(cd), n, ptr(x), ptr(ws), nbytes),
                   "zf_flow_sample")
        return x


def _wants_grad(a) -> bool:
    return isinstance(a, torch.Tensor) and a.requires_grad


def _grad_like(g: Optional[torch.Tensor], like) -> Optional[torch.Tensor]:
    """A float32 device gradient in the device, dtype and shape of the tensor it belongs to."""
    if g is None:
        return None
    return g.to(device=like.device, dtype=like.dtype).reshape(like.shape)


class _FlowLogProb(torch.autograd.Function):
    """Flow.__call__(x, c, train=False) as a differentiable op: forward = zf_flow_log_prob (the non-grad call, so lp is
    bit-identical to it), backward = one zf_flow_log_prob_vjp with the incoming gradient as the cotangent of lp.
    ``leaves`` are the torch tensors among the couplings' params leaves, in ``spec.param_slots`` order."""

    @staticmethod
    def forward(ctx, spec, latent_kind, peakness, x, c, *leaves):
        xd, cd = spec._inputs(x, c)
        ctx.spec, ctx.latent = spec, (latent_kind, peakness)
        ctx.x_like = x.detach() if isinstance(x, torch.Tensor) else None
        ctx.c_like = c.detach() if isinstance(c, torch.Tensor) else None
        ctx.save_for_backward(xd, cd)
        return spec.log_prob(xd, cd, latent_kind, peakness)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g_lp):
        xd, cd = ctx.saved_tensors
        spec = ctx.spec
        need = ctx.needs_input_grad
        want_p = any(need[5:])
        gx, gc, grads, _ = spec.log_prob_vjp(xd, cd, *ctx.latent, g_lp, want_gx=need[3], want_gc=need[4],
                                             want_params=want_p)
        out_p = []
        for i, (k, j) in enumerate(spec.param_slots):
            out_p.append(_grad_like(grads[k][j], spec.coupling_params[k][0][j]) if need[5 + i] else None)
        return (None, None, None, _grad_like(gx, ctx.x_like) if need[3] else None,
                _grad_like(gc, ctx.c_like) if need[4] else None, *out_p)


def flow_log_prob_differentiable(spec: ChainSpec, x, c, latent_kind: int, peakness: float) -> torch.Tensor:
    """The eval log-density with a grad_fn wrt every torch tensor among x, c and the couplings' params leaves."""
    return _FlowLogProb.apply(spec, latent_kind, peakness, x, c, *_param_leaves(spec))


class _FlowInverse(torch.autograd.Function):
    """Chain.inverse(z, c) (``draw`` None) or Flow.sample's inverse pass (``draw = (n, latent_kind, peakness, seed)``,
    z None) as a differentiable op: forward = zf_chain_inverse / zf_flow_sample (the non-grad calls, so x is
    bit-identical to them), backward = one zf_chain_inverse_vjp with the incoming gradient as the cotangent of x.
    ``leaves`` are the torch tensors among the couplings' params leaves, in ``spec.param_slots`` order."""

    @staticmethod
    def forward(ctx, spec, draw, z, c, *leaves):
        if draw is None:
            zd, cd = spec._inputs(z, c)
            x = spec.inverse(zd, cd)
        else:
            zd, cd = None, spec._conditions(int(draw[0]), c)
            x = spec.sample(int(draw[0]), cd, *draw[1:])
        ctx.spec, ctx.draw = spec, draw
        ctx.z_like = z.detach() if isinstance(z, torch.Tensor) else None
        ctx.c_like = c.detach() if isinstance(c, torch.Tensor) else None
        ctx.save_for_backward(zd, cd)
        return x

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g_x):
        zd, cd = ctx.saved_tensors
        spec = ctx.spec
        need = ctx.needs_input_grad
        gz, gc, grads, _ = spec.inverse_vjp(zd, cd, g_x, draw=ctx.draw, want_gz=need[2], want_gc=need[3],
                                            want_params=any(need[4:]))
        out_p = []
        for i, (k, j) in enumerate(spec.param_slots):
            out_p.append(_grad_like(grads[k][j], spec.coupling_params[k][0][j]) if need[4 + i] else None)
        return (None, None, _grad_like(gz, ctx.z_like) if need[2] else None,
                _grad_like(gc, ctx.c_like) if need[3] else None, *out_p)


def _param_leaves(spec: ChainSpec) -> list:
    spec.param_slots = [(k, j) for k, (src, _) in enumerate(spec.coupling_params)
                        for j, leaf in enumerate(src) if isinstance(leaf, torch.Tensor)]
    return [spec.coupling_params[k][0][j] for k, j in spec.param_slots]


def flow_inverse_differentiable(spec: ChainSpec, z, c) -> torch.Tensor:
    """Chain.inverse(z, c) with a grad_fn wrt every torch tensor among z, c and the couplings' params leaves."""
    return _FlowInverse.apply(spec, None, z, c, *_param_leaves(spec))


def flow_sample_differentiable(spec: ChainSpec, n: int, c, latent_kind: int, peakness: float, seed: int) -> torch.Tensor:
    """Flow.sample's draw and inverse pass with a grad_fn wrt c and the couplings' params leaves (the draw is a constant)."""
    return _FlowInverse.apply(spec, (int(n), int(latent_kind), float(peakness), int(seed)), None, c, *_param_leaves(spec))


class _FlowSampleLogProb(torch.autograd.Function):
    """Flow.inverse_and_log_prob (``n`` None: the given draw z) or Flow.sample_and_log_prob (``n`` rows drawn in-kernel
    with ``seed``, z None) as a differentiable op with two outputs (x, lp): forward = zf_flow_sample_log_prob (the
    non-grad call, so both are bit-identical to it), backward = one zf_flow_sample_log_prob_vjp with the incoming
    gradients as the cotangents; a gradient autograd does not provide is passed as NULL."""

    @staticmethod
    def forward(ctx, spec, latent, n, seed, z, c, *leaves):
        zd, cd, _ = spec._draw_inputs(z, c, n)   # the device tensors the backward reads
        x, lp = spec.sample_log_prob(zd, cd, *latent, draw_seed=seed, n=n)
        ctx.spec, ctx.latent, ctx.n, ctx.seed = spec, latent, n, seed
        ctx.z_like = z.detach() if isinstance(z, torch.Tensor) else None
        ctx.c_like = c.detach() if isinstance(c, torch.Tensor) else None
        ctx.set_materialize_grads(False)
        ctx.save_for_backward(zd, cd)
        return x, lp

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g_x, g_lp):
        zd, cd = ctx.saved_tensors
        spec = ctx.spec
        need = ctx.needs_input_grad
        n_in = 6 + len(spec.param_slots)
        if g_x is None and g_lp is None:
            return (None,) * n_in
        gz, gc, grads, _, _ = spec.sample_log_prob_vjp(zd, cd, *ctx.latent, g_x, g_lp, draw_seed=ctx.seed, n=ctx.n,
                                                       want_gz=need[4], want_gc=need[5], want_params=any(need[6:]))
        out_p = []
        for i, (k, j) in enumerate(spec.param_slots):
            out_p.append(_grad_like(grads[k][j], spec.coupling_params[k][0][j]) if need[6 + i] else None)
        return (None, None, None, None, _grad_like(gz, ctx.z_like) if need[4] else None,
                _grad_like(gc, ctx.c_like) if need[5] else None, *out_p)


def flow_inverse_log_prob_differentiable(spec: ChainSpec, z, c, latent_kind: int, peakness: float):
    """(Chain.inverse(z, c), its log-density) with grad_fns wrt every torch tensor among z, c and the params leaves."""
    return _FlowSampleLogProb.apply(spec, (int(latent_kind), float(peakness)), None, 0, z, c, *_param_leaves(spec))


def flow_sample_log_prob_differentiable(spec: ChainSpec, n: int, c, latent_kind: int, peakness: float, seed: int):
    """Flow.sample's draw, inverse pass and log-density with grad_fns wrt c and the params leaves (the draw is a constant)."""
    return _FlowSampleLogProb.apply(spec, (int(latent_kind), float(peakness)), int(n), int(seed), None, c,
                                    *_param_leaves(spec))
