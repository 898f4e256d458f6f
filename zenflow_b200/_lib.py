"""ctypes binding of libzenflow_b200.so (the C ABI in include/zenflow_b200.h).

There is no CPU fallback: if the shared library is missing and cannot be built, or a call
returns a non-zero status, this module raises.  PyTorch is used by the callers only to own
device memory and streams; no torch type crosses this boundary (pointers and sizes only).
"""
from __future__ import annotations

import ctypes as C
import os
import threading

from . import build as _build

ABI_VERSION = 3
DP_UNIQUE_ID_BYTES = 128
ZF_MAX_LAYERS = 8
ZF_MAX_DIM = 64

OP_SHIFT_BOUNDS, OP_ROLL, OP_COUPLING = 0, 1, 2
LATENT_KINDS = {"beta": 0, "normal": 1, "truncnorm": 2, "uniform": 3}
ACT_KINDS = {"swish": 0, "relu": 1, "tanh": 2, "sigmoid": 3, "gelu": 4, "elu": 5, "softplus": 6, "leaky_relu": 7}
BOUND_NONE, BOUND_BOTH, BOUND_LOWER, BOUND_UPPER = 0, 1, 2, 3

c_float_p = C.POINTER(C.c_float)


class ZfShiftBounds(C.Structure):
    _fields_ = [
        ("kind", C.c_int32 * ZF_MAX_DIM),
        ("lo", C.c_double * ZF_MAX_DIM),
        ("hi", C.c_double * ZF_MAX_DIM),
        ("margin", C.c_double),
        ("xmin", C.c_void_p),
        ("xmax", C.c_void_p),
    ]


class ZfCoupling(C.Structure):
    _fields_ = [
        ("knots", C.c_int32),
        ("n_hidden", C.c_int32),
        ("hidden", C.c_int32 * ZF_MAX_LAYERS),
        ("bn_scale", C.c_void_p),
        ("bn_bias", C.c_void_p),
        ("bn_mean", C.c_void_p),
        ("bn_var", C.c_void_p),
        ("kernel", C.c_void_p * (ZF_MAX_LAYERS + 1)),
        ("bias", C.c_void_p * (ZF_MAX_LAYERS + 1)),
        ("act", C.c_int32),
    ]


class ZfCouplingGrads(C.Structure):
    _fields_ = [
        ("bn_scale", C.c_void_p),
        ("bn_bias", C.c_void_p),
        ("kernel", C.c_void_p * (ZF_MAX_LAYERS + 1)),
        ("bias", C.c_void_p * (ZF_MAX_LAYERS + 1)),
    ]


class ZfPhi(C.Structure):
    _fields_ = [
        ("in_dim", C.c_int32),
        ("out_dim", C.c_int32),
        ("n_hidden", C.c_int32),
        ("hidden", C.c_int32 * ZF_MAX_LAYERS),
        ("bn_scale", C.c_void_p),
        ("bn_bias", C.c_void_p),
        ("bn_mean", C.c_void_p),
        ("bn_var", C.c_void_p),
        ("kernel", C.c_void_p * (ZF_MAX_LAYERS + 1)),
        ("bias", C.c_void_p * (ZF_MAX_LAYERS + 1)),
    ]


class ZfOp(C.Structure):
    _fields_ = [
        ("kind", C.c_int32),
        ("shift", C.c_int32),
        ("shift_bounds", C.POINTER(ZfShiftBounds)),
        ("coupling", C.POINTER(ZfCoupling)),
    ]


class ZfChain(C.Structure):
    _fields_ = [
        ("dim", C.c_int32),
        ("cdim", C.c_int32),
        ("n_ops", C.c_int32),
        ("ops", C.POINTER(ZfOp)),
    ]


class ZenflowNativeError(RuntimeError):
    """A C-ABI call returned a non-zero zf_status."""


_lock = threading.Lock()
_lib = None

# name -> (restype, argtypes); every symbol include/zenflow_b200.h declares
SIGNATURES = {
    "zf_abi_version": (C.c_int32, []),
    "zf_last_error": (C.c_char_p, []),
    "zf_launch_count": (C.c_int64, []),
    "zf_launch_count_add": (None, [C.c_int64]),
    "zf_rqs_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32,
                                 C.c_void_p, C.c_void_p, C.c_void_p]),
    "zf_rqs_inverse": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32,
                                 C.c_void_p, C.c_void_p]),
    "zf_squareplus": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "zf_normalize_spline_params": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p,
                                             C.c_void_p]),
    "zf_rqs_forward_normalized": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                            C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "zf_rqs_inverse_normalized": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                            C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "zf_selftest_exact_math": (C.c_int, [C.c_void_p, C.c_void_p]),
    "zf_selftest_umma": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int32]),
    "zf_selftest_umma_f16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int32]),
    "zf_selftest_umma_bf16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int32]),
    "zf_selftest_umma_gemm": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p,
                                        C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int64,
                                        C.c_int64, C.c_int64, C.c_int64]),
    "zf_chain_workspace_bytes": (C.c_size_t, [C.POINTER(ZfChain), C.c_int64]),
    "zf_chain_forward": (C.c_int, [C.c_void_p, C.POINTER(ZfChain), C.c_void_p, C.c_void_p, C.c_int64,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "zf_debug_set_impl": (C.c_int, [C.c_char_p, C.c_char_p]),
    "zf_chain_pack": (C.c_int, [C.c_void_p, C.POINTER(ZfChain), C.c_void_p, C.c_size_t]),
    "zf_chain_forward_packed": (C.c_int, [C.c_void_p, C.POINTER(ZfChain), C.c_void_p, C.c_void_p, C.c_int64,
                                          C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "zf_chain_inverse_packed": (C.c_int, [C.c_void_p, C.POINTER(ZfChain), C.c_void_p, C.c_void_p, C.c_int64,
                                          C.c_void_p, C.c_void_p, C.c_size_t]),
    "zf_flow_log_prob_packed": (C.c_int, [C.c_void_p, C.POINTER(ZfChain), C.c_int32, C.c_float, C.c_void_p,
                                          C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_size_t]),
    "zf_flow_sample_packed": (C.c_int, [C.c_void_p, C.POINTER(ZfChain), C.c_int32, C.c_float, C.c_uint64, C.c_void_p,
                                        C.c_int64, C.c_void_p, C.c_void_p, C.c_size_t]),
    "zf_chain_bin_indices": (C.c_int, [C.c_void_p, C.POINTER(ZfChain), C.c_void_p, C.c_void_p, C.c_int64,
                                       C.c_void_p, C.c_void_p, C.c_size_t]),
    "zf_flow_sample": (C.c_int, [C.c_void_p, C.POINTER(ZfChain), C.c_int32, C.c_float, C.c_uint64, C.c_void_p, C.c_int64,
                                 C.c_void_p, C.c_void_p, C.c_size_t]),
    "zf_chain_forward_acc": (C.c_int, [C.c_void_p, C.POINTER(ZfChain), C.c_void_p, C.c_void_p, C.c_int64,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "zf_shift_bounds_minmax": (C.c_int, [C.c_void_p, C.POINTER(ZfShiftBounds), C.c_void_p, C.c_int64, C.c_int32,
                                         C.c_void_p, C.c_void_p]),
    "zf_shift_bounds_update": (C.c_int, [C.c_void_p, C.POINTER(ZfShiftBounds), C.c_int32, C.c_void_p]),
    "zf_bn_moments": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p]),
    "zf_bn_finalize": (C.c_int, [C.c_void_p, C.c_void_p, C.c_double, C.c_int32, C.c_float, C.c_void_p, C.c_void_p,
                                 C.c_void_p, C.c_void_p]),
    "zf_flow_loss_grad": (C.c_int, [C.c_void_p, C.c_int32, C.c_float, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32,
                                    C.c_double, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "zf_flow_loss_grad_ct": (C.c_int, [C.c_void_p, C.c_int32, C.c_float, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32,
                                       C.c_double, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "zf_dp_unique_id": (C.c_int, [C.c_void_p]),
    "zf_dp_comm_create": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.POINTER(C.c_void_p)]),
    "zf_dp_comm_destroy": (C.c_int, [C.c_void_p]),
    "zf_dp_comm_size": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32)]),
    "zf_dp_allreduce_sum_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64]),
    "zf_dp_allreduce_sum_f64": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64]),
    "zf_dp_allreduce_minmax_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32]),
    "zf_flow_value_and_grad_workspace_bytes": (C.c_size_t, [C.POINTER(ZfChain), C.c_int64, C.c_int64]),
    "zf_flow_value_and_grad": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(ZfChain), C.POINTER(ZfCouplingGrads),
                                         C.c_int32, C.c_float, C.c_void_p, C.c_void_p, C.c_int64, C.c_double,
                                         C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int64]),
    "zf_flow_log_prob_vjp_workspace_bytes": (C.c_size_t, [C.POINTER(ZfChain), C.c_int64, C.c_int64]),
    "zf_flow_log_prob_vjp": (C.c_int, [C.c_void_p, C.POINTER(ZfChain), C.POINTER(ZfCouplingGrads), C.c_int32, C.c_float,
                                       C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_size_t, C.c_int64]),
    "zf_chain_inverse_vjp_workspace_bytes": (C.c_size_t, [C.POINTER(ZfChain), C.c_int64, C.c_int64]),
    "zf_chain_inverse_vjp": (C.c_int, [C.c_void_p, C.POINTER(ZfChain), C.POINTER(ZfCouplingGrads), C.c_void_p, C.c_int32,
                                       C.c_float, C.c_uint64, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_size_t, C.c_int64]),
    "zf_flow_sample_log_prob": (C.c_int, [C.c_void_p, C.POINTER(ZfChain), C.c_int32, C.c_float, C.c_uint64, C.c_void_p,
                                          C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "zf_flow_sample_log_prob_vjp_workspace_bytes": (C.c_size_t, [C.POINTER(ZfChain), C.c_int64, C.c_int64]),
    "zf_flow_sample_log_prob_vjp": (C.c_int, [C.c_void_p, C.POINTER(ZfChain), C.POINTER(ZfCouplingGrads), C.c_void_p,
                                              C.c_int32, C.c_float, C.c_uint64, C.c_void_p, C.c_int64, C.c_void_p,
                                              C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                              C.c_size_t, C.c_int64]),
    "zf_phi_workspace_bytes": (C.c_size_t, [C.POINTER(ZfPhi), C.c_int64]),
    "zf_phi_forward": (C.c_int, [C.c_void_p, C.POINTER(ZfPhi), C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64,
                                 C.c_int64, C.c_int32, C.c_float, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_size_t]),
    "zf_phi_backward": (C.c_int, [C.c_void_p, C.POINTER(ZfPhi), C.POINTER(ZfCouplingGrads), C.c_void_p, C.c_int64,
                                  C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_float, C.c_uint64, C.c_void_p,
                                  C.c_void_p, C.c_void_p, C.c_size_t]),
    "zf_coupling_backward_workspace_bytes": (C.c_size_t, [C.POINTER(ZfCoupling), C.c_int32, C.c_int32, C.c_int64]),
    "zf_coupling_backward": (C.c_int, [C.c_void_p, C.POINTER(ZfCoupling), C.POINTER(ZfCouplingGrads), C.c_int32,
                                       C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int64,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int64]),
    "zf_bn_param_grads": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "zf_bn_backward_apply": (C.c_int, [C.c_void_p, C.POINTER(ZfCoupling), C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_double, C.c_int64, C.c_void_p, C.c_void_p]),
    "zf_nadamw_update": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                   C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, C.c_int32]),
    "zf_nadamw_update_dev": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, C.c_int32]),
    "zf_permute_rows": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_uint64, C.c_void_p]),
    "zf_neg_sum": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "zf_chain_inverse": (C.c_int, [C.c_void_p, C.POINTER(ZfChain), C.c_void_p, C.c_void_p, C.c_int64,
                                   C.c_void_p, C.c_void_p, C.c_size_t]),
    "zf_flow_log_prob": (C.c_int, [C.c_void_p, C.POINTER(ZfChain), C.c_int32, C.c_float, C.c_void_p,
                                   C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_size_t]),
}


def library_path() -> str:
    return _build.LIB_PATH


def load():
    """Load (building first if the in-tree .so is absent or stale and nvcc exists)."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        path = _build.LIB_PATH
        if os.environ.get("ZENFLOW_B200_NO_BUILD") != "1":
            try:
                _build.nvcc_path()
                have_nvcc = True
            except RuntimeError:
                have_nvcc = False
            if have_nvcc:
                path = _build.build()   # a compile error on edited sources must surface, never a stale library
            elif not os.path.exists(path):
                raise ImportError(f"zenflow_b200: native library {path} is missing and there is no nvcc to build it")
            elif not _build.is_fresh():
                import warnings

                warnings.warn(f"zenflow_b200: {path} was not built from the sources in this tree (build.stamp differs) "
                              "and there is no nvcc to rebuild it", RuntimeWarning)
        if not os.path.exists(path):
            raise ImportError(f"zenflow_b200: native library {path} is missing (run python -m zenflow_b200.build)")
        lib = C.CDLL(path)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        ver = lib.zf_abi_version()
        if ver != ABI_VERSION:
            raise ImportError(f"zenflow_b200: ABI version {ver} != {ABI_VERSION} (stale {path}? run python -m zenflow_b200.build)")
        _lib = lib
        return lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().zf_last_error().decode(errors="replace")
        raise ZenflowNativeError(f"{what or 'zenflow_b200'} failed (status {rc}): {msg}")


def set_impl(chain_impl=None, gemm_impl=None) -> None:
    """Developer switch: force a chain kernel / train GEMM implementation (None = automatic)."""
    enc = lambda v: None if not v else v.encode()
    check(load().zf_debug_set_impl(enc(chain_impl), enc(gemm_impl)), "zf_debug_set_impl")


def launch_count() -> int:
    return int(load().zf_launch_count())
