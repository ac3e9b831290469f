"""ctypes binding of the C-ABI shared library (include/gnnjet_b200.h).

The library is the product: there is NO fallback.  If ``libgnnjet_b200.so`` is missing the import
raises with the build command; if a call returns a non-zero status a ``GnnJetError`` carries the
library's ``gj_last_error()`` text.  Only raw device pointers, sizes and the CUDA stream handle
cross this boundary -- no torch types.
"""
from __future__ import annotations

import ctypes as C
import os

GJ_MAX_LAYERS = 8
GJ_PREC_FP32, GJ_PREC_BF16 = 0, 1
GJ_METRIC_EUCLIDEAN, GJ_METRIC_MINKOWSKIAN = 0, 1
GJ_EMD_NORM, GJ_EMD_PERIODIC_PHI = 1, 2
GJ_EMD_COORDS_POLAR, GJ_EMD_COORDS_CARTESIAN = 0, 1
GJ_HMSE_ABS_CARTESIAN, GJ_HMSE_ABS_POLAR, GJ_HMSE_REL_POLAR, GJ_HMSE_REL_CARTESIAN = 0, 1, 2, 3

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgnnjet_b200.so")


class GnnJetError(RuntimeError):
    pass


class MPDesc(C.Structure):
    """``gj_mp_desc`` of include/gnnjet_b200.h (one iteration of reference graphnet.py:154-168)."""
    _fields_ = [
        ("batch", C.c_int32), ("num_nodes", C.c_int32), ("node_in", C.c_int32),
        ("n_edge_layers", C.c_int32), ("edge_widths", C.c_int32 * GJ_MAX_LAYERS),
        ("n_node_layers", C.c_int32), ("node_widths", C.c_int32 * GJ_MAX_LAYERS),
        ("alpha", C.c_float), ("metric", C.c_int32), ("precision", C.c_int32),
        ("h_ld", C.c_int32), ("h_cols", C.c_int32),
    ]


_P = C.c_void_p
_I = C.c_int32
_F = C.c_float
_SZ = C.c_size_t

# name -> (restype, argtypes); every symbol declared in include/gnnjet_b200.h
SIGNATURES = {
    "gj_mp_param_count": (_SZ, [C.POINTER(MPDesc)]),
    "gj_mp_step_fwd_workspace": (_SZ, [C.POINTER(MPDesc)]),
    "gj_mp_step_fwd": (C.c_int, [C.POINTER(MPDesc), _P, _P, _P, _P, _P, _SZ, _P]),
    "gj_mp_step_saved_bytes": (_SZ, [C.POINTER(MPDesc)]),
    "gj_mp_step_launches": (C.c_int, [C.POINTER(MPDesc), C.c_int, C.c_int]),
    "gj_mp_step_fwd_saving": (C.c_int, [C.POINTER(MPDesc), _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "gj_mp_step_bwd_saved": (C.c_int, [C.POINTER(MPDesc), _P, _P, _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "gj_mp_step_partials_bytes": (_SZ, [C.POINTER(MPDesc)]),
    "gj_mp_steps_pack": (C.c_int, [_I, C.POINTER(C.POINTER(MPDesc)), C.POINTER(_P), C.POINTER(_P), _P]),
    "gj_mp_step_fwd_packed": (C.c_int, [C.POINTER(MPDesc), _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "gj_mp_step_bwd_deferred": (C.c_int, [C.POINTER(MPDesc), _P, _P, _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "gj_mp_steps_reduce": (C.c_int, [_I, C.POINTER(C.POINTER(MPDesc)), C.POINTER(_P), C.POINTER(_P), _P]),
    "gj_mp_step_bwd_workspace": (_SZ, [C.POINTER(MPDesc)]),
    "gj_mp_step_bwd": (C.c_int, [C.POINTER(MPDesc), _P, _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "gj_chamfer_fwd_bwd": (C.c_int, [_I, _I, _I, _I, _I, _F, _F, _P, _P, _P, _P, _P, _P]),
    "gj_pair_min_dist": (C.c_int, [_I, _I, _I, _I, _I, _P, _P, _P, _P, _P]),
    "gj_assignment": (C.c_int, [_I, _I, _I, _I, _P, _P, _P, _P, _P]),
    "gj_emd_workspace": (_SZ, [_I, _I, _I]),
    "gj_emd": (C.c_int, [_I, _I, _I, _P, _P, _F, _F, _I, _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "gj_emd_loss_workspace": (_SZ, [_I, _I]),
    "gj_emd_loss": (C.c_int, [_I, _I, _I, _I, _P, _P, _F, _F, _I, _F, _P, _P, _P, _P, _SZ, _P]),
    "gj_hungarian_mse_loss_workspace": (_SZ, [_I, _I]),
    "gj_hungarian_mse_loss": (C.c_int, [_I, _I, _I, _I, _P, _P, _F, _P, _P, _P, _P, _SZ, _P]),
    "gj_adam_step_flat": (C.c_int, [_P, _P, _P, _P, _SZ, _F, _F, _F, _F, _I, _F, _F, _F, _P]),
    "gj_param_norms": (C.c_int, [_P, _SZ, _P, _P, _SZ, _P]),
    "gj_optimizer_step_flat": (C.c_int, [_I, _P, _P, _P, _P, _SZ, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, _P]),
    "gj_param_norms_workspace": (_SZ, [_SZ]),
    "gj_latent_mean_fwd": (C.c_int, [_I, _I, _I, _P, _P, _P]),
    "gj_latent_mean_bwd": (C.c_int, [_I, _I, _I, _P, _P, _P]),
    "gj_latent_extreme_fwd": (C.c_int, [_I, _I, _I, _I, _P, _P, _P]),
    "gj_latent_extreme_bwd": (C.c_int, [_I, _I, _I, _P, _P, _P, _P, _P]),
    "gj_output_transform_fwd": (C.c_int, [_SZ, _I, _I, _I, C.c_float, _P, _P, _P]),
    "gj_output_transform_bwd": (C.c_int, [_SZ, _I, _I, _I, C.c_float, _P, _P, _P, _P]),
    "gj_mse_workspace": (_SZ, []),
    "gj_mse_fwd_bwd": (C.c_int, [_SZ, C.c_double, _P, _P, _P, _P, _P, _SZ, _P]),
    "gj_linear_fwd": (C.c_int, [_I, _I, _I, _P, _P, _P, _P, _P]),
    "gj_linear_bwd_workspace": (_SZ, [_I, _I, _I]),
    "gj_linear_bwd": (C.c_int, [_I, _I, _I, _P, _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "gj_bench_edge_fwd_only": (C.c_int, [C.POINTER(MPDesc), _P, _P, _P, _P, _SZ, _P]),
    "gj_bench_edge_bwd_only": (C.c_int, [C.POINTER(MPDesc), _P, _P, _P, _P, _P, _SZ, _P]),
    "gj_bench_edge_bwd_saved_only": (C.c_int, [C.POINTER(MPDesc), _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "gj_mp_plan_info": (C.c_int, [C.POINTER(MPDesc), C.POINTER(C.c_int32)]),
    "gj_umma_selftest": (C.c_int, [_I, _I, _I, _I, _I, _P, _P, _P, _P]),
    "gj_dense_gemm": (C.c_int, [_I, _I, _I, _I, _P, _P, _P, _I, _F, _P, _I, _P, _P, _SZ, _I, _P]),
    "gj_dense_gemm_workspace": (_SZ, [_I, _I, _I, _I]),
    "gj_set_deterministic": (_I, [_I]),
    "gj_last_error": (C.c_char_p, []),
    "gj_abi_version": (_I, []),
    "gj_build_arch": (C.c_char_p, []),
}

_lib = None


def load():
    """Load the shared library once; raise loudly if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise GnnJetError(
            f"{LIB_PATH} not found: the CUDA library is the product and there is no fallback. "
            "Build it with `python -c 'import __graft_entry__ as g; g.build()'` or "
            "`make -C gnn_jet_autoencoder_b200/csrc`.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error() -> str:
    return load().gj_last_error().decode("utf-8", "replace")


def check(status: int, what: str) -> None:
    if status != 0:
        raise GnnJetError(f"{what} failed with status {status}: {last_error()}")


def make_desc(batch, num_nodes, node_in, edge_widths, node_widths, alpha, metric, precision,
              h_ld=0, h_cols=0) -> MPDesc:
    if len(edge_widths) > GJ_MAX_LAYERS or len(node_widths) > GJ_MAX_LAYERS:
        raise GnnJetError(f"at most {GJ_MAX_LAYERS} layers per edge / node network are supported")
    d = MPDesc()
    d.batch, d.num_nodes, d.node_in = int(batch), int(num_nodes), int(node_in)
    d.n_edge_layers = len(edge_widths)
    d.n_node_layers = len(node_widths)
    for i, w in enumerate(edge_widths):
        d.edge_widths[i] = int(w)
    for i, w in enumerate(node_widths):
        d.node_widths[i] = int(w)
    d.alpha = float(alpha)
    d.metric, d.precision = int(metric), int(precision)
    d.h_ld, d.h_cols = int(h_ld), int(h_cols)
    return d
