"""ctypes binding of ``include/b200icp.h`` (the drop-in C ABI).

There is NO fallback: if ``lib/libb200icp.so`` is missing or does not export every
symbol the header declares, importing this module's :func:`lib` raises.
"""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

c_i32p = C.POINTER(C.c_int32)
c_f64p = C.POINTER(C.c_double)

OK = 0
F32, F64 = 0, 1
PAIR_ROWWISE, PAIR_EXPLICIT, PAIR_TRIANGLE = 0, 1, 2
FLAG_DENSE_SWEEP = 1
FLAG_NO_SWEEP_REUSE = 2
FLAG_WARP_KERNEL = 4
FLAG_CTA_KERNEL = 8
FLAG_PAIR_WARPS_SHIFT = 8

STATUS_NAMES = {0: "OK", 1: "INVALID_ARGUMENT", 2: "UNSUPPORTED_SHAPE", 3: "CUDA", 4: "NO_DEVICE"}


class Problem(C.Structure):
    _fields_ = [
        ("src_points", C.c_void_p), ("tgt_points", C.c_void_p),
        ("src_len", C.c_void_p), ("tgt_len", C.c_void_p),
        ("src_pitch", C.c_int32), ("tgt_pitch", C.c_int32),
        ("dtype", C.c_int32), ("pairing", C.c_int32),
        ("src_row", C.c_void_p), ("tgt_row", C.c_void_p),
        ("first_pair", C.c_int64), ("n_rows", C.c_int32), ("reserved", C.c_int32),
    ]


class Options(C.Structure):
    _fields_ = [
        ("max_iterations", C.c_int32), ("flags", C.c_int32),
        ("tolerance", C.c_double), ("max_corr_dist", C.c_double),
        ("init_pose", C.c_void_p),
    ]


class Outputs(C.Structure):
    _fields_ = [
        ("pose_total", C.c_void_p), ("pose_last", C.c_void_p), ("error", C.c_void_p),
        ("rmse", C.c_void_p), ("inliers", C.c_void_p), ("iterations", C.c_void_p),
        ("indices", C.c_void_p), ("src_final", C.c_void_p), ("index_history", C.c_void_p),
        ("evaluated_pairs", C.c_void_p),
    ]


class GicpOptions(C.Structure):
    _fields_ = [
        ("max_iterations", C.c_int32), ("reserved", C.c_int32),
        ("max_corr_dist", C.c_double), ("relative_fitness", C.c_double), ("relative_rmse", C.c_double),
        ("init_pose", C.c_void_p),
    ]


class PolarFilter(C.Structure):
    _fields_ = [
        ("min_dist", C.c_double), ("max_dist", C.c_double), ("min_quality", C.c_double),
        ("arc_lo", C.c_double), ("arc_hi", C.c_double), ("use_arc", C.c_int32), ("y_sign", C.c_int32),
    ]


class S2MShard(C.Structure):
    _fields_ = [
        ("points", C.c_void_p), ("m", C.c_int64), ("global_offset", C.c_int64),
        ("dtype", C.c_int32), ("reserved", C.c_int32),
        ("chunk_circle", C.c_void_p), ("super_circle", C.c_void_p),
        ("sorted_points", C.c_void_p), ("order", C.c_void_p),
    ]


class S2MTables(C.Structure):
    _fields_ = [
        ("chunk_circle", C.c_void_p), ("super_circle", C.c_void_p),
        ("n_chunks_total", C.c_int32), ("first_local_chunk", C.c_int32),
        ("n_local_chunks", C.c_int32), ("reserved", C.c_int32),
    ]


class OccGrid(C.Structure):
    _fields_ = [
        ("probs", C.c_void_p), ("image", C.c_void_p), ("h", C.c_int32), ("w", C.c_int32),
        ("center_x", C.c_double), ("center_y", C.c_double), ("resolution", C.c_double),
        ("area", C.c_int32), ("p_occ_inc", C.c_float), ("p_free_dec", C.c_float),
        ("threshold_up", C.c_float),
    ]


# symbol -> (restype, argtypes); must list EVERY function include/b200icp.h declares
SYMBOLS = {
    "b200icp_version": (C.c_int, []),
    "b200icp_last_error": (C.c_char_p, []),
    "b200icp_max_src_pitch": (C.c_int, []),
    "b200icp_max_tgt_pitch": (C.c_int, []),
    "b200icp_nn_batch": (C.c_int, [C.POINTER(Problem), C.c_int64, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "b200icp_align_batch": (C.c_int, [C.POINTER(Problem), C.c_int64, C.POINTER(Options),
                                      C.POINTER(Outputs), C.c_void_p]),
    "b200icp_estimate_covariances": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                               C.c_double, C.c_void_p, C.c_void_p]),
    "b200icp_gicp_batch": (C.c_int, [C.POINTER(Problem), C.c_int64, C.POINTER(GicpOptions), C.c_void_p, C.c_void_p,
                                     C.POINTER(Outputs), C.c_void_p]),
    "b200icp_best_fit_batch": (C.c_int, [C.POINTER(Problem), C.c_int64, C.c_void_p, C.c_void_p]),
    "b200icp_polar_to_cartesian": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p,
                                             C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "b200icp_ffma_probe": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(C.c_int64), C.c_void_p]),
    "b200icp_select_points": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64, C.c_int32, C.c_void_p, C.c_double,
                                        C.c_double, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200icp_chain_poses": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "b200icp_voxel_workspace_bytes": (C.c_int64, [C.c_int64]),
    "b200icp_voxel_downsample": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64, C.c_double, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.c_int64, C.c_void_p]),
    "b200icp_occ_update": (C.c_int, [C.POINTER(OccGrid), C.c_int32, C.c_void_p, C.c_int32, C.c_void_p,
                                     C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]),
    "b200icp_occ_filter_points": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int64, C.c_void_p,
                                            C.c_int32, C.c_int32, C.c_double, C.c_double, C.c_double,
                                            C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200icp_s2m_chunk": (C.c_int, []),
    "b200icp_s2m_padded_chunks": (C.c_int64, [C.c_int64]),
    "b200icp_s2m_scratch_bytes": (C.c_int64, [C.c_int32]),
    "b200icp_s2m_inbox_bytes": (C.c_int64, [C.c_int32, C.c_int32]),
    "b200icp_s2m_prepare_workspace_bytes": (C.c_int64, [C.c_int64]),
    "b200icp_s2m_prepare_map": (C.c_int, [C.POINTER(S2MShard), C.c_void_p, C.c_int64, C.c_void_p]),
    "b200icp_s2m_init": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200icp_s2m_search": (C.c_int, [C.POINTER(S2MShard), C.POINTER(S2MTables), C.c_void_p, C.c_void_p,
                                     C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p,
                                     C.c_void_p, C.c_void_p]),
    "b200icp_s2m_update": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32,
                                     C.c_int32, C.c_double, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_void_p]),
    "b200icp_s2m_finish": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200icp_peer_alloc": (C.c_int, [C.c_int64, C.POINTER(C.c_void_p), C.c_void_p]),
    "b200icp_peer_open": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "b200icp_peer_close": (C.c_int, [C.c_void_p]),
    "b200icp_peer_free": (C.c_int, [C.c_void_p]),
}

_lib = None


class B200IcpError(RuntimeError):
    pass


def library_path() -> str:
    """In-tree library; ``B200ICP_LIB`` points at an alternative build (kernel A/B runs)."""
    return os.environ.get("B200ICP_LIB") or _build.LIB_PATH


def lib():
    """Load (once) and return the CUDA library.  Raises if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not os.path.exists(path):
        raise B200IcpError(
            f"{path} is missing: the CUDA library has not been built and there is no CPU "
            "fallback.  Run `python -c \"import __graft_entry__ as g; g.build()\"` in the repo root.")
    handle = C.CDLL(path)
    for name, (restype, argtypes) in SYMBOLS.items():
        try:
            fn = getattr(handle, name)
        except AttributeError as e:
            raise B200IcpError(f"{path} does not export {name}; rebuild it") from e
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = handle
    return _lib


def check(status: int, what: str) -> None:
    if status != OK:
        msg = lib().b200icp_last_error().decode("utf-8", "replace")
        raise B200IcpError(f"{what} failed: {STATUS_NAMES.get(status, status)}: {msg}")
