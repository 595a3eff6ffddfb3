"""ctypes binding of libtgn_b200.so (include/tgn_b200.h).

The library is the product: if it is missing or a call fails this module raises -- there is no
CPU or PyTorch fallback.  PyTorch is used only for device memory and streams.
"""
from __future__ import annotations

import ctypes
import os
from typing import Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_lib", "libtgn_b200.so")
_lib: Optional[ctypes.CDLL] = None

_vp, _i, _f = ctypes.c_void_p, ctypes.c_int, ctypes.c_float

# name -> argument types of the status-returning (part 2) entry points
_SIGS = {
    "tgn_furthestsampling": [_i, _i, _vp, _vp, _vp, _vp, _vp, _i, _vp],
    "tgn_knnquery": [_i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "tgn_crop_knn": [_i, _i, _i, _i, _vp, _vp, _vp, _i, _vp],
    "tgn_pt_layer_set_cta_threshold": [_i],
    "tgn_dbscan": [_i, _vp, ctypes.c_double, _i, _vp, _vp, _vp, _vp, _vp],
    "tgn_csr_build": [ctypes.c_longlong, _i, _vp, _vp, _vp],
    "tgn_gather_backward_det": [ctypes.c_longlong, _i, _i, _vp, _vp, _vp, _vp],
    "tgn_weighted_gather_backward_det": [ctypes.c_longlong, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp],
    "tgn_knn_grid_build": [_i, _i, _vp, _vp, _vp, _vp],
    "tgn_knn_grid_query": [_i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "tgn_knn_f64_build": [_i, _vp, _vp, _vp],
    "tgn_knn_f64_query": [_i, _i, _i, _vp, _vp, _vp, _vp, _vp, ctypes.c_double, _vp, _vp, _vp, _vp],
    "tgn_grouping_forward": [_i, _i, _i, _vp, _vp, _vp, _vp],
    "tgn_grouping_backward": [_i, _i, _i, _vp, _vp, _vp, _vp],
    "tgn_interpolation_forward": [_i, _i, _i, _vp, _vp, _vp, _vp, _vp],
    "tgn_interpolation_backward": [_i, _i, _i, _vp, _vp, _vp, _vp, _vp],
    "tgn_weighted_gather": [_i, _i, _i, _vp, _vp, _vp, _vp, _i, _vp],
    "tgn_subtraction_forward": [_i, _i, _i, _vp, _vp, _vp, _vp, _vp],
    "tgn_subtraction_backward": [_i, _i, _i, _vp, _vp, _vp, _vp, _vp],
    "tgn_aggregation_forward": [_i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp],
    "tgn_aggregation_backward": [_i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "tgn_ball_query": [_i, _i, _i, _f, _i, _vp, _vp, _vp, _i, _vp],
    "tgn_three_nn": [_i, _i, _i, _vp, _vp, _vp, _vp, _vp],
    "tgn_three_nn_ex": [_i, _i, _i, _vp, _vp, _vp, _vp, _i, _vp],
    "tgn_square_distance": [_i, _i, _i, _vp, _vp, _vp, _i, _vp],
    "tgn_three_interpolate": [_i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp],
    "tgn_three_interpolate_ex": [_i, _i, _i, _i, _vp, _vp, _vp, _vp, _i, _vp],
    "tgn_gather_rows": [_i, _i, _i, _i, _vp, _vp, _vp, _vp],
    "tgn_transpose_cn": [_i, _i, _i, _vp, _vp, _vp],
    "tgn_sa_group_mlp_max": [_i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _i, _i, _i, _vp],
    "tgn_pt_layer_forward": [_vp, _vp],
    "tgn_pw_pack_weights": [_i, _i, _vp, _vp, _vp],
    "tgn_pw_layer_forward": [_vp, _vp],
    "tgn_pw_apply": [_vp, _vp],
    "tgn_pw_fill": [_vp, ctypes.c_longlong, _f, _vp],
}



class PwLayer(ctypes.Structure):
    """tgn_pw_layer_t (include/tgn_b200.h)."""
    _fields_ = [
        ("rows", _i), ("rows_per_batch", _i), ("cin", _i), ("cout", _i), ("mode", _i),
        ("seg_ptr", _vp * 2), ("seg_channels", _i * 2),
        ("seg_batch_stride", ctypes.c_longlong * 2), ("seg_row_stride", ctypes.c_longlong * 2), ("seg_chan_stride", ctypes.c_longlong * 2),
        ("xyz", _vp), ("feats", _vp), ("new_xyz", _vp), ("gidx", _vp),
        ("N", _i), ("S", _i), ("K", _i), ("D", _i), ("xyz_first", _i),
        ("in_affine", _i), ("in_update_running", _i),
        ("in_stats", _vp), ("in_gamma", _vp), ("in_beta", _vp), ("in_running_mean", _vp), ("in_running_var", _vp),
        ("in_eps", _f), ("in_momentum", _f),
        ("w_packed", _vp), ("bias", _vp), ("y", _vp), ("stats", _vp), ("ymax", _vp), ("ymin", _vp),
        ("group", _i), ("extrema_atomic", _i), ("precision", _i),
    ]


class PwApply(ctypes.Structure):
    """tgn_pw_apply_t (include/tgn_b200.h)."""
    _fields_ = [
        ("rows", _i), ("rows_per_batch", _i), ("channels", _i), ("out_channels", _i), ("out_c_offset", _i), ("relu", _i),
        ("src", _vp), ("ymin", _vp), ("out", _vp),
        ("affine", _i), ("update_running", _i),
        ("stats", _vp), ("stat_rows", ctypes.c_longlong),
        ("gamma", _vp), ("beta", _vp), ("running_mean", _vp), ("running_var", _vp),
        ("eps", _f), ("momentum", _f),
    ]


class PtLayer(ctypes.Structure):
    """tgn_pt_layer_t (include/tgn_b200.h)."""
    _fields_ = [
        ("n", _i), ("c", _i), ("K", _i),
        ("p", _vp), ("xq", _vp), ("xk", _vp), ("xv", _vp), ("idx", _vp), ("out", _vp),
        ("p_w0", _vp), ("p_b0", _vp), ("p_w1", _vp), ("p_b1", _vp),
        ("p_gamma", _vp), ("p_beta", _vp), ("p_rmean", _vp), ("p_rvar", _vp), ("p_eps", _f), ("p_momentum", _f),
        ("a_gamma", _vp), ("a_beta", _vp), ("a_rmean", _vp), ("a_rvar", _vp), ("a_eps", _f), ("a_momentum", _f),
        ("a_w", _vp), ("a_b", _vp),
        ("b_gamma", _vp), ("b_beta", _vp), ("b_rmean", _vp), ("b_rvar", _vp), ("b_eps", _f), ("b_momentum", _f),
        ("b_w", _vp), ("b_b", _vp),
        ("stats_p", _vp), ("stats_a", _vp), ("stats_b", _vp),
        ("bn_mode", _i * 3), ("update_running", _i),
    ]


# the reference's ten extern "C" launchers (part 1): void return, legacy default stream
REFERENCE_LAUNCHERS = [
    "furthestsampling_cuda_launcher", "knnquery_cuda_launcher",
    "grouping_forward_cuda_launcher", "grouping_backward_cuda_launcher",
    "interpolation_forward_cuda_launcher", "interpolation_backward_cuda_launcher",
    "subtraction_forward_cuda_launcher", "subtraction_backward_cuda_launcher",
    "aggregation_forward_cuda_launcher", "aggregation_backward_cuda_launcher",
]
EXPORTS = list(_SIGS) + REFERENCE_LAUNCHERS + ["tgn_version", "tgn_last_error", "tgn_launch_count", "tgn_pw_packed_bytes", "tgn_pw_struct_size", "tgn_knn_grid_bytes", "tgn_csr_bytes", "tgn_pt_layer_struct_size", "tgn_dbscan_bytes",
                                                  "tgn_knn_f64_bytes"]


class TgnError(RuntimeError):
    pass


def load() -> ctypes.CDLL:
    """Load the CUDA library; raise loudly if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise TgnError(
            f"{LIB_PATH} is missing: build it with `python -m toothgroupnetwork_b200.build` "
            "(nvcc, sm_100a).  toothgroupnetwork_b200 has no CPU / PyTorch fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, args in _SIGS.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = _i
    lib.tgn_last_error.restype = ctypes.c_char_p
    lib.tgn_version.restype = _i
    lib.tgn_launch_count.restype = _i
    lib.tgn_pw_packed_bytes.argtypes = [_i, _i]
    lib.tgn_pw_packed_bytes.restype = ctypes.c_size_t
    lib.tgn_csr_bytes.argtypes = [ctypes.c_longlong, _i]
    lib.tgn_csr_bytes.restype = ctypes.c_size_t
    lib.tgn_knn_grid_bytes.argtypes = [_i, _i]
    lib.tgn_knn_grid_bytes.restype = ctypes.c_size_t
    lib.tgn_dbscan_bytes.argtypes = [_i]
    lib.tgn_knn_f64_bytes.argtypes = [_i]
    lib.tgn_knn_f64_bytes.restype = ctypes.c_size_t
    lib.tgn_dbscan_bytes.restype = ctypes.c_size_t
    lib.tgn_pw_struct_size.argtypes = [_i]
    lib.tgn_pw_struct_size.restype = _i
    lib.tgn_pt_layer_struct_size.restype = _i
    if (lib.tgn_pw_struct_size(0) != ctypes.sizeof(PwLayer) or lib.tgn_pw_struct_size(1) != ctypes.sizeof(PwApply)
            or lib.tgn_pt_layer_struct_size() != ctypes.sizeof(PtLayer)):
        raise TgnError("ctypes mirror of tgn_pw_layer_t / tgn_pw_apply_t / tgn_pt_layer_t is out of date with include/tgn_b200.h")
    _lib = lib
    return lib


def launch_count() -> int:
    return int(load().tgn_launch_count())


def stream_ptr() -> int:
    return torch.cuda.current_stream().cuda_stream


def ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def call(name: str, *args) -> None:
    lib = load()
    status = getattr(lib, name)(*args)
    if status != 0:
        raise TgnError(f"{name} failed ({status}): {lib.tgn_last_error().decode()}")


def require_cuda(*tensors: Optional[torch.Tensor]) -> None:
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise TgnError("toothgroupnetwork_b200 operators need CUDA tensors (no CPU path)")
