"""ctypes binding of libgsx.so (the C ABI declared in include/gsx.h).

There is deliberately NO fallback here: if the shared library is missing, or a tensor handed to a compute
op is not a CUDA tensor, the call raises.  Build the library with `python __graft_entry__.py build` (or
`python -m gradslam_b200.build`).
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# GSX_LIB_PATH selects another build of the same ABI (kernel tuning variants); never a fallback.
LIB_PATH = os.environ.get("GSX_LIB_PATH") or os.path.join(_HERE, "_lib", "libgsx.so")

c_f32p = ctypes.c_void_p
c_i32p = ctypes.c_void_p
c_i64 = ctypes.c_int64
c_int = ctypes.c_int
c_float = ctypes.c_float
c_double = ctypes.c_double
c_u32 = ctypes.c_uint32
c_vp = ctypes.c_void_p

# name -> (restype, argtypes); must list every symbol include/gsx.h declares (tests/test_abi.py checks)
SIGNATURES = {
    "gsx_version": (c_int, []),
    "gsx_last_error": (ctypes.c_char_p, []),
    "gsx_backproject_normals_fwd": (
        c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_int, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "gsx_backproject_normals_bwd_scratch_bytes": (c_i64, [c_int, c_int, c_int, c_int]),
    "gsx_backproject_normals_bwd": (
        c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_int, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp,
                c_vp, c_i64, c_vp]),
    "gsx_fusion_workspace_bytes": (c_i64, [c_int, c_int, c_int]),
    "gsx_fusion_workspace_stats_offset": (c_i64, [c_int, c_int, c_int]),
    "gsx_fusion_frame_records": (
        c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_double, c_vp, c_vp]),
    "gsx_fusion_project_select": (
        c_int, [c_vp, c_vp, c_i64, c_i64, c_vp, c_i64, c_vp, c_i64, c_int, c_int, c_int, c_float, c_float, c_vp, c_vp]),
    "gsx_fusion_merge_append": (
        c_int, [c_vp, c_vp, c_int, c_vp, c_vp, c_i64, c_vp, c_i64, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp]),
    "gsx_fusion_merge_append_bwd": (
        c_int, [c_vp, c_vp, c_vp, c_vp, c_int, c_i64, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int,
                c_double, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "gsx_pointfusion_sequence_groups": (c_int, [c_int]),
    "gsx_pointfusion_sequence_workspace_bytes": (c_i64, [c_int, c_int, c_int]),
    "gsx_pointfusion_sequence_gt": (
        c_int, [c_vp, c_vp, c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_int, c_int, c_int,
                c_float, c_float, c_double, c_vp, c_vp, c_vp]),
    "gsx_debug_fail_at_frame": (None, [c_int]),
    "gsx_peer_export": (c_int, [c_vp, c_vp, c_vp, c_vp]),
    "gsx_peer_open": (c_int, [c_vp, c_i64, c_vp]),
    "gsx_peer_close_all": (c_int, []),
    "gsx_peer_copy_rows": (c_int, [c_vp, c_i64, c_vp, c_i64, c_i64, c_i64, c_vp]),
    "gsx_ingest_raw": (c_int, [c_vp, c_vp, c_i64, c_double, c_int, c_vp, c_vp, c_vp]),
    "gsx_ingest_calibration": (c_int, [c_vp, c_i64, c_int, c_double, c_double, c_vp, c_vp, c_int, c_int, c_vp, c_vp,
                                       c_vp]),
    "gsx_compact_scratch_bytes": (c_i64, [c_i64]),
    "gsx_compact_indices": (c_int, [c_vp, c_i64, c_vp, c_vp, c_vp, c_u32, c_vp]),
    "gsx_active_eval": (c_int, [c_vp, c_vp, c_i64, c_i64, c_vp, c_i64, c_vp, c_i64, c_int, c_int, c_int, c_vp, c_vp,
                                c_vp]),
    "gsx_similar_eval": (c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_int, c_int, c_int, c_float, c_float, c_vp,
                                 c_vp]),
    "gsx_unique_select": (c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp]),
    "gsx_records_from_table": (c_int, [c_vp, c_i64, c_i64, c_int, c_int, c_int, c_vp, c_vp]),
    "gsx_knn1_scratch_bytes": (c_i64, [c_int, c_int, c_int]),
    "gsx_icp_tgt_scratch_bytes": (c_i64, [c_int, c_i64]),
    "gsx_knn1": (c_int, [c_vp, c_vp, c_int, c_vp, c_vp, c_int, c_int, c_vp, c_vp, c_vp, c_i64, c_int, c_vp]),
    "gsx_icp_normal_eq_scratch_bytes": (c_i64, [c_int]),
    "gsx_icp_normal_eq_batched_fwd": (c_int, [c_vp, c_vp, c_int, c_vp, c_vp, c_int, c_int, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "gsx_icp_normal_eq_batched_bwd": (c_int, [c_vp, c_vp, c_int, c_vp, c_vp, c_int, c_int, c_vp, c_vp, c_vp, c_vp, c_vp,
                                              c_vp]),
    "gsx_icp_solve_fwd": (c_int, [c_vp, c_vp, c_int, c_vp, c_vp, c_vp]),
    "gsx_icp_solve_bwd": (c_int, [c_vp, c_vp, c_int, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "gsx_icp_update_fwd": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_float, c_float, c_float, c_float,
                                   c_vp, c_vp, c_vp, c_vp]),
    "gsx_icp_update_bwd": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_float, c_float, c_float, c_float,
                                   c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "gsx_rigid_transform_bwd_scratch_bytes": (c_i64, [c_i64]),
    "gsx_rigid_transform_batched_fwd": (c_int, [c_vp, c_vp, c_i64, c_int, c_vp, c_vp, c_vp]),
    "gsx_rigid_transform_batched_bwd": (c_int, [c_vp, c_vp, c_i64, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "gsx_icp_align_scratch_bytes": (c_i64, [c_int, c_int, c_int]),
    "gsx_icp_align": (
        c_int, [c_vp, c_vp, c_int, c_vp, c_vp, c_vp, c_int, c_int, c_vp, c_int, c_int, c_float, c_int, c_float,
                c_float, c_float, c_float, c_float, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "gsx_icp_workspace_bytes": (c_i64, [c_int, c_int, c_int, c_int, c_i64]),
    "gsx_icp_localize": (
        c_int, [c_vp, c_vp, c_i64, c_i64, c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_int, c_int, c_int, c_int,
                c_int, c_int, c_float, c_int, c_float, c_float, c_float, c_float, c_float, c_vp, c_i64, c_vp, c_i64,
                c_vp, c_i64, c_u32, c_vp, c_vp]),
}

_lib = None


def lib():
    """Loads libgsx.so (once).  Raises RuntimeError if it has not been built — never falls back."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "gradslam_b200: CUDA extension %s is missing. Build it with `python __graft_entry__.py build`. "
                "There is no CPU fallback." % LIB_PATH
            )
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(rc, what):
    if rc != 0:
        raise RuntimeError("%s failed (status %d): %s" % (what, rc, lib().gsx_last_error().decode()))


def require_cuda(t, name):
    if not t.is_cuda:
        raise RuntimeError(
            "gradslam_b200: `%s` must be a CUDA tensor (got device %s); the engine has no CPU path." % (name, t.device)
        )
    if t.dtype != torch.float32:
        raise TypeError("gradslam_b200: `%s` must be float32 (got %s)." % (name, t.dtype))


def ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def stream_ptr(device=None):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)
