"""
ctypes binding of the C ABI declared in include/shotfpfh_b200.h (csrc/libshotfpfh_b200.so, built for sm_100a by
`__graft_entry__.build()`).

There is no CPU fallback: importing this module without the built library, or calling into it without a CUDA
device, raises.
"""

from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_float, c_int32, c_int64, c_uint64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libshotfpfh_b200.so")
ABI_VERSION = 15

SF_OK, SF_ERR_CUDA, SF_ERR_ARG, SF_ERR_CAPACITY = 0, 1, 2, 3


class SfError(RuntimeError):
    """An SF_ERR_* status returned by the native library."""


def _load() -> ctypes.CDLL:
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing. shot_fpfh_b200 has no CPU fallback: build the CUDA library first with "
            "`python -c 'import __graft_entry__ as g; g.build()'` (needs nvcc, cross-compiles sm_100a without a GPU)."
        )
    lib = ctypes.CDLL(LIB_PATH)
    lib.sf_last_error.restype = c_char_p
    lib.sf_abi_version.restype = c_int32
    if lib.sf_abi_version() != ABI_VERSION:
        raise ImportError(f"{LIB_PATH}: ABI version {lib.sf_abi_version()} != {ABI_VERSION}; rebuild the library")
    p_i64, p_f64, p_i32 = POINTER(c_int64), POINTER(c_double), POINTER(c_int32)
    sig = {
        "sf_grid_create": [POINTER(c_void_p)],
        "sf_grid_destroy": [c_void_p],
        "sf_grid_build": [c_void_p, c_void_p, c_void_p, c_int64, c_double, c_void_p],
        "sf_grid_info": [c_void_p, p_i64, p_i64, p_f64, p_i32],
        "sf_grid_build_in_box": [c_void_p, c_void_p, c_void_p, c_int64, c_double, p_f64, p_f64, c_void_p],
        "sf_grid_geometry": [p_f64, p_f64, c_double, p_f64, p_i32, p_i64],
        "sf_grid_set_speculative": [c_void_p, c_int32],
        "sf_grid_poll": [c_void_p, p_i32],
        "sf_grid_permutation": [c_void_p, c_void_p, c_void_p, c_void_p],
        "sf_grid_arrays": [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
        "sf_radius_count": [c_void_p, c_void_p, c_int64, c_int64, c_double, c_void_p, p_i64, c_void_p],
        "sf_radius_fill": [
            c_void_p, c_void_p, c_int64, c_int64, c_double, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
        ],
        "sf_voxel_subsample": [c_void_p, c_int64, c_double, c_void_p, c_void_p, p_i64, c_void_p],
        "sf_knn": [c_void_p, c_void_p, c_int64, c_int32, c_double, c_void_p, c_void_p, c_void_p],
        "sf_pca_normals": [c_void_p, c_int64, c_void_p, c_int32, c_void_p, c_void_p, c_void_p, c_void_p],  # xyz first
        "sf_iss_saliency": [c_void_p, c_double, c_int32, c_double, c_double, c_void_p, c_void_p, c_void_p, c_void_p],
        "sf_iss_select": [c_void_p, c_void_p, c_double, c_int32, c_void_p, p_i64, c_void_p],
        "sf_orient_normals": [c_void_p, c_void_p, c_int64, c_void_p, c_int32, p_f64, c_void_p, p_i64, c_void_p],
        "sf_shot_lrf": [c_void_p, c_void_p, c_int64, c_double, c_void_p, c_void_p, c_void_p, c_void_p],
        "sf_shot_descriptor": [
            c_void_p, c_void_p, c_int64, c_double, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_void_p, c_int32,
            c_void_p,
        ],
        "sf_shot_single_scale": [
            c_void_p, c_void_p, c_int64, c_double, c_int32, c_int32, c_void_p, c_int32, c_void_p, p_i64, c_void_p,
        ],
        "sf_shot_last_deferred": [p_i64],
        "sf_profile_enable": [c_int32],
        "sf_profile_read": [POINTER(c_float)],
        "sf_spfh": [c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_int32, c_int32, p_f64, c_void_p, c_void_p],
        "sf_fpfh": [
            c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_void_p, c_int32, c_void_p, c_int64, c_void_p, c_int32,
            c_void_p,
        ],
        "sf_fpfh_cloud": [c_void_p, c_double, c_int32, c_int32, p_f64, c_void_p, c_int64, c_void_p, c_int32, p_i64, c_void_p],
        "sf_nonempty_rows": [c_void_p, c_int64, c_int32, c_void_p, p_i64, p_f64, c_void_p],
        "sf_match_certify": [c_void_p, c_int32, c_void_p, c_void_p, c_void_p, c_int64, c_double, c_double, c_int32, c_int64,
                             c_int32, c_void_p, c_void_p],
        "sf_match_exhaustive": [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_int64, c_int32,
                                c_double, c_double, c_void_p, c_void_p],
        "sf_match_exhaustive_topk": [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_int32, c_int32,
                                     c_void_p, c_void_p],
        "sf_match_pack": [c_void_p, c_int32, c_void_p, c_int64, c_double, c_void_p, c_int32, c_void_p, c_void_p],
        "sf_match_topk": [
            c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_int32,
            c_void_p,
        ],
        "sf_topk_merge": [c_void_p, c_void_p, c_int32, c_int64, c_int32, c_void_p, c_void_p, c_void_p],
        "sf_nearest_merge": [c_void_p, c_int32, c_int64, c_void_p, c_void_p, c_void_p, c_void_p],
        "sf_match_rerank": [
            c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int32, c_void_p, c_int32, c_void_p, c_void_p, c_void_p,
            c_void_p,
        ],
        "sf_ransac_count_inliers": [c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_double, c_void_p, c_void_p],
        "sf_ransac_adaptive": [c_void_p, c_void_p, c_int64, c_double, c_double, c_uint64, c_int64, c_double, p_f64,
                               p_i64, p_i64, p_i64, p_i64, c_void_p, c_void_p],
        "sf_ransac_adaptive_batch": [c_void_p, c_void_p, c_int64, c_double, c_double, c_uint64, c_int64, c_int64,
                                     c_void_p, c_void_p, c_void_p, c_void_p, p_i64, c_void_p],
        "sf_icp_plane_step": [c_void_p, c_void_p, c_int64, p_f64, c_double, p_f64, c_void_p, c_void_p],
        "sf_fpfh_row_stride": [c_int32, POINTER(c_int32)],
        "sf_fpfh_block_begin": [c_void_p, c_double, c_int64, c_int64, c_void_p, p_i64, c_void_p],
        "sf_fpfh_block_spfh": [c_void_p, c_double, c_int32, c_int32, p_f64, c_int64, c_int64, c_void_p, c_void_p,
                               c_void_p, c_void_p, c_void_p, p_i64, c_void_p],
        "sf_fpfh_block_rows": [c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int32,
                               c_void_p, c_int64, c_void_p, c_int32, c_void_p],
        "sf_rows_compact_count": [c_void_p, c_int64, c_int32, c_void_p, p_i64, c_void_p],
        "sf_rows_compact_fill": [c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_void_p],
        "sf_host_expand_rows_begin": [c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_void_p, c_int32],
        "sf_host_widen_begin": [c_void_p, c_int64, c_void_p, c_int32],
        "sf_host_copy_begin": [c_void_p, c_void_p, c_int64, c_int32],
        "sf_host_advise_huge": [c_void_p, c_int64],
        "sf_host_wait": [],
    }
    for name, argtypes in sig.items():
        fn = getattr(lib, name)  # AttributeError here = the library does not export what the header declares
        fn.argtypes = argtypes
        fn.restype = c_int32
    return lib


lib = _load()
EXPORTS = (
    "sf_last_error sf_abi_version sf_grid_create sf_grid_destroy sf_grid_build sf_grid_info sf_grid_build_in_box sf_grid_geometry sf_grid_set_speculative sf_grid_poll sf_grid_permutation sf_grid_arrays "
    "sf_radius_count sf_radius_fill sf_voxel_subsample sf_knn sf_pca_normals sf_iss_saliency sf_iss_select sf_orient_normals sf_shot_lrf sf_shot_descriptor sf_shot_single_scale sf_shot_last_deferred sf_profile_enable sf_profile_read sf_spfh sf_fpfh sf_fpfh_cloud sf_fpfh_row_stride sf_fpfh_block_begin sf_fpfh_block_spfh sf_fpfh_block_rows sf_nonempty_rows sf_match_certify sf_match_exhaustive sf_match_exhaustive_topk sf_match_pack "
    "sf_match_topk sf_topk_merge sf_nearest_merge sf_match_rerank sf_ransac_count_inliers sf_ransac_adaptive sf_ransac_adaptive_batch sf_icp_plane_step sf_rows_compact_count sf_rows_compact_fill "
    "sf_host_expand_rows_begin sf_host_widen_begin sf_host_copy_begin sf_host_advise_huge sf_host_wait"
).split()


def check(status: int) -> None:
    if status != SF_OK:
        raise SfError(f"shotfpfh_b200 status {status}: {lib.sf_last_error().decode(errors='replace')}")


__all__ = ["lib", "check", "SfError", "LIB_PATH", "EXPORTS", "c_float"]
