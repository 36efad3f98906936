"""ctypes binding of libvggsfm_b200.so (the C ABI declared in include/vggsfm_b200.h).

The product path has NO fallback: if the shared library is missing this raises, it never routes to
PyTorch eager or to the CPU oracle.
"""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libvggsfm_b200.so")

# every symbol include/vggsfm_b200.h declares (tests/test_abi.py checks the two lists agree)
EXPORTS = [
    "vgg_last_error", "vgg_version",
    "vgg_ba_default_options", "vgg_ba_dims", "vgg_ba_workspace_bytes", "vgg_ba_camrec_len",
    "vgg_ba_build_blocks", "vgg_ba_schur", "vgg_cholesky_lower", "vgg_ba_solve",
    "vgg_ba_reduced_system_doubles", "vgg_ba_fabric_doubles", "vgg_ba_solve_fabric",
    "vgg_pose_default_options", "vgg_pose_refinement", "vgg_pnp_workspace_bytes", "vgg_absolute_pose_estimation", "vgg_syrk_ozaki_workspace_bytes", "vgg_syrk_ozaki",
    "vgg_tri_workspace_bytes", "vgg_triangulate_tracks", "vgg_triangulate_by_pair", "vgg_filter_points3d",
    "vgg_project_points", "vgg_normalize_tracks", "vgg_undistort_simple_radial",
    "vgg_corr_pyramid_bytes", "vgg_corr_build_pyramid", "vgg_corr_sample", "vgg_sample_features4d",
    "vgg_corr_tc_supported", "vgg_corr_tc_bytes", "vgg_corr_tc_build", "vgg_corr_tc_sample",
]


# development probes (csrc/dev_probes.h): exported, not part of the public header
DEV_EXPORTS = ["vgg_syrk_ozaki_mma_rate", "vgg_dev_blocks_timing", "vgg_dev_blocks_last_ms",
               "vgg_dev_chol128_probe", "vgg_dev_set_syrk_ranges", "vgg_dev_trsv_probe", "vgg_dev_set_chol_band"]


class BAProblem(ctypes.Structure):
    _fields_ = [
        ("S", ctypes.c_int32), ("N", ctypes.c_int32),
        ("camera_model", ctypes.c_int32), ("intr_mode", ctypes.c_int32),
        ("uv", ctypes.c_void_p), ("mask", ctypes.c_void_p),
        ("param_const", ctypes.c_void_p), ("point_const", ctypes.c_void_p),
        ("poses", ctypes.c_void_p), ("intr", ctypes.c_void_p), ("points", ctypes.c_void_p),
    ]


class BAOptions(ctypes.Structure):
    _fields_ = [
        ("max_num_iterations", ctypes.c_int32),
        ("max_num_consecutive_invalid_steps", ctypes.c_int32),
        ("jacobi_scaling", ctypes.c_int32),
        ("reserved", ctypes.c_int32),
        ("function_tolerance", ctypes.c_double),
        ("gradient_tolerance", ctypes.c_double),
        ("parameter_tolerance", ctypes.c_double),
        ("initial_trust_region_radius", ctypes.c_double),
        ("max_trust_region_radius", ctypes.c_double),
        ("min_trust_region_radius", ctypes.c_double),
        ("min_relative_decrease", ctypes.c_double),
        ("min_lm_diagonal", ctypes.c_double),
        ("max_lm_diagonal", ctypes.c_double),
    ]


class BASummary(ctypes.Structure):
    _fields_ = [
        ("iterations", ctypes.c_int32), ("successful", ctypes.c_int32),
        ("termination", ctypes.c_int32), ("reserved", ctypes.c_int32),
        ("initial_cost", ctypes.c_double), ("final_cost", ctypes.c_double),
        ("final_radius", ctypes.c_double), ("device_ms", ctypes.c_double),
        ("kernel_launches", ctypes.c_int64),
    ]


class BAFabric(ctypes.Structure):
    _fields_ = [("ar_local", ctypes.c_void_p), ("ar_multicast", ctypes.c_void_p), ("ar_doubles", ctypes.c_size_t),
                ("world", ctypes.c_int32), ("rank", ctypes.c_int32), ("peer_base", ctypes.c_void_p * 8),
                ("total_doubles", ctypes.c_size_t)]


class PoseOptions(ctypes.Structure):
    _fields_ = [
        ("max_num_iterations", ctypes.c_int32),
        ("max_num_consecutive_invalid_steps", ctypes.c_int32),
        ("min_inliers", ctypes.c_int32),
        ("reserved", ctypes.c_int32),
        ("function_tolerance", ctypes.c_double),
        ("gradient_tolerance", ctypes.c_double),
        ("parameter_tolerance", ctypes.c_double),
        ("initial_trust_region_radius", ctypes.c_double),
        ("max_trust_region_radius", ctypes.c_double),
        ("min_trust_region_radius", ctypes.c_double),
        ("min_relative_decrease", ctypes.c_double),
        ("min_lm_diagonal", ctypes.c_double),
        ("max_lm_diagonal", ctypes.c_double),
        ("loss_function_scale", ctypes.c_double),
        ("max_reproj_error", ctypes.c_double),
    ]


ALLREDUCE_FN = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t,
                                ctypes.c_int, ctypes.c_void_p)

_lib = None


class NativeLibraryMissing(RuntimeError):
    pass


def lib() -> ctypes.CDLL:
    """Load (once) and return the shared library; raises NativeLibraryMissing if it was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeLibraryMissing(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make`. vggsfm_b200 has no CPU/PyTorch fallback.")
    L = ctypes.CDLL(LIB_PATH, mode=ctypes.RTLD_GLOBAL)
    L.vgg_last_error.restype = ctypes.c_char_p
    L.vgg_version.restype = ctypes.c_int
    L.vgg_ba_default_options.argtypes = [ctypes.POINTER(BAOptions)]
    L.vgg_ba_default_options.restype = None
    L.vgg_ba_dims.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int)]
    L.vgg_ba_workspace_bytes.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                         ctypes.POINTER(ctypes.c_size_t)]
    L.vgg_ba_camrec_len.argtypes = [ctypes.c_int, ctypes.c_int]
    L.vgg_ba_build_blocks.argtypes = [ctypes.POINTER(BAProblem)] + [ctypes.c_void_p] * 6 + [ctypes.c_int, ctypes.c_void_p]
    L.vgg_ba_schur.argtypes = ([ctypes.POINTER(BAProblem)] + [ctypes.c_void_p] * 6 +
                               [ctypes.c_double] * 3 + [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p,
                                                        ctypes.c_void_p, ctypes.POINTER(ctypes.c_int), ctypes.c_void_p])
    L.vgg_ba_solve.argtypes = [ctypes.POINTER(BAProblem), ctypes.POINTER(BAOptions), ctypes.c_void_p, ctypes.c_size_t,
                               ALLREDUCE_FN, ctypes.c_void_p, ctypes.POINTER(BASummary), ctypes.c_void_p,
                               ctypes.c_void_p]
    vp, ci, cd, cs = ctypes.c_void_p, ctypes.c_int, ctypes.c_double, ctypes.c_size_t
    L.vgg_ba_reduced_system_doubles.argtypes = [ci, ci, ci, ctypes.POINTER(cs)]
    L.vgg_ba_fabric_doubles.argtypes = [ci, ci, ci, ctypes.POINTER(cs)]
    L.vgg_ba_solve_fabric.argtypes = [ctypes.POINTER(BAProblem), ctypes.POINTER(BAOptions), vp, cs, ALLREDUCE_FN, vp,
                                      ctypes.POINTER(BAFabric), ctypes.POINTER(BASummary), vp, vp]
    L.vgg_pose_default_options.argtypes = [ctypes.POINTER(PoseOptions)]
    L.vgg_pose_default_options.restype = None
    L.vgg_pose_refinement.argtypes = [ci, ci, ci, vp, vp, vp, vp, vp, vp, ctypes.POINTER(PoseOptions), vp, vp, vp, vp]
    L.vgg_pnp_workspace_bytes.argtypes = [ci, ci, ctypes.POINTER(cs)]
    L.vgg_absolute_pose_estimation.argtypes = [ci, ci, ci, vp, vp, vp, vp, vp, vp, ci, ci, cd, vp, vp, vp, vp, vp, cs, vp]
    L.vgg_syrk_ozaki_workspace_bytes.argtypes = [ci, ci, ci, ctypes.POINTER(cs)]
    L.vgg_syrk_ozaki_mma_rate.argtypes = [ci, ci, ctypes.POINTER(cd), vp]
    L.vgg_dev_blocks_timing.argtypes = [ci]
    L.vgg_dev_blocks_last_ms.argtypes = [ctypes.POINTER(cd)]
    L.vgg_dev_chol128_probe.argtypes = [ci, vp, vp, vp]
    L.vgg_dev_set_syrk_ranges.argtypes = [vp, ci]
    L.vgg_dev_trsv_probe.argtypes = [ci, ci, vp, vp, vp, vp]
    L.vgg_dev_set_chol_band.argtypes = [vp, ci, ci]
    L.vgg_syrk_ozaki.argtypes = [ci, ci, vp, vp, ci, vp, cs, vp]
    L.vgg_cholesky_lower.argtypes = [ci, ci, vp, vp, cs, ctypes.POINTER(ci), vp]
    L.vgg_tri_workspace_bytes.argtypes = [ci, ci, ci, ci, ctypes.POINTER(cs)]
    L.vgg_triangulate_tracks.argtypes = [ci, ci, vp, vp, vp, vp, vp, ci, ci, cd, cd, vp, vp, vp, vp, cs, vp]
    L.vgg_triangulate_by_pair.argtypes = [ci, ci, vp, vp, vp, vp, vp, vp, cs, vp]
    L.vgg_filter_points3d.argtypes = [ci, ci, vp, vp, ci, vp, vp, vp, cd, cd, ci, cd, vp, vp, vp, cs, vp]
    L.vgg_project_points.argtypes = [ci, ci, vp, vp, vp, vp, vp, vp, vp]
    L.vgg_normalize_tracks.argtypes = [ci, ci, vp, vp, vp, ci, vp, vp]
    L.vgg_undistort_simple_radial.argtypes = [ci, ci, vp, vp, ci, cd, cd, vp, ctypes.POINTER(ci), vp, cs, vp]
    L.vgg_corr_pyramid_bytes.argtypes = [ci, ci, ci, ci, ci, ci, ctypes.POINTER(cs), ctypes.POINTER(cs)]
    L.vgg_corr_build_pyramid.argtypes = [ci, ci, ci, ci, ci, vp, ci, vp, vp, vp]
    L.vgg_sample_features4d.argtypes = [ci, ci, ci, ci, ci, vp, vp, vp, vp]
    L.vgg_corr_sample.argtypes = [ci, ci, ci, ci, ci, ci, ci, vp, ci, vp, vp, ci, vp, vp]
    L.vgg_corr_tc_supported.argtypes = [ci, ci, ci, ci, ci]
    L.vgg_corr_tc_bytes.argtypes = [ci, ci, ci, ci, ci, ci, ctypes.POINTER(cs), ctypes.POINTER(cs)]
    L.vgg_corr_tc_build.argtypes = [ci, ci, ci, ci, ci, vp, vp, vp]
    L.vgg_corr_tc_sample.argtypes = [ci, ci, ci, ci, ci, ci, ci, vp, vp, vp, vp, vp, vp]
    _lib = L
    return L


def check(rc: int, what: str) -> None:
    if rc != 0:
        raise RuntimeError(f"{what} failed (rc={rc}): {lib().vgg_last_error().decode(errors='replace')}")
