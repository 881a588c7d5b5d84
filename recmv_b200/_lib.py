"""ctypes binding of librecmv_b200.so (the C ABI declared in include/recmv_b200.h).

There is NO fallback: if the shared library is missing or a call returns a non-zero status the
caller gets an exception (the reference's pybind modules raise RuntimeError the same way,
FastMinv/M3x3Inv.cpp:4-6).
"""
import ctypes
import os
from ctypes import (POINTER, Structure, c_char_p, c_float, c_int, c_int64, c_size_t,
                    c_void_p)

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "librecmv_b200.so")

F32, F64 = 0, 1
LAYOUT_NCDHW, LAYOUT_NDHWC = 0, 1
MLP_FP32_SIMT, MLP_TC_F16X3, MLP_TC_F16X1 = 0, 1, 2


RECMV_E_RANGE = -4


class RecmvError(RuntimeError):
    pass


class Voxel(Structure):
    _fields_ = [("ws_cl", c_void_p), ("D", c_int), ("H", c_int), ("W", c_int),
                ("center", c_float * 3), ("extend", c_float)]


class RayMarch(Structure):
    _fields_ = [("cam_pos", c_float * 3), ("t_near", c_float), ("t_far", c_float),
                ("samples_per_ray", c_int)]


# name -> (restype, argtypes); must list every symbol of include/recmv_b200.h
SIGNATURES = {
    "recmv_version": (c_int, []),
    "recmv_error_string": (c_char_p, [c_int]),
    "recmv_launch_count": (c_int64, []),
    "recmv_minv3x3_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int, c_void_p]),
    "recmv_minv3x3_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int, c_void_p]),
    "recmv_gridsample3d_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                                       c_int, c_int64, c_int, c_int, c_void_p]),
    "recmv_gridsample3d_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int,
                                       c_int, c_int, c_int, c_int, c_int64, c_int, c_int, c_void_p]),
    "recmv_gridsample3d_bwd2": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                        c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int,
                                        c_int64, c_int, c_int, c_void_p]),
    "recmv_voxel_to_channels_last": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                                             c_void_p]),
    "recmv_mc_scratch_bytes": (c_int, [c_int, c_int, c_int, POINTER(c_size_t)]),
    "recmv_mc_count": (c_int, [c_void_p, c_int, c_int, c_int, c_float, c_void_p, POINTER(c_int64),
                               POINTER(c_int64), c_void_p]),
    "recmv_mc_emit": (c_int, [c_void_p, c_int, c_int, c_int, c_float, c_void_p, POINTER(c_float),
                              POINTER(c_float), c_void_p, c_void_p, c_void_p]),
    "recmv_mc_run": (c_int, [c_void_p, c_int, c_int, c_int, c_float, c_void_p, POINTER(c_float), POINTER(c_float), c_void_p,
                             c_int64, c_void_p, c_int64, c_void_p, c_void_p]),
    "recmv_lbs_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int,
                              POINTER(Voxel), c_void_p, c_void_p, c_int64, c_void_p]),
    "recmv_lbs_inverse": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int,
                                  POINTER(Voxel), c_void_p, c_void_p, c_int64, c_void_p]),
    "recmv_bone_matrices": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "recmv_sdf_packed_bytes": (c_size_t, []),
    "recmv_sdf_pack_weights": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "recmv_sdf_mlp_fwd": (c_int, [c_void_p, c_void_p, POINTER(c_float), c_void_p, c_void_p, c_int64,
                                  c_int, c_void_p]),
    "recmv_sdf_mlp_fwd_grad": (c_int, [c_void_p, c_void_p, POINTER(c_float), c_void_p, c_void_p, c_void_p, c_int64,
                                       c_int, c_void_p]),
    "recmv_mlp_fwd_layer": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_int, c_void_p,
                                    c_int64, c_void_p, c_int64, c_int64, c_void_p]),
    "recmv_pe_forward": (c_int, [c_void_p, POINTER(c_float), c_int, c_void_p, c_int64, c_void_p, c_int64, c_int64, c_void_p]),
    "recmv_mlp_bwd_data_layer": (c_int, [c_void_p, c_int64, c_void_p, c_int, c_int, c_void_p, c_int64, c_int, c_int,
                                         c_void_p, c_int64, c_void_p, c_int64, c_float, c_void_p, c_int64, c_void_p]),
    "recmv_mlp_bwd_weight": (c_int, [c_int, POINTER(c_void_p), POINTER(c_int64), POINTER(c_void_p), POINTER(c_int64),
                                     POINTER(c_int), POINTER(c_int), POINTER(c_void_p), POINTER(c_void_p),
                                     POINTER(c_float), c_void_p, c_int64, c_void_p]),
    "recmv_pe_backward": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int64, POINTER(c_float), c_int, c_void_p,
                                  c_int, c_int64, c_void_p]),
    "recmv_split_planes": (c_int, [c_void_p, c_int64, c_int64, c_int, c_float, c_void_p, c_int, c_void_p, c_void_p, c_int64,
                                   c_void_p]),
    "recmv_pe_forward_planes": (c_int, [c_void_p, POINTER(c_float), c_int, c_void_p, c_int64, c_void_p, c_void_p, c_int64,
                                        c_int64, c_void_p]),
    "recmv_mlp_layer_planes": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_int64, c_int, c_int, c_int,
                                       c_void_p, c_void_p, c_int64, c_float, c_void_p, c_int, c_int, c_void_p, c_int64,
                                       c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_int, c_void_p]),
    "recmv_translator_packed_bytes": (c_size_t, []),
    "recmv_translator_pack_weights": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "recmv_deformer_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int, c_void_p, POINTER(c_float),
                                   c_void_p, c_void_p, POINTER(Voxel), c_void_p, c_void_p, c_void_p, c_int64,
                                   c_int, c_void_p]),
    "recmv_deformer_fwd_jac": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int, c_void_p, POINTER(c_float),
                                       c_void_p, c_void_p, POINTER(Voxel), c_void_p, c_void_p, c_void_p, c_void_p,
                                       c_int64, c_int, c_void_p]),
    "recmv_rendernet_packed_bytes": (c_size_t, []),
    "recmv_rendernet_pack_weights": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "recmv_rendernet_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, POINTER(c_float), c_void_p, c_int64,
                                    c_int, c_void_p]),
    "recmv_interp2x_boundary3d_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_float, c_int,
                                              c_void_p]),
    "recmv_interp2x_boundary3d_bwd": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "recmv_c2f_todo_mask": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "recmv_mlp_wgrad_workspace_floats": (c_size_t, []),
    "recmv_mlp_wgrad_planes": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_int64, c_int, c_int, c_float,
                                       c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "recmv_colsum": (c_int, [c_void_p, c_int64, c_int64, c_int, c_void_p, c_void_p, c_void_p]),
    "recmv_softplus_tangent_planes": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_int64, c_int, c_float,
                                              c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_void_p]),
    "recmv_add_split_planes": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_int64, c_int, c_float, c_void_p, c_void_p,
                                       c_void_p, c_int64, c_void_p]),
    "recmv_svd3x3": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p]),
    "recmv_svd3x3_backward_s": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "recmv_fragment_decode_scratch_bytes": (c_size_t, [c_int64]),
    "recmv_fragment_decode": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int64, c_void_p,
                                      POINTER(c_float), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                      c_void_p, c_void_p]),
    "recmv_raster_scratch_bytes": (c_int, [c_int, c_int, c_int, POINTER(c_size_t)]),
    "recmv_rasterize": (c_int, [c_void_p, c_void_p, c_int, c_int64, c_int64, POINTER(c_float), c_void_p, c_void_p, c_int,
                                c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "recmv_points_scratch_bytes": (c_int, [c_int, c_int64, c_int, c_int, POINTER(c_size_t)]),
    "recmv_points_count": (c_int, [c_void_p, c_int, c_int64, POINTER(c_float), c_void_p, c_void_p, c_int, c_int, c_int,
                                   c_float, c_void_p, POINTER(c_int64), c_void_p]),
    "recmv_points_render": (c_int, [c_void_p, c_int, c_int, c_int64, c_int, c_int, c_float, c_int, c_void_p, c_void_p,
                                    c_int64, c_void_p, c_void_p]),
    "recmv_points_render_backward": (c_int, [c_void_p, c_int, c_int64, POINTER(c_float), c_void_p, c_void_p, c_int, c_int,
                                             c_int, c_float, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p,
                                             c_void_p, c_void_p]),
    "recmv_points_fragments": (c_int, [c_int, c_int64, c_int, c_int, c_float, c_int, c_void_p, c_void_p, c_void_p,
                                       c_void_p, c_void_p, c_void_p]),
    "recmv_c2f_done_up": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "recmv_c2f_compact": (c_int, [c_void_p, POINTER(c_int), POINTER(c_int), POINTER(c_float), POINTER(c_float), c_void_p,
                                  c_void_p, c_void_p, c_int, c_void_p]),
    "recmv_c2f_scatter": (c_int, [c_void_p, c_void_p, c_void_p, c_int, POINTER(c_int), POINTER(c_int), c_void_p, c_void_p,
                                  c_void_p, c_void_p, c_float, c_void_p, c_void_p]),
    "recmv_c2f_conflict_todo": (c_int, [c_void_p, c_void_p, POINTER(c_int), POINTER(c_int), c_void_p, c_void_p]),
    "recmv_c2f_refine": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, POINTER(c_int), POINTER(c_float), POINTER(c_float),
                                 c_float, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "recmv_c2f_scatter_list": (c_int, [c_void_p, c_void_p, c_void_p, c_int, POINTER(c_int), POINTER(c_int), c_void_p,
                                       c_void_p, c_void_p, c_void_p, c_float, c_void_p, c_void_p, c_void_p, c_void_p]),
    "recmv_c2f_mark_conflicts": (c_int, [c_void_p, c_void_p, c_int, c_void_p, POINTER(c_int), POINTER(c_int),
                                         POINTER(c_float), POINTER(c_float), c_void_p, c_void_p, c_void_p, c_void_p, c_int,
                                         c_void_p]),
    "recmv_sdf_mlp_fwd_counted": (c_int, [c_void_p, c_void_p, POINTER(c_float), c_void_p, c_void_p, c_int64, c_void_p, c_int,
                                          c_void_p]),
    "recmv_surface_solve_workspace": (c_size_t, [c_int64]),
    "recmv_surface_solve": (c_int, [POINTER(c_float), c_void_p, c_void_p, c_void_p, c_void_p, POINTER(c_float), c_void_p,
                                    POINTER(c_float), c_void_p, c_int, c_void_p, c_void_p, POINTER(Voxel), c_float, c_float,
                                    c_float, c_float, c_int, c_int, c_void_p, c_size_t, c_void_p, c_int64, c_void_p]),
    "recmv_surface_grad_coeffs": (c_int, [c_void_p] * 9 + [c_int64, c_void_p]),
    "recmv_tc_set_acc_gain": (c_int, [c_int, c_float]),
    "recmv_check_async_errors": (c_int, [POINTER(c_int), c_int]),
    "recmv_render_sdf": (c_int, [c_void_p, POINTER(RayMarch), c_void_p, c_void_p, c_void_p, c_int64,
                                 c_int, POINTER(Voxel), c_void_p, POINTER(c_float), c_void_p,
                                 c_void_p, c_void_p, c_void_p, c_int64, c_int, c_void_p]),
    "recmv_ray_first_hit": (c_int, [c_void_p, POINTER(RayMarch), c_void_p, c_void_p, c_int64,
                                    c_void_p]),
}

# diagnostics (include/recmv_b200_diag.h), not part of the product ABI
DIAG_SIGNATURES = {
    "recmv_sdf_mlp_tc_debug": (c_int, [c_void_p, c_void_p, POINTER(c_float), c_void_p, c_void_p, c_int64,
                                       c_int, c_int, c_void_p, POINTER(c_int), c_void_p, c_void_p]),
}
DIAG_LIB_SIGNATURES = {
    "recmv_tc_microbench": (c_int, [c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
}
DIAG_LIB_PATH = os.path.join(_HERE, "librecmv_b200_diag.so")

_lib = None
_diag = None


def load():
    """Load the shared library once; raises RecmvError with build instructions if it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RecmvError(
            f"{LIB_PATH} not found: the CUDA extension is not built. Run "
            "`python -c 'import __graft_entry__ as g; g.build()'` (or `make -C recmv_b200/csrc`). "
            "There is no CPU fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in list(SIGNATURES.items()) + list(DIAG_SIGNATURES.items()):
        fn = getattr(lib, name)  # AttributeError if the .so lacks a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def load_diag():
    """librecmv_b200_diag.so (tools only): the tcgen05 issue-rate microbenchmark."""
    global _diag
    if _diag is None:
        lib = ctypes.CDLL(DIAG_LIB_PATH)
        for name, (res, args) in DIAG_LIB_SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _diag = lib
    return _diag


def check(status, what=""):
    if status != 0:
        msg = load().recmv_error_string(int(status)).decode()
        raise RecmvError(f"{what or 'recmv call'} failed with status {status}: {msg}")


def header_symbols():
    """Function names declared in include/recmv_b200.h (used by the CPU export test)."""
    import re
    hdr = os.path.join(_HERE, "..", "include", "recmv_b200.h")
    return re.findall(r"RECMV_API [\w\* ]+?\b(recmv_\w+)\(", open(hdr).read())
