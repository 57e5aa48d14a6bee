"""ctypes binding of libp3p.so (include/p3p.h).  No torch types cross this boundary: device pointers are
passed as integers, the CUDA stream as a void*."""
from __future__ import annotations

import ctypes as C
import os

from .build import LIB_PATH

P3P_PRECISION = {"fp32": 0, "tf32": 1, "bf16": 2, "fp16": 3}
P3P_LAYOUT_NCHW, P3P_LAYOUT_NLC = 0, 1
P3P_DTYPE_F32, P3P_DTYPE_BF16, P3P_DTYPE_F16 = 0, 1, 2
P3P_GRID_DROP_OVERFLOW = 1

EXPORTED = [
    "p3p_last_error", "p3p_version", "p3p_workspace_bytes", "p3p_pfn_blob_bytes", "p3p_pfn_prepare",
    "p3p_voxelize", "p3p_pillar_features", "p3p_encode", "p3p_encode_tokens", "p3p_patch_embed", "p3p_las_to_pixels",
    "p3p_profile_begin", "p3p_profile_end", "p3p_conv3x3_blob_bytes", "p3p_conv3x3_prepare", "p3p_conv3x3", "p3p_conv3x3_vit_tokens",
    "p3p_nchw_to_nhwc16", "p3p_upsample_bilinear_nhwc16", "p3p_las_packed_to_pixels",
    "p3p_patch_embed_blob_bytes", "p3p_patch_embed_prepare", "p3p_patch_embed_prepared",
    "p3p_encode_workspace", "p3p_pfn_train_state_doubles", "p3p_pfn_train_route_bytes", "p3p_pfn_train_stats0",
    "p3p_pfn_train_stats1", "p3p_pfn_train_stats2", "p3p_pfn_train_forward", "p3p_pfn_backward1", "p3p_pfn_backward2", "p3p_pfn_backward3",
]


class LasTile(C.Structure):
    _fields_ = [("scale", C.c_double * 3), ("offset", C.c_double * 3), ("left", C.c_double), ("top", C.c_double),
                ("res", C.c_double), ("height", C.c_double), ("width", C.c_double), ("origin_from_min", C.c_int32),
                ("clip", C.c_int32), ("d4", C.c_int32), ("reserved", C.c_int32), ("center_x", C.c_double),
                ("center_y", C.c_double)]


P3P_D4 = {None: 0, "none": 0, "e": 1, "r90": 2, "r180": 3, "r270": 4, "v": 5, "hvt": 6, "h": 7, "t": 8}


class Grid(C.Structure):
    _fields_ = [("range_min", C.c_float * 3), ("range_max", C.c_float * 3), ("voxel_size", C.c_float * 3),
                ("max_points", C.c_int32), ("max_voxels", C.c_int32), ("ny", C.c_int32), ("nx", C.c_int32),
                ("flags", C.c_int32)]


class PfnParams(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "linear0_weight", "norm0_weight", "norm0_bias", "norm0_mean", "norm0_var",
        "linear1_weight", "norm1_weight", "norm1_bias", "norm1_mean", "norm1_var")] + [
        ("eps", C.c_float), ("channels", C.c_int32), ("center_alias", C.c_int32)]


class ConvParams(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("weight", "bias", "norm_weight", "norm_bias", "norm_mean", "norm_var")] + [
        ("eps", C.c_float), ("in_channels", C.c_int32), ("out_channels", C.c_int32)]


class VoxelOutputs(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "point_hash", "num_pillars", "pillar_coords", "pillar_num_points", "pillar_point_idx", "pillar_points",
        "cell_owner")]


class P3PError(RuntimeError):
    pass


_lib = None


def lib():
    """The loaded library.  Fails loudly when it has not been built: there is no fallback path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise P3PError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `python -m pixelspointspolygons_b200.build`). This package has no CPU or eager fallback.")
    l = C.CDLL(LIB_PATH)
    vp, i32, i64, sz = C.c_void_p, C.c_int32, C.c_int64, C.c_size_t
    l.p3p_last_error.restype = C.c_char_p
    l.p3p_last_error.argtypes = []
    l.p3p_version.restype = C.c_int
    l.p3p_version.argtypes = []
    l.p3p_workspace_bytes.restype = sz
    l.p3p_workspace_bytes.argtypes = [C.POINTER(Grid), i32, i64]
    l.p3p_pfn_blob_bytes.restype = sz
    l.p3p_pfn_blob_bytes.argtypes = [i32]
    l.p3p_pfn_prepare.restype = C.c_int
    l.p3p_pfn_prepare.argtypes = [C.POINTER(PfnParams), i32, vp, sz, vp]
    l.p3p_voxelize.restype = C.c_int
    l.p3p_voxelize.argtypes = [vp, i32, vp, i32, i64, C.POINTER(Grid), C.POINTER(VoxelOutputs), vp, sz, vp]
    l.p3p_pillar_features.restype = C.c_int
    l.p3p_pillar_features.argtypes = [C.POINTER(Grid), i32, i64, vp, i32, i32, vp, vp, sz, vp]
    l.p3p_encode.restype = C.c_int
    l.p3p_encode.argtypes = [vp, i32, vp, i32, i64, C.POINTER(Grid), vp, i32, i32, vp, i32, i32, i32, i32, i32, vp, sz, vp]
    l.p3p_encode_tokens.restype = C.c_int
    l.p3p_encode_tokens.argtypes = [vp, i32, vp, i32, i64, C.POINTER(Grid), vp, i32, i32, vp, vp, vp, vp, sz, vp]
    l.p3p_las_to_pixels.restype = C.c_int
    l.p3p_las_to_pixels.argtypes = [vp, vp, vp, vp, i32, i64, vp, C.c_double, vp, vp, vp]
    l.p3p_las_packed_to_pixels.restype = C.c_int
    l.p3p_las_packed_to_pixels.argtypes = [vp, vp, vp, i32, i64, vp, C.c_double, vp, vp, vp]
    l.p3p_patch_embed.restype = C.c_int
    l.p3p_patch_embed.argtypes = [vp, i32, i32, i32, i32, i32, vp, vp, i32, i32, vp, i32, i32, i32, i32, vp]
    l.p3p_patch_embed_blob_bytes.restype = sz
    l.p3p_patch_embed_blob_bytes.argtypes = [i32, i32, i32]
    l.p3p_patch_embed_prepare.restype = C.c_int
    l.p3p_patch_embed_prepare.argtypes = [vp, vp, i32, i32, i32, i32, vp, sz, vp]
    l.p3p_patch_embed_prepared.restype = C.c_int
    l.p3p_patch_embed_prepared.argtypes = [vp, i32, i32, i32, i32, i32, vp, vp, vp, i32, i32, vp, i32, i32, i32, i32, vp]
    l.p3p_conv3x3_blob_bytes.restype = sz
    l.p3p_conv3x3_blob_bytes.argtypes = [i32, i32]
    l.p3p_conv3x3_prepare.restype = C.c_int
    l.p3p_conv3x3_prepare.argtypes = [C.POINTER(ConvParams), i32, vp, sz, vp]
    l.p3p_conv3x3.restype = C.c_int
    l.p3p_conv3x3.argtypes = [vp, i32, i32, i32, i32, vp, i32, i32, i32, vp, i32, i32, i32, vp]
    l.p3p_conv3x3_vit_tokens.restype = C.c_int
    l.p3p_conv3x3_vit_tokens.argtypes = [vp, i32, i32, i32, i32, vp, i32, i32, vp, vp, vp, vp]
    l.p3p_nchw_to_nhwc16.restype = C.c_int
    l.p3p_nchw_to_nhwc16.argtypes = [vp, i32, i32, i32, i32, i32, vp, i32, i32, vp]
    l.p3p_upsample_bilinear_nhwc16.restype = C.c_int
    l.p3p_upsample_bilinear_nhwc16.argtypes = [vp, i32, i32, i32, i32, i64, i32, i32, i32, vp, vp]
    l.p3p_encode_workspace.restype = C.c_int
    l.p3p_encode_workspace.argtypes = [C.POINTER(Grid), i32, i64, vp, i32, i32, vp, i32, i32, i32, i32, vp, sz, vp]
    l.p3p_pfn_train_state_doubles.restype = i64
    l.p3p_pfn_train_state_doubles.argtypes = [i32, C.POINTER(i64)]
    l.p3p_pfn_train_route_bytes.restype = sz
    l.p3p_pfn_train_route_bytes.argtypes = [C.POINTER(Grid), i32, i32]
    for name in ("p3p_pfn_train_stats0", "p3p_pfn_train_stats1"):
        getattr(l, name).restype = C.c_int
        getattr(l, name).argtypes = [C.POINTER(Grid), i32, i64, C.POINTER(PfnParams), vp, vp, sz, vp]
    l.p3p_pfn_train_stats2.restype = C.c_int
    l.p3p_pfn_train_stats2.argtypes = [C.POINTER(PfnParams), vp, vp, vp, vp, vp, vp]
    l.p3p_pfn_backward1.restype = C.c_int
    l.p3p_pfn_backward1.argtypes = [C.POINTER(Grid), i32, i64, C.POINTER(PfnParams), vp, vp, vp, vp, vp, sz, vp]
    l.p3p_pfn_train_forward.restype = C.c_int
    l.p3p_pfn_train_forward.argtypes = [C.POINTER(Grid), i32, i64, C.POINTER(PfnParams), vp, vp, vp, vp, sz, vp]
    l.p3p_pfn_backward2.restype = C.c_int
    l.p3p_pfn_backward2.argtypes = [C.POINTER(Grid), i32, i64, C.POINTER(PfnParams), vp, vp, vp, sz, vp]
    l.p3p_pfn_backward3.restype = C.c_int
    l.p3p_pfn_backward3.argtypes = [C.POINTER(PfnParams), vp, vp, vp, vp, vp, vp, vp, vp]
    l.p3p_profile_begin.restype = C.c_int
    l.p3p_profile_begin.argtypes = [i32]
    l.p3p_profile_end.restype = C.c_int
    l.p3p_profile_end.argtypes = [vp, vp, i32, C.POINTER(i32)]
    _lib = l
    return l


def check(rc: int, what: str = "p3p call"):
    if rc != 0:
        msg = lib().p3p_last_error().decode("utf-8", "replace")
        raise P3PError(f"{what} failed (code {rc}): {msg}")


def make_grid(range_min, range_max, voxel_size, max_points, max_voxels, ny, nx, flags=0) -> Grid:
    g = Grid()
    for i in range(3):
        g.range_min[i] = float(range_min[i])
        g.range_max[i] = float(range_max[i])
        g.voxel_size[i] = float(voxel_size[i])
    g.max_points, g.max_voxels, g.ny, g.nx, g.flags = int(max_points), int(max_voxels), int(ny), int(nx), int(flags)
    return g
