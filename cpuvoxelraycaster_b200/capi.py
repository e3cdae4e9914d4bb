"""ctypes binding of libvrt.so (include/vrt.h).  Loading fails loudly: there is no CPU fallback."""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("VRT_LIBRARY", os.path.join(HERE, "libvrt.so"))    # override: A/B builds in tools/

VRT_OK = 0

LNODE = np.dtype([("color", "u1"), ("child_mask", "u1"), ("leaf_mask", "u1"), ("pad", "u1"), ("child_offset", "u4")])
HIT = np.dtype([("position", "f4", 3), ("distance", "f4"), ("normal", "f4", 3), ("complexity", "u4"),
                ("voxel_coord", "f4", 2), ("flags", "u4"), ("scale", "i4"), ("voxel", "i4", 3), ("face", "u4")])
SHADE_JOB = np.dtype([("start", "f4", 3), ("pixel", "u4"), ("direction", "f4", 3), ("sample", "u4")])
SHADE_RESULT = np.dtype([("r", "u1"), ("g", "u1"), ("b", "u1"), ("hit", "u1"), ("distance", "f4"), ("complexity", "u4"), ("reserved", "u4")])
POINT_LIGHT = np.dtype([("position", "f4", 3), ("color", "f4", 3), ("range", "f4"), ("reserved", "u4")])
assert HIT.itemsize == 64 and LNODE.itemsize == 8 and SHADE_JOB.itemsize == 32 and SHADE_RESULT.itemsize == 16
assert POINT_LIGHT.itemsize == 32


class Camera(C.Structure):
    _fields_ = [("position", C.c_float * 3), ("rot_mat", C.c_float * 9), ("fov", C.c_float),
                ("aperture", C.c_float), ("focal_length", C.c_float)]


class RenderParams(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("row_begin", C.c_int32), ("row_end", C.c_int32),
                ("spp", C.c_int32), ("sample_offset", C.c_int32), ("seed_lo", C.c_uint32), ("seed_hi", C.c_uint32),
                ("light_position", C.c_float * 3), ("use_gi", C.c_int32), ("gi_bounces", C.c_int32),
                ("use_samples", C.c_int32), ("accum_in", C.c_int32), ("tile_step", C.c_int32), ("tile_index", C.c_int32),
                ("roughness", C.c_float), ("max_bounds", C.c_int32),
                ("checker", C.c_int32), ("checker_area_height", C.c_int32), ("mirror_y1", C.c_int32), ("autofocus", C.c_int32)]


class PresentParams(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("median", C.c_int32),
                ("old_value_conservation", C.c_float)]


class RenderStats(C.Structure):
    _fields_ = [("rays", C.c_uint64 * 6), ("complexity", C.c_uint64 * 6)]


class VrtError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libvrt error %d: %s" % (code, msg))
        self.code = code


_lib = None

_vp, _u64, _u32, _i32, _f = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int32, C.c_float
_SIGNATURES = {
    "vrt_abi_version": (C.c_int, []),
    "vrt_last_error": (C.c_char_p, []),
    "vrt_build_info": (C.c_char_p, []),
    "vrt_context_create": (C.c_int, [C.c_int, _vp, C.POINTER(_vp)]),
    "vrt_context_destroy": (C.c_int, [_vp]),
    "vrt_context_synchronize": (C.c_int, [_vp]),
    "vrt_context_set_stream": (C.c_int, [_vp, _vp]),
    "vrt_context_launch_count": (_u64, [_vp]),
    "vrt_context_set_option": (C.c_int, [_vp, C.c_char_p, C.c_int]),
    "vrt_context_take_timings": (C.c_int, [_vp, _vp, _i32, C.POINTER(_i32)]),
    "vrt_host_terrain_heights": (C.c_int, [_i32, _vp]),
    "vrt_host_noise2d": (_f, [_f, _f]),
    "vrt_host_build_terrain_lsvo": (C.c_int, [_u32, _vp, _vp, _u64, C.POINTER(_u64)]),
    "vrt_host_build_lsvo_from_voxels": (C.c_int, [_u32, _vp, _u64, _vp, _u64, C.POINTER(_u64)]),
    "vrt_host_camera_rotation": (C.c_int, [_vp, _vp, _vp]),
    "vrt_lsvo_create": (C.c_int, [_vp, _vp, _u64, _u32, _i32, C.POINTER(_vp)]),
    "vrt_lsvo_create_terrain": (C.c_int, [_vp, _u32, _i32, C.POINTER(_vp)]),
    "vrt_scene_set_layout": (C.c_int, [_vp, _i32, _i32]),
    "vrt_scene_download_nodes": (C.c_int, [_vp, _vp, _u64, C.POINTER(_u64)]),
    "vrt_grid_create": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, C.POINTER(_vp)]),
    "vrt_svo_create": (C.c_int, [_vp, _vp, _u32, C.POINTER(_vp)]),
    "vrt_scene_destroy": (C.c_int, [_vp]),
    "vrt_scene_info": (C.c_int, [_vp, C.POINTER(_i32), C.POINTER(_u32), C.POINTER(_u64)]),
    "vrt_cast_rays": (C.c_int, [_vp, _vp, _vp, _f, _f, _u64, _vp]),
    "vrt_cast_rays_device": (C.c_int, [_vp, _vp, _vp, _f, _f, _u64, _vp]),
    "vrt_cast_rays_svo": (C.c_int, [_vp, _vp, _vp, _u32, _u64, _vp]),
    "vrt_scene_last_complexity": (C.c_int, [_vp, C.POINTER(_u64)]),
    "vrt_scene_set_textures": (C.c_int, [_vp, _vp, _vp]),
    "vrt_scene_set_palette": (C.c_int, [_vp, _vp]),
    "vrt_scene_set_cell_types": (C.c_int, [_vp, _vp]),
    "vrt_scene_set_point_lights": (C.c_int, [_vp, _vp, _u32]),
    "vrt_scene_paint_cells": (C.c_int, [_vp, _vp, _vp, _u64, C.POINTER(_u64)]),
    "vrt_scene_cell_colors": (C.c_int, [_vp, _vp, _u64, _vp]),
    "vrt_render_accumulate_device": (C.c_int, [_vp, C.POINTER(Camera), C.POINTER(RenderParams), _vp]),
    "vrt_render_resolve_device": (C.c_int, [_vp, C.POINTER(RenderParams), _vp, _vp]),
    "vrt_render": (C.c_int, [_vp, C.POINTER(Camera), C.POINTER(RenderParams), _vp, _vp, C.POINTER(RenderStats)]),
    "vrt_scene_last_render_stats": (C.c_int, [_vp, C.POINTER(RenderStats)]),
    "vrt_scene_last_render_culled": (C.c_int, [_vp, C.POINTER(C.c_uint64)]),
    "vrt_shade_rays": (C.c_int, [_vp, C.POINTER(RenderParams), _u64, _vp, _vp]),
    "vrt_beam_floors": (C.c_int, [_vp, C.POINTER(Camera), C.POINTER(RenderParams), _i32, _vp]),
    "vrt_autofocus": (C.c_int, [_vp, C.POINTER(Camera), C.POINTER(_f)]),
    "vrt_lsvo_create_from_voxels": (C.c_int, [_vp, _u32, _vp, _u64, _i32, C.POINTER(_vp)]),
    "vrt_scene_set_cells": (C.c_int, [_vp, _vp, _u64, _i32]),
    "vrt_scene_voxel_count": (C.c_int, [_vp, C.POINTER(_u64)]),
    "vrt_lsvo_create_heightfield": (C.c_int, [_vp, _u32, _vp, _i32, C.POINTER(_vp)]),
    "vrt_scene_edit_heights": (C.c_int, [_vp, _u32, _u32, _u32, _u32, _vp]),
    "vrt_scene_download_heights": (C.c_int, [_vp, _vp]),
    "vrt_present_device": (C.c_int, [_vp, _vp, _vp, C.POINTER(PresentParams)]),
    "vrt_present": (C.c_int, [_vp, _vp, _vp, C.POINTER(PresentParams)]),
    "vrt_comm_create_local": (C.c_int, [C.POINTER(_vp), C.c_int, C.c_int, C.c_int, C.POINTER(_vp)]),
    "vrt_comm_create": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(_vp)]),
    "vrt_comm_export": (C.c_int, [_vp, _vp]),
    "vrt_comm_connect": (C.c_int, [_vp, _vp]),
    "vrt_comm_destroy": (C.c_int, [_vp]),
    "vrt_comm_info": (C.c_int, [_vp, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(_u64)]),
    "vrt_render_distributed": (C.c_int, [_vp, _vp, C.POINTER(Camera), C.POINTER(RenderParams), C.c_int, C.c_int, _vp]),
    "vrt_comm_frame_wait": (C.c_int, [_vp]),
    "vrt_comm_frame_device": (C.c_int, [_vp, C.c_int, C.POINTER(_vp)]),
}
COMM_HANDLE_BYTES = 256
SPLIT_TILES, SPLIT_SAMPLES = 0, 1


def declared_symbols():
    """Every entry point include/vrt.h declares (kept in sync by tests/test_capi_symbols.py)."""
    return sorted(_SIGNATURES)


def lib():
    """Load libvrt.so; raises if the CUDA extension has not been built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError("libvrt.so is missing (%s): run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "or `make -C cpuvoxelraycaster_b200`. There is no CPU fallback." % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            if os.environ.get("VRT_ALLOW_OLD_LIBRARY") and not hasattr(L, name):
                continue                   # A/B tools only (tools/probe_policies.py against an earlier build)
            fn = getattr(L, name)          # AttributeError here = header/library mismatch: fail loudly
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(code):
    if code != VRT_OK:
        raise VrtError(code, lib().vrt_last_error().decode("utf-8", "replace"))


def ptr(a):
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data_as(C.c_void_p)
    if isinstance(a, int):
        return C.c_void_p(a)
    # torch tensor
    return C.c_void_p(a.data_ptr())
