"""TEST INFRASTRUCTURE ONLY: ctypes binding of tests/point_lights_oracle.c (vo_render_point_lights, the CPU specification of point
lights).  The library is compiled on first use with the oracle's flags into a temporary directory: the tree may be read-only."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from oracle.loader import PortRenderParams, PortRenderStats

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE = os.path.join(os.path.dirname(HERE), "oracle")
_lib = None

# vrt_point_light / vo_point_light: 32 bytes
LIGHT_DTYPE = np.dtype([("position", "<f4", 3), ("color", "<f4", 3), ("range", "<f4"), ("reserved", "<u4")])


def lib():
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="vrt_point_lights_oracle_"), "libvrt_point_lights_oracle.so")
        subprocess.run([os.environ.get("CC", "gcc"), "-O2", "-std=c11", "-ffp-contract=off", "-fPIC", "-shared", "-Wall", "-Wextra",
                        "-pthread", "-I" + ORACLE, "-I" + HERE, "-o", out, os.path.join(HERE, "point_lights_oracle.c"), "-lm"], check=True)
        L = C.CDLL(out)
        L.vo_render_point_lights.argtypes = [C.c_void_p, C.POINTER(PortRenderParams), C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32,
                                             C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(PortRenderStats)]
        _lib = L
    return _lib


def pack_lights(positions, colors, ranges):
    """(n,3), (n,3), (n,) -> a contiguous LIGHT_DTYPE array (None or n == 0 -> None)."""
    if positions is None:
        return None
    pos = np.asarray(positions, np.float32).reshape(-1, 3)
    if len(pos) == 0:
        return None
    a = np.zeros(len(pos), LIGHT_DTYPE)
    a["position"] = pos
    a["color"] = np.asarray(colors, np.float32).reshape(-1, 3)
    a["range"] = np.asarray(ranges, np.float32).reshape(-1)
    return a


def render_point_lights(nodes, params, palette, types, lights, tex_top, tex_side, prev_rgba=None):
    """vo_render_point_lights: palette uint8 [256, 3] or None; types 256 ints or None; lights a LIGHT_DTYPE array (pack_lights) or
    None.  Returns (accum uint32 [H,W,4], rgba uint8 [H,W,4], stats) like oracle.loader.Port.render."""
    H, W = params.height, params.width
    accum = np.zeros((H, W, 4), np.uint32)
    rgba = np.zeros((H, W, 4), np.uint8) if prev_rgba is None else np.ascontiguousarray(prev_rgba).copy()
    stats = PortRenderStats()
    nodes = np.ascontiguousarray(nodes)
    pal = None if palette is None else np.ascontiguousarray(palette, np.uint8).reshape(768)
    ty = None if types is None else np.ascontiguousarray(types, np.uint8).reshape(256)
    li = None if lights is None or len(lights) == 0 else np.ascontiguousarray(lights, LIGHT_DTYPE)
    tt, ts = np.ascontiguousarray(tex_top, np.uint8), np.ascontiguousarray(tex_side, np.uint8)
    ptr = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)   # noqa: E731
    lib().vo_render_point_lights(ptr(nodes), C.byref(params), ptr(pal), ptr(ty), ptr(li), 0 if li is None else len(li), ptr(tt),
                                 ptr(ts), ptr(accum), ptr(rgba), C.byref(stats))
    return accum, rgba, stats
