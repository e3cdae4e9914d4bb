"""TEST INFRASTRUCTURE ONLY: ctypes binding of tests/cell_types_oracle.c (vo_render_cell_types, the CPU specification of mirror
voxels).  The library is compiled on first use with the oracle's flags into a temporary directory: the tree may be read-only."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from oracle.loader import PortRenderParams, PortRenderStats

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE = os.path.join(os.path.dirname(HERE), "oracle")
_lib = None


def lib():
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="vrt_cell_types_oracle_"), "libvrt_cell_types_oracle.so")
        subprocess.run([os.environ.get("CC", "gcc"), "-O2", "-std=c11", "-ffp-contract=off", "-fPIC", "-shared", "-Wall", "-Wextra",
                        "-pthread", "-I" + ORACLE, "-I" + HERE, "-o", out, os.path.join(HERE, "cell_types_oracle.c"), "-lm"], check=True)
        L = C.CDLL(out)
        L.vo_render_cell_types.argtypes = [C.c_void_p, C.POINTER(PortRenderParams), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.c_void_p, C.POINTER(PortRenderStats)]
        _lib = L
    return _lib


def render_cell_types(nodes, params, palette, types, tex_top, tex_side, prev_rgba=None):
    """vo_render_cell_types: palette uint8 [256, 3] or None for the textures; types 256 ints (1 = Solid, 2 = Mirror) or None
    for all Solid.  Returns (accum uint32 [H,W,4], rgba uint8 [H,W,4], stats) like oracle.loader.Port.render."""
    H, W = params.height, params.width
    accum = np.zeros((H, W, 4), np.uint32)
    rgba = np.zeros((H, W, 4), np.uint8) if prev_rgba is None else np.ascontiguousarray(prev_rgba).copy()
    stats = PortRenderStats()
    nodes = np.ascontiguousarray(nodes)
    pal = None if palette is None else np.ascontiguousarray(palette, np.uint8).reshape(768)
    ty = None if types is None else np.ascontiguousarray(types, np.uint8).reshape(256)
    tt, ts = np.ascontiguousarray(tex_top, np.uint8), np.ascontiguousarray(tex_side, np.uint8)
    ptr = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)   # noqa: E731
    lib().vo_render_cell_types(ptr(nodes), C.byref(params), ptr(pal), ptr(ty), ptr(tt), ptr(ts), ptr(accum), ptr(rgba), C.byref(stats))
    return accum, rgba, stats
