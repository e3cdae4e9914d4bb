"""TEST INFRASTRUCTURE ONLY: ctypes bindings for the two CPU checkers under oracle/.

  port()        oracle/libvrt_oracle.so   — the C restatement (oracle/port.c)
  ref()         oracle/_ref/libvrt_ref.so — the reference's own sources, compiled (may be absent)
  ref_patched() oracle/_ref/libvrt_ref_patched.so — Grid3D / intended-SVO variants
  ref_depth(d)  oracle/_ref/libvrt_ref_d{d}.so    — RayCaster/Camera rebuilt for octree depth d

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs import this.
The product package never does.
"""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))

PORT_HIT = np.dtype([("position", "f4", 3), ("normal", "f4", 3), ("voxel_coord", "f4", 2), ("distance", "f4"),
                     ("complexity", "u4"), ("hit", "u4"), ("scale", "i4"), ("voxel", "i4", 3), ("face", "u4")])
REF_HIT = np.dtype([("position", "f4", 3), ("normal", "f4", 3), ("voxel_coord", "f4", 2), ("distance", "f4"),
                    ("complexity", "u4"), ("hit", "u4"), ("pad", "u4")])
LNODE = np.dtype([("color", "u1"), ("child_mask", "u1"), ("leaf_mask", "u1"), ("pad", "u1"), ("child_offset", "u4")])


class PortRenderParams(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("depth", C.c_int32), ("guard", C.c_int32),
                ("cam_position", C.c_float * 3), ("rot_mat", C.c_float * 9),
                ("fov", C.c_float), ("aperture", C.c_float), ("focal_length", C.c_float),
                ("light_position", C.c_float * 3),
                ("use_gi", C.c_int32), ("gi_bounces", C.c_int32), ("use_samples", C.c_int32), ("spp", C.c_int32),
                ("seed_lo", C.c_uint32), ("seed_hi", C.c_uint32), ("sample_offset", C.c_int32),
                ("row_begin", C.c_int32), ("row_end", C.c_int32), ("threads", C.c_int32),
                ("tile_step", C.c_int32), ("tile_index", C.c_int32), ("roughness", C.c_float), ("max_bounds", C.c_int32),
                ("checker", C.c_int32), ("checker_area_height", C.c_int32), ("mirror_y1", C.c_int32)]


class PortRenderStats(C.Structure):
    _fields_ = [("rays", C.c_uint64 * 6), ("complexity", C.c_uint64 * 6)]


class RefRenderParams(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("cam_position", C.c_float * 3),
                ("view_angle", C.c_float * 2), ("fov", C.c_float), ("aperture", C.c_float),
                ("focal_length", C.c_float), ("light_position", C.c_float * 3),
                ("use_gi", C.c_int32), ("use_samples", C.c_int32), ("spp", C.c_int32), ("threads", C.c_int32),
                ("row_begin", C.c_int32), ("row_end", C.c_int32), ("tile_step", C.c_int32), ("tile_index", C.c_int32),
                ("checker", C.c_int32), ("checker_area_height", C.c_int32), ("frames", C.c_int32)]


class RefRayCounts(C.Structure):
    _fields_ = [("cone0_calls", C.c_uint64), ("cone_gi_calls", C.c_uint64)]


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def build(quiet=True):
    """(Re)build the checkers: the port always, oracle/_ref only where $VRT_REFERENCE names the reference tree."""
    subprocess.run(["make", "-s" if quiet else "-j1", "-C", HERE, "all"], check=True,
                   stdout=subprocess.DEVNULL if quiet else None)


_cache = {}


def _load(path):
    if path not in _cache:
        _cache[path] = C.CDLL(path) if os.path.exists(path) else None
    return _cache[path]


class Port:
    def __init__(self, lib):
        self.lib = L = lib
        L.vo_build_terrain_lsvo.restype = C.c_uint64
        L.vo_build_terrain_lsvo.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_uint64]
        L.vo_build_dense_lsvo.restype = C.c_uint64
        L.vo_build_dense_lsvo.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_uint64]
        L.vo_noise2d.restype = C.c_float
        L.vo_noise2d.argtypes = [C.c_float, C.c_float]
        L.vo_terrain_heights.argtypes = [C.c_int32, C.c_void_p]
        L.vo_lsvo_cast.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_float, C.c_float,
                                   C.c_uint64, C.c_void_p, C.c_int]
        L.vo_lsvo_cast_restructured.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_float, C.c_float, C.c_int,
                                                C.c_uint64, C.c_void_p, C.c_int]
        L.vo_grid_cast.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_uint64,
                                   C.c_void_p, C.c_void_p, C.c_int]
        L.vo_grid_miss_test.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                        C.c_void_p, C.c_uint64, C.c_void_p, C.c_int]
        L.vo_svo_cast.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint64, C.c_void_p,
                                  C.c_int]
        L.vo_render.argtypes = [C.c_void_p, C.POINTER(PortRenderParams), C.c_void_p, C.c_void_p, C.c_void_p,
                                C.c_void_p, C.POINTER(PortRenderStats)]
        L.vo_grid_render.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(PortRenderParams), C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.POINTER(PortRenderStats)]
        L.vo_camera_ray.argtypes = [C.POINTER(PortRenderParams), C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                    C.c_void_p]
        L.vo_philox4x32_10.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]

    def terrain_heights(self, size):
        out = np.zeros((size, size), np.int32)
        self.lib.vo_terrain_heights(size, _p(out))
        return out

    def build_terrain(self, depth, heights=None):
        if heights is None:
            heights = self.terrain_heights(1 << depth)
        heights = np.ascontiguousarray(heights, np.int32)
        n = self.lib.vo_build_terrain_lsvo(depth, _p(heights), None, 0)
        nodes = np.zeros(n, LNODE)
        self.lib.vo_build_terrain_lsvo(depth, _p(heights), _p(nodes), n)
        return nodes

    def build_dense(self, depth, occ):
        occ = np.ascontiguousarray(occ, np.uint8)
        n = self.lib.vo_build_dense_lsvo(depth, _p(occ), None, 0)
        nodes = np.zeros(n, LNODE)
        self.lib.vo_build_dense_lsvo(depth, _p(occ), _p(nodes), n)
        return nodes

    def lsvo_cast(self, nodes, depth, origin, direction, coef=0.0, bias=0.0, guard=None, threads=1):
        o, d = _f32(origin), _f32(direction)
        out = np.zeros(len(o), PORT_HIT)
        self.lib.vo_lsvo_cast(_p(nodes), depth, depth if guard is None else guard, _p(o), _p(d), coef, bias, len(o),
                              _p(out), threads)
        return out

    def lsvo_cast_restructured(self, nodes, depth, origin, direction, coef=0.0, bias=0.0, guard=None, unit=False, threads=1):
        """The walk with the device loop's structural changes (port.c: lsvo_cast_one_restructured); must equal lsvo_cast."""
        o, d = _f32(origin), _f32(direction)
        out = np.zeros(len(o), PORT_HIT)
        self.lib.vo_lsvo_cast_restructured(_p(nodes), depth, depth if guard is None else guard, _p(o), _p(d), coef, bias,
                                           1 if unit else 0, len(o), _p(out), threads)
        return out

    def grid_cast(self, cells, origin, direction, threads=1):
        cells = np.ascontiguousarray(cells, np.uint8)
        o, d = _f32(origin), _f32(direction)
        out = np.zeros(len(o), PORT_HIT)
        steps = np.zeros(len(o), np.uint32)
        X, Y, Z = cells.shape
        self.lib.vo_grid_cast(_p(cells), X, Y, Z, _p(o), _p(d), len(o), _p(out), _p(steps), threads)
        return out, steps

    def grid_miss_test(self, cells, shift, origin, direction, threads=1):
        """Prototype (port.c grid_miss_one): 1 where a ray certainly misses the dense grid, judged on the OR-pyramid level `shift`
        dilated by two cubes; 0 = has to be walked."""
        cells = np.ascontiguousarray(cells, np.uint8)
        X, Y, Z = cells.shape
        k = 1 << shift
        assert X % k == 0 and Y % k == 0 and Z % k == 0
        coarse = cells.reshape(X // k, k, Y // k, k, Z // k, k).max(axis=(1, 3, 5)) != 0
        dil = coarse.copy()
        for axis in range(3):                                   # box dilation by two cubes, axis by axis
            acc = dil.copy()
            for s in (1, 2):
                a = np.zeros_like(dil); b = np.zeros_like(dil)
                sl_to = [slice(None)] * 3; sl_from = [slice(None)] * 3
                sl_to[axis], sl_from[axis] = slice(s, None), slice(None, -s)
                a[tuple(sl_to)] = dil[tuple(sl_from)]
                b[tuple(sl_from)] = dil[tuple(sl_to)]
                acc |= a | b
            dil = acc
        dil = np.ascontiguousarray(dil, np.uint8)
        o, d = _f32(origin), _f32(direction)
        out = np.zeros(len(o), np.uint8)
        self.lib.vo_grid_miss_test(_p(dil), dil.shape[0], dil.shape[1], dil.shape[2], shift, X, Y, Z, _p(o), _p(d), len(o), _p(out), threads)
        return out

    def svo_cast(self, occ, depth, origin, direction, max_iter=1 << 30, threads=1):
        occ = np.ascontiguousarray(occ, np.uint8)
        o, d = _f32(origin), _f32(direction)
        out = np.zeros(len(o), PORT_HIT)
        self.lib.vo_svo_cast(_p(occ), depth, _p(o), _p(d), max_iter, len(o), _p(out), threads)
        return out

    def render(self, nodes, params, tex_top, tex_side, prev_rgba=None):
        """Returns (accum uint32 [H,W,4], rgba uint8 [H,W,4], stats)."""
        H, W = params.height, params.width
        accum = np.zeros((H, W, 4), np.uint32)
        rgba = np.zeros((H, W, 4), np.uint8) if prev_rgba is None else np.ascontiguousarray(prev_rgba).copy()
        stats = PortRenderStats()
        tt, ts = np.ascontiguousarray(tex_top, np.uint8), np.ascontiguousarray(tex_side, np.uint8)
        self.lib.vo_render(_p(nodes), C.byref(params), _p(tt), _p(ts), _p(accum), _p(rgba), C.byref(stats))
        return accum, rgba, stats

    def grid_render(self, cells, params, tex_top, tex_side):
        """Grid shading with mirror reflections (extension). Returns (accum, rgba, stats)."""
        cells = np.ascontiguousarray(cells, np.uint8)
        X, Y, Z = cells.shape
        H, W = params.height, params.width
        accum = np.zeros((H, W, 4), np.uint32)
        rgba = np.zeros((H, W, 4), np.uint8)
        stats = PortRenderStats()
        tt, ts = np.ascontiguousarray(tex_top, np.uint8), np.ascontiguousarray(tex_side, np.uint8)
        self.lib.vo_grid_render(_p(cells), X, Y, Z, C.byref(params), _p(tt), _p(ts), _p(accum), _p(rgba), C.byref(stats))
        return accum, rgba, stats

    def present(self, frame, display, median=0, old_value_conservation=0.1):
        """main.cpp:159-177: returns the new display image (uint8 [H,W,4])."""
        frame = np.ascontiguousarray(frame, np.uint8)
        out = np.ascontiguousarray(display, np.uint8).copy()
        H, W = frame.shape[:2]
        self.lib.vo_present(_p(frame), _p(out), W, H, int(median), C.c_float(old_value_conservation))
        return out

    def camera_ray(self, params, x, y, sample=0):
        o = np.zeros(3, np.float32)
        d = np.zeros(3, np.float32)
        self.lib.vo_camera_ray(C.byref(params), x, y, sample, _p(o), _p(d))
        return o, d

    def philox(self, ctr, key):
        c = np.asarray(ctr, np.uint32)
        k = np.asarray(key, np.uint32)
        out = np.zeros(4, np.uint32)
        self.lib.vo_philox4x32_10(_p(c), _p(k), _p(out))
        return out


class Ref:
    """The reference's own code (verbatim headers; RayCaster/Camera at the depth the .so was built for)."""

    def __init__(self, lib):
        self.lib = L = lib
        for f in ("vrt_ref_scene_terrain", "vrt_ref_scene_from_voxels", "vrt_ref_scene_from_nodes"):
            getattr(L, f).restype = C.c_void_p
        L.vrt_ref_scene_terrain.argtypes = [C.c_int]
        L.vrt_ref_scene_from_voxels.argtypes = [C.c_int, C.c_void_p, C.c_uint64]
        L.vrt_ref_scene_from_nodes.argtypes = [C.c_int, C.c_void_p, C.c_uint64]
        L.vrt_ref_scene_destroy.argtypes = [C.c_void_p]
        L.vrt_ref_scene_node_count.restype = C.c_uint64
        L.vrt_ref_scene_node_count.argtypes = [C.c_void_p]
        L.vrt_ref_scene_copy_nodes.argtypes = [C.c_void_p, C.c_void_p]
        L.vrt_ref_terrain_heights.argtypes = [C.c_int, C.c_void_p]
        L.vrt_ref_noise2d.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]
        L.vrt_ref_lsvo_cast.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_float, C.c_uint64,
                                        C.c_void_p, C.c_int]
        L.vrt_ref_camera_basis.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.vrt_ref_camera_rays.argtypes = [C.POINTER(RefRenderParams), C.c_void_p, C.c_void_p]
        L.vrt_ref_autofocus.restype = C.c_float
        L.vrt_ref_autofocus.argtypes = [C.c_void_p, C.POINTER(RefRenderParams)]
        L.vrt_ref_render.argtypes = [C.c_void_p, C.POINTER(RefRenderParams), C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.POINTER(C.c_double), C.POINTER(RefRayCounts)]
        L.vrt_ref_register_texture.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_void_p]
        L.vrt_ref_getrand.argtypes = [C.c_uint64, C.c_void_p]
        self.depth = L.vrt_ref_compiled_depth()

    def register_textures(self, tex_top, tex_side):
        tt, ts = np.ascontiguousarray(tex_top, np.uint8), np.ascontiguousarray(tex_side, np.uint8)
        self.lib.vrt_ref_register_texture(b"grass_top_16x16.bmp", 16, 16, _p(tt))
        self.lib.vrt_ref_register_texture(b"grass_side_16x16.bmp", 16, 16, _p(ts))

    def scene_terrain(self, depth):
        return self.lib.vrt_ref_scene_terrain(depth)

    def scene_from_voxels(self, depth, xyz):
        xyz = np.ascontiguousarray(xyz, np.uint32).reshape(-1, 3)
        return self.lib.vrt_ref_scene_from_voxels(depth, _p(xyz), len(xyz))

    def scene_from_nodes(self, depth, nodes):
        nodes = np.ascontiguousarray(nodes)
        return self.lib.vrt_ref_scene_from_nodes(depth, _p(nodes), len(nodes))

    def scene_destroy(self, s):
        self.lib.vrt_ref_scene_destroy(s)

    def nodes(self, scene):
        n = self.lib.vrt_ref_scene_node_count(scene)
        out = np.zeros(n, LNODE)
        self.lib.vrt_ref_scene_copy_nodes(scene, _p(out))
        return out

    def terrain_heights(self, size):
        out = np.zeros((size, size), np.int32)
        self.lib.vrt_ref_terrain_heights(size, _p(out))
        return out

    def noise2d(self, x, y):
        x, y = _f32(x), _f32(y)
        out = np.zeros(len(x), np.float32)
        self.lib.vrt_ref_noise2d(_p(x), _p(y), len(x), _p(out))
        return out

    def lsvo_cast(self, scene, origin, direction, coef=0.0, bias=0.0, threads=1):
        o, d = _f32(origin), _f32(direction)
        out = np.zeros(len(o), REF_HIT)
        code = self.lib.vrt_ref_lsvo_cast(scene, _p(o), _p(d), coef, bias, len(o), _p(out), threads)
        if code < 0:
            raise RuntimeError("reference swarm dropped part of the job")
        return out

    def camera_basis(self, view_angle):
        va = _f32(view_angle)
        m = np.zeros(9, np.float32)
        v = np.zeros(3, np.float32)
        self.lib.vrt_ref_camera_basis(_p(va), _p(m), _p(v))
        return m, v

    def camera_rays(self, params):
        n = params.width * params.height
        o = np.zeros((n, 3), np.float32)
        d = np.zeros((n, 3), np.float32)
        self.lib.vrt_ref_camera_rays(C.byref(params), _p(o), _p(d))
        return o, d

    def autofocus(self, scene, params):
        return float(self.lib.vrt_ref_autofocus(scene, C.byref(params)))

    def render(self, scene, params, want_raw=False):
        """Returns dict(raw, image, samples, seconds, code)."""
        H, W = params.height, params.width
        raw = np.zeros((H, W, 4), np.uint8) if want_raw else None
        img = np.zeros((H, W, 4), np.uint8)
        smp = np.zeros((H, W, 4), np.float64)
        sec = C.c_double(0)
        cnt = RefRayCounts()
        code = self.lib.vrt_ref_render(scene, C.byref(params), _p(raw), _p(img), _p(smp), C.byref(sec), C.byref(cnt))
        if code < 0:
            raise RuntimeError("reference render failed (code %d)" % code)
        return dict(raw=raw, image=img, samples=smp, seconds=sec.value, code=code,
                    cone0_calls=cnt.cone0_calls, cone_gi_calls=cnt.cone_gi_calls)

    def getrand(self, n):
        out = np.zeros(n, np.float32)
        self.lib.vrt_ref_getrand(n, _p(out))
        return out


class RefPatched:
    def __init__(self, lib):
        self.lib = L = lib
        L.vrt_ref_grid_create.restype = C.c_void_p
        L.vrt_ref_grid_create.argtypes = [C.c_int, C.c_void_p]
        L.vrt_ref_grid_destroy.argtypes = [C.c_void_p]
        L.vrt_ref_grid_cast.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]
        L.vrt_ref_svo_create.restype = C.c_void_p
        L.vrt_ref_svo_create.argtypes = [C.c_int, C.c_void_p]
        L.vrt_ref_svo_destroy.argtypes = [C.c_void_p]
        L.vrt_ref_svo_cast.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint64, C.c_void_p]

    def grid_create(self, occ):
        occ = np.ascontiguousarray(occ, np.uint8)
        n = occ.shape[0]
        assert occ.shape == (n, n, n) and n & (n - 1) == 0
        return self.lib.vrt_ref_grid_create(n.bit_length() - 1, _p(occ))

    def grid_destroy(self, g):
        self.lib.vrt_ref_grid_destroy(g)

    def grid_cast(self, g, origin, direction):
        o, d = _f32(origin), _f32(direction)
        out = np.zeros(len(o), REF_HIT)
        self.lib.vrt_ref_grid_cast(g, _p(o), _p(d), len(o), _p(out))
        return out

    def svo_create(self, occ):
        occ = np.ascontiguousarray(occ, np.uint8)
        n = occ.shape[0]
        return self.lib.vrt_ref_svo_create(n.bit_length() - 1, _p(occ))

    def svo_destroy(self, s):
        self.lib.vrt_ref_svo_destroy(s)

    def svo_cast(self, s, origin, direction, max_iter=1 << 30):
        o, d = _f32(origin), _f32(direction)
        out = np.zeros(len(o), REF_HIT)
        self.lib.vrt_ref_svo_cast(s, _p(o), _p(d), max_iter, len(o), _p(out))
        return out


def port():
    path = os.path.join(HERE, "libvrt_oracle.so")
    if not os.path.exists(path):
        build()
    return Port(C.CDLL(path))


def ref():
    lib = _load(os.path.join(HERE, "_ref", "libvrt_ref.so"))
    return Ref(lib) if lib is not None else None


def ref_depth(depth):
    if depth == 9:
        return ref()
    lib = _load(os.path.join(HERE, "_ref", "libvrt_ref_d%d.so" % depth))
    return Ref(lib) if lib is not None else None


def ref_patched():
    lib = _load(os.path.join(HERE, "_ref", "libvrt_ref_patched.so"))
    return RefPatched(lib) if lib is not None else None
