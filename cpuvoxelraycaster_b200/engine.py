"""Host-side mirror of the reference's hot-path interface over libvrt's C ABI.

Names follow the reference (file:line under the reference tree):
  Volumetric.castRay        include/volumetric.hpp:55-61
  LSVO                      include/lsvo.hpp:10-24, castRay :33
  Grid3D / MipmapGrid3D     include/grid_3d.hpp:10-27, include/mipmap_grid3D.hpp:14-17
  SVO                       include/svo.hpp:29, castRay :62, setCell :72
  Camera                    include/camera_controller.hpp:16-61
  RayCaster                 include/raycaster.hpp:43-282 (renderRay :67 → render(): whole frames)
Batched entry points (cast_rays, render) are the additions: the reference casts one ray per call from
a swarm worker (src/main.cpp:139-152); here one call is one kernel launch.
"""
import ctypes as C
import os
import weakref

import numpy as np

from . import capi
from .capi import HIT, LNODE, check, lib, ptr


def _f32(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float32)
    if shape is not None:
        a = a.reshape(shape)
    return a


# ---- host-side scene construction (src/main.cpp:59-86) ----------------------------------------------
def host_terrain_heights(size):
    out = np.zeros((size, size), np.int32)
    check(lib().vrt_host_terrain_heights(size, ptr(out)))
    return out


def host_build_terrain_lsvo(depth, heights=None):
    if heights is None:
        heights = host_terrain_heights(1 << depth)
    heights = np.ascontiguousarray(heights, np.int32)
    n = C.c_uint64(0)
    check(lib().vrt_host_build_terrain_lsvo(depth, ptr(heights), None, 0, C.byref(n)))
    nodes = np.zeros(n.value, LNODE)
    check(lib().vrt_host_build_terrain_lsvo(depth, ptr(heights), ptr(nodes), n.value, C.byref(n)))
    return nodes[:n.value]


def host_build_lsvo_from_voxels(depth, xyz):
    xyz = np.ascontiguousarray(xyz, np.uint32).reshape(-1, 3)
    n = C.c_uint64(0)
    check(lib().vrt_host_build_lsvo_from_voxels(depth, ptr(xyz), len(xyz), None, 0, C.byref(n)))
    nodes = np.zeros(n.value, LNODE)
    check(lib().vrt_host_build_lsvo_from_voxels(depth, ptr(xyz), len(xyz), ptr(nodes), n.value, C.byref(n)))
    return nodes[:n.value]


# ---- execution resource -------------------------------------------------------------------------------
class Context:
    """One CUDA device + stream (replaces swrm::Swarm, src/main.cpp:90-92). Not thread-safe."""

    def __init__(self, device=0, stream=None):
        h = C.c_void_p()
        check(lib().vrt_context_create(int(device), C.c_void_p(stream) if stream else None, C.byref(h)))
        self.handle = h
        self.device = int(device)
        self._scenes = weakref.WeakSet()      # scenes hold a pointer to the context: they must die first

        for key in ("cast_variant", "render_variant", "refill_cast", "refill_render", "spp_chunks", "samples_per_warp", "sort_bins1", "sort_bins2"):      # measurement overrides (tools/, profiles/)
            v = os.environ.get("VRT_" + key.upper())
            if v is not None:
                self.set_option(key, int(v))

    def set_option(self, key, value):
        check(lib().vrt_context_set_option(self.handle, key.encode(), int(value)))

    def take_kernel_timings(self):
        """Device times (ms) of the frame-kernel calls bracketed since the last take (option "time_frame_kernels" = 1)."""
        n = C.c_int32(0)
        buf = (C.c_float * 4096)()
        check(lib().vrt_context_take_timings(self.handle, buf, 4096, C.byref(n)))
        return [float(buf[i]) for i in range(min(n.value, 4096))]

    def synchronize(self):
        check(lib().vrt_context_synchronize(self.handle))

    def set_stream(self, stream):
        check(lib().vrt_context_set_stream(self.handle, C.c_void_p(stream) if stream else None))

    @property
    def launch_count(self):
        return int(lib().vrt_context_launch_count(self.handle))

    def close(self):
        if getattr(self, "handle", None):
            for sc in list(self._scenes):
                sc.close()
            lib().vrt_context_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class HitPoint:
    """include/volumetric.hpp:7-22 for one ray; `cell` is truthy on a hit."""

    __slots__ = ("position", "normal", "voxel_coord", "cell", "distance", "complexity")

    def __init__(self, rec):
        self.position = rec["position"].copy()
        self.normal = rec["normal"].copy()
        self.voxel_coord = rec["voxel_coord"].copy()
        self.cell = bool(rec["flags"] & 1)
        self.distance = float(rec["distance"])
        self.complexity = int(rec["complexity"])


class Volumetric:
    """include/volumetric.hpp:55-61."""

    def __init__(self, ctx):
        self.ctx = ctx
        self.handle = None
        ctx._scenes.add(self)

    # -- batched: n rays, one launch --
    def cast_rays(self, origin, direction, ray_size_coef=0.0, ray_size_bias=0.0):
        o, d = _f32(origin, (-1, 3)), _f32(direction, (-1, 3))
        if o.shape != d.shape:
            raise ValueError("origin and direction must have the same shape")
        out = np.zeros(len(o), HIT)
        check(lib().vrt_cast_rays(self.handle, ptr(o), ptr(d), ray_size_coef, ray_size_bias, len(o), ptr(out)))
        return out

    def cast_rays_device(self, d_origin, d_dir, n, d_out, ray_size_coef=0.0, ray_size_bias=0.0):
        """Device pointers (ints or torch tensors); enqueues on the context stream."""
        check(lib().vrt_cast_rays_device(self.handle, ptr(d_origin), ptr(d_dir), ray_size_coef, ray_size_bias, int(n),
                                         ptr(d_out)))

    # -- reference signature: one ray --
    def castRay(self, position, direction, ray_size_coef=0.0, ray_size_bias=0.0):
        return HitPoint(self.cast_rays([position], [direction], ray_size_coef, ray_size_bias)[0])

    def set_textures(self, top_rgb, side_rgb):
        """RayCaster::image_top / image_side (raycaster.hpp:53-54): 16x16 RGB, top-down rows."""
        t, s = np.ascontiguousarray(top_rgb, np.uint8), np.ascontiguousarray(side_rgb, np.uint8)
        if t.size != 768 or s.size != 768:
            raise ValueError("textures must be 16x16 RGB")
        check(lib().vrt_scene_set_textures(self.handle, ptr(t), ptr(s)))

    def last_complexity(self):
        v = C.c_uint64(0)
        check(lib().vrt_scene_last_complexity(self.handle, C.byref(v)))
        return v.value

    def info(self):
        k, d, b = C.c_int32(0), C.c_uint32(0), C.c_uint64(0)
        check(lib().vrt_scene_info(self.handle, C.byref(k), C.byref(d), C.byref(b)))
        return dict(kind=k.value, depth=d.value, device_bytes=b.value)

    def close(self):
        if getattr(self, "handle", None):
            lib().vrt_scene_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class LSVO(Volumetric):
    """LSVO<MAX_DEPTH> (include/lsvo.hpp:10). `nodes` is the reference's flattened layout (LNode[])."""

    def __init__(self, ctx, nodes, depth, guard=0):
        super().__init__(ctx)
        nodes = np.ascontiguousarray(nodes)
        if nodes.dtype.itemsize != 8:
            raise ValueError("nodes must be 8-byte LNode records")
        h = C.c_void_p()
        check(lib().vrt_lsvo_create(ctx.handle, ptr(nodes), len(nodes), int(depth), int(guard), C.byref(h)))
        self.handle = h
        self.depth = int(depth)
        self.n_nodes = len(nodes)
        self._layout_from_env()

    def _layout_from_env(self):
        v = os.environ.get("VRT_LAYOUT")                       # measurement override: "1" compact, "1p" compact + L2 window
        if v:
            self.set_layout(int(v[0]), v.endswith("p"))

    @classmethod
    def from_terrain(cls, ctx, depth, guard=0, on_device=True):
        """The demo scene T(D): src/main.cpp:59-83.  Built on the GPU by default (byte-identical to the host builder)."""
        if not on_device:
            return cls(ctx, host_build_terrain_lsvo(depth), depth, guard)
        self = cls.__new__(cls)
        Volumetric.__init__(self, ctx)
        h = C.c_void_p()
        check(lib().vrt_lsvo_create_terrain(ctx.handle, int(depth), int(guard), C.byref(h)))
        self.handle = h
        self.depth = int(depth)
        self.n_nodes = len(self)
        self._layout_from_env()
        return self

    @classmethod
    def from_heightfield(cls, ctx, depth, heights=None, guard=0):
        """A world given by column heights[x, z] with the demo's fill rule (src/main.cpp:70-76), flattened on the GPU and
        editable afterwards (edit_heights).  heights=None: the demo's FastNoise terrain."""
        S = 1 << int(depth)
        self = cls.__new__(cls)
        Volumetric.__init__(self, ctx)
        h = C.c_void_p()
        hp = None
        if heights is not None:
            hh = np.ascontiguousarray(heights, np.int32)
            if hh.shape != (S, S):
                raise ValueError("heights must be [2^depth, 2^depth]")
            hp = ptr(hh)
        check(lib().vrt_lsvo_create_heightfield(ctx.handle, int(depth), hp, int(guard), C.byref(h)))
        self.handle = h
        self.depth = int(depth)
        self.n_nodes = len(self)
        self._layout_from_env()
        return self

    def edit_heights(self, x0, z0, heights):
        """Dynamic scene (the reference's LSVO::setCell is a no-op, lsvo.hpp:26): replaces the heights of the columns
        [x0, x0+nx) x [z0, z0+nz) and re-flattens the world on the device."""
        hh = np.ascontiguousarray(heights, np.int32)
        check(lib().vrt_scene_edit_heights(self.handle, int(x0), int(z0), hh.shape[0], hh.shape[1], ptr(hh)))
        self.n_nodes = len(self)

    def heights(self):
        S = 1 << self.depth
        out = np.zeros((S, S), np.int32)
        check(lib().vrt_scene_download_heights(self.handle, ptr(out)))
        return out

    def set_layout(self, layout, l2_persist=False):
        """0 = the reference's LNode array, 1 = compact breadth-first live nodes (same results, 8x smaller)."""
        check(lib().vrt_scene_set_layout(self.handle, int(layout), int(bool(l2_persist))))

    def __len__(self):
        n = C.c_uint64(0)
        check(lib().vrt_scene_download_nodes(self.handle, None, 0, C.byref(n)))
        return int(n.value)

    def download_nodes(self):
        """LSVO::data (lsvo.hpp:287)."""
        n = C.c_uint64(0)
        check(lib().vrt_scene_download_nodes(self.handle, None, 0, C.byref(n)))
        nodes = np.zeros(n.value, LNODE)
        check(lib().vrt_scene_download_nodes(self.handle, ptr(nodes), n.value, C.byref(n)))
        return nodes

    @classmethod
    def from_voxels(cls, ctx, depth, xyz, guard=0, on_device=False, colors=None):
        """SVO::setCell for every voxel (svo.hpp:72) followed by LSVO(const SVO&) (lsvo.hpp:12).  on_device=True: the
        voxel list is flattened on the GPU (byte-identical) and stays editable through set_cells.  colors (uint8 per voxel,
        optional): painted afterwards (paint_cells)."""
        if not on_device:
            self = cls(ctx, host_build_lsvo_from_voxels(depth, xyz), depth, guard)
        else:
            v = np.ascontiguousarray(np.asarray(xyz, np.uint32).reshape(-1, 3))
            self = cls.__new__(cls)
            Volumetric.__init__(self, ctx)
            h = C.c_void_p()
            check(lib().vrt_lsvo_create_from_voxels(ctx.handle, int(depth), ptr(v) if len(v) else None, len(v), int(guard), C.byref(h)))
            self.handle = h
            self.depth = int(depth)
            self.n_nodes = len(self)
            self._layout_from_env()
        if colors is not None:
            self.paint_cells(xyz, colors)
        return self

    def paint_cells(self, xyz, colors):
        """Per-voxel colours (extension): sets the `color` byte of the leaf slots of the solid voxels xyz (setCell
        coordinates).  Empty voxels are skipped; a voxel listed twice takes its last colour.  Returns the number of distinct
        solid voxels painted.  Frames show the colours through set_palette."""
        v = np.ascontiguousarray(np.asarray(xyz, np.uint32).reshape(-1, 3))
        c = np.ascontiguousarray(np.broadcast_to(np.asarray(colors, np.uint8), (len(v),)))
        n = C.c_uint64(0)
        check(lib().vrt_scene_paint_cells(self.handle, ptr(v) if len(v) else None, ptr(c) if len(v) else None, len(v), C.byref(n)))
        return int(n.value)

    def cell_colors(self, xyz):
        """int16 per voxel: its colour, or -1 where the voxel is empty."""
        v = np.ascontiguousarray(np.asarray(xyz, np.uint32).reshape(-1, 3))
        out = np.zeros(len(v), np.int16)
        check(lib().vrt_scene_cell_colors(self.handle, ptr(v) if len(v) else None, len(v), ptr(out) if len(v) else None))
        return out

    def set_palette(self, rgb):
        """rgb: uint8 [256, 3] (entry c is the albedo of colour c) — frames take the albedo from it instead of the textures;
        None = back to the textures."""
        if rgb is None:
            check(lib().vrt_scene_set_palette(self.handle, None))
            return
        p = np.ascontiguousarray(rgb, np.uint8)
        if p.size != 768:
            raise ValueError("the palette must be 256 RGB entries")
        check(lib().vrt_scene_set_palette(self.handle, ptr(p)))

    def set_cell_types(self, types):
        """types: 256 ints, the Cell::Type of the voxels of each colour (1 = Solid, 2 = Mirror) — camera rays reflect off mirror
        voxels (vrt_scene_set_cell_types); None = all Solid."""
        if types is None:
            check(lib().vrt_scene_set_cell_types(self.handle, None))
            return
        t = np.asarray(types).reshape(-1)
        if t.size != 256:
            raise ValueError("the cell-type table must have 256 entries")
        if not np.isin(t, (1, 2)).all():
            raise ValueError("cell types must be 1 (Solid) or 2 (Mirror)")
        t = np.ascontiguousarray(t, np.uint8)
        check(lib().vrt_scene_set_cell_types(self.handle, ptr(t)))

    def set_point_lights(self, positions, colors=None, ranges=None):
        """Point lights (vrt_scene_set_point_lights): positions (n,3) in the normalised castRay frame of light_position, colors (n,3)
        linear RGB >= 0 (1,1,1 = white), ranges (n,) > 0 (inf allowed); n <= 16.  None (or n = 0) clears them."""
        if positions is None:
            check(lib().vrt_scene_set_point_lights(self.handle, None, 0))
            return
        pos = np.asarray(positions, np.float32)
        n = len(pos) if pos.ndim == 2 else -1
        col = np.asarray(colors, np.float32) if colors is not None else None
        rng = np.asarray(ranges, np.float32) if ranges is not None else None
        if n < 0 or pos.shape != (n, 3) or col is None or col.shape != (n, 3) or rng is None or rng.shape != (n,):
            raise ValueError("point lights need positions (n,3), colors (n,3) and ranges (n,)")
        if n > 16:
            raise ValueError("at most 16 point lights")
        if not np.isfinite(pos).all():
            raise ValueError("light positions must be finite")
        if not (np.isfinite(col).all() and (col >= 0).all()):
            raise ValueError("light colours must be finite and >= 0")
        if not (rng > 0).all():
            raise ValueError("light ranges must be > 0 (inf allowed)")
        a = np.zeros(n, capi.POINT_LIGHT)
        a["position"], a["color"], a["range"] = pos, col, rng
        check(lib().vrt_scene_set_point_lights(self.handle, ptr(a) if n else None, n))

    def set_cells(self, xyz, solid=True):
        """Dynamic scene: adds (solid) or removes voxels of a from_voxels(on_device=True) world and re-flattens it on
        the device — what LSVO::setCell would do if it were not a no-op (lsvo.hpp:26)."""
        v = np.ascontiguousarray(np.asarray(xyz, np.uint32).reshape(-1, 3))
        check(lib().vrt_scene_set_cells(self.handle, ptr(v) if len(v) else None, len(v), int(bool(solid))))
        self.n_nodes = len(self)

    def voxel_count(self):
        n = C.c_uint64(0)
        check(lib().vrt_scene_voxel_count(self.handle, C.byref(n)))
        return int(n.value)

    def setCell(self, *a):
        """No-op, as in the reference (lsvo.hpp:26); see set_cells."""


class Grid3D(Volumetric):
    """Grid3D<X,Y,Z> (include/grid_3d.hpp:10). cells[x,y,z] = Cell::Type (0 Empty, 1 Solid, 2 Mirror)."""

    mip_levels = 0

    def __init__(self, ctx, cells):
        super().__init__(ctx)
        cells = np.ascontiguousarray(cells, np.uint8)
        X, Y, Z = cells.shape
        h = C.c_void_p()
        check(lib().vrt_grid_create(ctx.handle, ptr(cells), X, Y, Z, int(self.mip_levels), C.byref(h)))
        self.handle = h
        self.shape = (X, Y, Z)

    def castRay(self, position, direction):  # grid_3d.hpp:16 takes no cone arguments
        return HitPoint(self.cast_rays([position], [direction])[0])


class MipmapGrid3D(Grid3D):
    """MipmapGrid3D<X,Y,Z,MipmapDepth> (include/mipmap_grid3D.hpp:14-17; an empty stub in the reference).
    Results are bit-identical to Grid3D; the occupancy pyramid only removes memory fetches."""

    def __init__(self, ctx, cells, mip_levels=3):
        self.mip_levels = int(mip_levels)
        super().__init__(ctx, cells)


class SVO(Volumetric):
    """SVO<N> (include/svo.hpp:29) with the hit fill of svo.hpp:116-138 restored ("intended SVO")."""

    def __init__(self, ctx, occ):
        super().__init__(ctx)
        occ = np.ascontiguousarray(occ, np.uint8)
        S = occ.shape[0]
        if occ.shape != (S, S, S) or S & (S - 1):
            raise ValueError("occupancy must be a cube with a power-of-two edge")
        h = C.c_void_p()
        check(lib().vrt_svo_create(ctx.handle, ptr(occ), S.bit_length() - 1, C.byref(h)))
        self.handle = h
        self.depth = S.bit_length() - 1

    def cast_rays(self, origin, direction, max_iter=1 << 30):
        o, d = _f32(origin, (-1, 3)), _f32(direction, (-1, 3))
        out = np.zeros(len(o), HIT)
        check(lib().vrt_cast_rays_svo(self.handle, ptr(o), ptr(d), int(max_iter), len(o), ptr(out)))
        return out

    def castRay(self, position, direction, max_iter):  # svo.hpp:62
        return HitPoint(self.cast_rays([position], [direction], max_iter)[0])


# ---- camera -------------------------------------------------------------------------------------------
class Camera:
    """include/camera_controller.hpp:16-61."""

    def __init__(self, position=(256.0, 200.0, 256.0), view_angle=(0.0, 0.0), fov=1.0, aperture=0.0, focal_length=1.0):
        self.position = np.asarray(position, np.float32)
        self.fov = float(fov)
        self.aperture = float(aperture)
        self.focal_length = float(focal_length)
        self.setViewAngle(view_angle)

    def setViewAngle(self, angle):
        """camera_controller.hpp:27-32 + generateRotationMatrix (utils.cpp:94-100), computed by libvrt's host code
        with the C library's cosf/sinf like the reference."""
        self.view_angle = np.asarray(angle, np.float32)
        m = np.zeros(9, np.float32)
        v = np.zeros(3, np.float32)
        check(lib().vrt_host_camera_rotation(ptr(self.view_angle), ptr(m), ptr(v)))
        self.rot_mat = m
        self.camera_vec = v

    def as_struct(self):
        c = capi.Camera()
        c.position[:] = [float(x) for x in self.position]
        c.rot_mat[:] = [float(x) for x in self.rot_mat]
        c.fov, c.aperture, c.focal_length = self.fov, self.aperture, self.focal_length
        return c

    def getClosestPoint(self, volume):
        """camera_controller.hpp:56-60 (the centre ray)."""
        scale = np.float32(1.0) / np.float32(1 << volume.depth)
        return volume.castRay(self.position * scale + np.float32(1.0), self.camera_vec, 0.0, 0.0)

    def autofocus(self, volume):
        """src/main.cpp:115-121, evaluated on the device."""
        f = C.c_float(0)
        check(lib().vrt_autofocus(volume.handle, C.byref(self.as_struct()), C.byref(f)))
        self.focal_length = f.value
        return f.value


class CameraController:
    """include/camera_controller.hpp:64-78."""
    movement_speed = 1.0

    def updateCameraView(self, d_view_angle, camera):
        new_angle = camera.view_angle + np.asarray(d_view_angle, np.float32)
        half_pi = np.float32(3.141592653) * np.float32(0.5)          # PI, camera_controller.hpp:8
        new_angle[1] = min(max(new_angle[1], -half_pi), half_pi)
        camera.setViewAngle(new_angle)

    def move(self, move_vector, camera):
        raise NotImplementedError


class FlyController(CameraController):
    """include/fly_controller.hpp:6-12."""

    def move(self, move_vector, camera):
        camera.position = camera.position + np.asarray(move_vector, np.float32)


class ReplayElements:
    """include/replay.hpp:8-33: one tick of a recorded camera path, `timestamp x y z view_x view_y` per line."""
    __slots__ = ("timestamp", "x", "y", "z", "view_x", "view_y")

    def __init__(self, timestamp, x, y, z, view_x, view_y):
        self.timestamp, self.x, self.y, self.z, self.view_x, self.view_y = (float(np.float32(v)) for v in (timestamp, x, y, z, view_x, view_y))

    @staticmethod
    def loadFromFile(filename):
        """Whitespace-separated floats, six per tick; reading stops at the first token that is not a number or at an
        incomplete tick, like `file >> ...` (replay.hpp:26).  A missing file gives an empty list (:24)."""
        try:
            with open(filename) as f:
                tokens = f.read().split()
        except OSError:
            return []
        values = []
        for t in tokens:
            try:
                values.append(float(t))
            except ValueError:
                break
        return [ReplayElements(*values[i:i + 6]) for i in range(0, len(values) - len(values) % 6, 6)]

    def apply(self, camera):
        """Puts the camera where the tick was recorded."""
        camera.position = np.float32([self.x, self.y, self.z])
        camera.setViewAngle((self.view_x, self.view_y))


# ---- renderer -----------------------------------------------------------------------------------------
class RayCaster:
    """include/raycaster.hpp:43.  render() replaces the swarm lambda of src/main.cpp:139-154."""

    def __init__(self, svo, render_size, tex_top=None, tex_side=None):
        self.svo = svo
        self.render_size = (int(render_size[0]), int(render_size[1]))
        W, H = self.render_size
        self.render_image = np.zeros((H, W, 4), np.uint8)     # sf::Image render_image (raycaster.hpp:261)
        self.colors = np.zeros((H, W, 4), np.uint32)          # Sample accumulators r,g,b,count (raycaster.hpp:259)
        self.light_position = np.zeros(3, np.float32)
        self.use_gi = False
        self.use_samples = False
        self.gi_bounces = 1
        self.roughness = 0.0            # blur of Cell::Mirror reflections (extension)
        self.mirror_y = None            # LSVO volumes: voxel layer (castRay y) whose top faces are mirrors; None = no mirrors
        self.max_bounds = 4             # raycaster.hpp:277
        self.checker_board_offset = None   # None = every pixel; 0 / 1 = the checkerboard of main.cpp:137,143
        self.checker_area_height = 0       # RENDER_HEIGHT / area_count (main.cpp:132); 0 = one area
        self.display = None                # denoised_tex of main.cpp:159-177, made by present()
        self.autofocus = False             # True: focal length from the centre ray on the device (main.cpp:114-121)
        self.seed = (0x5EED, 0)
        self.sample_count = 0
        self.frame_index = 0               # frames rendered in blend mode: selects the random stream of the frame
        self.last_stats = None
        if tex_top is not None:
            svo.set_textures(tex_top, tex_side)

    def setLightPosition(self, position):                       # raycaster.hpp:62
        self.light_position = np.asarray(position, np.float32)

    def resetSamples(self):                                     # raycaster.hpp:105-116
        self.colors[...] = 0
        self.sample_count = 0

    def params(self, spp=1, row_begin=0, row_end=0, sample_offset=None):
        p = capi.RenderParams()
        p.width, p.height = self.render_size
        p.row_begin, p.row_end = int(row_begin), int(row_end) if row_end else self.render_size[1]
        p.spp = int(spp)
        if sample_offset is None:
            sample_offset = self.sample_count if self.use_samples else self.frame_index
        p.sample_offset = int(sample_offset)
        p.seed_lo, p.seed_hi = self.seed
        p.light_position[:] = [float(x) for x in self.light_position]
        p.use_gi, p.gi_bounces, p.use_samples = int(self.use_gi), int(self.gi_bounces), int(self.use_samples)
        p.roughness, p.max_bounds = float(self.roughness), int(self.max_bounds)
        p.checker = 0 if self.checker_board_offset is None else 1 + (int(self.checker_board_offset) & 1)
        p.checker_area_height = int(self.checker_area_height)
        p.mirror_y1 = 0 if self.mirror_y is None else int(self.mirror_y) + 1
        p.autofocus = int(bool(self.autofocus))
        return p

    def render(self, camera, spp=1, row_begin=0, row_end=0):
        """One frame: `spp` renderRay passes per pixel (every pixel, or the checkerboard half selected by
        checker_board_offset), then samples_to_image when use_samples, else the 0.4/0.6 temporal blend into
        render_image (raycaster.hpp:77-91)."""
        p = self.params(spp, row_begin, row_end)
        stats = capi.RenderStats()
        if self.use_samples:
            p.accum_in = 1                                      # progressive: sums carry over (raycaster.hpp:87-90)
        else:
            self.colors[...] = 0
        check(lib().vrt_render(self.svo.handle, C.byref(camera.as_struct()), C.byref(p), ptr(self.render_image),
                               ptr(self.colors), C.byref(stats)))
        if self.use_samples:
            self.sample_count += int(spp)
        else:
            self.frame_index += 1
        culled = C.c_uint64(0)          # primary rays answered by the beam search instead of a walk (vrt_scene_last_render_culled)
        check(lib().vrt_scene_last_render_culled(self.svo.handle, C.byref(culled)))
        self.last_stats = dict(rays=list(stats.rays), complexity=list(stats.complexity), culled_primary=int(culled.value))
        return self.render_image

    def beam_floors(self, camera, tile=8):
        """Diagnostic (vrt_beam_floors): per-tile start distances of the camera rays, float32 [tiles_y, tiles_x]."""
        W, H = self.render_size
        tx, ty = (W + tile - 1) // tile, (H + tile - 1) // tile
        out = np.zeros((ty, tx), np.float32)
        check(lib().vrt_beam_floors(self.svo.handle, C.byref(camera.as_struct()), C.byref(self.params(1)), int(tile), ptr(out)))
        return out

    def present(self, median=0, old_value_conservation=None):
        """The presentation step of the main loop (src/main.cpp:159-177): optional 3x3 / 5x5 median
        (res/median_3.frag, res/median.frag) and the persistence blend into `display`."""
        if old_value_conservation is None:
            old_value_conservation = 0.0 if self.use_samples else 0.1          # main.cpp:160
        W, H = self.render_size
        if self.display is None:
            self.display = np.zeros((H, W, 4), np.uint8)
        p = capi.PresentParams(W, H, int(median), float(old_value_conservation))
        check(lib().vrt_present(self.svo.ctx.handle, ptr(self.render_image), ptr(self.display), C.byref(p)))
        return self.display

    def samples_to_image(self):
        """raycaster.hpp:94-103 — already applied on the device by render() when use_samples."""
        return self.render_image
