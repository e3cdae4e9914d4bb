r"""Per-voxel colours (DESIGN.md §2, "Per-voxel colours"): vrt_scene_paint_cells / vrt_scene_cell_colors write and read the `color`
byte of a solid voxel's leaf slot, vrt_scene_set_palette turns it into the albedo of frames.

| test                                       | what it pins                                                                         |
|--------------------------------------------|--------------------------------------------------------------------------------------|
| test_paint_writes_leaf_slots               | voxel set, T(9) and a host array: only the painted voxels' leaf-slot colour bytes change (slots from a numpy getAtRayHit descent); counts, last occurrence wins, empty voxels, -1 |
| test_paint_argument_checks                 | VRT_ERR_INVALID for bad arguments, VRT_ERR_UNSUPPORTED for heightfield, grid and SVO scenes |
| test_colours_survive_set_cells             | paint, add and remove voxels: the array equals a scene built and painted from scratch |
| test_painting_changes_no_cast_or_textured_frame | casts (cast_variant 0-3, both layouts) and K4 / K6 frames (beam floors and bounds exits off and on) |
| test_palette_frames_match_the_oracle       | K4 (spp 1, 4) and K6 (spp 16) against vo_render_palette: GI 1 / 2 bounces, DOF, mirrors, checkerboard, autofocus, binding guard, temporal blend, product defaults |
| test_clearing_the_palette                  | set_palette(None) gives the textured frame back byte for byte                        |
| test_shade_rays_with_palette               | vrt_shade_rays against the oracle's 1-sample palette frames, reference and compact layout |
| test_palette_refusals_and_no_textures      | compact layout and render_variant 1 / 3 refuse palette frames; no textures needed     |
| test_communicator_palette_frame            | a world-1 vrt_comm_create_local frame equals the vrt_render frame                    |
| test_cpp_dropin_palette                    | tests/cpp/palette_test.cpp: paintCells, getCellColors, setPalette through RayCaster   |

Contexts are created without beam floors and bounds exits (tests/conftest.py); the product-default rows turn them back on.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, golden
from palette_oracle import render_palette

pytestmark = pytest.mark.gpu

INVALID, UNSUPPORTED = -1, -4
DEMO_VIEW = dict(position=(256, 200, 256), view_angle=(0.3, -0.35))
W, H = 96, 54
SHADE_JOB = np.dtype([("start", "f4", 3), ("pixel", "u4"), ("direction", "f4", 3), ("sample", "u4")])
SHADE_RESULT = np.dtype([("r", "u1"), ("g", "u1"), ("b", "u1"), ("hit", "u1"), ("distance", "f4"), ("complexity", "u4"),
                         ("reserved", "u4")])


def default_light(depth=9):
    return np.float32([-200, -1000, -300]) * np.float32(1.0 / (1 << depth)) + np.float32(1.0)


def make_palette(seed=7):
    return np.random.default_rng(seed).integers(0, 256, (256, 3), dtype=np.uint8)


def leaf_slots(nodes, depth, xyz):
    """LSVO::getAtRayHit's descent in numpy, setCell coordinates: leaf slot per voxel, -1 where a child bit is missing."""
    xyz = np.asarray(xyz, np.int64).reshape(-1, 3)
    node = np.zeros(len(xyz), np.int64)
    out = np.full(len(xyz), -1, np.int64)
    live = np.ones(len(xyz), bool)
    for b in range(depth - 1, -1, -1):
        slot = ((xyz[:, 0] >> b) & 1) | (((xyz[:, 1] >> b) & 1) << 1) | (((xyz[:, 2] >> b) & 1) << 2)
        nd = nodes[node]
        has = ((nd["child_mask"].astype(np.int64) >> slot) & 1) != 0
        live &= has
        child = node + nd["child_offset"].astype(np.int64) + slot
        leaf = live & (((nd["leaf_mask"].astype(np.int64) >> slot) & 1) != 0) & (out < 0)
        out[leaf] = child[leaf]
        node = np.where(live & (out < 0), child, 0)
    return out


def height_band_cells(depth=9, seed=3, n=60000):
    """Voxels of T(depth)'s hills and some air, coloured by height band, with repeats (the last one wins)."""
    rng = np.random.default_rng(seed)
    S = 1 << depth
    xyz = np.stack([rng.integers(0, S, n), rng.integers(S // 2, S // 2 + 90, n), rng.integers(0, S, n)], 1).astype(np.uint32)
    colors = (2 + (xyz[:, 1] - S // 2) // 6).astype(np.uint8)
    xyz = np.concatenate([xyz, xyz[:500]])
    colors = np.concatenate([colors, (colors[:500] + 100).astype(np.uint8)])
    return xyz, colors


def expected_paint(nodes, depth, xyz, colors):
    slots = leaf_slots(nodes, depth, xyz)
    want = nodes.copy()
    last = {}
    for i, s in enumerate(slots):
        if s >= 0:
            last[int(s)] = colors[i]
    idx = np.fromiter(last.keys(), np.int64, len(last))
    want["color"][idx] = np.fromiter(last.values(), np.uint8, len(last))
    return want, len(last), slots


def port_params(vrt, depth, cam, use_gi=1, bounces=2, use_samples=True, spp=1, offset=0, guard=None, mirror_y1=0):
    from oracle import loader
    p = loader.PortRenderParams()
    p.width, p.height, p.depth, p.guard = W, H, depth, depth if guard is None else guard
    p.cam_position[:] = [float(x) for x in cam.position]
    p.rot_mat[:] = [float(x) for x in cam.rot_mat]
    p.fov, p.aperture, p.focal_length = cam.fov, cam.aperture, cam.focal_length
    p.light_position[:] = [float(x) for x in default_light(depth)]
    p.use_gi, p.gi_bounces, p.use_samples, p.spp = int(use_gi), bounces, int(use_samples), spp
    p.seed_lo, p.seed_hi, p.sample_offset = 0x5EED, 0, offset
    p.threads = 8
    p.roughness, p.max_bounds, p.mirror_y1 = 0.05, 4, mirror_y1
    return p


def ray_caster(vrt, scene, use_gi=True, bounces=2, use_samples=True, mirror_y=None):
    rc = vrt.RayCaster(scene, (W, H))
    rc.setLightPosition(default_light(scene.depth))
    rc.use_samples, rc.use_gi, rc.gi_bounces = use_samples, use_gi, bounces
    rc.mirror_y, rc.roughness = mirror_y, 0.05
    return rc


@pytest.fixture(scope="module")
def painted9(vrt, terrain9_nodes):
    """T(9) painted by height band: (nodes, xyz, colors)."""
    xyz, colors = height_band_cells()
    want, count, _ = expected_paint(terrain9_nodes, 9, xyz, colors)
    assert count > 20000
    return want, xyz, colors


def painted_scene(vrt, c, painted9, textures=None, guard=0):
    nodes, xyz, colors = painted9
    s = vrt.LSVO(c, vrt.host_build_terrain_lsvo(9), 9, guard)
    s.paint_cells(xyz, colors)
    if textures is not None:
        s.set_textures(*textures)
    return s


# ---- 1: painting ----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["voxels", "terrain", "host"])
def test_paint_writes_leaf_slots(vrt, ctx, terrain9_nodes, kind):
    rng = np.random.default_rng(11)
    if kind == "voxels":
        depth = 6
        solid = np.unique(rng.integers(0, 64, (3000, 3)).astype(np.uint32), axis=0)
        s = vrt.LSVO.from_voxels(ctx, depth, solid, on_device=True)
        empty = np.uint32([[v, 63 - v, v] for v in range(64)])
        empty = empty[leaf_slots(s.download_nodes(), depth, empty) < 0][:20]
        xyz = np.concatenate([solid[rng.permutation(len(solid))[:1200]], empty, solid[:50]])
    else:
        depth = 9
        s = vrt.LSVO.from_terrain(ctx, 9) if kind == "terrain" else vrt.LSVO(ctx, terrain9_nodes, 9)
        xyz, _ = height_band_cells(n=20000, seed=5)
    colors = rng.integers(0, 256, len(xyz)).astype(np.uint8)
    colors[colors == 1] = 2
    before = s.download_nodes()
    want, count, slots = expected_paint(before, depth, xyz, colors)
    assert 0 < count < len(xyz) and (slots < 0).any()
    assert s.paint_cells(xyz, colors) == count
    got = s.download_nodes()
    assert np.array_equal(got.view(np.uint64), want.view(np.uint64))
    changed = np.flatnonzero(got["color"] != before["color"])
    assert set(changed.tolist()) <= set(slots[slots >= 0].tolist())
    cc = s.cell_colors(xyz)
    assert np.array_equal(cc[slots < 0], np.full(int((slots < 0).sum()), -1, np.int16))
    assert np.array_equal(cc[slots >= 0], want["color"][slots[slots >= 0]].astype(np.int16))
    # last occurrence wins: the voxels listed twice carry the colour of their second entry
    if kind == "voxels":
        dup = solid[:50]
        assert np.array_equal(s.cell_colors(dup), colors[-50:].astype(np.int16))
        assert (s.cell_colors(solid) >= 0).all()


def test_paint_argument_checks(vrt, ctx, terrain9_nodes):
    lib = vrt.capi.lib()
    n = C.c_uint64(0)
    s = vrt.LSVO.from_voxels(ctx, 5, [[1, 2, 3], [4, 5, 6]], on_device=True)
    xyz = np.uint32([[1, 2, 3], [32, 0, 0]])
    col = np.uint8([9, 9])
    assert lib.vrt_scene_paint_cells(s.handle, vrt.capi.ptr(xyz), vrt.capi.ptr(col), 2, C.byref(n)) == INVALID
    assert s.cell_colors([[1, 2, 3]])[0] == 1                    # nothing was painted
    assert lib.vrt_scene_paint_cells(s.handle, None, vrt.capi.ptr(col), 1, None) == INVALID
    assert lib.vrt_scene_paint_cells(s.handle, vrt.capi.ptr(xyz), None, 1, None) == INVALID
    assert lib.vrt_scene_paint_cells(None, vrt.capi.ptr(xyz), vrt.capi.ptr(col), 1, None) == INVALID
    out = np.zeros(2, np.int16)
    assert lib.vrt_scene_cell_colors(s.handle, vrt.capi.ptr(xyz), 2, vrt.capi.ptr(out)) == INVALID
    assert lib.vrt_scene_cell_colors(s.handle, None, 1, vrt.capi.ptr(out)) == INVALID
    assert lib.vrt_scene_cell_colors(None, vrt.capi.ptr(xyz), 1, vrt.capi.ptr(out)) == INVALID
    assert lib.vrt_scene_set_palette(None, None) == INVALID
    assert lib.vrt_scene_paint_cells(s.handle, None, None, 0, C.byref(n)) == 0 and n.value == 0
    hf = vrt.LSVO.from_heightfield(ctx, 6, np.full((64, 64), 40, np.int32))
    assert lib.vrt_scene_paint_cells(hf.handle, vrt.capi.ptr(xyz), vrt.capi.ptr(col), 1, None) == UNSUPPORTED
    grid = vrt.Grid3D(ctx, np.ones((8, 8, 8), np.uint8))
    svo = vrt.SVO(ctx, np.ones((8, 8, 8), np.uint8))
    pal = make_palette()
    for g in (grid, svo):
        assert lib.vrt_scene_paint_cells(g.handle, vrt.capi.ptr(xyz), vrt.capi.ptr(col), 1, None) == UNSUPPORTED
        assert lib.vrt_scene_cell_colors(g.handle, vrt.capi.ptr(xyz), 1, vrt.capi.ptr(out)) == UNSUPPORTED
        assert lib.vrt_scene_set_palette(g.handle, vrt.capi.ptr(pal)) == UNSUPPORTED
    for sc in (hf, grid, svo, s):
        sc.close()


# ---- 2: persistence across set_cells --------------------------------------------------------------------------------------------
def test_colours_survive_set_cells(vrt, ctx):
    rng = np.random.default_rng(21)
    depth = 6
    base = np.unique(rng.integers(0, 64, (4000, 3)).astype(np.uint32), axis=0)
    s = vrt.LSVO.from_voxels(ctx, depth, base, on_device=True)
    bytes0 = s.info()["device_bytes"]
    colors = rng.integers(2, 256, len(base)).astype(np.uint8)
    s.paint_cells(base, colors)
    assert s.info()["device_bytes"] == bytes0 + len(base)          # one colour byte per resident key
    colour = {tuple(v): int(c) for v, c in zip(base.tolist(), colors)}
    removed = base[:300]
    s.set_cells(removed, solid=False)
    for v in removed.tolist():
        colour.pop(tuple(v))
    added = np.concatenate([removed[:100], np.unique(rng.integers(0, 64, (500, 3)).astype(np.uint32), axis=0)])
    s.set_cells(added, solid=True)
    for v in added.tolist():
        colour.setdefault(tuple(v), 1)                              # new, or removed and added again: LNode()'s colour
    final = np.uint32(sorted(colour.keys()))
    fresh = vrt.LSVO.from_voxels(ctx, depth, final, on_device=True)
    fc = np.uint8([colour[tuple(v)] for v in final.tolist()])
    fresh.paint_cells(final, fc)
    assert np.array_equal(s.download_nodes().view(np.uint64), fresh.download_nodes().view(np.uint64))
    assert (s.cell_colors(removed[:100]) == 1).all()
    assert np.array_equal(s.cell_colors(final), fc.astype(np.int16))
    assert s.info()["device_bytes"] == fresh.info()["device_bytes"]
    s.close()
    fresh.close()


# ---- 3: nothing changes without a palette ---------------------------------------------------------------------------------------
def test_painting_changes_no_cast_or_textured_frame(vrt, terrain9_nodes, textures, painted9):
    rng = np.random.default_rng(0)
    n = 70000
    o = rng.uniform(1, 2, (n, 3)).astype(np.float32)
    o[:, 1] = rng.uniform(1.0, 1.45, n)
    d = rng.normal(size=(n, 3)).astype(np.float32)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    c = vrt.Context(0)
    try:
        plain = vrt.LSVO(c, terrain9_nodes, 9)
        plain.set_textures(*textures)
        paint = painted_scene(vrt, c, painted9, textures)
        for layout in (0, 1):
            plain.set_layout(layout)
            paint.set_layout(layout)
            for variant in range(4):
                c.set_option("cast_variant", variant)
                for coef in (0.0, 0.5):
                    want = plain.cast_rays(o, d, coef)
                    got = paint.cast_rays(o, d, coef)
                    assert np.array_equal(got.view(np.uint8), want.view(np.uint8)), (layout, variant, coef)
        plain.set_layout(0)
        paint.set_layout(0)
        cam = vrt.Camera(aperture=0.5, focal_length=60.0, **DEMO_VIEW)
        for beam in (0, 1):
            c.set_option("beam_tile", 8 * beam)
            c.set_option("bounds_exit", beam)
            for spp in (2, 16):                                     # K4, K6
                frames = []
                for s in (plain, paint):
                    rc = ray_caster(vrt, s)
                    frames.append((rc.render(cam, spp).copy(), rc.colors.copy(), rc.last_stats))
                assert np.array_equal(frames[0][0], frames[1][0]) and np.array_equal(frames[0][1], frames[1][1]), (beam, spp)
                assert frames[0][2] == frames[1][2], (beam, spp)
    finally:
        c.close()


# ---- 4: palette frames against the oracle ---------------------------------------------------------------------------------------
CONFIGS = {
    "gi1":      dict(bounces=1),
    "gi2":      dict(bounces=2),
    "nogi":     dict(use_gi=False),
    "dof":      dict(bounces=2, aperture=2.0, focal_length=40.0),
    "mirror":   dict(bounces=2, mirror_y=240),
    "checker":  dict(bounces=1, checker=True),
    "autofocus": dict(bounces=2, autofocus=True),
    "guard":    dict(bounces=2, guard=14),
    "blend":    dict(bounces=1, use_samples=False),
    "defaults": dict(bounces=2, product=True),
}


@pytest.mark.parametrize("config", sorted(CONFIGS))
def test_palette_frames_match_the_oracle(vrt, port, textures, painted9, config):
    cfg = CONFIGS[config]
    nodes = painted9[0]
    pal = make_palette()
    c = vrt.Context(0)
    if cfg.get("product"):
        c.set_option("beam_tile", 8)
        c.set_option("bounds_exit", 1)
    try:
        s = painted_scene(vrt, c, painted9, textures, guard=cfg.get("guard", 0))
        s.set_palette(pal)
        cam = vrt.Camera(aperture=cfg.get("aperture", 0.5), focal_length=cfg.get("focal_length", 60.0), **DEMO_VIEW)
        if cfg.get("autofocus"):
            cam.autofocus(s)
        use_samples = cfg.get("use_samples", True)
        for spp in ((1, 4, 16) if use_samples else (1,)):
            rc = ray_caster(vrt, s, use_gi=cfg.get("use_gi", True), bounces=cfg.get("bounces", 1), use_samples=use_samples,
                            mirror_y=cfg.get("mirror_y"))
            rc.autofocus = bool(cfg.get("autofocus"))
            if cfg.get("checker"):
                rc.checker_board_offset, rc.checker_area_height = 1, 18
            prev = np.zeros((H, W, 4), np.uint8)
            for frame in range(1 if use_samples else 2):
                img = rc.render(cam, spp).copy()
                p = port_params(vrt, 9, cam, cfg.get("use_gi", True), cfg.get("bounces", 1), use_samples, spp,
                                offset=frame, guard=cfg.get("guard"), mirror_y1=cfg.get("mirror_y", -1) + 1)
                if cfg.get("checker"):
                    p.checker, p.checker_area_height = 2, 18
                accum, rgba, st = render_palette(nodes, p, pal, *textures, prev_rgba=prev)
                label = "%s, spp %d, frame %d" % (config, spp, frame)
                if use_samples:
                    assert np.array_equal(rc.colors, accum), "%s: accumulators differ on %d pixels" % (label, int((rc.colors != accum).any(-1).sum()))
                    done = accum[..., 3] > 0
                    assert np.array_equal(img[done], rgba[done]), label
                else:
                    assert np.array_equal(img, rgba), label
                    prev = rgba
                assert rc.last_stats["rays"] == list(st.rays), label
                if cfg.get("product"):
                    assert all(x <= y for x, y in zip(rc.last_stats["complexity"], st.complexity)), label
                else:
                    assert rc.last_stats["complexity"] == list(st.complexity), label
                if config not in ("guard",):
                    assert accum[..., :3].max() > 0 or rgba[..., :3].max() > 0, label
    finally:
        c.close()


def test_palette_frame_uses_the_colours(vrt, textures, painted9):
    """A palette frame differs from the textured one."""
    c = vrt.Context(0)
    try:
        s = painted_scene(vrt, c, painted9, textures)
        cam = vrt.Camera(aperture=0.0, focal_length=60.0, **DEMO_VIEW)
        rc = ray_caster(vrt, s, use_gi=False)
        textured = rc.render(cam, 1).copy()
        s.set_palette(make_palette())
        rc.resetSamples()
        pal_img = rc.render(cam, 1).copy()
        assert (pal_img != textured).any(-1).mean() > 0.2
    finally:
        c.close()


# ---- 5: clearing --------------------------------------------------------------------------------------------------------------
def test_clearing_the_palette(vrt, textures, painted9):
    c = vrt.Context(0)
    try:
        s = painted_scene(vrt, c, painted9, textures)
        cam = vrt.Camera(aperture=0.5, focal_length=60.0, **DEMO_VIEW)
        out = []
        for pal in (None, make_palette(), None):
            s.set_palette(pal)
            for spp in (2, 16):
                rc = ray_caster(vrt, s)
                out.append((pal is None, spp, rc.render(cam, spp).copy(), rc.colors.copy()))
        assert not np.array_equal(out[0][2], out[2][2])
        for a, b in ((out[0], out[4]), (out[1], out[5])):
            assert np.array_equal(a[2], b[2]) and np.array_equal(a[3], b[3]), a[1]
    finally:
        c.close()


# ---- 6: vrt_shade_rays --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("layout", [0, 1])
def test_shade_rays_with_palette(vrt, port, textures, painted9, layout):
    nodes = painted9[0]
    pal = make_palette()
    c = vrt.Context(0)
    try:
        s = painted_scene(vrt, c, painted9, textures)
        s.set_palette(pal)
        if layout:
            s.set_layout(1)
        cam = vrt.Camera(aperture=0.5, focal_length=60.0, **DEMO_VIEW)
        for sample in (0, 3):
            p0 = port_params(vrt, 9, cam, spp=1, offset=sample)
            rays = [port.camera_ray(p0, x, y, sample) for y in range(H) for x in range(W)]
            jobs = np.zeros(W * H, SHADE_JOB)
            jobs["start"] = [o for o, _ in rays]
            jobs["direction"] = [d for _, d in rays]
            jobs["pixel"] = np.arange(W * H)
            jobs["sample"] = sample
            for use_gi, bounces in ((0, 1), (1, 2)):
                p = port_params(vrt, 9, cam, use_gi, bounces, True, 1, offset=sample)
                accum, _, _ = render_palette(nodes, p, pal, *textures)
                q = vrt.capi.RenderParams()
                q.width, q.height, q.spp, q.use_samples = W, H, 1, 1
                q.seed_lo, q.seed_hi = 0x5EED, 0
                q.light_position[:] = [float(x) for x in default_light()]
                q.use_gi, q.gi_bounces = use_gi, bounces
                out = np.zeros(len(jobs), SHADE_RESULT)
                vrt.capi.check(vrt.capi.lib().vrt_shade_rays(s.handle, C.byref(q), len(jobs), vrt.capi.ptr(jobs), vrt.capi.ptr(out)))
                rgb = np.stack([out["r"], out["g"], out["b"]], -1)
                assert np.array_equal(rgb, accum.reshape(-1, 4)[:, :3]), (layout, sample, use_gi)
                assert 0.2 < (out["hit"] != 0).mean() < 0.95
    finally:
        c.close()


# ---- 7: refusals, textures ----------------------------------------------------------------------------------------------------
def test_palette_refusals_and_no_textures(vrt, port, textures, painted9):
    nodes = painted9[0]
    pal = make_palette()
    lib = vrt.capi.lib()
    c = vrt.Context(0)
    try:
        s = painted_scene(vrt, c, painted9)                         # no textures
        cam = vrt.Camera(aperture=0.5, focal_length=60.0, **DEMO_VIEW)
        rc = ray_caster(vrt, s)
        with pytest.raises(vrt.VrtError):
            rc.render(cam, 1)                                       # neither textures nor a palette
        s.set_palette(pal)
        img = rc.render(cam, 4).copy()
        accum, rgba, _ = render_palette(nodes, port_params(vrt, 9, cam, 1, 2, True, 4), pal, *textures)
        assert np.array_equal(rc.colors, accum) and np.array_equal(img, rgba)
        cs = cam.as_struct()
        p = rc.params(1)
        buf = np.zeros((H, W, 4), np.uint8)
        for variant in (1, 3):
            c.set_option("render_variant", variant)
            assert lib.vrt_render(s.handle, C.byref(cs), C.byref(p), vrt.capi.ptr(buf), None, None) == UNSUPPORTED
        c.set_option("render_variant", 0)
        s.set_layout(1)
        assert lib.vrt_render(s.handle, C.byref(cs), C.byref(p), vrt.capi.ptr(buf), None, None) == UNSUPPORTED
        s.set_palette(None)
        with pytest.raises(vrt.VrtError):
            rc.render(cam, 1)                                       # textures again, and there are none
    finally:
        c.close()


# ---- 8: the communicator ------------------------------------------------------------------------------------------------------
def test_communicator_palette_frame(vrt, textures, painted9):
    capi = vrt.capi
    pal = make_palette()
    c = vrt.Context(0)
    comm = None
    try:
        s = painted_scene(vrt, c, painted9, textures)
        s.set_palette(pal)
        cam = vrt.Camera(aperture=0.5, focal_length=60.0, **DEMO_VIEW).as_struct()
        p = capi.RenderParams()
        p.width, p.height, p.row_begin, p.row_end = W, H, 0, H
        p.spp, p.seed_lo, p.seed_hi = 16, 0x5EED, 0
        p.light_position[:] = [float(x) for x in default_light()]
        p.use_gi, p.gi_bounces, p.use_samples, p.max_bounds = 1, 2, 1, 4
        want = np.zeros((H, W, 4), np.uint8)
        capi.check(capi.lib().vrt_render(s.handle, C.byref(cam), C.byref(p), capi.ptr(want), None, None))
        ctxs = (C.c_void_p * 1)(c.handle.value)
        out = (C.c_void_p * 1)()
        capi.check(capi.lib().vrt_comm_create_local(ctxs, 1, W, H, out))
        comm = C.c_void_p(out[0])
        for split in (capi.SPLIT_TILES, capi.SPLIT_SAMPLES):
            host = np.zeros((H, W, 4), np.uint8)
            capi.check(capi.lib().vrt_render_distributed(comm, s.handle, C.byref(cam), C.byref(p), split, 0, capi.ptr(host)))
            capi.check(capi.lib().vrt_comm_frame_wait(comm))
            assert np.array_equal(host, want), split
        assert want[..., :3].max() > 0
    finally:
        if comm is not None:
            capi.lib().vrt_comm_destroy(comm)
        c.close()


# ---- 9: the C++ drop-in -------------------------------------------------------------------------------------------------------
def test_cpp_dropin_palette(vrt, ctx, textures, tmp_path):
    exe, tex = str(tmp_path / "palette_test"), str(tmp_path / "textures.bin")
    lib_dir = os.path.join(ROOT, "cpuvoxelraycaster_b200")
    subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-I" + os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "tests", "cpp", "palette_test.cpp"), "-o", exe, "-L" + lib_dir, "-lvrt",
                    "-Wl,-rpath," + lib_dir], check=True)
    t = golden("textures.npz")
    with open(tex, "wb") as f:
        f.write(t["top"].tobytes() + t["side"].tobytes())
    r = subprocess.run([exe, tex], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    out = {line.split(" ", 1)[0]: line.split(" ", 1)[1] for line in r.stdout.strip().splitlines()}
    # the same in Python (the C++ program runs with the product defaults: beam floors and bounds exits on)
    c = vrt.Context(0)
    c.set_option("beam_tile", 8)
    c.set_option("bounds_exit", 1)
    try:
        s = vrt.LSVO(c, vrt.host_build_terrain_lsvo(9), 9)
        g = np.mgrid[160:352, 256:352, 160:352].reshape(3, -1).T.astype(np.uint32)
        painted = s.paint_cells(g, (2 + (g[:, 1] - 256) // 4).astype(np.uint8))
        coloured = int((s.download_nodes()["color"] != 1).sum())
        probe = s.cell_colors([[200, 257, 200], [0, 511, 0]])
        assert out["paint"] == "painted=%d coloured=%d probe=%d,%d" % (painted, coloured, probe[0], probe[1])
        assert painted > 100000 and probe[1] == -1
        cc = np.arange(256)
        pal = np.stack([cc * 37, cc * 91 + 40, cc * 53 + 90], -1).astype(np.uint8)
        s.set_palette(pal)
        rc = vrt.RayCaster(s, (W, H), *textures)
        rc.setLightPosition(default_light())
        rc.use_samples, rc.use_gi = True, True
        cam = vrt.Camera(aperture=0.5, focal_length=60.0, **DEMO_VIEW)

        def fnv(a):
            h = 1469598103934665603
            for b in a.tobytes():
                h = ((h ^ b) * 1099511628211) & 0xFFFFFFFFFFFFFFFF
            return "hash=%016x" % h
        assert out["frame"] == fnv(rc.render(cam, 2))
        s.set_palette(None)
        rc.resetSamples()
        assert out["textured"] == fnv(rc.render(cam, 2))
        assert out["frame"] != out["textured"]
    finally:
        c.close()
