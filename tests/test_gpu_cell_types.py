r"""Mirror voxels (DESIGN.md §2, "Mirror voxels"): vrt_scene_set_cell_types gives each colour a Cell::Type, and camera-chain
rays reflect off the voxels whose colour is Cell::Mirror.  Frames are compared with tests/cell_types_oracle.c vo_render_cell_types.

| test                                       | what it pins                                                                         |
|--------------------------------------------|--------------------------------------------------------------------------------------|
| test_frames_match_the_oracle               | K4 (spp 1, 4) and K6 (spp 16) on walls facing x / y / z, a cube and facing mirrors: GI 1 / 2 bounces, roughness 0 / 0.3, DOF, palette, lake + table, checkerboard, autofocus, temporal blend, product defaults |
| test_facing_mirrors_max_bounds             | two facing mirrors with max_bounds 0, 1, 4 and 16                                     |
| test_edge_and_zero_normal_hits             | frames with edge hits and zero-normal hits on mirror voxels (shown by a cast of the camera rays) |
| test_slab_equals_the_lake                  | a complete layer painted Mirror renders the lake frame of that layer                 |
| test_heightfield_colour_one                | a heightfield with types[1] = Mirror: every voxel is a mirror                        |
| test_mirrors_survive_set_cells             | set_cells on a painted scene: mirror voxels stay mirrors, added voxels follow types[1] |
| test_shade_rays_with_mirror_voxels         | vrt_shade_rays against the oracle's 1-sample frames, reference and compact layout     |
| test_communicator_frame                    | a world-1 vrt_comm_create_local frame equals the vrt_render frame                    |
| test_refusals                              | values 0 and 3, grid and SVO scenes, compact layout, render_variant 1 / 3, max_bounds 17 |
| test_clearing_and_all_solid                | clearing the table (or an all-Solid one) gives the frame without it byte for byte     |
| test_casts_unchanged                       | cast_variant 0-3: the table changes no cast                                           |
| test_cpp_dropin_cell_types                 | tests/cpp/cell_types_test.cpp: setCellTypes / clearCellTypes through RayCaster       |

Contexts are created without beam floors and bounds exits (tests/conftest.py); the product-default rows turn them back on.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import cell_types_scenes as cts
from conftest import ROOT, golden
from cell_types_oracle import render_cell_types

pytestmark = pytest.mark.gpu

INVALID, UNSUPPORTED = -1, -4
W, H = 52, 30
SHADE_JOB = np.dtype([("start", "f4", 3), ("pixel", "u4"), ("direction", "f4", 3), ("sample", "u4")])
SHADE_RESULT = np.dtype([("r", "u1"), ("g", "u1"), ("b", "u1"), ("hit", "u1"), ("distance", "f4"), ("complexity", "u4"),
                         ("reserved", "u4")])


def gpu_scene(vrt, c, xyz, colours, textures=None):
    """A painted voxel-set scene; its node array must equal the host-painted one the oracle renders."""
    s = vrt.LSVO.from_voxels(c, cts.DEPTH, xyz, on_device=True, colors=colours)
    nodes = cts.host_nodes(vrt, xyz, colours)
    assert np.array_equal(s.download_nodes().view(np.uint64), nodes.view(np.uint64))
    if textures is not None:
        s.set_textures(*textures)
    return s, nodes


def ray_caster(vrt, scene, cfg):
    rc = vrt.RayCaster(scene, (W, H))
    rc.setLightPosition(cts.default_light())
    rc.use_samples = cfg.get("use_samples", True)
    rc.use_gi, rc.gi_bounces = cfg.get("use_gi", True), cfg.get("bounces", 2)
    rc.roughness, rc.max_bounds = cfg.get("roughness", 0.0), cfg.get("max_bounds", 4)
    rc.mirror_y = cfg.get("mirror_y")
    rc.autofocus = bool(cfg.get("autofocus"))
    if cfg.get("checker"):
        rc.checker_board_offset, rc.checker_area_height = 1, 18
    return rc


def check_frames(vrt, scene, nodes, cam, cfg, textures, palette=None, types=None, spps=(1, 4, 16), label="", lit=True):
    """Renders spps (K4 below 8 samples, K6 at 16) and compares each frame with vo_render_cell_types.  Returns (primary rays,
    camera rays) of the oracle per frame: the primary rays count the reflected ones too."""
    types = cts.mirror_types() if types is None else types
    use_samples = cfg.get("use_samples", True)
    primaries = []
    for spp in (spps if use_samples else (1,)):
        rc = ray_caster(vrt, scene, cfg)
        prev = np.zeros((H, W, 4), np.uint8)
        for frame in range(1 if use_samples else 2):
            img = rc.render(cam, spp).copy()
            p = cts.port_params(vrt, cam, W, H, use_gi=cfg.get("use_gi", True), bounces=cfg.get("bounces", 2), use_samples=use_samples,
                                spp=spp, offset=frame, roughness=cfg.get("roughness", 0.0), max_bounds=cfg.get("max_bounds", 4),
                                mirror_y1=cfg.get("mirror_y", -1) + 1)
            if cfg.get("checker"):
                p.checker, p.checker_area_height = 2, 18
            accum, rgba, st = render_cell_types(nodes, p, palette, types, *textures, prev_rgba=prev)
            where = "%s spp %d frame %d" % (label, spp, frame)
            if use_samples:
                assert np.array_equal(rc.colors, accum), "%s: accumulators differ on %d pixels" % (where, int((rc.colors != accum).any(-1).sum()))
                done = accum[..., 3] > 0
                assert np.array_equal(img[done], rgba[done]), where
            else:
                assert np.array_equal(img, rgba), where
                prev = rgba
            assert rc.last_stats["rays"] == list(st.rays), where
            if cfg.get("product"):
                assert all(x <= y for x, y in zip(rc.last_stats["complexity"], st.complexity)), where
            else:
                assert rc.last_stats["complexity"] == list(st.complexity), where
            assert rgba[..., :3].max() > 0 or not lit, where
            primaries.append((st.rays[0], int(accum[..., 3].sum()) if use_samples else W * H))   # (primary rays, camera rays)
    return primaries


CONFIGS = {
    "gi2":       dict(bounces=2),
    "gi1_rough": dict(bounces=1, roughness=0.3),
    "dof":       dict(bounces=2, aperture=2.0, focal_length=20.0, roughness=0.3),
    "palette":   dict(bounces=2, palette=True),
    "lake":      dict(bounces=1, mirror_y=cts.FLOOR_Y, palette=True),
    "checker":   dict(bounces=1, checker=True),
    "autofocus": dict(bounces=2, autofocus=True),
    "blend":     dict(bounces=1, use_samples=False),
    "defaults":  dict(bounces=2, product=True, roughness=0.3),
}


def camera(vrt, pos, angle, cfg):
    return vrt.Camera(position=pos, view_angle=angle, aperture=cfg.get("aperture", 0.5), focal_length=cfg.get("focal_length", 30.0))


@pytest.mark.parametrize("config", sorted(CONFIGS))
@pytest.mark.parametrize("world", cts.WORLDS)
def test_frames_match_the_oracle(vrt, textures, world, config):
    cfg = CONFIGS[config]
    (xyz, colours), pos, angle = cts.world(world)
    c = vrt.Context(0)
    if cfg.get("product"):
        c.set_option("beam_tile", 8)
        c.set_option("bounds_exit", 1)
    try:
        s, nodes = gpu_scene(vrt, c, xyz, colours, textures)
        pal = cts.make_palette() if cfg.get("palette") else None
        if pal is not None:
            s.set_palette(pal)
        s.set_cell_types(cts.mirror_types())
        cam = camera(vrt, pos, angle, cfg)
        if cfg.get("autofocus"):
            cam.autofocus(s)
        prim = check_frames(vrt, s, nodes, cam, cfg, textures, pal, label="%s/%s" % (world, config))
        assert any(n > base for n, base in prim), "no reflections"
    finally:
        c.close()


@pytest.mark.parametrize("max_bounds", [0, 1, 4, 16])
def test_facing_mirrors_max_bounds(vrt, textures, max_bounds):
    (xyz, colours), pos, angle = cts.world("facing")
    c = vrt.Context(0)
    try:
        s, nodes = gpu_scene(vrt, c, xyz, colours, textures)
        s.set_cell_types(cts.mirror_types())
        cfg = dict(bounces=2, max_bounds=max_bounds, roughness=0.05)
        prim = check_frames(vrt, s, nodes, camera(vrt, pos, angle, cfg), cfg, textures)
        for n, base in prim:
            assert (n == base) if max_bounds == 0 else (base < n <= base * (max_bounds + 1))
    finally:
        c.close()


def test_edge_and_zero_normal_hits(vrt, port, textures):
    c = vrt.Context(0)
    try:
        for make, faces_wanted in ((cts.edge_world, 2), (cts.inside_world, 0)):
            (xyz, colours), pos, angle = make()
            s, nodes = gpu_scene(vrt, c, xyz, colours, textures)
            s.set_cell_types(cts.mirror_types())
            cfg = dict(bounces=2, aperture=0.0, max_bounds=4)
            cam = camera(vrt, pos, angle, cfg)
            # the hits are there: a cast of the camera rays on the device, equal to the oracle's walk
            o, d = cts.camera_rays(port, cts.port_params(vrt, cam, W, H))
            got = s.cast_rays(o, d)
            want = port.lsvo_cast(nodes, cts.DEPTH, o, d)
            hit = (got["flags"] & 1) != 0
            assert np.array_equal(hit, want["hit"] != 0)
            assert np.array_equal(got["normal"][hit], want["normal"][hit])
            faces = (want["normal"] != 0).sum(1)
            mirror = np.isin(cts.hit_colours(nodes, want), cts.MIRROR_COLOURS)
            assert (mirror & hit & (faces == faces_wanted)).sum() > 10, make.__name__
            for spp in (1, 4, 16):
                check_frames(vrt, s, nodes, cam, cfg, textures, spps=(spp,), label=make.__name__, lit=make is cts.edge_world)
            s.close()
    finally:
        c.close()


@pytest.mark.parametrize("product", [False, True])
def test_slab_equals_the_lake(vrt, textures, product):
    (xyz, colours), pos, angle = cts.slab_world(layer_y=40)
    c = vrt.Context(0)
    if product:
        c.set_option("beam_tile", 8)
        c.set_option("bounds_exit", 1)
    try:
        s, nodes = gpu_scene(vrt, c, xyz, colours, textures)
        cfg = dict(bounces=2, roughness=0.3, product=product)
        cam = camera(vrt, pos, angle, cfg)
        for spp in (2, 16):
            out = []
            for table in (True, False):
                s.set_cell_types(cts.mirror_types((9,)) if table else None)
                rc = ray_caster(vrt, s, dict(cfg, mirror_y=None if table else 40))
                out.append((rc.render(cam, spp).copy(), rc.colors.copy(), rc.last_stats))
            assert np.array_equal(out[0][0], out[1][0]) and np.array_equal(out[0][1], out[1][1]), spp
            assert out[0][2] == out[1][2], spp
            assert out[0][2]["rays"][0] > W * H * spp
        s.set_cell_types(cts.mirror_types((9,)))
        check_frames(vrt, s, nodes, cam, cfg, textures, types=cts.mirror_types((9,)), spps=(4, 16))
    finally:
        c.close()


def test_heightfield_colour_one(vrt, textures):
    heights = np.full((64, 64), 10, np.int32)
    heights[20:30, 20:44] = 30
    c = vrt.Context(0)
    try:
        s = vrt.LSVO.from_heightfield(c, cts.DEPTH, heights)
        s.set_textures(*textures)
        nodes = s.download_nodes()
        types = cts.mirror_types((1,))
        s.set_cell_types(types)
        cfg = dict(bounces=2, roughness=0.05)
        cam = camera(vrt, (32.0, 8.0, 2.0), (0.2, -0.6), cfg)
        # every hit reflects until max_bounds binds, and the reflected rays mostly leave the world: a dark frame
        prim = check_frames(vrt, s, nodes, cam, cfg, textures, types=types, spps=(1, 16), lit=False)
        assert all(n > base for n, base in prim)
    finally:
        c.close()


@pytest.mark.parametrize("types1", [1, 2])
def test_mirrors_survive_set_cells(vrt, textures, types1):
    (xyz, colours), pos, angle = cts.world("cube")
    types = cts.mirror_types()
    types[1] = types1
    c = vrt.Context(0)
    try:
        s, _ = gpu_scene(vrt, c, xyz, colours, textures)
        s.set_cell_types(types)
        colour = {tuple(v): int(k) for v, k in zip(xyz.tolist(), colours)}
        removed = cts.to_set_cell(cts.box(28, 34, 42, 48, 30, 36))               # a corner bite out of the mirror cube
        s.set_cells(removed, solid=False)
        for v in removed.tolist():
            colour.pop(tuple(v))
        added = cts.to_set_cell(np.concatenate([cts.box(12, 18, 40, 56, 44, 50), cts.box(30, 32, 44, 46, 32, 34)]))
        s.set_cells(added, solid=True)
        for v in added.tolist():
            colour.setdefault(tuple(v), 1)
        final = np.uint32(sorted(colour.keys()))
        fc = np.uint8([colour[tuple(v)] for v in final.tolist()])
        fresh, nodes = gpu_scene(vrt, c, final, fc, textures)
        fresh.set_cell_types(types)
        assert np.array_equal(s.download_nodes().view(np.uint64), nodes.view(np.uint64))
        cfg = dict(bounces=2, roughness=0.05)
        cam = camera(vrt, pos, angle, cfg)
        for spp in (2, 16):
            frames = []
            for sc in (s, fresh):
                rc = ray_caster(vrt, sc, cfg)
                frames.append((rc.render(cam, spp).copy(), rc.colors.copy(), rc.last_stats))
            assert np.array_equal(frames[0][0], frames[1][0]) and np.array_equal(frames[0][1], frames[1][1])
            assert frames[0][2] == frames[1][2]
        check_frames(vrt, s, nodes, cam, cfg, textures, types=types, spps=(4, 16))
    finally:
        c.close()


@pytest.mark.parametrize("layout", [0, 1])
def test_shade_rays_with_mirror_voxels(vrt, port, textures, layout):
    (xyz, colours), pos, angle = cts.world("cube")
    c = vrt.Context(0)
    try:
        s, nodes = gpu_scene(vrt, c, xyz, colours, textures)
        s.set_cell_types(cts.mirror_types())
        if layout:
            s.set_layout(1)
        cam = camera(vrt, pos, angle, dict(aperture=0.5))
        for pal in (None, cts.make_palette()):
            s.set_palette(pal)
            for sample in (0, 3):
                p0 = cts.port_params(vrt, cam, W, H, offset=sample)
                o, d = cts.camera_rays(port, p0)
                jobs = np.zeros(W * H, SHADE_JOB)
                jobs["start"], jobs["direction"] = o, d
                jobs["pixel"] = np.arange(W * H)
                jobs["sample"] = sample
                first = port.lsvo_cast(nodes, cts.DEPTH, o, d)
                for use_gi, bounces, roughness in ((0, 1, 0.0), (1, 2, 0.3)):
                    p = cts.port_params(vrt, cam, W, H, use_gi=use_gi, bounces=bounces, offset=sample, roughness=roughness)
                    accum, _, st = render_cell_types(nodes, p, pal, cts.mirror_types(), *textures)
                    assert st.rays[0] > W * H
                    q = vrt.capi.RenderParams()
                    q.width, q.height, q.spp, q.use_samples = W, H, 1, 1
                    q.seed_lo, q.seed_hi = 0x5EED, 0
                    q.light_position[:] = [float(x) for x in cts.default_light()]
                    q.use_gi, q.gi_bounces, q.roughness, q.max_bounds = use_gi, bounces, roughness, 4
                    out = np.zeros(len(jobs), SHADE_RESULT)
                    vrt.capi.check(vrt.capi.lib().vrt_shade_rays(s.handle, C.byref(q), len(jobs), vrt.capi.ptr(jobs), vrt.capi.ptr(out)))
                    rgb = np.stack([out["r"], out["g"], out["b"]], -1)
                    assert np.array_equal(rgb, accum.reshape(-1, 4)[:, :3]), (layout, sample, use_gi)
                    # distance and complexity are the camera ray's
                    assert np.array_equal(out["complexity"], first["complexity"])
                    h = first["hit"] != 0
                    assert np.array_equal(out["distance"][h], first["distance"][h])
        s.set_palette(None)
    finally:
        c.close()


def test_communicator_frame(vrt, textures):
    capi = vrt.capi
    (xyz, colours), pos, angle = cts.world("wall_x")
    c = vrt.Context(0)
    comm = None
    try:
        s, _ = gpu_scene(vrt, c, xyz, colours, textures)
        s.set_cell_types(cts.mirror_types())
        cam = camera(vrt, pos, angle, dict(aperture=0.5)).as_struct()
        p = capi.RenderParams()
        p.width, p.height, p.row_begin, p.row_end = W, H, 0, H
        p.spp, p.seed_lo, p.seed_hi = 16, 0x5EED, 0
        p.light_position[:] = [float(x) for x in cts.default_light()]
        p.use_gi, p.gi_bounces, p.use_samples, p.max_bounds, p.roughness = 1, 2, 1, 4, 0.3
        want = np.zeros((H, W, 4), np.uint8)
        stats = capi.RenderStats()
        capi.check(capi.lib().vrt_render(s.handle, C.byref(cam), C.byref(p), capi.ptr(want), None, C.byref(stats)))
        assert stats.rays[0] > W * H * 16
        ctxs = (C.c_void_p * 1)(c.handle.value)
        out = (C.c_void_p * 1)()
        capi.check(capi.lib().vrt_comm_create_local(ctxs, 1, W, H, out))
        comm = C.c_void_p(out[0])
        for split in (capi.SPLIT_TILES, capi.SPLIT_SAMPLES):
            host = np.zeros((H, W, 4), np.uint8)
            capi.check(capi.lib().vrt_render_distributed(comm, s.handle, C.byref(cam), C.byref(p), split, 0, capi.ptr(host)))
            capi.check(capi.lib().vrt_comm_frame_wait(comm))
            assert np.array_equal(host, want), split
    finally:
        if comm is not None:
            capi.lib().vrt_comm_destroy(comm)
        c.close()


def test_refusals(vrt, textures):
    lib, capi = vrt.capi.lib(), vrt.capi
    (xyz, colours), pos, angle = cts.world("wall_x")
    c = vrt.Context(0)
    try:
        s, _ = gpu_scene(vrt, c, xyz, colours, textures)
        for bad in (0, 3):
            t = cts.mirror_types()
            t[5] = bad
            assert lib.vrt_scene_set_cell_types(s.handle, capi.ptr(t)) == INVALID
            with pytest.raises(ValueError):
                s.set_cell_types(t)
        assert lib.vrt_scene_set_cell_types(None, None) == INVALID
        t = cts.mirror_types()
        grid = vrt.Grid3D(c, np.ones((8, 8, 8), np.uint8))
        svo = vrt.SVO(c, np.ones((8, 8, 8), np.uint8))
        for g in (grid, svo):
            assert lib.vrt_scene_set_cell_types(g.handle, capi.ptr(t)) == UNSUPPORTED
            assert lib.vrt_scene_set_cell_types(g.handle, None) == UNSUPPORTED
            g.close()
        cam = camera(vrt, pos, angle, dict(aperture=0.5)).as_struct()
        rc = ray_caster(vrt, s, dict(bounces=2))
        buf = np.zeros((H, W, 4), np.uint8)
        p = rc.params(1)
        for variant in (1, 3):                                   # the plain frame renders; the one with the table is refused
            c.set_option("render_variant", variant)
            s.set_cell_types(None)
            assert lib.vrt_render(s.handle, C.byref(cam), C.byref(p), capi.ptr(buf), None, None) == 0
            s.set_cell_types(t)
            assert lib.vrt_render(s.handle, C.byref(cam), C.byref(p), capi.ptr(buf), None, None) == UNSUPPORTED
        c.set_option("render_variant", 0)
        s.set_layout(1)
        assert lib.vrt_render(s.handle, C.byref(cam), C.byref(p), capi.ptr(buf), None, None) == UNSUPPORTED
        s.set_layout(0)
        assert lib.vrt_render(s.handle, C.byref(cam), C.byref(p), capi.ptr(buf), None, None) == 0
        p.max_bounds = 17
        assert lib.vrt_render(s.handle, C.byref(cam), C.byref(p), capi.ptr(buf), None, None) == INVALID
        job = np.zeros(1, SHADE_JOB)
        res = np.zeros(1, SHADE_RESULT)
        assert lib.vrt_shade_rays(s.handle, C.byref(p), 1, capi.ptr(job), capi.ptr(res)) == INVALID
        s.set_cell_types(None)                                   # without mirror voxels max_bounds is not read
        assert lib.vrt_render(s.handle, C.byref(cam), C.byref(p), capi.ptr(buf), None, None) == 0
    finally:
        c.close()


def test_clearing_and_all_solid(vrt, textures):
    (xyz, colours), pos, angle = cts.world("cube")
    c = vrt.Context(0)
    try:
        s, _ = gpu_scene(vrt, c, xyz, colours, textures)
        s.set_palette(cts.make_palette())
        cfg = dict(bounces=2, roughness=0.3)
        cam = camera(vrt, pos, angle, cfg)
        out = []
        for types in (None, cts.mirror_types(), None, np.ones(256, np.uint8)):
            s.set_cell_types(types)
            for spp in (2, 16):
                rc = ray_caster(vrt, s, cfg)
                out.append((rc.render(cam, spp).copy(), rc.colors.copy(), rc.last_stats))
        assert not np.array_equal(out[0][1], out[2][1])
        for i in (4, 6):                                         # cleared, all Solid: the frames without a table
            for k in (0, 1):
                assert np.array_equal(out[k][0], out[i + k][0]) and np.array_equal(out[k][1], out[i + k][1])
                assert out[k][2] == out[i + k][2]
    finally:
        c.close()


def test_casts_unchanged(vrt, textures):
    (xyz, colours), _, _ = cts.world("facing")
    rng = np.random.default_rng(0)
    n = 50000
    o = rng.uniform(1, 2, (n, 3)).astype(np.float32)
    d = rng.normal(size=(n, 3)).astype(np.float32)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    c = vrt.Context(0)
    try:
        s, _ = gpu_scene(vrt, c, xyz, colours, textures)
        for variant in range(4):
            c.set_option("cast_variant", variant)
            for coef in (0.0, 0.5):
                s.set_cell_types(None)
                want = s.cast_rays(o, d, coef)
                s.set_cell_types(cts.mirror_types())
                got = s.cast_rays(o, d, coef)
                assert np.array_equal(got.view(np.uint8), want.view(np.uint8)), (variant, coef)
                assert ((want["flags"] & 1) != 0).mean() > 0.1
    finally:
        c.close()


def test_cpp_dropin_cell_types(vrt, textures, tmp_path):
    exe, tex = str(tmp_path / "cell_types_test"), str(tmp_path / "textures.bin")
    lib_dir = os.path.join(ROOT, "cpuvoxelraycaster_b200")
    subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-I" + os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "tests", "cpp", "cell_types_test.cpp"), "-o", exe, "-L" + lib_dir, "-lvrt",
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
        xyz, colours = cts._world([(cts.box(0, 64, 56, 64, 0, 64), 3), (cts.box(50, 53, 18, 56, 6, 58), 9),
                                   (cts.box(20, 25, 30, 56, 30, 35), 4)])
        s = vrt.LSVO(c, vrt.host_build_lsvo_from_voxels(cts.DEPTH, xyz), cts.DEPTH)
        assert out["paint"] == "painted=%d" % s.paint_cells(xyz, colours)
        s.set_cell_types(cts.mirror_types((9,)))
        rc = vrt.RayCaster(s, (96, 54), *textures)
        rc.setLightPosition(cts.default_light())
        rc.use_samples, rc.use_gi, rc.roughness = True, True, 0.3
        cam = vrt.Camera(position=(14.0, 30.0, 8.0), view_angle=(0.9, -0.3), aperture=0.5, focal_length=30.0)

        def fnv(a):
            h = 1469598103934665603
            for b in a.tobytes():
                h = ((h ^ b) * 1099511628211) & 0xFFFFFFFFFFFFFFFF
            return "hash=%016x" % h
        assert out["frame"] == fnv(rc.render(cam, 2))
        assert rc.last_stats["rays"][0] > 96 * 54 * 2
        s.set_cell_types(None)
        rc.resetSamples()
        assert out["cleared"] == fnv(rc.render(cam, 2))
        assert out["frame"] != out["cleared"]
    finally:
        c.close()
