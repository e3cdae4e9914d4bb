r"""Point lights (DESIGN.md §2, "Point lights"): vrt_scene_set_point_lights gives an LSVO scene up to 16 coloured, shadowed point
lights that light the final camera-chain hit after the sun.  Frames are compared with tests/point_lights_oracle.c
vo_render_point_lights: accumulators, 8-bit image, rays per class, and loop trips (equal with the shortcuts off, at most the
specification's with beam floors and bounds exits on).

| test                                  | what it pins                                                                          |
|---------------------------------------|---------------------------------------------------------------------------------------|
| test_frames_match_the_oracle          | K4 (spp 1, 4) and K6 (spp 16) with 1, 4 and 16 lights (some culled, some shadowed): GI 0 / 1 / 2, DOF, palette, cell types + lake, checkerboard, autofocus, temporal blend, product defaults |
| test_night_floor_known_answer         | the wall and overhang worlds lit by one light each: the floor is what light_terms computes |
| test_heightfield_before_and_after_edit | a heightfield before and after edit_heights                                          |
| test_voxel_set_after_set_cells        | a voxel set after set_cells                                                           |
| test_shade_rays_with_point_lights     | vrt_shade_rays against the 1-sample specification, reference and compact layout       |
| test_communicator_frame               | a world-1 vrt_comm_create_local frame equals the vrt_render frame                     |
| test_refusals                         | every argument check of vrt_scene_set_point_lights and LSVO.set_point_lights; compact layout and render_variant 1 / 3 |
| test_clearing_restores_the_unlit_frame | clearing the lights (None or n = 0) gives the frame without them byte for byte       |
| test_cpp_dropin_point_lights          | tests/cpp/point_lights_test.cpp: setPointLights / clearPointLights through render() and the queued renderRay path |

Contexts are created without beam floors and bounds exits (tests/conftest.py); the product-default rows turn them back on.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import cell_types_scenes as cts
import point_lights_scenes as pls
from conftest import ROOT, golden
from point_lights_oracle import LIGHT_DTYPE, render_point_lights

pytestmark = pytest.mark.gpu

INVALID, UNSUPPORTED = -1, -4
W, H = 52, 30
SHADE_JOB = np.dtype([("start", "f4", 3), ("pixel", "u4"), ("direction", "f4", 3), ("sample", "u4")])
SHADE_RESULT = np.dtype([("r", "u1"), ("g", "u1"), ("b", "u1"), ("hit", "u1"), ("distance", "f4"), ("complexity", "u4"),
                         ("reserved", "u4")])


def set_lights(scene, lts):
    if lts is None:
        scene.set_point_lights(None)
    else:
        scene.set_point_lights(lts["position"], lts["color"], lts["range"])


def gpu_scene(vrt, c, xyz, colours, textures):
    s = vrt.LSVO.from_voxels(c, cts.DEPTH, xyz, on_device=True, colors=colours)
    nodes = cts.host_nodes(vrt, xyz, colours)
    assert np.array_equal(s.download_nodes().view(np.uint64), nodes.view(np.uint64))
    s.set_textures(*textures)
    return s, nodes


def ray_caster(vrt, scene, cfg):
    rc = vrt.RayCaster(scene, (W, H))
    rc.setLightPosition(cfg.get("sun", cts.default_light()))
    rc.use_samples = cfg.get("use_samples", True)
    rc.use_gi, rc.gi_bounces = cfg.get("use_gi", True), cfg.get("bounces", 2)
    rc.roughness, rc.max_bounds = cfg.get("roughness", 0.0), cfg.get("max_bounds", 4)
    rc.mirror_y = cfg.get("mirror_y")
    rc.autofocus = bool(cfg.get("autofocus"))
    if cfg.get("checker"):
        rc.checker_board_offset, rc.checker_area_height = 1, 18
    return rc


def check_frames(vrt, scene, nodes, cam, cfg, textures, lts, palette=None, types=None, spps=(1, 4, 16), label=""):
    """Renders spps (K4 below 8 samples, K6 at 16) and compares each frame with vo_render_point_lights.  The first frame must
    cast more shadow rays than the same frame without the lights."""
    use_samples = cfg.get("use_samples", True)
    first = True
    for spp in (spps if use_samples else (1,)):
        rc = ray_caster(vrt, scene, cfg)
        prev = np.zeros((H, W, 4), np.uint8)
        for frame in range(1 if use_samples else 2):
            img = rc.render(cam, spp).copy()
            p = cts.port_params(vrt, cam, W, H, use_gi=cfg.get("use_gi", True), bounces=cfg.get("bounces", 2),
                                use_samples=use_samples, spp=spp, offset=frame, roughness=cfg.get("roughness", 0.0),
                                max_bounds=cfg.get("max_bounds", 4), mirror_y1=cfg.get("mirror_y", -1) + 1)
            p.light_position[:] = [float(x) for x in cfg.get("sun", cts.default_light())]
            if cfg.get("checker"):
                p.checker, p.checker_area_height = 2, 18
            accum, rgba, st = render_point_lights(nodes, p, palette, types, lts, *textures, prev_rgba=prev)
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
            assert rgba[..., :3].max() > 0, where
            if first:
                assert st.rays[1] > render_point_lights(nodes, p, palette, types, None, *textures)[2].rays[1], where
                first = False


CONFIGS = {
    "gi0":       dict(use_gi=False),
    "gi1":       dict(bounces=1),
    "gi2_dof":   dict(bounces=2, aperture=2.0, focal_length=20.0),
    "palette":   dict(bounces=2, palette=True),
    "types_lake": dict(bounces=1, mirror_y=cts.FLOOR_Y, types=True, roughness=0.3),
    "checker":   dict(bounces=1, checker=True, spps=(1, 4)),
    "autofocus": dict(bounces=2, autofocus=True, spps=(1, 4)),
    "blend":     dict(bounces=1, use_samples=False),
    "defaults":  dict(bounces=2, product=True),
    "night":     dict(use_gi=False, sun=pls.NIGHT_SUN),
}


def camera(vrt, pos, angle, cfg):
    return vrt.Camera(position=pos, view_angle=angle, aperture=cfg.get("aperture", 0.5), focal_length=cfg.get("focal_length", 30.0))


def product_context(vrt, on):
    c = vrt.Context(0)
    if on:
        c.set_option("beam_tile", 8)
        c.set_option("bounds_exit", 1)
    return c


@pytest.mark.parametrize("config", sorted(CONFIGS))
@pytest.mark.parametrize("n", [1, 4, 16])
def test_frames_match_the_oracle(vrt, textures, n, config):
    cfg = CONFIGS[config]
    (xyz, colours), pos, angle = pls.world("room")
    c = product_context(vrt, cfg.get("product"))
    try:
        s, nodes = gpu_scene(vrt, c, xyz, colours, textures)
        pal = cts.make_palette() if cfg.get("palette") or cfg.get("types") else None
        types = cts.mirror_types((4,)) if cfg.get("types") else None
        s.set_palette(pal)
        s.set_cell_types(types)
        lts = pls.room_lights(n)
        set_lights(s, lts)
        cam = camera(vrt, pos, angle, cfg)
        if cfg.get("autofocus"):
            cam.autofocus(s)
        check_frames(vrt, s, nodes, cam, cfg, textures, lts, pal, types, spps=cfg.get("spps", (1, 4, 16)), label="%d lights/%s" % (n, config))
    finally:
        c.close()


@pytest.mark.parametrize("product", [False, True])
def test_night_floor_known_answer(vrt, port, textures, product):
    c = product_context(vrt, product)
    try:
        for name, lts in (("wall", pls.lights([[20.5, 44.5, 32.5]], [[1.0, 0.6, 0.3]], [np.inf])),
                          ("overhang", pls.lights([[32.5, 28.5, 20.5]], [[0.8, 0.8, 1.2]], [np.inf]))):
            (xyz, colours), pos, angle = pls.world(name)
            s, nodes = gpu_scene(vrt, c, xyz, colours, textures)
            pal = cts.make_palette()
            s.set_palette(pal)
            set_lights(s, lts)
            cfg = dict(use_gi=False, sun=pls.NIGHT_SUN, aperture=0.0, focal_length=60.0, product=product)
            cam = camera(vrt, pos, angle, cfg)
            check_frames(vrt, s, nodes, cam, cfg, textures, lts, pal, spps=(1, 16), label=name)
            rc = ray_caster(vrt, s, cfg)
            img = rc.render(cam, 1).copy()
            p = cts.port_params(vrt, cam, W, H, use_gi=False)
            p.light_position[:] = [float(x) for x in pls.NIGHT_SUN]
            h, terms = pls.light_terms(port, nodes, p, lts)
            top = (h["hit"] != 0) & (h["normal"][:, 1] != 0) & (h["voxel"][:, 1] == 56)
            want = pls.predicted_rgb(pal[np.maximum(cts.hit_colours(nodes, h), 0)], terms)
            assert top.sum() > 300 and np.array_equal(img[..., :3].reshape(-1, 3)[top], want[top]), name
            s.close()
    finally:
        c.close()


def test_heightfield_before_and_after_edit(vrt, textures):
    heights = np.full((64, 64), 10, np.int32)
    heights[20:30, 20:44] = 30
    c = vrt.Context(0)
    try:
        s = vrt.LSVO.from_heightfield(c, cts.DEPTH, heights)
        s.set_textures(*textures)
        lts = pls.room_lights(16)
        set_lights(s, lts)
        cfg = dict(bounces=2)
        cam = camera(vrt, (32.0, 8.0, 2.0), (0.2, -0.6), cfg)
        check_frames(vrt, s, s.download_nodes(), cam, cfg, textures, lts, label="heightfield")
        s.edit_heights(8, 30, np.full((20, 12), 24, np.int32))
        check_frames(vrt, s, s.download_nodes(), cam, cfg, textures, lts, label="edited")
    finally:
        c.close()


def test_voxel_set_after_set_cells(vrt, textures):
    (xyz, colours), pos, angle = pls.world("room")
    c = vrt.Context(0)
    try:
        s, _ = gpu_scene(vrt, c, xyz, colours, textures)
        pal = cts.make_palette()
        s.set_palette(pal)
        lts = pls.room_lights(4)
        set_lights(s, lts)
        s.set_cells(cts.to_set_cell(cts.box(30, 32, 20, 56, 20, 44)), solid=False)          # a door through the wall
        s.set_cells(cts.to_set_cell(cts.box(40, 48, 36, 56, 40, 48)), solid=True)           # a block of colour 1
        cfg = dict(bounces=2)
        check_frames(vrt, s, s.download_nodes(), camera(vrt, pos, angle, cfg), cfg, textures, lts, pal, label="set_cells")
    finally:
        c.close()


@pytest.mark.parametrize("layout", [0, 1])
def test_shade_rays_with_point_lights(vrt, port, textures, layout):
    (xyz, colours), pos, angle = pls.world("room")
    c = vrt.Context(0)
    try:
        s, nodes = gpu_scene(vrt, c, xyz, colours, textures)
        lts = pls.room_lights(16)
        set_lights(s, lts)
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
                for use_gi, bounces in ((0, 1), (1, 2)):
                    p = cts.port_params(vrt, cam, W, H, use_gi=use_gi, bounces=bounces, offset=sample)
                    accum, _, st = render_point_lights(nodes, p, pal, None, lts, *textures)
                    q = vrt.capi.RenderParams()
                    q.width, q.height, q.spp, q.use_samples = W, H, 1, 1
                    q.seed_lo, q.seed_hi = 0x5EED, 0
                    q.light_position[:] = [float(x) for x in cts.default_light()]
                    q.use_gi, q.gi_bounces, q.max_bounds = use_gi, bounces, 4
                    out = np.zeros(len(jobs), SHADE_RESULT)
                    vrt.capi.check(vrt.capi.lib().vrt_shade_rays(s.handle, C.byref(q), len(jobs), vrt.capi.ptr(jobs), vrt.capi.ptr(out)))
                    rgb = np.stack([out["r"], out["g"], out["b"]], -1)
                    assert np.array_equal(rgb, accum.reshape(-1, 4)[:, :3]), (layout, sample, use_gi)
                    assert np.array_equal(out["complexity"], first["complexity"])
                    h = first["hit"] != 0
                    assert np.array_equal(out["distance"][h], first["distance"][h])
    finally:
        c.close()


def test_communicator_frame(vrt, textures):
    capi = vrt.capi
    (xyz, colours), pos, angle = pls.world("room")
    c = vrt.Context(0)
    comm = None
    try:
        s, _ = gpu_scene(vrt, c, xyz, colours, textures)
        set_lights(s, pls.room_lights(16))
        cam = camera(vrt, pos, angle, dict(aperture=0.5)).as_struct()
        p = capi.RenderParams()
        p.width, p.height, p.row_begin, p.row_end = W, H, 0, H
        p.spp, p.seed_lo, p.seed_hi = 16, 0x5EED, 0
        p.light_position[:] = [float(x) for x in cts.default_light()]
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
    finally:
        if comm is not None:
            capi.lib().vrt_comm_destroy(comm)
        c.close()


def test_refusals(vrt, textures):
    lib, capi = vrt.capi.lib(), vrt.capi
    (xyz, colours), pos, angle = pls.world("room")
    c = vrt.Context(0)
    try:
        s, _ = gpu_scene(vrt, c, xyz, colours, textures)
        good = pls.room_lights(4)
        set_light = lambda scene, a, n: lib.vrt_scene_set_point_lights(scene, None if a is None else capi.ptr(a), n)   # noqa: E731
        assert set_light(None, good, 4) == INVALID
        assert set_light(s.handle, None, 1) == INVALID
        assert set_light(s.handle, np.concatenate([good] * 5), 17) == INVALID
        for field, k, value in (("position", 1, np.inf), ("position", 2, np.nan), ("color", 0, -0.5), ("color", 1, np.inf),
                                ("color", 2, np.nan), ("range", None, 0.0), ("range", None, -1.0), ("range", None, np.nan)):
            bad = good.copy()
            if k is None:
                bad[field][2] = value
            else:
                bad[field][2, k] = value
            assert set_light(s.handle, bad, 4) == INVALID, (field, value)
            with pytest.raises(ValueError):
                set_lights(s, bad)
        for args in ((np.zeros((2, 3)), np.zeros((3, 3)), np.ones(2)), (np.zeros((2, 3)), np.zeros((2, 3)), np.ones(3)),
                     (np.zeros(3), np.zeros(3), np.ones(1)), (np.zeros((2, 3)), None, None), (np.zeros((17, 3)), np.zeros((17, 3)), np.ones(17))):
            with pytest.raises(ValueError):
                s.set_point_lights(*args)
        grid = vrt.Grid3D(c, np.ones((8, 8, 8), np.uint8))
        svo = vrt.SVO(c, np.ones((8, 8, 8), np.uint8))
        for g in (grid, svo):
            assert set_light(g.handle, good, 4) == UNSUPPORTED
            assert set_light(g.handle, None, 0) == UNSUPPORTED
            g.close()
        inf_range = good.copy()
        inf_range["range"] = np.inf
        assert set_light(s.handle, inf_range, 4) == 0
        cam = camera(vrt, pos, angle, dict(aperture=0.5)).as_struct()
        rc = ray_caster(vrt, s, dict(bounces=2))
        buf = np.zeros((H, W, 4), np.uint8)
        p = rc.params(1)
        for variant in (1, 3):                                   # the plain frame renders; the one with lights is refused
            c.set_option("render_variant", variant)
            s.set_point_lights(None)
            assert lib.vrt_render(s.handle, C.byref(cam), C.byref(p), capi.ptr(buf), None, None) == 0
            set_lights(s, good)
            assert lib.vrt_render(s.handle, C.byref(cam), C.byref(p), capi.ptr(buf), None, None) == UNSUPPORTED
        c.set_option("render_variant", 0)
        s.set_layout(1)
        assert lib.vrt_render(s.handle, C.byref(cam), C.byref(p), capi.ptr(buf), None, None) == UNSUPPORTED
        s.set_point_lights(None)
        assert lib.vrt_render(s.handle, C.byref(cam), C.byref(p), capi.ptr(buf), None, None) == 0
        s.set_layout(0)
    finally:
        c.close()


def test_clearing_restores_the_unlit_frame(vrt, textures):
    (xyz, colours), pos, angle = pls.world("room")
    c = vrt.Context(0)
    try:
        s, _ = gpu_scene(vrt, c, xyz, colours, textures)
        cfg = dict(bounces=2)
        cam = camera(vrt, pos, angle, cfg)
        empty = np.zeros(0, LIGHT_DTYPE)
        out = []
        for step in ("none", "lit", "cleared", "lit", "empty"):
            if step == "lit":
                set_lights(s, pls.room_lights(16))
            elif step == "cleared":
                s.set_point_lights(None)
            elif step == "empty":
                set_lights(s, empty)
            for spp in (2, 16):
                rc = ray_caster(vrt, s, cfg)
                out.append((rc.render(cam, spp).copy(), rc.colors.copy(), rc.last_stats))
        assert not np.array_equal(out[0][1], out[2][1])
        for i in (4, 8):
            for k in (0, 1):
                assert np.array_equal(out[k][0], out[i + k][0]) and np.array_equal(out[k][1], out[i + k][1])
                assert out[k][2] == out[i + k][2]
    finally:
        c.close()


def test_cpp_dropin_point_lights(vrt, textures, tmp_path):
    exe, tex = str(tmp_path / "point_lights_test"), str(tmp_path / "textures.bin")
    lib_dir = os.path.join(ROOT, "cpuvoxelraycaster_b200")
    subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-I" + os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "tests", "cpp", "point_lights_test.cpp"), "-o", exe, "-L" + lib_dir, "-lvrt",
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
        xyz, _ = cts._world([(cts.box(0, 64, 56, 64, 0, 64), 3), (cts.box(30, 32, 20, 56, 0, 64), 4)])
        s = vrt.LSVO(c, vrt.host_build_lsvo_from_voxels(cts.DEPTH, xyz), cts.DEPTH)
        set_lights(s, pls.lights([[20.5, 44.5, 32.5], [44.5, 40.5, 20.5]], [[1.0, 0.6, 0.3], [0.2, 0.4, 1.0]], [np.inf, 20.0 / 64]))
        rc = vrt.RayCaster(s, (96, 54), *textures)
        rc.setLightPosition(cts.default_light())
        rc.use_samples, rc.use_gi = True, True
        cam = vrt.Camera(position=(31.0, 8.0, 4.0), view_angle=(0.0, -0.9), aperture=0.0, focal_length=30.0)

        def fnv(a):
            h = 1469598103934665603
            for b in a.tobytes():
                h = ((h ^ b) * 1099511628211) & 0xFFFFFFFFFFFFFFFF
            return "hash=%016x" % h
        assert out["frame"] == fnv(rc.render(cam, 2))
        lit_shadow = rc.last_stats["rays"][1]
        s.set_point_lights(None)
        rc.resetSamples()
        assert out["cleared"] == fnv(rc.render(cam, 2))
        assert out["frame"] != out["cleared"] and lit_shadow > rc.last_stats["rays"][1]
        assert out["queued"] == out["frame"]
    finally:
        c.close()
