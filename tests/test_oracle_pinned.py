"""Pins the CPU restatement (oracle/port.c) against the reference's OWN compiled sources (oracle/_ref, built by
oracle/Makefile from the checkout $VRT_REFERENCE names).  Skipped where oracle/_ref has not been built.  Bit-exact, except the
stochastic frame, which the reference cannot reproduce even against itself (racy global RNG): PSNR there."""
import numpy as np
import pytest

from conftest import assert_hits_equal


def rays(rng, n, lo, hi):
    o = rng.uniform(lo, hi, (n, 3)).astype(np.float32)
    d = rng.normal(size=(n, 3)).astype(np.float32)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    return o, d.astype(np.float32)


def test_noise_and_heights(port, ref):
    rng = np.random.default_rng(0)
    x, y = rng.uniform(-500, 3000, 20000).astype(np.float32), rng.uniform(-500, 3000, 20000).astype(np.float32)
    got = np.array([port.lib.vo_noise2d(float(a), float(b)) for a, b in zip(x[:2000], y[:2000])], np.float32)
    assert np.array_equal(got.view(np.uint32), ref.noise2d(x[:2000], y[:2000]).view(np.uint32))
    assert np.array_equal(port.terrain_heights(512), ref.terrain_heights(512))


@pytest.mark.parametrize("depth", [1, 2, 4, 6])
def test_flattening_and_cast_random_scenes(port, ref, depth):
    rng = np.random.default_rng(depth)
    S = 1 << depth
    occ = (rng.random((S, S, S)) < 0.2).astype(np.uint8)
    xyz = np.argwhere(occ).astype(np.uint32)
    rng.shuffle(xyz)
    sc = ref.scene_from_voxels(depth, xyz)
    rn = ref.nodes(sc)
    rn["pad"] = 0
    pn = port.build_dense(depth, occ)
    assert np.array_equal(pn.view(np.uint64), rn.view(np.uint64))
    o, d = rays(rng, 20000, 0.7, 2.3)
    d[:200, rng.integers(0, 3)] = 0.0
    for coef, bias in ((0.0, 0.0), (0.5, 0.0), (0.1, 0.01)):
        want = ref.lsvo_cast(sc, o, d, coef, bias)
        got = port.lsvo_cast(pn, depth, o, d, coef, bias)
        assert_hits_equal(got, want, got["hit"] != 0, "depth %d coef %g" % (depth, coef))
    ref.scene_destroy(sc)


def test_terrain_scene_and_cast(port, ref):
    sc = ref.scene_terrain(9)
    rn = ref.nodes(sc)
    rn["pad"] = 0
    pn = port.build_terrain(9)
    assert np.array_equal(pn.view(np.uint64), rn.view(np.uint64))
    o, d = rays(np.random.default_rng(2), 100000, (1, 1, 1), (2, 1.45, 2))
    want = ref.lsvo_cast(sc, o, d, 0.0, 0.0, threads=4)
    got = port.lsvo_cast(pn, 9, o, d, threads=4)
    assert_hits_equal(got, want, got["hit"] != 0, "terrain")
    ref.scene_destroy(sc)


def test_depth12_guard_quirk(port, ref):
    """lsvo.hpp:72 `scale > MAX_DEPTH`: at depth 12 the walk stops one level above the leaves, every ray misses;
    the port reproduces it with guard = depth and reaches the leaves with the guard lifted."""
    occ = np.zeros((16, 16, 16), np.uint8)            # a depth-4 pattern reused at depth 12 through a voxel list
    xyz = np.array([[4095, 0, 0], [100, 2000, 300], [2048, 2048, 2048]], np.uint32)
    sc = ref.scene_from_voxels(12, xyz)
    rn = ref.nodes(sc)
    rn["pad"] = 0
    o = np.float32([[1 + (4095 - 100 + 0.5) / 4096, 1 + (4095 - 2000 + 0.5) / 4096, 1.0]])
    d = np.float32([[0, 0, 1]])
    want = ref.lsvo_cast(sc, o, d)
    assert want["hit"][0] == 0
    got = port.lsvo_cast(rn, 12, o, d, guard=12)
    assert_hits_equal(got, want, got["hit"] != 0, "guard 12")
    lifted = port.lsvo_cast(rn, 12, o, d, guard=0)
    assert lifted["hit"][0] == 1 and list(lifted["voxel"][0]) == [4095 - 100, 4095 - 2000, 4095 - 300]
    ref.scene_destroy(sc)


def test_grid_and_svo(port, ref_patched):
    rng = np.random.default_rng(4)
    occ = (rng.random((64, 64, 64)) < 0.02).astype(np.uint8)
    occ[:, :2, :] = 1
    o = rng.uniform(-2, 66, (30000, 3)).astype(np.float32)
    d = rng.normal(size=(30000, 3)).astype(np.float32)
    d[:300, 1] = 0.0
    o[:300] = np.floor(o[:300])
    g = ref_patched.grid_create(occ)
    want = ref_patched.grid_cast(g, o, d)
    got, _ = port.grid_cast(occ, o, d)
    assert_hits_equal(got, want, got["hit"] != 0, "grid")
    ref_patched.grid_destroy(g)
    s = ref_patched.svo_create(occ)
    oi = rng.uniform(0, 64, (30000, 3)).astype(np.float32)
    for mi in (1 << 20, 40):
        want = ref_patched.svo_cast(s, oi, d, mi)
        got = port.svo_cast(occ, 6, oi, d, mi)
        assert_hits_equal(got, want, got["hit"] != 0, "svo max_iter %d" % mi)
    ref_patched.svo_destroy(s)


def _ref_params(loader, W, H, view, aperture, use_gi, use_samples, spp, light, focal=60.0):
    p = loader.RefRenderParams()
    p.width, p.height = W, H
    p.cam_position[:] = [256.0, 200.0, 256.0]
    p.view_angle[:] = view
    p.fov, p.aperture, p.focal_length = 1.0, aperture, focal
    p.light_position[:] = [float(x) for x in light]
    p.use_gi, p.use_samples, p.spp, p.threads = use_gi, use_samples, spp, 1
    return p


def _port_params(loader, ref, W, H, view, aperture, use_gi, use_samples, spp, light, focal=60.0):
    p = loader.PortRenderParams()
    p.width, p.height, p.depth, p.guard = W, H, 9, 9
    p.cam_position[:] = [256.0, 200.0, 256.0]
    rot, _ = ref.camera_basis(np.float32(view))
    p.rot_mat[:] = [float(x) for x in rot]
    p.fov, p.aperture, p.focal_length = 1.0, aperture, focal
    p.light_position[:] = [float(x) for x in light]
    p.use_gi, p.gi_bounces, p.use_samples, p.spp = use_gi, 1, use_samples, spp
    p.seed_lo, p.threads = 0x5EED, 8
    return p


def test_raycaster_deterministic_frame_and_camera(port, ref, textures):
    from oracle import loader
    ref.register_textures(*textures)
    light = np.float32([-200, -1000, -300]) * np.float32(1 / 512.0) + np.float32(1)
    sc = ref.scene_terrain(9)
    nodes = port.build_terrain(9)
    W, H, view = 128, 72, [0.7, -0.4]
    want = ref.render(sc, _ref_params(loader, W, H, view, 0.0, 0, 1, 1, light))
    accum, rgba, _ = port.render(nodes, _port_params(loader, ref, W, H, view, 0.0, 0, 1, 1, light), *textures)
    assert np.array_equal(accum, want["samples"].astype(np.uint32)) and np.array_equal(rgba, want["image"])
    # temporal-blend mode (use_samples off): two frames, u8-exact
    pr = _ref_params(loader, W, H, view, 0.0, 0, 0, 2, light)
    want2 = ref.render(sc, pr)
    pp = _port_params(loader, ref, W, H, view, 0.0, 0, 0, 1, light)
    _, f1, _ = port.render(nodes, pp, *textures)
    _, f2, _ = port.render(nodes, pp, *textures, prev_rgba=f1)
    assert np.array_equal(f2, want2["image"])
    # Camera::getRay with aperture 0: rays bit-exact for every pixel
    p0 = _ref_params(loader, W, H, view, 0.0, 0, 1, 1, light)
    ro, rd = ref.camera_rays(p0)
    for (x, y) in ((0, 0), (17, 5), (127, 71), (64, 36)):
        o, d = port.camera_ray(pp, x, y, 0)
        i = y * W + x
        assert np.array_equal(o.view(np.uint32), ro[i].view(np.uint32)) and np.array_equal(d.view(np.uint32), rd[i].view(np.uint32))
    # autofocus rule (main.cpp:115-121)
    pa = _ref_params(loader, W, H, [0.0, -0.6], 0.0, 0, 1, 1, light)
    f = ref.autofocus(sc, pa)
    rot, cv = ref.camera_basis(np.float32([0.0, -0.6]))
    h = port.lsvo_cast(nodes, 9, [np.float32([256, 200, 256]) * np.float32(1 / 512.0) + np.float32(1)], [cv])[0]
    assert h["hit"] and np.float32(f) == np.float32(h["distance"]) * np.float32(512.0)
    ref.scene_destroy(sc)


@pytest.mark.parametrize("W,H,area_height", [(128, 72, 18), (96, 60, 15), (64, 36, 0)])
def test_checkerboard_frames_match_the_reference_loop(port, ref, textures, W, H, area_height):
    """main.cpp:137-143 on the reference's own RayCaster: alternating checkerboard halves with the 0.4/0.6 temporal
    blend (raycaster.hpp:79-85), 4 frames; area heights even, odd (the demo's 135 is odd) and a single area."""
    from oracle import loader
    ref.register_textures(*textures)
    light = np.float32([-200, -1000, -300]) * np.float32(1 / 512.0) + np.float32(1)
    sc = ref.scene_terrain(9)
    nodes = port.build_terrain(9)
    view = [0.7, -0.4]
    pr = _ref_params(loader, W, H, view, 0.0, 0, 0, 1, light)
    pr.checker, pr.checker_area_height, pr.frames = 2, area_height, 4       # main.cpp:98,137: the first frame has offset 1
    want = ref.render(sc, pr)["image"]
    pp = _port_params(loader, ref, W, H, view, 0.0, 0, 0, 1, light)
    pp.checker_area_height = area_height
    img = None
    for frame in range(4):
        pp.checker = 1 + ((1 + frame) & 1)
        _, img, _ = port.render(nodes, pp, *textures, prev_rgba=img)
    assert np.array_equal(img, want)
    # sample mode: each half accumulates its own pixels
    pr = _ref_params(loader, W, H, view, 0.0, 0, 1, 1, light)
    pr.checker, pr.checker_area_height, pr.frames = 1, area_height, 2
    want = ref.render(sc, pr)
    pp = _port_params(loader, ref, W, H, view, 0.0, 0, 1, 1, light)
    pp.checker_area_height = area_height
    acc = np.zeros((H, W, 4), np.uint32)
    for frame in range(2):
        pp.checker = 1 + (frame & 1)
        a, _, _ = port.render(nodes, pp, *textures)
        acc += a
    assert np.array_equal(acc, want["samples"].astype(np.uint32)) and (acc[..., 3] == 1).all()
    ref.scene_destroy(sc)


def test_present_restatement(port):
    """vo_present against an independent numpy statement of main.cpp:159-177 (median_3.frag / median.frag windows)."""
    rng = np.random.default_rng(5)
    H, W = 37, 53
    frame = rng.integers(0, 256, (H, W, 4), dtype=np.uint8)
    display = rng.integers(0, 256, (H, W, 4), dtype=np.uint8)
    for median in (0, 3, 5):
        for ovc in (0.1, 0.0, 0.5, 1.0):
            got = port.present(frame, display, median, ovc)
            r = median // 2
            pad = np.pad(frame[..., :3], ((r, r), (r, r), (0, 0)), mode="edge")
            win = np.stack([pad[dy:dy + H, dx:dx + W] for dy in range(2 * r + 1) for dx in range(2 * r + 1)], 0)
            f = np.sort(win, axis=0)[win.shape[0] // 2].astype(np.uint32)
            c1, c2 = int(np.float32(255) * np.float32(ovc)), int(np.float32(255) * (np.float32(1.0) - np.float32(ovc)))
            want = np.minimum(255, (display[..., :3].astype(np.uint32) * c1 + 127) // 255 + (f * c2 + 127) // 255)
            assert np.array_equal(got[..., :3], want.astype(np.uint8)), (median, ovc)
            assert (got[..., 3] == 255).all()


def psnr(a, b):
    mse = np.mean((a.astype(np.float64) - b.astype(np.float64)) ** 2)
    return 99.0 if mse == 0 else 10 * np.log10(255.0 ** 2 / mse)


def test_stochastic_frame_distribution(port, ref, textures):
    """GI + DOF at matched spp: the port (Philox lattice) against the reference's RayCaster (global xorshf96).
    Same estimator, different random numbers → compare images statistically.  Threshold: the port-vs-reference
    PSNR must be no worse than 1.5 dB below the reference-vs-reference PSNR of two different RNG offsets."""
    from oracle import loader
    ref.register_textures(*textures)
    light = np.float32([-200, -1000, -300]) * np.float32(1 / 512.0) + np.float32(1)
    sc = ref.scene_terrain(9)
    nodes = port.build_terrain(9)
    W, H, view, spp = 96, 54, [0.3, -0.35], 64
    r1 = ref.render(sc, _ref_params(loader, W, H, view, 0.5, 1, 1, spp, light))["image"][..., :3]
    ref.getrand(12345)                                   # advance the global RNG: an independent second run
    r2 = ref.render(sc, _ref_params(loader, W, H, view, 0.5, 1, 1, spp, light))["image"][..., :3]
    _, p1, _ = port.render(nodes, _port_params(loader, ref, W, H, view, 0.5, 1, 1, spp, light), *textures)
    p1 = p1[..., :3]
    rr, pr = psnr(r1, r2), psnr(p1, r1)
    assert pr >= rr - 1.5, "port vs reference %.2f dB, reference vs reference %.2f dB" % (pr, rr)
    assert abs(p1.mean() - r1.mean()) < 1.0              # no brightness bias
    ref.scene_destroy(sc)


def test_lattice_rng_matches_getrand_distribution(port, ref):
    g = ref.getrand(200000)
    levels = np.round((g + 0.5) * 100).astype(int)
    assert levels.min() == 0 and levels.max() == 99 and len(np.unique(levels)) == 100
    assert np.allclose(np.unique((g + 0.5) * 100 - levels), 0, atol=1e-4)     # 100-point lattice
    counts = np.bincount(levels, minlength=100)
    assert counts.min() > 1600 and counts.max() < 2400


# ---- the benchmark depth: oracle/port.c against the reference's RayCaster rebuilt at depth 11 (oracle/_ref/libvrt_ref_d11.so) ----
def _c11_params(loader, R, W, H, view, aperture, use_gi, spp, light, focal, threads=8):
    S = 2048.0
    pr = loader.RefRenderParams()
    pr.width, pr.height = W, H
    pr.cam_position[:] = [S / 2, S / 2 - 56.0, S / 2]
    pr.view_angle[:] = view
    pr.fov, pr.aperture, pr.focal_length = 1.0, aperture, focal
    pr.light_position[:] = [float(x) for x in light]
    pr.use_gi, pr.use_samples, pr.spp, pr.threads = use_gi, 1, spp, threads
    pp = loader.PortRenderParams()
    pp.width, pp.height, pp.depth, pp.guard = W, H, 11, 11
    pp.cam_position[:] = [S / 2, S / 2 - 56.0, S / 2]
    rot, _ = R.camera_basis(np.float32(view))
    pp.rot_mat[:] = [float(x) for x in rot]
    pp.fov, pp.aperture, pp.focal_length = 1.0, aperture, focal
    pp.light_position[:] = [float(x) for x in light]
    pp.use_gi, pp.gi_bounces, pp.use_samples, pp.spp = use_gi, 1, 1, spp
    pp.seed_lo, pp.threads = 0x5EED, threads
    return pr, pp


def test_depth11_raycaster_matches_the_reference_build(port, textures):
    """The depth-dependent constants of the shading path (SCALE = 1/2^D, n_norm, the 512s of camera_controller.hpp:36,58
    and raycaster.hpp:171) at the BENCHMARK depth: deterministic frames u8- and accumulator-exact, the autofocus rule
    exact, and the 1-bounce GI + DOF frame within the reference's own run-to-run PSNR."""
    from oracle import loader
    R = loader.ref_depth(11)
    if R is None:
        pytest.skip("oracle/_ref/libvrt_ref_d11.so not built")
    assert R.depth == 11
    R.register_textures(*textures)
    light = np.float32([-200, -1000, -300]) * np.float32(1 / 2048.0) + np.float32(1)
    nodes = port.build_terrain(11)
    sc = R.scene_from_nodes(11, nodes)
    for (W, H, view) in ((160, 90, [0.0, 0.0]), (128, 72, [0.7, -0.4])):
        pr, pp = _c11_params(loader, R, W, H, view, 0.0, 0, 1, light, 100.0)
        want = R.render(sc, pr)
        accum, rgba, _ = port.render(nodes, pp, *textures)
        assert np.array_equal(accum, want["samples"].astype(np.uint32)) and np.array_equal(rgba, want["image"])
        assert 0.2 < (accum[..., :3].sum(-1) > 0).mean() < 0.99         # lit terrain, and sky or shadow
    # main.cpp:115-121 at depth 11
    pr, pp = _c11_params(loader, R, 160, 90, [0.0, 0.0], 0.5, 0, 1, light, 100.0)
    f = R.autofocus(sc, pr)
    _, cv = R.camera_basis(np.float32([0.0, 0.0]))
    h = port.lsvo_cast(nodes, 11, [np.float32([1024, 968, 1024]) * np.float32(1 / 2048.0) + np.float32(1)], [cv])[0]
    assert h["hit"] and np.float32(f) == np.float32(h["distance"]) * np.float32(2048.0)
    # stochastic: GI (one bounce, the reference's) + DOF, 64 spp
    W, H, view, spp = 96, 54, [0.0, 0.0], 64
    pr, pp = _c11_params(loader, R, W, H, view, 0.5, 1, spp, light, f)
    r1 = R.render(sc, pr)["image"][..., :3]
    R.getrand(12345)
    r2 = R.render(sc, pr)["image"][..., :3]
    _, p1, _ = port.render(nodes, pp, *textures)
    rr, pq = psnr(r1, r2), psnr(p1[..., :3], r1)
    assert pq >= rr - 1.5, "port vs reference %.2f dB, reference vs reference %.2f dB" % (pq, rr)
    assert abs(float(p1[..., :3].mean()) - float(r1.mean())) < 1.0
    R.scene_destroy(sc)


def test_cfg1_full_frame_known_answers(port, textures):
    """BASELINE configs[0] at its full size against the values frozen from the reference's own RayCaster / Camera /
    LSVO<9>::castRay (tests/golden/cfg1_full.json, made by make_golden.py): 468 025 primary hits, frame and hit hashes."""
    import hashlib
    import json
    import os
    from conftest import GOLDEN
    from oracle import loader
    g = json.load(open(os.path.join(GOLDEN, "cfg1_full.json")))
    assert g["primary_hits"] == 468025
    import cpuvoxelraycaster_b200 as vrt
    cam = vrt.Camera(position=g["cam_position"], view_angle=g["view_angle"], focal_length=g["focal_length"])   # host code only
    nodes = port.build_terrain(9)
    pp = loader.PortRenderParams()
    pp.width, pp.height, pp.depth, pp.guard = g["width"], g["height"], 9, 9
    pp.cam_position[:] = g["cam_position"]
    pp.rot_mat[:] = [float(x) for x in cam.rot_mat]
    pp.fov, pp.aperture, pp.focal_length = 1.0, 0.0, g["focal_length"]
    pp.light_position[:] = g["light"]
    pp.use_gi, pp.gi_bounces, pp.use_samples, pp.spp, pp.seed_lo, pp.threads = 0, 1, 1, 1, 0x5EED, 8
    accum, rgba, st = port.render(nodes, pp, *textures)
    assert hashlib.sha256(rgba.tobytes()).hexdigest() == g["sha256_image"]
    assert hashlib.sha256(accum.tobytes()).hexdigest() == g["sha256_samples_u32"]
    assert st.rays[0] == g["width"] * g["height"] and st.rays[1] == g["primary_hits"] and st.complexity[0] == g["sum_complexity"]
