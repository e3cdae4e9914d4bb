"""The CPU restatement (oracle/port.c) against the committed golden vectors, which were produced by the
reference's own compiled sources (tests/golden/make_golden.py).  Bit-exact."""
import hashlib

import numpy as np

from conftest import assert_hits_equal, golden


def test_philox_known_answers(port):
    # Random123 kat_vectors, philox4x32 10 rounds
    assert list(port.philox([0, 0, 0, 0], [0, 0])) == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    assert list(port.philox([0xffffffff] * 4, [0xffffffff] * 2)) == [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]
    assert list(port.philox([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0])) == [
        0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]


def test_terrain_heights_match_fastnoise(port):
    g = golden("terrain_heights.npz")
    assert np.array_equal(port.terrain_heights(256), g["heights8"])
    assert hashlib.sha256(port.terrain_heights(512).tobytes()).hexdigest() == str(g["sha_heights9"])
    assert hashlib.sha256(port.terrain_heights(1024).tobytes()).hexdigest() == str(g["sha_heights10"])


def test_terrain_flattening_matches_compileSVO(port):
    g = golden("terrain_heights.npz")
    nodes = port.build_terrain(9)
    assert len(nodes) == int(g["n_nodes9"]) == 10528393          # SURVEY.md §8c known answer
    assert hashlib.sha256(nodes.tobytes()).hexdigest() == str(g["sha_nodes9"])
    assert int(g["solid_voxels9"]) == 8583552


def test_single_voxel_known_answers(port):
    g = golden("lsvo_kat.npz")
    occ = np.zeros((512, 512, 512), np.uint8)
    occ[100, 200, 300] = 1
    nodes = port.build_dense(9, occ)
    assert len(nodes) == 73                                       # SURVEY.md §8c
    ref_nodes = g["nodes"].copy()
    ref_nodes["pad"] = 0
    assert np.array_equal(nodes.view(np.uint64), ref_nodes.view(np.uint64))
    hits = port.lsvo_cast(nodes, 9, g["origin"], g["dir"])
    assert_hits_equal(hits, g["hits"], hits["hit"] != 0, "kat")
    # point mirroring: setCell(100,200,300) is seen at (411,311,211)
    assert list(hits["voxel"][0]) == [411, 311, 211] and hits["distance"][1] == 0.0
    assert hits["hit"][3] == 0 and hits["hit"][4] == 0           # t > 1 is a miss; un-mirrored column misses


def test_lsvo_terrain_rays(port):
    g = golden("lsvo_terrain9.npz")
    nodes = port.build_terrain(9)
    for key, coef, bias in (("hits_coef0", 0.0, 0.0), ("hits_coef05", 0.5, 0.0), ("hits_bias", 0.25, 0.001)):
        hits = port.lsvo_cast(nodes, 9, g["origin"], g["dir"], coef, bias, threads=4)
        assert_hits_equal(hits, g[key], hits["hit"] != 0, key)
    assert 0.2 < (g["hits_coef0"]["hit"] != 0).mean() < 0.9


def test_lsvo_random_scene(port):
    g = golden("lsvo_random6.npz")
    occ = np.zeros((64, 64, 64), np.uint8)
    v = g["voxels"]
    occ[v[:, 0], v[:, 1], v[:, 2]] = 1
    nodes = port.build_dense(6, occ)
    assert np.array_equal(nodes.view(np.uint64), g["nodes"].view(np.uint64))
    for key, coef in (("hits_coef0", 0.0), ("hits_coef05", 0.5)):
        hits = port.lsvo_cast(nodes, 6, g["origin"], g["dir"], coef, 0.0)
        assert_hits_equal(hits, g[key], hits["hit"] != 0, key)


def _unit(v):
    v = np.asarray(v, np.float32)
    return (v / np.sqrt((v * v).sum(1, keepdims=True, dtype=np.float32))).astype(np.float32)


def test_restructured_walk_equals_the_reference_walk(port):
    """The device loop (csrc/lsvo_step.cuh, Trav2) differs from lsvo.hpp:72-146 in structure, not in arithmetic: unconditional
    stack writes (no `h`), one exit for cone and leaf hits, the hit read off the final state instead of a flag, no loop guard where
    it cannot bind, fmaf(half, tc, c) for the child selection of unit directions, the node fetched when the parent changes.
    port.c restates exactly those changes on the CPU; here every field of every record AND the trip counts must equal the
    reference-shaped walk's — on the T(9) terrain (camera-like, random, surface-skimming cone rays), on a random voxel set with
    binding and lifted guards, and on degenerate rays (axis-parallel, zero components, origins on cell planes, inside solids,
    outside the cube, huge and tiny direction magnitudes, non-finite)."""
    rng = np.random.default_rng(11)
    t9 = port.build_terrain(9)
    g6 = golden("lsvo_random6.npz")
    r6 = g6["nodes"].copy()

    def check(nodes, depth, o, d, coef, guard=None, unit=False, label=""):
        want = port.lsvo_cast(nodes, depth, o, d, coef=coef, guard=guard, threads=4)
        got = port.lsvo_cast_restructured(nodes, depth, o, d, coef=coef, guard=guard, unit=unit, threads=4)
        assert np.array_equal(got.view(np.uint8), want.view(np.uint8)), (label, int((got["complexity"] != want["complexity"]).sum()),
                                                                          int((got["hit"] != want["hit"]).sum()))
        return want

    # camera-like rays over the terrain (unit directions, origin above the ground), coef 0
    n = 200_000
    o = np.float32([256, 200, 256]) / np.float32(512) + np.float32(1) + rng.uniform(-0.002, 0.002, (n, 3)).astype(np.float32)
    d = _unit(np.stack([rng.uniform(-0.8, 0.8, n), rng.uniform(-0.45, 0.45, n), np.ones(n)], 1))
    prim = check(t9, 9, o, d, 0.0, unit=True, label="camera")
    assert 0.2 < prim["hit"].mean() < 0.9
    # secondary rays from the hits: sun-like shadow rays (coef 0) and tangent cone rays (coef 0.5), both from just above the surface
    m = prim["hit"] != 0
    so = (prim["position"][m] + prim["normal"][m] * np.float32(1.0 / 512 * 0.001)).astype(np.float32)
    light = np.float32([-200, -1000, -300]) / np.float32(512) + np.float32(1)
    check(t9, 9, so, _unit(light - so), 0.0, unit=True, label="shadow")
    go = (prim["position"][m] + prim["normal"][m] * np.float32(1.0 / 512 / 64)).astype(np.float32)
    gd = _unit(prim["normal"][m] + rng.uniform(-1000, 1000, (int(m.sum()), 3)).astype(np.float32) * (prim["normal"][m] == 0))
    cone = check(t9, 9, go, gd, 0.5, unit=True, label="gi")
    assert cone["hit"].mean() > 0.3
    # random rays through the cube, un-normalised directions (no fmaf), both coefficients
    o = rng.uniform(0.9, 2.1, (200_000, 3)).astype(np.float32)
    d = (rng.standard_normal((200_000, 3)) * rng.choice([1e-3, 1.0, 50.0], (200_000, 1))).astype(np.float32)
    check(t9, 9, o, d, 0.0, label="random")
    check(t9, 9, o, d, 0.5, label="random cone")
    # the random voxel set at depth 6: reference guard (6), a guard that binds (17 = 23 - 6: the walk stops above the voxels), lifted
    o = rng.uniform(0.95, 2.05, (100_000, 3)).astype(np.float32)
    d = rng.standard_normal((100_000, 3)).astype(np.float32)
    for guard in (None, 17, 18, 21, 22, -1):
        check(r6, 6, o, d, 0.0, guard=guard, label="depth 6 guard %s" % guard)
        check(r6, 6, o, _unit(d), 0.5, guard=guard, unit=True, label="depth 6 cone guard %s" % guard)
    # degenerate rays: origins on cell planes / inside solid voxels / outside, axis-parallel and zero components, extreme magnitudes
    vox = g6["voxels"].astype(np.float32)
    planes = (rng.integers(0, 65, (20_000, 3)) / np.float32(64) + np.float32(1)).astype(np.float32)
    inside = ((vox[rng.integers(0, len(vox), 20_000)] + rng.uniform(0, 1, (20_000, 3)).astype(np.float32)) / np.float32(64) + np.float32(1)).astype(np.float32)
    o = np.concatenate([planes, inside, rng.uniform(-1, 4, (20_000, 3)).astype(np.float32)])
    axis = np.zeros((len(o), 3), np.float32)
    axis[np.arange(len(o)), rng.integers(0, 3, len(o))] = rng.choice([-1.0, 1.0], len(o))
    two = rng.standard_normal((len(o), 3)).astype(np.float32)
    two[np.arange(len(o)), rng.integers(0, 3, len(o))] = 0.0
    for d in (axis, two, (two * np.float32(1e30)).astype(np.float32), (two * np.float32(1e-30)).astype(np.float32)):
        check(r6, 6, o, d, 0.0, label="degenerate")
        check(r6, 6, o, d, 0.5, label="degenerate cone")
    bad = np.float32([[np.nan, 1, 1], [1.5, np.inf, 1.5], [1.5, 1.5, 1.5]])
    check(r6, 6, bad, np.float32([[0, 0, 1], [0, 1, 0], [np.nan, 0, 1]]), 0.0, label="non-finite")


def test_grid_dda(port):
    g = golden("grid_random5.npz")
    hits, steps = port.grid_cast(g["occ"], g["origin"], g["dir"])
    assert_hits_equal(hits, g["hits"], hits["hit"] != 0, "grid")
    assert np.all(steps[hits["hit"] != 0] == hits["complexity"][hits["hit"] != 0])


def test_dilated_pyramid_answers_grid_misses_exactly(port):
    """Groundwork for DESIGN.md §7 (6), on the CPU only: Grid3D::castRay's per-cell recurrence cannot be shortened for a HIT, but a
    MISS can be answered from the pyramid.  A ray whose exact path meets no cube of an OR-pyramid level dilated by two cubes is a
    miss of the reference's fp DDA (its cells stay within one cell per axis of the exact ray's).  Checked here against the oracle's
    DDA on the T(8) terrain grid: never a false "miss" on camera-like rays (half sky), random rays, near-axis rays and extreme
    direction magnitudes, at 4^3-, 8^3- and 16^3-cell cubes — and the test is worth having: at 8^3 cubes it answers 80 % of a camera's
    misses, which are 48 % of all the cell steps the reference's walk takes for the frame's rays."""
    size = 256
    h = np.maximum(16, np.minimum(size, port.terrain_heights(size)))
    y = np.arange(size)[None, :, None]
    cells = np.ascontiguousarray(((y >= size // 2 + 1) & (y <= (size // 2 + h - 1)[:, None, :])).astype(np.uint8))
    rng = np.random.default_rng(21)
    n = 150_000
    cam_o = np.broadcast_to(np.float32([128.3, 100.6, 20.9]), (n, 3)).copy()        # above the ground (solid cells start at y = 129, up = -y)
    cam_d = _unit(np.stack([rng.uniform(-1.0, 1.0, n), rng.uniform(-0.3, 0.9, n), np.ones(n)], 1))
    rnd_o = rng.uniform(0, size, (n, 3)).astype(np.float32)
    rnd_o[:, 1] = rng.uniform(0, size // 2, n)                                      # in the air
    rnd_d = rng.standard_normal((n, 3)).astype(np.float32)
    near_axis = rnd_d.copy()
    near_axis[np.arange(n), rng.integers(0, 3, n)] *= np.float32(1e-6)
    cases = [("camera", cam_o, cam_d), ("random", rnd_o, rnd_d), ("near-axis", rnd_o, near_axis),
             ("tiny |d|", rnd_o, (rnd_d * np.float32(1e-20)).astype(np.float32)), ("huge |d|", rnd_o, (rnd_d * np.float32(1e20)).astype(np.float32)),
             ("outside", rng.uniform(-40, size + 40, (n, 3)).astype(np.float32), rnd_d)]
    for label, o, d in cases:
        hits, steps = port.grid_cast(cells, o, d, threads=4)
        missed = hits["hit"] == 0
        for shift in (2, 3, 4):
            sure = port.grid_miss_test(cells, shift, o, d, threads=4) != 0
            assert not (sure & ~missed).any(), (label, shift, int((sure & ~missed).sum()))
            if label == "camera" and shift < 4:        # (16^3 cubes dilated by two swallow a camera 28 cells above the ground)
                answered = (sure & missed).sum() / max(1, missed.sum())
                saved = steps[sure].sum() / steps.sum()                      # cell steps the reference's walk spends on those rays
                assert 0.25 < missed.mean() < 0.5 and answered > (0.8, 0.7)[shift - 2] and saved > 0.4, (shift, float(answered), float(saved))


def test_svo_intended(port):
    g = golden("svo_random5.npz")
    hits = port.svo_cast(g["occ"], 5, g["origin"], g["dir"], 1 << 20)
    assert_hits_equal(hits, g["hits"], hits["hit"] != 0, "svo")
    hits = port.svo_cast(g["occ"], 5, g["origin"], g["dir"], 16)
    assert_hits_equal(hits, g["hits_iter16"], hits["hit"] != 0, "svo max_iter=16")


def test_frame_primary_shadow(port, textures):
    """Deterministic RayCaster frame (primary + sun shadow): u8-exact against the reference's RayCaster."""
    from oracle import loader
    g = golden("frame_cfg1_small.npz")
    p = loader.PortRenderParams()
    p.width, p.height, p.depth, p.guard = int(g["width"]), int(g["height"]), 9, 9
    p.cam_position[:] = [float(x) for x in g["cam_position"]]
    p.rot_mat[:] = [float(x) for x in g["rot_mat"]]
    p.fov, p.aperture, p.focal_length = 1.0, 0.0, 100.0
    p.light_position[:] = [float(x) for x in g["light"]]
    p.use_gi, p.gi_bounces, p.use_samples, p.spp = 0, 1, 1, 1
    p.seed_lo, p.seed_hi, p.threads = 0x5EED, 0, 4
    nodes = port.build_terrain(9)
    accum, rgba, stats = port.render(nodes, p, *textures)
    assert np.array_equal(accum, g["samples"])
    assert np.array_equal(rgba, g["image"])
    assert stats.rays[0] == p.width * p.height and 0 < stats.rays[1] < stats.rays[0]


def test_checkerboard_frames(port, vrt, textures):
    """The interactive loop's checkerboard halves (main.cpp:137-143) with the temporal blend, 4 frames, and two half frames in
    sample mode: the oracle against frames produced by the reference's own RayCaster (golden)."""
    from oracle import loader
    g = golden("frame_checker_small.npz")
    nodes = port.build_terrain(9)
    cam = vrt.Camera(position=g["cam_position"], view_angle=g["view_angle"], focal_length=100.0)   # host-side basis only
    for tag in ("a", "b"):
        W, H, area = (int(v) for v in g["size_" + tag])
        p = loader.PortRenderParams()
        p.width, p.height, p.depth, p.guard = W, H, 9, 9
        p.cam_position[:] = [float(x) for x in g["cam_position"]]
        p.rot_mat[:] = [float(x) for x in cam.rot_mat]
        p.fov, p.aperture, p.focal_length = 1.0, 0.0, 100.0
        p.light_position[:] = [float(x) for x in g["light"]]
        p.use_gi, p.gi_bounces, p.use_samples, p.spp = 0, 1, 0, 1
        p.seed_lo, p.threads, p.checker_area_height = 0x5EED, 4, area
        img = None
        for frame in range(4):
            p.checker = 1 + ((1 + frame) & 1)
            _, img, _ = port.render(nodes, p, *textures, prev_rgba=img)
        assert np.array_equal(img, g["blend4_" + tag]), tag
        p.use_samples = 1
        acc = np.zeros((H, W, 4), np.uint32)
        for frame in range(2):
            p.checker = 1 + (frame & 1)
            acc += port.render(nodes, p, *textures)[0]
        assert np.array_equal(acc, g["samples2_" + tag]), tag


def test_grid_render_checkerboard_halves(port):
    """vo_grid_render with the checkerboard of main.cpp:143 (the rule vo_render applies): it touches exactly the pixels the rule
    selects, those pixels equal the full frame's, the others are left alone, and the two halves add up to the full frame."""
    h = port.terrain_heights(64)
    y = np.arange(64)[None, :, None]
    cells = (y <= (20 + np.clip(h, 0, 30))[:, None, :]).astype(np.uint8)
    xs, zs = np.nonzero(h <= 12)
    cells[xs, 20 + np.clip(h, 0, 30)[xs, zs], zs] = 2               # a mirror lake on the lowest columns
    from oracle import loader
    W, H = 53, 31
    p = loader.PortRenderParams()
    p.width, p.height, p.depth, p.guard = W, H, 6, 6
    p.cam_position[:] = [32.0, 60.0, 4.0]
    p.rot_mat[:] = [1.0, 0.0, 0.0, 0.0, 0.6, -0.8, 0.0, 0.8, 0.6]                 # looking down towards +z
    p.fov, p.aperture, p.focal_length = 1.0, 0.3, 30.0
    p.light_position[:] = [100.0, 300.0, -50.0]
    p.use_gi, p.gi_bounces, p.use_samples, p.spp = 0, 1, 1, 2
    p.seed_lo, p.threads, p.roughness, p.max_bounds = 0x5EED, 4, 0.1, 4
    full, full_rgba, _ = port.grid_render(cells, p, np.full(768, 200, np.uint8), np.full(768, 120, np.uint8))
    assert (full[..., 3] == 2).all() and full_rgba[..., :3].max() > 0
    xs, ys = np.meshgrid(np.arange(W), np.arange(H))
    for area in (0, 7):
        rel = ys % area if area else ys
        halves = np.zeros_like(full)
        for checker in (1, 2):
            p.checker, p.checker_area_height = checker, area
            accum, rgba, _ = port.grid_render(cells, p, np.full(768, 200, np.uint8), np.full(768, 120, np.uint8))
            rule = (rel & 1) == ((xs + checker - 1) & 1)
            assert np.array_equal(accum[..., 3] > 0, rule), (area, checker)
            assert np.array_equal(accum[rule], full[rule]) and np.array_equal(rgba[rule], full_rgba[rule])
            assert not accum[~rule].any() and not rgba[~rule].any()
            halves += accum
        assert np.array_equal(halves, full)
