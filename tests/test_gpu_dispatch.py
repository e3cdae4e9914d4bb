r"""The frame, shade and grid launchers choose among many template instances (node layout, render_variant, trav_policy, whether
the loop guard can bind, mirrors, checkerboard / device autofocus, grid_variant).  Every instance below is reachable through the
C ABI and is held to the contract of the default one: accumulators, 8-bit image, ray counts and loop-trip counts exact against
oracle/port.c.  Rows, the test that runs each, and the launcher line that selects its instance:

| row | test                                          | instance                                             | selected at                                  |
|-----|-----------------------------------------------|------------------------------------------------------|----------------------------------------------|
| 1   | test_compact_layout_frames (variant 0/4, 16)  | render_rounds_kernel<CompactNodes, 0> (K6)           | render_kernels.cu launch_render_accumulate_ref: `if (compact) launch6(render_rounds_kernel<CompactNodes, 0>` |
| 1   | test_compact_layout_frames (variant 0/2, 3)   | render_accumulate_kernel<CompactNodes, false> (K4)   | launch_render_accumulate_ref: `else launch4(render_accumulate_kernel<CompactNodes, false>` |
| 1   | test_compact_layout_frames (variant 3)        | render_sorted_kernel<CompactNodes> (K5)              | launch_render_accumulate_ref: `if (compact) render_sorted_kernel<CompactNodes>` |
| 1   | test_compact_layout_frames (variant 1)        | render_persistent (K4p, reference array)             | capi.cu vrt_render_accumulate_device: `launch_render_persistent(sc->d_nodes` |
| 1   | test_compact_layout_checkerboard              | render_accumulate_kernel<CompactNodes, true>         | launch_render_accumulate_ref: `if (live) launch4(render_accumulate_kernel<CompactNodes, true>` |
| 1   | test_compact_layout_device_autofocus          | autofocus_kernel<CompactNodes> + the live K4 / K6     | launch_autofocus: `if (compact) autofocus_kernel<CompactNodes>` |
| 1   | test_compact_layout_refuses_mirrors           | (refused)                                            | capi.cu check_render_args: `if (sc->use_compact \|\| ...` |
| 2   | test_k6_traversal_policies (policy 0)         | render_rounds_kernel<RefNodes, 0>                    | launch_render_accumulate_ref: `case 0: launch6(render_rounds_kernel<RefNodes, 0>` |
| 2   | test_k6_traversal_policies (policy 1)         | render_rounds_kernel<RefNodes, 1>                    | launch_render_accumulate_ref: `case 1: launch6(render_rounds_kernel<RefNodes, 1>` |
| 2   | test_k6_traversal_policies (policy 2)         | render_rounds_kernel<RefNodes, 2, false, false>      | launch_render_accumulate_ref: `default:` ... `else launch6(render_rounds_kernel<RefNodes, 2, false, false>` |
| 2   | test_k6_help_window                           | the helper scan of render_rounds_kernel              | render_rounds_kernel: `const int W = L.help_window > groups ? ...` |
| 3a  | test_binding_guard_casts                      | K1 / K1p / K1b with the guard kept                   | capi.cu vrt_cast_rays_device (cast_variant 0..3) |
| 3b  | test_binding_guard_frames (K4, mirrors off)   | render_accumulate_kernel<RefNodes, false, false, true> | launch_render_accumulate_ref: `else { if (guarded) launch4(render_accumulate_kernel<RefNodes, false, false, true>` |
| 3b  | test_binding_guard_frames (K4, mirrors on)    | render_accumulate_kernel<RefNodes, false, true, true>  | launch_render_accumulate_ref: `else { if (guarded) launch4(render_accumulate_kernel<RefNodes, false, true, true>` |
| 3b  | test_binding_guard_frames (K6, mirrors off)   | render_rounds_kernel<RefNodes, 2, false, true>       | launch_render_accumulate_ref: `if (guard_binds(L)) launch6(render_rounds_kernel<RefNodes, 2, false, true>` |
| 3b  | test_binding_guard_frames (K6, mirrors on)    | render_rounds_kernel<RefNodes, 2, true, true>        | launch_render_accumulate_ref: `if (guard_binds(L)) launch6(render_rounds_kernel<RefNodes, 2, true, true>` |
| 3c  | test_reference_guard_at_depth_12              | the same guarded instances; then the kGuard = false ones with the guard lifted | guard_binds (render_kernels.cu) |
| 4   | test_shade_rays_match_the_oracle (reference)  | shade_rays_kernel<RefNodes, false>                   | launch_shade_rays: `else shade_rays_kernel<RefNodes, false>` |
| 4   | test_shade_rays_match_the_oracle (compact)    | shade_rays_kernel<CompactNodes, true>                | launch_shade_rays: `if (compact) shade_rays_kernel<CompactNodes, true>` |
| 4   | test_shade_rays_match_the_oracle (guard)      | shade_rays_kernel<RefNodes, true>                    | launch_shade_rays: `else if (guard_binds(L)) shade_rays_kernel<RefNodes, true>` |
| 4   | test_shade_rays_non_finite_rays, test_shade_rays_argument_checks | the same kernel; capi.cu vrt_shade_rays | vrt_shade_rays |
| 5   | test_degenerate_camera_through_k6             | K6 policies 0 / 1 / 2, compact K6, K6 with beam floors and bounds exits | launch_render_accumulate_ref (K6 branch); beam_kernels.cu launch_beam_floor |
| 6   | test_grid_frames_on_the_generic_loops (Grid3D) | grid_render_kernel<0>                               | grid_kernels.cu launch_grid_render: `else grid_render_kernel<0>` |
| 6   | test_grid_frames_on_the_generic_loops (mip)   | grid_render_kernel<1>                                | launch_grid_render: `else if (use_mip && g.n_levels > 1) grid_render_kernel<1>` |
| 6   | test_grid_checkerboard_frames                 | the checker test of grid_render_kernel, modes 2, 0, 1 | grid_render_kernel: `(!L.checker \|\| (x & 1) == checker_x_parity(...))` |

Contexts are created without beam floors and bounds exits (tests/conftest.py), so ray and trip counts equal the oracle's; rows that
need the product defaults turn them on explicitly.
"""
import ctypes as C

import numpy as np
import pytest

from conftest import assert_hits_equal

pytestmark = pytest.mark.gpu

SHADE_JOB = np.dtype([("start", "f4", 3), ("pixel", "u4"), ("direction", "f4", 3), ("sample", "u4")])                 # vrt_shade_job
SHADE_RESULT = np.dtype([("r", "u1"), ("g", "u1"), ("b", "u1"), ("hit", "u1"), ("distance", "f4"), ("complexity", "u4"),
                         ("reserved", "u4")])                                                                            # vrt_shade_result
assert SHADE_JOB.itemsize == 32 and SHADE_RESULT.itemsize == 16

DEMO_VIEW = dict(position=(256, 200, 256), view_angle=(0.3, -0.35))
INSIDE_HILL = dict(position=(307.2727, 210.45, 400.7897), view_angle=(2.801253, -0.355602))


def port_params(W, H, depth, cam, light, use_gi, bounces, use_samples, spp, seed=(0x5EED, 0), offset=0, rows=(0, 0)):
    from oracle import loader
    p = loader.PortRenderParams()
    p.width, p.height, p.depth, p.guard = W, H, depth, depth
    p.cam_position[:] = [float(x) for x in cam.position]
    p.rot_mat[:] = [float(x) for x in cam.rot_mat]
    p.fov, p.aperture, p.focal_length = cam.fov, cam.aperture, cam.focal_length
    p.light_position[:] = [float(x) for x in light]
    p.use_gi, p.gi_bounces, p.use_samples, p.spp = int(use_gi), bounces, int(use_samples), spp
    p.seed_lo, p.seed_hi, p.sample_offset = seed[0], seed[1], offset
    p.row_begin, p.row_end, p.threads = rows[0], rows[1], 8
    return p


def default_light(depth=9):
    return np.float32([-200, -1000, -300]) * np.float32(1.0 / (1 << depth)) + np.float32(1.0)


_oracle_frames = {}


def oracle_render(port, nodes, p, textures):
    """port.render, memoised on the parameter block (several instances are compared with the same oracle frame)."""
    key = (id(nodes), C.string_at(C.addressof(p), C.sizeof(p)))
    if key not in _oracle_frames:
        _oracle_frames[key] = port.render(nodes, p, *textures)
    return _oracle_frames[key]


def render(vrt, scene, size, cam, spp, light=None, use_gi=True, bounces=2, mirror_y=None, autofocus=False):
    rc = vrt.RayCaster(scene, size)
    rc.setLightPosition(default_light(scene.depth) if light is None else light)
    rc.use_samples, rc.use_gi, rc.gi_bounces = True, use_gi, bounces
    rc.mirror_y, rc.roughness, rc.autofocus = mirror_y, 0.05, autofocus
    img = rc.render(cam, spp=spp).copy()
    return rc, img


def assert_frame(rc, img, want, label, counts=True):
    accum, rgba, st = want
    assert np.array_equal(rc.colors, accum), "%s: accumulators differ on %d pixels" % (label, int((rc.colors != accum).any(-1).sum()))
    assert np.array_equal(img, rgba), label
    assert rc.last_stats["rays"] == list(st.rays), (label, rc.last_stats["rays"], list(st.rays))
    if counts:
        assert rc.last_stats["complexity"] == list(st.complexity), (label, rc.last_stats["complexity"], list(st.complexity))


def lsvo_scene(vrt, ctx, nodes, depth, textures, guard=0, layout=0):
    s = vrt.LSVO(ctx, nodes, depth, guard)
    s.set_textures(*textures)
    if layout:
        s.set_layout(layout)
    return s


# ---- row 1: the compact node layout ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("spp", [3, 16])
def test_compact_layout_frames(vrt, ctx, port, terrain9_nodes, textures, spp):
    """K4, K5, K6 (and K4p, which reads the reference array whatever the layout) on the compact array: GI with 2 bounces, depth of
    field, ragged frame; render_variant 0 picks K4 at 3 and K6 at 16 samples per pixel."""
    W, H = 203, 77
    cam = vrt.Camera(aperture=0.5, focal_length=60.0, **DEMO_VIEW)
    want = oracle_render(port, terrain9_nodes, port_params(W, H, 9, cam, default_light(), 1, 2, True, spp), textures)
    assert want[1][..., :3].max() > 0
    c = vrt.Context(0)
    try:
        s = lsvo_scene(vrt, c, terrain9_nodes, 9, textures, layout=1)
        for variant in (0, 2, 3, 1, 4):
            c.set_option("render_variant", variant)
            rc, img = render(vrt, s, (W, H), cam, spp)
            assert_frame(rc, img, want, "compact, render_variant %d, spp %d" % (variant, spp))
    finally:
        c.close()


@pytest.mark.parametrize("W,H,area_height,use_samples", [(161, 75, 15, False), (70, 44, 11, True)])
def test_compact_layout_checkerboard(vrt, ctx, port, terrain9_nodes, textures, W, H, area_height, use_samples):
    """The checkerboard sequence of test_gpu_render.py::test_checkerboard_frames on the compact layout (the live K4 instance)."""
    c = vrt.Context(0)
    try:
        s = lsvo_scene(vrt, c, terrain9_nodes, 9, textures, layout=1)
        cam = vrt.Camera(position=(256, 200, 256), view_angle=(0.3, -0.35), focal_length=80.0, aperture=0.4)
        rc = vrt.RayCaster(s, (W, H))
        rc.setLightPosition(default_light())
        rc.use_samples, rc.use_gi = use_samples, True
        rc.checker_area_height = area_height
        prev, acc = None, np.zeros((H, W, 4), np.uint32)
        spp = 2 if use_samples else 1
        for frame in range(4):
            rc.checker_board_offset = 1 - (frame & 1)
            img = rc.render(cam, spp=spp).copy()
            p = port_params(W, H, 9, cam, default_light(), 1, 1, use_samples, spp, offset=2 * frame if use_samples else frame)
            p.checker, p.checker_area_height = 1 + (1 - (frame & 1)), area_height
            a, want, st = port.render(terrain9_nodes, p, *textures, prev_rgba=prev)
            assert rc.last_stats["rays"] == list(st.rays) and rc.last_stats["complexity"] == list(st.complexity), "frame %d" % frame
            if use_samples:
                acc += a
                assert np.array_equal(rc.colors, acc), "frame %d" % frame
                rendered = acc[..., 3] > 0
                assert np.array_equal(img[rendered][:, :3], (acc[rendered][:, :3] // acc[rendered][:, 3:4]).astype(np.uint8))
            else:
                assert np.array_equal(img, want), "frame %d" % frame
                prev = want
    finally:
        c.close()


@pytest.mark.parametrize("view", [(0.0, -0.6), (0.3, -0.35)])
def test_compact_layout_device_autofocus(vrt, ctx, port, terrain9_nodes, textures, view):
    """vrt_render_params::autofocus on the compact layout (autofocus_kernel<CompactNodes>, then the live K4 and K6) gives the frame
    that Camera.autofocus's focal length gives on the reference layout; Camera.autofocus agrees in both layouts."""
    W, H = 128, 72
    c = vrt.Context(0)
    try:
        s = lsvo_scene(vrt, c, terrain9_nodes, 9, textures)
        cam = vrt.Camera(position=(256, 200, 256), view_angle=view, aperture=0.5, focal_length=3.0)
        f_ref = cam.autofocus(s)
        s.set_layout(1)
        cam.focal_length = 3.0
        assert cam.autofocus(s) == f_ref != 3.0
        for spp in (3, 16):
            cam.focal_length = 3.0
            rc, img = render(vrt, s, (W, H), cam, spp, autofocus=True)
            cam.focal_length = f_ref
            want = oracle_render(port, terrain9_nodes, port_params(W, H, 9, cam, default_light(), 1, 2, True, spp), textures)
            assert_frame(rc, img, want, "compact autofocus, spp %d" % spp)
            s.set_layout(0)
            rc0, img0 = render(vrt, s, (W, H), cam, spp)
            s.set_layout(1)
            assert np.array_equal(img, img0) and np.array_equal(rc.colors, rc0.colors)
    finally:
        c.close()


def test_compact_layout_refuses_mirrors(vrt, ctx, terrain9_nodes, textures):
    c = vrt.Context(0)
    try:
        s = lsvo_scene(vrt, c, terrain9_nodes, 9, textures, layout=1)
        cam = vrt.Camera(aperture=0.5, focal_length=60.0, **DEMO_VIEW)
        for spp in (1, 16):
            with pytest.raises(vrt.VrtError) as e:
                render(vrt, s, (64, 36), cam, spp, mirror_y=240)
            assert e.value.code == -4                                    # VRT_ERR_UNSUPPORTED
    finally:
        c.close()


# ---- row 2: K6 traversal loops and helping order ----------------------------------------------------------------------------------
@pytest.mark.parametrize("spp", [16, 70])
def test_k6_traversal_policies(vrt, ctx, port, terrain9_nodes, textures, spp):
    """K6 on Trav (0), Trav2 (1) and Trav2 without the cone test in the coef-0 casts (2).  Then 0 and 1 with the product defaults
    (beam floors, bounds exits): those loops ignore both, but the sort kernel still answers the samples of empty beam tiles — same
    frame and rays, the secondary trip counts of the reference, fewer primary trips."""
    W, H = 150, 70
    cam = vrt.Camera(aperture=0.5, focal_length=60.0, **DEMO_VIEW)
    want = oracle_render(port, terrain9_nodes, port_params(W, H, 9, cam, default_light(), 1, 2, True, spp), textures)
    c = vrt.Context(0)
    try:
        c.set_option("render_variant", 4)
        s = lsvo_scene(vrt, c, terrain9_nodes, 9, textures)
        for policy in (0, 1, 2):
            c.set_option("trav_policy", policy)
            rc, img = render(vrt, s, (W, H), cam, spp)
            assert_frame(rc, img, want, "trav_policy %d, spp %d" % (policy, spp))
        c.set_option("beam_tile", 8)
        c.set_option("bounds_exit", 1)
        for policy in (0, 1):
            c.set_option("trav_policy", policy)
            rc, img = render(vrt, s, (W, H), cam, spp)
            assert_frame(rc, img, want, "trav_policy %d with beam floors and bounds exits" % policy, counts=False)
            assert rc.last_stats["complexity"][1:] == list(want[2].complexity)[1:]
            assert rc.last_stats["complexity"][0] <= want[2].complexity[0]
    finally:
        c.close()


def test_k6_help_window(vrt, ctx, port, terrain9_nodes, textures):
    """Helping CTAs that all start at the last block (0), that spread over 1, 64 (default) or 4096 groups: one frame."""
    W, H, spp = 150, 70, 16
    cam = vrt.Camera(aperture=0.5, focal_length=60.0, **DEMO_VIEW)
    want = oracle_render(port, terrain9_nodes, port_params(W, H, 9, cam, default_light(), 1, 2, True, spp), textures)
    c = vrt.Context(0)
    try:
        c.set_option("render_variant", 4)
        s = lsvo_scene(vrt, c, terrain9_nodes, 9, textures)
        for window in (0, 1, 64, 4096):
            c.set_option("help_window", window)
            rc, img = render(vrt, s, (W, H), cam, spp)
            assert_frame(rc, img, want, "help_window %d" % window)
    finally:
        c.close()


# ---- row 3: a loop guard that binds ------------------------------------------------------------------------------------------------
def _rays(rng, n):
    o = rng.uniform(1, 2, (n, 3)).astype(np.float32)
    o[:, 1] = rng.uniform(1.0, 1.45, n)
    d = rng.normal(size=(n, 3)).astype(np.float32)
    return o, d / np.linalg.norm(d, axis=1, keepdims=True)


def _casts_match(vrt, port, c, s, nodes, depth, guard, o, d, coef, label):
    want = port.lsvo_cast(nodes, depth, o, d, coef, 0.0, guard=guard, threads=8)
    for variant in (0, 1, 2, 3):
        c.set_option("cast_variant", variant)
        got = s.cast_rays(o, d, coef, 0.0)
        assert_hits_equal(got, want, (got["flags"] & 1) != 0, "%s, cast_variant %d, coef %g" % (label, variant, coef))
        assert s.last_complexity() == int(want["complexity"].sum())
    return want


@pytest.mark.parametrize("guard", [14, 16])
def test_binding_guard_casts(vrt, ctx, port, terrain9_nodes, guard):
    """T(9) with guard 14 (= 23 - 9: the walk stops at the leaves' level) and 16: camera rays all miss, cone rays hit coarse nodes."""
    rng = np.random.default_rng(guard)
    c = vrt.Context(0)
    try:
        s = vrt.LSVO(c, terrain9_nodes, 9, guard)
        o, d = _rays(rng, 70000)                                    # >= 65536 coherent-gate rays: cast_variant 3 runs its classifier
        want = _casts_match(vrt, port, c, s, terrain9_nodes, 9, guard, o, d, 0.0, "guard %d" % guard)
        assert not want["hit"].any() and want["complexity"].min() > 0
        o, d = _rays(rng, 20000)
        want = _casts_match(vrt, port, c, s, terrain9_nodes, 9, guard, o, d, 0.5, "guard %d" % guard)
        assert 0.1 < (want["hit"] != 0).mean() < 0.99
    finally:
        c.close()


@pytest.mark.parametrize("guard", [14, 16])
def test_binding_guard_frames(vrt, ctx, port, terrain9_nodes, textures, guard):
    """Frames on the guarded scenes through K4 and K6, with and without mirrors.  Every camera ray misses, so what is pinned here
    is the rays and the loop-trip counts of the guarded walks."""
    W, H = 128, 72
    cam = vrt.Camera(aperture=0.5, focal_length=60.0, **DEMO_VIEW)
    c = vrt.Context(0)
    try:
        s = lsvo_scene(vrt, c, terrain9_nodes, 9, textures, guard=guard)
        for variant, spp in ((2, 3), (4, 16)):
            c.set_option("render_variant", variant)
            for mirror_y in (None, 240):
                p = port_params(W, H, 9, cam, default_light(), 1, 2, True, spp)
                p.guard = guard
                if mirror_y is not None:
                    p.mirror_y1, p.roughness, p.max_bounds = mirror_y + 1, 0.05, 4
                want = oracle_render(port, terrain9_nodes, p, textures)
                rc, img = render(vrt, s, (W, H), cam, spp, mirror_y=mirror_y)
                assert_frame(rc, img, want, "guard %d, render_variant %d, mirror %s" % (guard, variant, mirror_y))
                assert rc.last_stats["complexity"][0] > 0 and rc.last_stats["rays"][0] == W * H * spp
    finally:
        c.close()


def _sparse_depth12_voxels():
    """A few thousand random voxels and a 64 x 64 slab that a camera at z = 2990 (castRay frame, voxel units) looks at."""
    rng = np.random.default_rng(12)
    xs, ys = np.meshgrid(np.arange(2016, 2080), np.arange(2016, 2080), indexing="ij")
    slab = np.stack([xs.ravel(), ys.ravel(), np.full(xs.size, 1000)], 1)      # setCell z = 1000: castRay z = 4095 - 1000
    return np.concatenate([rng.integers(0, 4096, (3000, 3)), slab]).astype(np.uint32)


def test_reference_guard_at_depth_12(vrt, ctx, port, textures):
    """The reference's own guard binds at depth 12 (DESIGN.md §2): a sparse depth-12 scene with guard 0 (= the reference
    expression) misses everywhere, casts and frames equal to the oracle's; lifted (-1), the same scene shows its voxels."""
    vox = _sparse_depth12_voxels()
    nodes = vrt.host_build_lsvo_from_voxels(12, vox)
    assert len(nodes) < 1 << 20
    cam = vrt.Camera(position=(2048, 2048, 2990), view_angle=(0.0, 0.0), aperture=0.5, focal_length=100.0)
    rng = np.random.default_rng(4)
    n = 20000
    o = np.tile(cam.position * np.float32(1 / 4096) + np.float32(1), (n, 1)).astype(np.float32)
    towards_slab = np.stack([rng.normal(0, 0.25, n // 2), rng.normal(0, 0.25, n // 2), np.ones(n // 2)], 1)
    d = np.concatenate([towards_slab, rng.normal(size=(n // 2, 3))]).astype(np.float32)
    o[n // 2:] = rng.uniform(1, 2, (n // 2, 3))
    W, H = 96, 54
    c = vrt.Context(0)
    try:
        for guard, port_guard in ((0, 12), (-1, 0)):
            s = vrt.LSVO.from_voxels(c, 12, vox, guard=guard)
            s.set_textures(*textures)
            hits = []
            for coef in (0.0, 0.5):
                want = _casts_match(vrt, port, c, s, nodes, 12, port_guard, o, d, coef, "depth 12, guard %d" % guard)
                hits.append(int((want["hit"] != 0).sum()))
            for variant, spp in ((2, 3), (4, 16)):
                c.set_option("render_variant", variant)
                p = port_params(W, H, 12, cam, default_light(12), 1, 2, True, spp)
                p.guard = port_guard
                want = oracle_render(port, nodes, p, textures)
                rc, img = render(vrt, s, (W, H), cam, spp)
                assert_frame(rc, img, want, "depth 12, guard %d, render_variant %d" % (guard, variant))
                if guard == 0:
                    assert rc.last_stats["rays"][1] == 0 and rc.last_stats["complexity"][0] > 0
                else:
                    assert rc.last_stats["rays"][1] > W * H * spp // 8 and img[..., :3].max() > 0
            if guard == 0:
                assert hits[0] == 0
            else:
                assert hits[0] > 1000
            s.close()
    finally:
        c.close()


# ---- row 4: vrt_shade_rays -------------------------------------------------------------------------------------------------------
def shade_params(vrt, W, H, light, use_gi, bounces):
    p = vrt.capi.RenderParams()
    p.width, p.height, p.spp, p.use_samples = W, H, 1, 1
    p.seed_lo, p.seed_hi = 0x5EED, 0
    p.light_position[:] = [float(x) for x in light]
    p.use_gi, p.gi_bounces = int(use_gi), bounces
    return p


def shade(vrt, scene, p, jobs):
    out = np.zeros(len(jobs), SHADE_RESULT)
    vrt.capi.check(vrt.capi.lib().vrt_shade_rays(scene.handle, C.byref(p), len(jobs), vrt.capi.ptr(jobs), vrt.capi.ptr(out)))
    return out


def camera_jobs(port, p, W, H, sample):
    rays = [port.camera_ray(p, x, y, sample) for y in range(H) for x in range(W)]
    jobs = np.zeros(W * H, SHADE_JOB)
    jobs["start"] = [o for o, _ in rays]
    jobs["direction"] = [d for _, d in rays]
    jobs["pixel"] = np.arange(W * H)                     # y * W + x
    jobs["sample"] = sample
    return jobs


def assert_shaded(port, nodes, got, jobs, accum, guard, label):
    rgb = np.stack([got["r"], got["g"], got["b"]], -1)
    want_rgb = accum.reshape(-1, 4)[:, :3]
    assert np.array_equal(rgb, want_rgb), "%s: colour differs on %d rays" % (label, int((rgb != want_rgb).any(-1).sum()))
    assert (accum.reshape(-1, 4)[:, 3] == 1).all()
    rec = port.lsvo_cast(nodes, 9, jobs["start"], jobs["direction"], guard=guard, threads=8)
    assert np.array_equal(got["hit"] != 0, rec["hit"] != 0), label
    assert np.array_equal(got["complexity"], rec["complexity"]), label
    want_d = np.where(rec["hit"] != 0, rec["distance"], np.float32(0))
    assert np.array_equal(got["distance"].view(np.uint32), want_d.astype(np.float32).view(np.uint32)), label
    assert (got["reserved"] == 0).all()


@pytest.mark.parametrize("instance", ["reference", "compact", "guard"])
def test_shade_rays_match_the_oracle(vrt, ctx, port, terrain9_nodes, textures, instance):
    """vrt_shade_rays fed with the oracle's camera rays of a 96 x 54 frame: colour = the oracle frame's 1-sample accumulator
    (sample_offset = s), hit / distance (bits) / complexity = the oracle's record of that primary ray.  Reference layout, compact
    layout, and a scene whose guard binds (guard 14 on T(9))."""
    W, H = 96, 54
    guard = 14 if instance == "guard" else 9
    cam = vrt.Camera(aperture=0.5, focal_length=60.0, **DEMO_VIEW)
    c = vrt.Context(0)
    try:
        s = lsvo_scene(vrt, c, terrain9_nodes, 9, textures, guard=14 if instance == "guard" else 0,
                       layout=1 if instance == "compact" else 0)
        for sample in (0, 5):
            p = port_params(W, H, 9, cam, default_light(), 0, 1, True, 1, offset=sample)
            p.guard = guard
            jobs = camera_jobs(port, p, W, H, sample)
            for use_gi, bounces in ((0, 1), (1, 1), (1, 2)):
                p = port_params(W, H, 9, cam, default_light(), use_gi, bounces, True, 1, offset=sample)
                p.guard = guard
                accum, _, _ = oracle_render(port, terrain9_nodes, p, textures)
                got = shade(vrt, s, shade_params(vrt, W, H, default_light(), use_gi, bounces), jobs)
                label = "%s, sample %d, use_gi %d, bounces %d" % (instance, sample, use_gi, bounces)
                assert_shaded(port, terrain9_nodes, got, jobs, accum, guard, label)
                if instance != "guard":
                    assert 0.2 < (got["hit"] != 0).mean() < 0.95 and accum[..., :3].max() > 0
                else:
                    assert not got["hit"].any()
    finally:
        c.close()


def test_shade_rays_non_finite_rays(vrt, ctx, port, terrain9_nodes, textures):
    """Camera inside a hill: autofocus gives focal length 0, and the lens samples with both numbers 0 normalise a zero vector
    (test_gpu_render.py::test_camera_inside_solid_terminates).  Those NaN rays come back black, hit 0, complexity 0."""
    W, H = 96, 54
    c = vrt.Context(0)
    try:
        for layout in (0, 1):
            s = lsvo_scene(vrt, c, terrain9_nodes, 9, textures, layout=layout)
            cam = vrt.Camera(aperture=0.3, **INSIDE_HILL)
            assert cam.autofocus(s) == 0.0
            nan_rays = 0
            for sample in (0, 5):
                p = port_params(W, H, 9, cam, default_light(), 1, 2, True, 1, offset=sample)
                jobs = camera_jobs(port, p, W, H, sample)
                accum, _, _ = oracle_render(port, terrain9_nodes, p, textures)
                got = shade(vrt, s, shade_params(vrt, W, H, default_light(), 1, 2), jobs)
                assert_shaded(port, terrain9_nodes, got, jobs, accum, 9, "inside a hill, layout %d, sample %d" % (layout, sample))
                bad = ~np.isfinite(jobs["direction"]).all(-1)
                nan_rays += int(bad.sum())
                assert not got["hit"][bad].any() and (got["complexity"][bad] == 0).all()
                assert not got["r"][bad].any() and not got["g"][bad].any() and not got["b"][bad].any()
            assert nan_rays > 0
            s.close()
    finally:
        c.close()


def test_shade_rays_argument_checks(vrt, ctx, terrain9_nodes, textures):
    lib, check = vrt.capi.lib(), vrt.capi.check
    jobs, out = np.zeros(4, SHADE_JOB), np.zeros(4, SHADE_RESULT)
    jobs["direction"] = [0.0, 0.0, 1.0]
    jobs["start"] = 1.5
    s = lsvo_scene(vrt, ctx, terrain9_nodes, 9, textures)
    p = shade_params(vrt, 8, 8, default_light(), 1, 3)
    with pytest.raises(vrt.VrtError) as e:
        check(lib.vrt_shade_rays(s.handle, C.byref(p), 4, vrt.capi.ptr(jobs), vrt.capi.ptr(out)))
    assert e.value.code == -1
    p.gi_bounces = 2
    check(lib.vrt_shade_rays(s.handle, C.byref(p), 0, None, None))                 # n = 0: nothing to do
    check(lib.vrt_shade_rays(s.handle, C.byref(p), 4, vrt.capi.ptr(jobs), vrt.capi.ptr(out)))
    bare = vrt.LSVO(ctx, terrain9_nodes, 9)                                        # no textures
    with pytest.raises(vrt.VrtError) as e:
        check(lib.vrt_shade_rays(bare.handle, C.byref(p), 4, vrt.capi.ptr(jobs), vrt.capi.ptr(out)))
    assert e.value.code == -1
    grid = vrt.Grid3D(ctx, np.ones((8, 8, 8), np.uint8))
    grid.set_textures(*textures)
    with pytest.raises(vrt.VrtError) as e:
        check(lib.vrt_shade_rays(grid.handle, C.byref(p), 4, vrt.capi.ptr(jobs), vrt.capi.ptr(out)))
    assert e.value.code == -4                                                      # VRT_ERR_UNSUPPORTED
    for sc in (s, bare, grid):
        sc.close()


# ---- row 5: a degenerate camera through K6 -----------------------------------------------------------------------------------------
def test_degenerate_camera_through_k6(vrt, ctx, port, terrain9_nodes, textures):
    """Focal length 0 from inside a hill, 16 samples per pixel: K6 on every traversal loop and on the compact layout equals the
    oracle, counts included.  With the product defaults the beam kernel widens the lens by a clamped focal length (its camera
    rays point along their lens offsets, not through their pixels); the frame and the rays still equal the oracle's."""
    W, H, spp = 128, 72, 16
    c = vrt.Context(0)
    try:
        s = lsvo_scene(vrt, c, terrain9_nodes, 9, textures)
        cam = vrt.Camera(aperture=0.3, **INSIDE_HILL)
        assert cam.autofocus(s) == 0.0
        want = oracle_render(port, terrain9_nodes, port_params(W, H, 9, cam, default_light(), 1, 2, True, spp), textures)
        c.set_option("render_variant", 4)
        for policy in (0, 1, 2):
            c.set_option("trav_policy", policy)
            rc, img = render(vrt, s, (W, H), cam, spp)
            assert_frame(rc, img, want, "inside a hill, trav_policy %d" % policy)
        s.set_layout(1)
        rc, img = render(vrt, s, (W, H), cam, spp)
        assert_frame(rc, img, want, "inside a hill, compact")
        s.set_layout(0)
        c.set_option("render_variant", 0)
        c.set_option("trav_policy", 2)
        c.set_option("beam_tile", 8)
        c.set_option("bounds_exit", 1)
        rc, img = render(vrt, s, (W, H), cam, spp)
        assert_frame(rc, img, want, "inside a hill, product defaults", counts=False)
        assert all(a <= b for a, b in zip(rc.last_stats["complexity"], want[2].complexity))
    finally:
        c.close()


# ---- row 6: grid frames on the generic loops ---------------------------------------------------------------------------------------
def mirror_scene(vrt, size=128):
    """Terrain columns over a flat lake of Cell::Mirror voxels (test_gpu_grid.py::mirror_scene)."""
    h = vrt.host_terrain_heights(256)[:size, :size]
    top = 30 + np.clip(h, 0, 70)
    y = np.arange(size)[None, :, None]
    cells = (y <= top[:, None, :]).astype(np.uint8)
    lake = h <= 18
    xs, zs = np.nonzero(lake)
    cells[xs, 30 + np.clip(h, 0, 70)[lake], zs] = 2
    return cells


def grid_params(W, H, cam, light, spp, roughness, offset=0):
    from oracle import loader
    p = loader.PortRenderParams()
    p.width, p.height, p.depth, p.guard = W, H, 7, 7
    p.cam_position[:] = [float(x) for x in cam.position]
    p.rot_mat[:] = [float(x) for x in cam.rot_mat]
    p.fov, p.aperture, p.focal_length = cam.fov, cam.aperture, cam.focal_length
    p.light_position[:] = [float(x) for x in light]
    p.use_gi, p.gi_bounces, p.use_samples, p.spp = 0, 1, 1, spp
    p.seed_lo, p.seed_hi, p.sample_offset, p.threads = 0x5EED, 0, offset, 8
    p.roughness, p.max_bounds = roughness, 4
    return p


GRID_LIGHT = np.float32([300.0, 900.0, -200.0])


def grid_frame(vrt, scene, size, cam, spp, roughness, checker=None, area=0):
    rc = vrt.RayCaster(scene, size)
    rc.setLightPosition(GRID_LIGHT)
    rc.use_samples, rc.roughness, rc.max_bounds = True, roughness, 4
    rc.checker_board_offset, rc.checker_area_height = checker, area
    img = rc.render(cam, spp=spp).copy()
    return rc, img


@pytest.mark.parametrize("roughness,aperture,spp", [(0.0, 0.0, 1), (0.15, 0.0, 2), (0.3, 0.4, 3)])
def test_grid_frames_on_the_generic_loops(vrt, ctx, port, textures, roughness, aperture, spp):
    """grid_variant 1: Grid3D renders on the flat generic DDA, MipmapGrid3D (3 levels) on the fetch-skipping pyramid — the oracle's
    frame and counts, and byte for byte the frame of the bordered DDA (grid_variant 0)."""
    cells = mirror_scene(vrt)
    W, H = 200, 120
    cam = vrt.Camera(position=(64.0, 118.0, 20.0), view_angle=(0.0, 0.75), aperture=aperture, focal_length=40.0)
    accum, rgba, st = port.grid_render(cells, grid_params(W, H, cam, GRID_LIGHT, spp, roughness), *textures)
    assert st.rays[2] > 0 and rgba[..., :3].max() > 0
    c = vrt.Context(0)
    try:
        for make in (lambda: vrt.Grid3D(c, cells), lambda: vrt.MipmapGrid3D(c, cells, 3)):
            scene = make()
            scene.set_textures(*textures)
            frames = []
            for variant in (1, 0):
                c.set_option("grid_variant", variant)
                rc, img = grid_frame(vrt, scene, (W, H), cam, spp, roughness)
                label = "%s, grid_variant %d" % (type(scene).__name__, variant)
                assert np.array_equal(rc.colors, accum) and np.array_equal(img, rgba), label
                assert rc.last_stats["rays"][:3] == list(st.rays)[:3], label
                assert rc.last_stats["complexity"][:3] == list(st.complexity)[:3], label
                frames.append(img)
            assert np.array_equal(frames[0], frames[1])
            scene.close()
    finally:
        c.close()


@pytest.mark.parametrize("area", [0, 15])
def test_grid_checkerboard_frames(vrt, ctx, port, textures, area):
    """Checkerboard halves of a grid frame (offsets 0 and 1) on the bordered DDA and both generic loops: the oracle's accumulators
    and counts, untouched pixels left at zero, and the two halves add up to the full frame."""
    cells = mirror_scene(vrt)
    W, H, spp = 161, 75, 2
    cam = vrt.Camera(position=(64.0, 118.0, 20.0), view_angle=(0.0, 0.75), aperture=0.4, focal_length=40.0)
    full, _, _ = port.grid_render(cells, grid_params(W, H, cam, GRID_LIGHT, spp, 0.15), *textures)
    c = vrt.Context(0)
    try:
        for make, variant in ((lambda: vrt.Grid3D(c, cells), 0), (lambda: vrt.Grid3D(c, cells), 1),
                              (lambda: vrt.MipmapGrid3D(c, cells, 3), 1)):
            c.set_option("grid_variant", variant)
            scene = make()
            scene.set_textures(*textures)
            halves = np.zeros_like(full)
            for offset in (0, 1):
                p = grid_params(W, H, cam, GRID_LIGHT, spp, 0.15)
                p.checker, p.checker_area_height = 1 + offset, area
                accum, rgba, st = port.grid_render(cells, p, *textures)
                rc, img = grid_frame(vrt, scene, (W, H), cam, spp, 0.15, checker=offset, area=area)
                label = "%s, grid_variant %d, offset %d" % (type(scene).__name__, variant, offset)
                assert np.array_equal(rc.colors, accum), label
                rendered = accum[..., 3] > 0
                assert np.array_equal(img[rendered], rgba[rendered]), label
                assert rc.last_stats["rays"][:3] == list(st.rays)[:3] and rc.last_stats["complexity"][:3] == list(st.complexity)[:3], label
                assert abs(int(rendered.sum()) - W * H // 2) <= H
                halves += rc.colors
            assert np.array_equal(halves, full)
            scene.close()
    finally:
        c.close()
