r"""Frames of edited and off-centre LSVO scenes against the oracle, with the product's two frame shortcuts on: beam floors
(`beam_tile` 8, beam_kernels.cu: a conservative start distance per screen tile, and K6 skips the samples of tiles whose frustum is
empty) and bounds exits (`bounds_exit` 1: a walk ends where its ray leaves the box of the solid voxels, scene_device.cu
device_scene_bounds, recomputed by capi.cu update_bounds after creation and after every edit).

Every frame is checked four ways against the oracle (port.render, or palette_oracle.render_palette for palette frames) fed a node
array built from scratch on the host (vrt.host_build_lsvo_from_voxels; heightfields through the fill rule of test_gpu_lsvo.py):
  (a) the accumulator and the 8-bit image are equal;
  (b) the ray counts are equal, and every loop-trip class is at most the oracle's (the shortcuts only remove trips);
  (c) with both shortcuts off, the trip counts are equal too;
  (d) the edited scene's stats (rays, complexity, culled_primary) equal those of a scene created from scratch on the device from
      the same voxels or heights, with the same options: bounds and floors are functions of the node array, so stale bounds show
      here even where the pixels are right.
K4 is run at 4 samples (no floors) and, forced by render_variant 2, at 8 (floors on); K6 at 16 (render_variant 0, floors on).

| test                                          | what it pins                                                                          |
|-----------------------------------------------|---------------------------------------------------------------------------------------|
| test_voxel_model_edits                        | vrt_scene_set_cells -> rebuild_from_keys -> update_bounds on a model in one corner of the cube: growth past each of the six box faces, removing the outer layer, removing everything (empty box), single voxels on the cube's corners, the model back |
| test_growth_is_in_view                        | the premise of the growth steps: each one changes the oracle's frame of some camera    |
| test_heightfield_edits                        | vrt_scene_edit_heights -> update_bounds: a raised rectangle, a flattened mirror lake, everything lowered, the compact layout (capi.cu rebuilds it, bounds exits only) |
| test_painted_model_edits                      | paint_cells, set_cells adding and removing voxels, palette frames with the product defaults; added voxels have colour 1 |
| test_frames_enqueued_before_an_edit           | frames enqueued on the stream (vrt_render_accumulate_device) before vrt_scene_edit_heights / vrt_scene_set_cells read the old world; the replaced array is the pool's spare |
| test_shallow_worlds                           | device_scene_bounds with stop_level 0 (depth <= 3) and at depth 4                      |
| test_bounds_queue_overflow                    | bounds_expand_kernel's full-queue branch (more than 2^19 occupied 16-voxel cubes): overflowed cubes are terminal |
| test_bounds_exits_shorten_walks               | the bounds are not the whole cube: fewer loop trips with bounds_exit 1 on the model    |

Each test renders on a context of its own and sets beam_tile, bounds_exit and render_variant on it explicitly.
"""
import ctypes as C

import numpy as np
import pytest

from palette_oracle import render_palette
from test_gpu_lsvo import _heightfield_voxels
from test_gpu_palette import leaf_slots

pytestmark = pytest.mark.gpu

KERNELS = ((4, 0), (8, 2), (16, 0))         # (spp, render_variant): K4, K4 with beam floors, K6 with beam floors
SIZES = ((96, 54), (131, 67), (160, 90))


def default_light(depth):
    return np.float32([-200, -1000, -300]) * np.float32(1.0 / (1 << depth)) + np.float32(1.0)


def look_at(vrt, position, target, aperture=0.5, focal_length=60.0):
    """A camera at `position` (world voxel units, as Camera.position) whose centre ray points at `target`."""
    d = np.float64(target) - np.float64(position)
    d /= np.linalg.norm(d)
    angle = (float(np.arctan2(d[0], d[2])), float(-np.arcsin(d[1])))      # camera_vec = (sin a0 cos a1, -sin a1, cos a0 cos a1)
    return vrt.Camera(position=position, view_angle=angle, aperture=aperture, focal_length=focal_length)


def world(S, c):
    """Centre of setCell voxel c in camera units: the tree stores the mirrored octant (world voxel index S - 1 - c)."""
    return S - 0.5 - np.float64(c)


def set_shortcuts(c, on):
    c.set_option("beam_tile", 8 if on else 0)
    c.set_option("bounds_exit", 1 if on else 0)


def oracle_params(depth, cam, size, spp, mirror_y=None, rows=(0, 0)):
    from oracle import loader
    p = loader.PortRenderParams()
    p.width, p.height, p.depth, p.guard = size[0], size[1], depth, depth
    p.cam_position[:] = [float(x) for x in cam.position]
    p.rot_mat[:] = [float(x) for x in cam.rot_mat]
    p.fov, p.aperture, p.focal_length = cam.fov, cam.aperture, cam.focal_length
    p.light_position[:] = [float(x) for x in default_light(depth)]
    p.use_gi, p.gi_bounces, p.use_samples, p.spp = 1, 2, 1, spp
    p.seed_lo, p.seed_hi, p.sample_offset = 0x5EED, 0, 0
    p.row_begin, p.row_end, p.threads = rows[0], rows[1], 8
    p.roughness, p.max_bounds, p.mirror_y1 = 0.05, 4, 0 if mirror_y is None else mirror_y + 1
    return p


def gpu_frame(vrt, scene, cam, size, spp, mirror_y=None, rows=(0, 0)):
    rc = vrt.RayCaster(scene, size)
    rc.setLightPosition(default_light(scene.depth))
    rc.use_samples, rc.use_gi, rc.gi_bounces = True, True, 2
    rc.mirror_y, rc.roughness, rc.max_bounds = mirror_y, 0.05, 4
    img = rc.render(cam, spp, *rows).copy()
    return rc.colors.copy(), img, rc.last_stats


def check_frame(vrt, c, edited, fresh, want, cam, size, spp, variant, label, mirror_y=None, rows=(0, 0)):
    """(a)-(d) for one frame, shortcuts on and off.  Returns the stats with the shortcuts on."""
    accum, rgba, st = want
    y0, y1 = rows if rows[1] else (0, size[1])
    c.set_option("render_variant", variant)
    out = None
    try:
        for on in (True, False):
            set_shortcuts(c, on)
            tag = "%s, spp %d, render_variant %d, shortcuts %s" % (label, spp, variant, "on" if on else "off")
            colors, img, stats = gpu_frame(vrt, edited, cam, size, spp, mirror_y, rows)
            bad = int((colors[y0:y1] != accum[y0:y1]).any(-1).sum())
            assert bad == 0, "%s: accumulators differ on %d pixels" % (tag, bad)
            assert np.array_equal(img[y0:y1], rgba[y0:y1]), tag
            assert stats["rays"] == list(st.rays), (tag, stats["rays"], list(st.rays))
            assert all(g <= w for g, w in zip(stats["complexity"], st.complexity)), (tag, stats["complexity"], list(st.complexity))
            if not on:
                assert stats["complexity"] == list(st.complexity), (tag, stats["complexity"], list(st.complexity))
                assert stats["culled_primary"] == 0, tag
            _, _, ref = gpu_frame(vrt, fresh, cam, size, spp, mirror_y, rows)
            assert stats == ref, (tag, "edited scene vs the same world created from scratch", stats, ref)
            if on:
                out = stats
    finally:
        set_shortcuts(c, False)
        c.set_option("render_variant", 0)
    return out


def voxel_scene(vrt, c, depth, vox, textures):
    s = vrt.LSVO.from_voxels(c, depth, np.asarray(vox, np.uint32).reshape(-1, 3), on_device=True)
    s.set_textures(*textures)
    return s


def as_set(vox):
    return set(map(tuple, np.asarray(vox, np.int64).reshape(-1, 3).tolist()))


def as_array(voxels):
    return np.array(sorted(voxels), np.uint32).reshape(-1, 3)


def box(x, y, z):
    """Voxels of the box [x0, x1) x [y0, y1) x [z0, z1)."""
    g = np.mgrid[x[0]:x[1], y[0]:y[1], z[0]:z[1]]
    return g.reshape(3, -1).T.astype(np.uint32)


# ---- the model: a hollow box with a rod along +x, in one corner of the depth-8 cube (setCell coordinates) ------------------------
DEPTH = 8
S = 1 << DEPTH


def model_voxels():
    shell = box((24, 48), (160, 184), (28, 52))
    inner = as_set(box((25, 47), (161, 183), (29, 51)))
    shell = np.array([v for v in shell.tolist() if tuple(v) not in inner], np.uint32)
    rod = box((48, 88), (171, 173), (39, 41))
    return np.concatenate([shell, rod])                        # 3176 + 160 voxels, 2+ voxels from every cube face


# Growth past each face of the box, one side per edit.  Every blob is 3 voxels deep and its outermost layer is alone in its 8-voxel
# cube of the bounds sweep, so removing the outer layer later shrinks the bounds by a whole cube on every side.
GROWTH = (("-x", box((15, 18), (168, 174), (36, 42))), ("+x", box((102, 105), (168, 174), (36, 42))),
          ("-y", box((50, 56), (143, 146), (36, 42))), ("+y", box((50, 56), (198, 201), (36, 42))),
          ("-z", box((50, 56), (168, 174), (15, 18))), ("+z", box((50, 56), (168, 174), (62, 65))))


def model_cameras(vrt):
    centre = (world(S, 56), world(S, 172), world(S, 40))
    return (("outside the cube", look_at(vrt, (400.0, -40.0, 330.0), centre)),
            ("inside the cube", look_at(vrt, (120.0, 40.0, 130.0), centre)),
            # in the plane of the top face of the bounds (8-voxel cubes less the 2-voxel margin), looking along it
            ("grazing the box", look_at(vrt, (120.0, S - 184 - 2.0, world(S, 40)), (230.0, S - 184 - 2.0, world(S, 40)))))


def outer_layer(voxels):
    a = as_array(voxels).astype(np.int64)
    lo, hi = a.min(0), a.max(0)
    return as_set(a[((a == lo) | (a == hi)).any(1)])


def test_voxel_model_edits(vrt, port, textures):
    """§1: a few thousand voxels in one corner of the cube, edited step by step; after every step, three cameras (outside the
    cube, inside it but outside the model's box, grazing a face of the bounds) each render one kernel configuration, in turn."""
    cams = model_cameras(vrt)
    model = as_set(model_voxels())
    steps = [("model", set(model))]
    current = set(model)
    for side, blob in GROWTH:
        current = current | as_set(blob)
        steps.append(("grow " + side, current))
    current = current - outer_layer(current)
    steps.append(("outer layer removed", current))
    steps.append(("everything removed", set()))
    steps.append(("cube corners", {(0, 0, 0), (S - 1, S - 1, S - 1)}))
    steps.append(("model back", steps[-1][1] | model))
    c = vrt.Context(0)
    try:
        s = voxel_scene(vrt, c, DEPTH, as_array(model), textures)
        previous = set(model)
        for k, (label, voxels) in enumerate(steps):
            added, removed = voxels - previous, previous - voxels
            if removed:
                s.set_cells(as_array(removed), solid=False)
            if added:
                s.set_cells(as_array(added), solid=True)
            previous = voxels
            assert s.voxel_count() == len(voxels), label
            nodes = vrt.host_build_lsvo_from_voxels(DEPTH, as_array(voxels))
            fresh = voxel_scene(vrt, c, DEPTH, as_array(voxels), textures)
            for i, (where, cam) in enumerate(cams):
                spp, variant = KERNELS[(k + i) % 3]
                size = SIZES[(k + 2 * i) % 3]
                want = port.render(nodes, oracle_params(DEPTH, cam, size, spp), *textures)
                stats = check_frame(vrt, c, s, fresh, want, cam, size, spp, variant, "%s, camera %s" % (label, where))
                if not voxels:
                    # all sky: every sample counted, no primary hit; K6 answers every sample from the empty beam tiles
                    assert (want[0][..., 3] == spp).all() and want[2].rays[1] == 0, label
                    assert stats["culled_primary"] == (stats["rays"][0] if (spp >= 8 and variant == 0) else 0), (label, where, stats)
            fresh.close()
    finally:
        c.close()


def grown_frames_change(vrt, port, textures):
    """Every growth step of the model changes the oracle's frame of at least one camera: the new voxels are in view."""
    cams = model_cameras(vrt)
    current = as_set(model_voxels())
    before = {w: port.render(vrt.host_build_lsvo_from_voxels(DEPTH, as_array(current)), oracle_params(DEPTH, cam, (96, 54), 4), *textures)[0]
              for w, cam in cams}
    for side, blob in GROWTH:
        current = current | as_set(blob)
        nodes = vrt.host_build_lsvo_from_voxels(DEPTH, as_array(current))
        changed = 0
        for w, cam in cams:
            acc = port.render(nodes, oracle_params(DEPTH, cam, (96, 54), 4), *textures)[0]
            changed += int((acc != before[w]).any(-1).sum())
            before[w] = acc
        assert changed > 0, side


def test_growth_is_in_view(vrt, port, textures):
    """The premise of the growth steps above (CPU oracle only, run with the GPU tests that rely on it)."""
    grown_frames_change(vrt, port, textures)


# ---- §2: heightfields -----------------------------------------------------------------------------------------------------------
def heightfield_nodes(vrt, depth, heights):
    return vrt.host_build_lsvo_from_voxels(depth, _heightfield_voxels(heights))


@pytest.mark.parametrize("depth", [8, 9])
def test_heightfield_edits(vrt, port, textures, depth):
    """§2: the demo terrain as an editable heightfield.  A rectangle raised above the old maximum (the box grows upwards), a region
    flattened to the 16-voxel floor and rendered as a mirror lake, everything lowered (the box shrinks), and the compact layout
    switched on between two edits (no mirrors there, no beam floors: bounds exits only)."""
    Sd = 1 << depth
    k = Sd // 256                                                # cameras and rectangles scale with the world
    c = vrt.Context(0)
    try:
        s = vrt.LSVO.from_heightfield(c, depth)
        s.set_textures(*textures)
        heights = s.heights()
        hi = int(heights.max())
        lake_y = Sd // 2 - 16                                    # the flat floor's top layer, setCell y = S/2 + 15 (240 for T(9))
        tower = look_at(vrt, (136.0 * k, 60.0 * k, 200.0 * k), (136.0 * k, 30.0 * k, 71.0 * k))
        over = look_at(vrt, (128.0 * k, 100.0 * k, 128.0 * k), (160.0 * k, 128.0 * k, 60.0 * k), aperture=0.7, focal_length=40.0 * k)
        lake = look_at(vrt, (155.0 * k, 10.0 * k, 250.0 * k), (155.0 * k, float(lake_y), 160.0 * k))
        steps = [
            ("raised", (100 * k, 170 * k, np.full((40 * k, 30 * k), min(Sd // 2, hi + 32 * k), np.int32)), False, [tower, over]),
            ("flattened", (40 * k, 20 * k, np.full((120 * k, 150 * k), 10, np.int32)), False, [lake]),
            ("compact layout", None, True, [over]),
            ("lowered", (0, 0, np.full((Sd, Sd), 20, np.int32)), True, [over]),
            ("raised again", (70 * k, 170 * k, np.full((50 * k, 50 * k), Sd // 2, np.int32)), True, [over]),
        ]
        compact = False
        for n, (label, edit, layout, cams) in enumerate(steps):
            if edit is not None:
                x0, z0, patch = edit
                heights[x0:x0 + patch.shape[0], z0:z0 + patch.shape[1]] = patch
                s.edit_heights(x0, z0, patch)
            if layout and not compact:
                s.set_layout(1)
                compact = True
            assert np.array_equal(s.heights(), heights), label
            nodes = heightfield_nodes(vrt, depth, heights)
            fresh = vrt.LSVO.from_heightfield(c, depth, heights)
            fresh.set_textures(*textures)
            if compact:
                fresh.set_layout(1)
            for i, cam in enumerate(cams):
                spp, variant = KERNELS[(n + i) % 3]
                size = SIZES[(n + i + depth) % 3]
                mirror_y = lake_y if label == "flattened" else None
                want = port.render(nodes, oracle_params(depth, cam, size, spp, mirror_y), *textures)
                assert want[2].rays[1] > 0, label
                stats = check_frame(vrt, c, s, fresh, want, cam, size, spp, variant, "depth %d, %s, camera %d" % (depth, label, i), mirror_y)
                if mirror_y is not None:
                    assert want[2].rays[0] > size[0] * size[1] * spp, label            # reflection rays were cast
                if compact:
                    assert stats["culled_primary"] == 0, label                         # no beam floors on the compact layout
            fresh.close()
    finally:
        c.close()


# ---- §3: a painted voxel set, edited, palette frames -----------------------------------------------------------------------------
def test_painted_model_edits(vrt, port, textures):
    """§3: the model painted by position, then voxels added and removed by set_cells; palette frames with the product defaults
    against render_palette on the host-built array coloured by the numpy leaf-slot descent.  Added voxels carry colour 1."""
    pal = np.random.default_rng(5).integers(0, 256, (256, 3), dtype=np.uint8)
    pal[1] = (250, 20, 200)                                      # colour 1 (new voxels) stands out
    vox = model_voxels()
    colors = (2 + (vox[:, 0] + 3 * vox[:, 1] + 7 * vox[:, 2]) % 250).astype(np.uint8)
    colour = {tuple(v): int(col) for v, col in zip(vox.tolist(), colors)}
    cams = model_cameras(vrt)
    c = vrt.Context(0)
    try:
        s = voxel_scene(vrt, c, DEPTH, vox, textures)
        s.paint_cells(vox, colors)
        s.set_palette(pal)
        removed = box((24, 36), (160, 184), (28, 52))            # the -x half of the shell and ...
        s.set_cells(removed, solid=False)
        for v in removed.tolist():
            colour.pop(tuple(v), None)
        added = np.concatenate([GROWTH[1][1], GROWTH[3][1], box((28, 32), (170, 176), (36, 42))])
        s.set_cells(added, solid=True)
        for v in added.tolist():
            colour.setdefault(tuple(v), 1)
        assert (s.cell_colors(added) == 1).all()
        final = as_array(colour.keys())
        fc = np.uint8([colour[tuple(v)] for v in final.tolist()])
        nodes = vrt.host_build_lsvo_from_voxels(DEPTH, final)
        slots = leaf_slots(nodes, DEPTH, final)
        assert (slots >= 0).all()
        nodes["color"][slots] = fc
        fresh = voxel_scene(vrt, c, DEPTH, final, textures)
        fresh.paint_cells(final, fc)
        fresh.set_palette(pal)
        assert np.array_equal(s.download_nodes().view(np.uint64), fresh.download_nodes().view(np.uint64))
        for i, (where, cam) in enumerate(cams):
            for spp, variant in KERNELS:
                size = SIZES[i]
                want = render_palette(nodes, oracle_params(DEPTH, cam, size, spp), pal, *textures)
                check_frame(vrt, c, s, fresh, want, cam, size, spp, variant, "painted, camera %s" % where)
        # the new voxels are in view and take palette[1]: without them the oracle frame is different
        plain = nodes.copy()
        plain["color"][leaf_slots(plain, DEPTH, added)] = 2
        where, cam = cams[1]
        p = oracle_params(DEPTH, cam, SIZES[1], 4)
        assert not np.array_equal(render_palette(plain, p, pal, *textures)[0], render_palette(nodes, p, pal, *textures)[0])
        fresh.close()
    finally:
        c.close()


# ---- §4: frames enqueued before an edit ------------------------------------------------------------------------------------------
def enqueued_frames(vrt, port, textures, scene, cam, size, worlds, edits):
    """Enqueues a frame of `scene`, then for each edit: the edit (no synchronisation in between) and the next frame into a
    further accumulator; one synchronisation at the end.  Frame i must be the oracle's frame of worlds[i]."""
    import torch
    from cpuvoxelraycaster_b200.capi import check, lib, ptr
    from cpuvoxelraycaster_b200.frame import FrameRenderer
    W, H = size
    fr = FrameRenderer(scene, W, H)
    fr.use_gi, fr.gi_bounces, fr.light = True, 2, default_light(scene.depth)
    spp = 16
    p = fr.params(spp)
    with torch.cuda.stream(fr.stream):
        accums = [torch.zeros_like(fr.accum) for _ in worlds]
        rgbas = [torch.zeros_like(fr.rgba) for _ in worlds]
    cs = cam.as_struct()
    for i, acc in enumerate(accums):
        if i:
            edits[i - 1]()
        check(lib().vrt_render_accumulate_device(scene.handle, C.byref(cs), C.byref(p), ptr(acc)))
        check(lib().vrt_render_resolve_device(scene.handle, C.byref(p), ptr(acc), ptr(rgbas[i])))
    fr.stream.synchronize()
    previous = None
    for i, nodes in enumerate(worlds):
        accum, rgba, _ = port.render(nodes, oracle_params(scene.depth, cam, size, spp), *textures)
        got = accums[i].cpu().numpy().view(np.uint32)[: H * W * 4].reshape(H, W, 4)
        assert np.array_equal(got, accum), "frame %d: accumulators differ on %d pixels" % (i, int((got != accum).any(-1).sum()))
        assert np.array_equal(rgbas[i].cpu().numpy()[: H * W * 4].reshape(H, W, 4), rgba), i
        assert previous is None or not np.array_equal(previous, accum), "edit %d is not in view" % i
        previous = accum


def test_frames_enqueued_before_an_edit(vrt, port, textures):
    """§4: frames enqueued on the device path before an edit read the world they were enqueued for; two edits of a heightfield
    and three set_cells edits in a row (the replaced array is the build pool's spare, reused on alternate edits).  K6 with the
    product defaults.  Run once: this is an ordering test."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    c = vrt.Context(0)
    try:
        set_shortcuts(c, True)
        depth = 8
        hf = vrt.LSVO.from_heightfield(c, depth)
        hf.set_textures(*textures)
        heights = hf.heights()
        patches = [(90, 150, np.full((50, 40), 120, np.int32)), (60, 120, np.full((60, 50), 5, np.int32))]
        worlds = [heightfield_nodes(vrt, depth, heights)]
        for x0, z0, patch in patches:
            heights[x0:x0 + patch.shape[0], z0:z0 + patch.shape[1]] = patch
            worlds.append(heightfield_nodes(vrt, depth, heights))
        edits = [lambda e=e: hf.edit_heights(*e) for e in patches]
        cam = look_at(vrt, (128.0, 10.0, 230.0), (141.0, 100.0, 96.0))
        enqueued_frames(vrt, port, textures, hf, cam, (131, 67), worlds, edits)

        c2 = vrt.Context(0)
        try:
            set_shortcuts(c2, True)
            model = as_set(model_voxels())
            s = voxel_scene(vrt, c2, DEPTH, as_array(model), textures)
            changes = [(GROWTH[0][1], True), (box((24, 48), (160, 184), (28, 36)), False), (GROWTH[4][1], True)]
            worlds, current = [vrt.host_build_lsvo_from_voxels(DEPTH, as_array(model))], set(model)
            for vox, solid in changes:
                current = (current | as_set(vox)) if solid else (current - as_set(vox))
                worlds.append(vrt.host_build_lsvo_from_voxels(DEPTH, as_array(current)))
            edits = [lambda v=v, solid=solid: s.set_cells(v, solid) for v, solid in changes]
            enqueued_frames(vrt, port, textures, s, model_cameras(vrt)[0][1], (96, 54), worlds, edits)
            set_shortcuts(c2, False)
        finally:
            c2.close()
        set_shortcuts(c, False)
    finally:
        c.close()


# ---- §5: the sweep's corner cases ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("depth", [1, 2, 3, 4])
def test_shallow_worlds(vrt, port, textures, depth):
    """device_scene_bounds with stop_level 0 (depth <= 3: voxel-exact bounds) and 3 (depth 4): random voxel worlds in part of the
    cube, the camera outside it; frames with and without the shortcuts equal the oracle's."""
    Sd = 1 << depth
    rng = np.random.default_rng(40 + depth)
    vox = rng.integers(0, max(1, Sd - Sd // 4), (max(2, Sd ** 3 // 6), 3)).astype(np.uint32)
    vox = np.unique(vox, axis=0)
    c = vrt.Context(0)
    try:
        s = voxel_scene(vrt, c, depth, vox, textures)
        nodes = vrt.host_build_lsvo_from_voxels(depth, vox)
        for i, (position, target) in enumerate((((1.15 * Sd, 0.8 * Sd, 1.1 * Sd), (0.5 * Sd,) * 3),
                                               ((1.25 * Sd, 0.4 * Sd, 0.3 * Sd), (0.6 * Sd, 0.6 * Sd, 0.7 * Sd)))):
            cam = look_at(vrt, position, target, aperture=0.02 * Sd, focal_length=1.5 * Sd)
            for spp, variant in KERNELS:
                size = SIZES[(i + spp) % 3]
                want = port.render(nodes, oracle_params(depth, cam, size, spp), *textures)
                assert want[2].rays[1] > 0
                check_frame(vrt, c, s, s, want, cam, size, spp, variant, "depth %d, camera %d" % (depth, i))
    finally:
        c.close()


def test_bounds_queue_overflow(vrt, port, textures):
    """More occupied 16-voxel cubes than the sweep's queue holds (2^19): the cubes that do not fit are taken whole.  A depth-11
    voxel set in an off-centre sub-box, plus a 16^3 cluster beyond its +x face (setCell) that only a walk leaving the dense part can
    reach; a 32-row crop of a K6 frame from inside the sub-box, looking at the cluster, against the oracle's crop."""
    depth = 11
    Sd = 1 << depth
    rng = np.random.default_rng(2048)
    n = 1_500_000
    vox = np.stack([rng.integers(0, 1200, n), rng.integers(0, Sd, n), rng.integers(300, Sd, n)], 1)
    cluster = box((1264, 1280), (1008, 1024), (1008, 1024)).astype(np.int64)   # 48 mod 64 on every axis
    vox = np.concatenate([vox, cluster]).astype(np.uint32)
    cubes = len(np.unique((vox >> 4).astype(np.int64) @ np.int64([1 << 14, 1 << 7, 1])))
    assert cubes > 1 << 19, cubes
    size, spp, rows = (160, 90), 16, (29, 61)
    cam = look_at(vrt, (1100.0, world(Sd, 1016), world(Sd, 1016)), (world(Sd, 1272), world(Sd, 1016), world(Sd, 1016)))
    nodes = vrt.host_build_lsvo_from_voxels(depth, vox)
    want = port.render(nodes, oracle_params(depth, cam, size, spp, rows=rows), *textures)
    accum, rgba, st = want
    assert st.rays[1] > 0
    c = vrt.Context(0)
    try:
        s = voxel_scene(vrt, c, depth, vox, textures)
        on = check_frame(vrt, c, s, s, want, cam, size, spp, 0, "overflow crop", rows=rows)
        set_shortcuts(c, False)
        _, _, off = gpu_frame(vrt, s, cam, size, spp, rows=rows)
        assert all(a >= b for a, b in zip(off["complexity"], on["complexity"])) and sum(off["complexity"]) > sum(on["complexity"]), (off, on)
    finally:
        c.close()


def test_bounds_exits_shorten_walks(vrt, textures):
    """On the model of test_voxel_model_edits, bounds exits cut the loop trips of a frame: a sweep that returned the whole cube would
    pass every frame comparison above.  Loop trips are a count, not a time, so the ratio does not depend on the GPU: measured
    1449950 / 1801027 = 0.805 (on a B200 at 1000 W)."""
    vox = model_voxels()
    c = vrt.Context(0)
    try:
        s = voxel_scene(vrt, c, DEPTH, vox, textures)
        cam = model_cameras(vrt)[1][1]
        totals = []
        for bounds in (0, 1):
            c.set_option("beam_tile", 0)
            c.set_option("bounds_exit", bounds)
            _, _, st = gpu_frame(vrt, s, cam, (160, 90), 16)
            totals.append(sum(st["complexity"]))
        set_shortcuts(c, False)
        assert totals[1] < totals[0], totals
        print("bounds exits: %d / %d loop trips = %.3f" % (totals[1], totals[0], totals[1] / totals[0]))
    finally:
        c.close()
