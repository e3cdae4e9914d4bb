"""Per-voxel colours in the CPU specification (tests/palette_oracle.c vo_render_palette, DESIGN.md §2): without a palette it is
vo_render, and a scene painted in one colour with a one-colour palette renders like vo_render with uniform textures of that
colour."""
import numpy as np

from palette_oracle import render_palette

DEMO_VIEW = dict(position=(256.0, 200.0, 256.0), view_angle=(0.3, -0.35))


def params(vrt, W=64, H=40, spp=2, mirror_y1=241):
    from oracle import loader
    cam = vrt.Camera(aperture=0.5, focal_length=60.0, **DEMO_VIEW)
    p = loader.PortRenderParams()
    p.width, p.height, p.depth, p.guard = W, H, 9, 9
    p.cam_position[:] = [float(x) for x in cam.position]
    p.rot_mat[:] = [float(x) for x in cam.rot_mat]
    p.fov, p.aperture, p.focal_length = cam.fov, cam.aperture, cam.focal_length
    p.light_position[:] = [float(x) for x in np.float32([-200, -1000, -300]) * np.float32(1 / 512.0) + np.float32(1)]
    p.use_gi, p.gi_bounces, p.use_samples, p.spp = 1, 2, 1, spp
    p.seed_lo, p.seed_hi, p.threads = 0x5EED, 0, 8
    p.roughness, p.max_bounds, p.mirror_y1 = 0.05, 4, mirror_y1
    return p


def leaf_slots(nodes):
    """Every leaf slot of a reference-layout array: parent + child_offset + s for each leaf bit s."""
    parents = np.flatnonzero(nodes["leaf_mask"])
    out = [parents[(nodes["leaf_mask"][parents] >> s) & 1 != 0] for s in range(8)]
    return np.concatenate([p + nodes["child_offset"][p].astype(np.int64) + s for s, p in enumerate(out)])


def same_frame(a, b):
    return np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and list(a[2].rays) == list(b[2].rays) and \
        list(a[2].complexity) == list(b[2].complexity)


def test_no_palette_is_vo_render(vrt, port, textures):
    nodes = port.build_terrain(9)
    nodes["color"][leaf_slots(nodes)[::3]] = 77            # colours are not read without a palette
    p = params(vrt)
    want = port.render(nodes, p, *textures)
    got = render_palette(nodes, p, None, *textures)
    assert want[1][..., :3].max() > 0
    assert same_frame(got, want)


def test_one_colour_equals_uniform_textures(vrt, port, textures):
    nodes = port.build_terrain(9)
    slots = leaf_slots(nodes)
    assert len(slots) > 1000000 and not nodes["child_mask"][slots].any()
    nodes["color"][slots] = 200
    rgb = np.uint8([180, 120, 40])
    palette = np.zeros((256, 3), np.uint8)
    palette[200] = rgb                                     # every other entry black: a wrong slot shows
    uniform = np.broadcast_to(rgb, (256, 3)).copy()
    for mirror_y1 in (0, 241):
        p = params(vrt, mirror_y1=mirror_y1)
        want = port.render(nodes, p, uniform, uniform)
        got = render_palette(nodes, p, palette, *textures)
        assert want[1][..., :3].max() > 0 and want[2].rays[2] > 0
        assert same_frame(got, want), "mirror_y1 %d" % mirror_y1
        if mirror_y1:
            assert want[2].rays[0] > p.width * p.height * p.spp    # reflections happened
