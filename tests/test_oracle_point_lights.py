"""Point lights in the CPU specification (tests/point_lights_oracle.c vo_render_point_lights, DESIGN.md §2 "Point lights"):

| test                                  | what it pins                                                                          |
|---------------------------------------|---------------------------------------------------------------------------------------|
| test_no_lights_is_vo_render_cell_types | no lights give vo_render_cell_types's frame: palette, cell types and the lake on / off, GI 0/1/2 |
| test_culled_lights_change_nothing     | 16 lights all out of range, or all below a floor, give the same frame and ray counts  |
| test_wall_shadows_the_floor_behind_it | the floor behind a wall is shadowed, the floor in front lit as the rule computes      |
| test_overhang_beyond_the_light_does_not_shadow | shadow rays that hit an overhang beyond the light leave the floor lit       |
| test_light_below_the_floor_casts_nothing | no ray for top-face hits of a light below them                                     |
| test_range_cuts_off                   | exactly the hits within range cast a ray and get light, weighted 1 - dist / range     |
| test_room_lights                      | 1, 4 and 16 lights in range, culled, behind a wall and below the floor: the floor is what the rule computes |
"""
import numpy as np
import pytest

import cell_types_scenes as cts
import point_lights_scenes as pls
from cell_types_oracle import render_cell_types
from point_lights_oracle import pack_lights, render_point_lights

W, H = 48, 32
DEMO_VIEW = dict(position=(256.0, 200.0, 256.0), view_angle=(0.3, -0.35))


def same_frame(a, b):
    return np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and list(a[2].rays) == list(b[2].rays) and \
        list(a[2].complexity) == list(b[2].complexity)


def painted_terrain(port):
    nodes = port.build_terrain(9)
    parents = np.flatnonzero(nodes["leaf_mask"])
    slots = np.concatenate([p + nodes["child_offset"][p].astype(np.int64) + s
                            for s in range(8) for p in [parents[(nodes["leaf_mask"][parents] >> s) & 1 != 0]]])
    nodes["color"][slots] = (2 + slots % 7).astype(np.uint8)
    return nodes


def night_params(vrt, cam, **kw):
    p = cts.port_params(vrt, cam, W, H, use_gi=False, **kw)
    p.light_position[:] = [float(x) for x in pls.NIGHT_SUN]
    return p


def scene(vrt, name):
    (xyz, colours), pos, angle = pls.world(name)
    nodes = cts.host_nodes(vrt, xyz, colours)
    return nodes, vrt.Camera(position=pos, view_angle=angle, aperture=0.0, focal_length=60.0)


def test_no_lights_is_vo_render_cell_types(vrt, port, textures):
    nodes = painted_terrain(port)
    cam = vrt.Camera(aperture=0.5, focal_length=60.0, **DEMO_VIEW)
    types = cts.mirror_types((4, 5))
    for palette, ty, mirror_y1 in ((None, None, 0), (cts.make_palette(), None, 241), (cts.make_palette(), types, 241), (None, types, 0)):
        for use_gi, bounces in ((False, 1), (True, 1), (True, 2)):
            p = cts.port_params(vrt, cam, 64, 40, depth=9, spp=2, use_gi=use_gi, bounces=bounces, roughness=0.05, mirror_y1=mirror_y1)
            p.light_position[:] = [float(x) for x in cts.default_light(9)]
            want = render_cell_types(nodes, p, palette, ty, *textures)
            assert want[1][..., :3].max() > 0
            for lts in (None, pls.lights(np.zeros((0, 3)), np.zeros((0, 3)), np.zeros(0))):
                assert same_frame(render_point_lights(nodes, p, palette, ty, lts, *textures), want), (palette is None, ty is None, use_gi)


def test_culled_lights_change_nothing(vrt, port, textures):
    nodes = painted_terrain(port)
    cam = vrt.Camera(aperture=0.5, focal_length=60.0, **DEMO_VIEW)
    p = cts.port_params(vrt, cam, 64, 40, depth=9, spp=2, use_gi=True, bounces=2, mirror_y1=241)
    p.light_position[:] = [float(x) for x in cts.default_light(9)]
    want = render_cell_types(nodes, p, cts.make_palette(), None, *textures)
    rng = np.random.default_rng(3)
    far = pack_lights(rng.uniform(1.0, 2.0, (16, 3)) + np.float32([0, -3.0, 0]), rng.uniform(0, 2, (16, 3)), np.full(16, 0.5))
    assert same_frame(render_point_lights(nodes, p, cts.make_palette(), None, far, *textures), want)
    # a flat floor lit from below: every hit is a top face, every light back-facing
    nodes, cam = scene(vrt, "floor")
    p = night_params(vrt, cam)
    want = render_cell_types(nodes, p, cts.make_palette(), None, *textures)
    below = pls.lights(np.column_stack([np.linspace(2, 60, 16), np.full(16, 70.0), np.linspace(60, 2, 16)]), np.ones((16, 3)),
                       np.full(16, np.inf))
    assert same_frame(render_point_lights(nodes, p, cts.make_palette(), None, below, *textures), want)


def known_answer(vrt, port, textures, name, lts):
    nodes, cam = scene(vrt, name)
    p = night_params(vrt, cam)
    pal = cts.make_palette()
    accum, rgba, st = render_point_lights(nodes, p, pal, None, lts, *textures)
    dark = render_cell_types(nodes, p, pal, None, *textures)
    h, terms = pls.light_terms(port, nodes, p, lts)
    colours = cts.hit_colours(nodes, h)
    got = rgba[..., :3].reshape(-1, 3)
    want = pls.predicted_rgb(pal[np.maximum(colours, 0)], terms)
    top = (h["hit"] != 0) & (h["normal"][:, 1] != 0) & (h["normal"][:, 0] == 0) & (h["normal"][:, 2] == 0) & (h["voxel"][:, 1] == 56)
    assert np.array_equal(got[top], want[top])                  # the floor: no sun, no GI, only the lights
    assert np.array_equal(dark[1][..., :3].reshape(-1, 3)[top], 0 * want[top])
    assert st.rays[1] == dark[2].rays[1] + sum(int(t["cast"].sum()) for t in terms)
    return nodes, h, terms, top, got


def test_wall_shadows_the_floor_behind_it(vrt, port, textures):
    lts = pls.lights([[20.5, 44.5, 32.5]], [[1.0, 0.6, 0.3]], [np.inf])
    nodes, h, (t,), top, got = known_answer(vrt, port, textures, "wall", lts)
    front, behind = top & (h["voxel"][:, 0] < 30), top & (h["voxel"][:, 0] >= 32)
    assert front.sum() > 100 and behind.sum() > 100
    assert t["cast"][front | behind].all()                      # every floor hit faces the light and is in range
    assert t["occluded"][behind].all() and not t["occluded"][front].any()
    assert (got[behind] == 0).all() and (got[front][:, 0] > 0).all()


def test_overhang_beyond_the_light_does_not_shadow(vrt, port, textures):
    lts = pls.lights([[32.5, 28.5, 20.5]], [[0.8, 0.8, 1.2]], [np.inf])
    nodes, h, (t,), top, got = known_answer(vrt, port, textures, "overhang", lts)
    under = top & (h["voxel"][:, 2] < 40)
    assert under.sum() > 100 and t["cast"][under].all() and not t["occluded"][under].any()
    # the shadow rays of the floor under the overhang do hit it — beyond the light
    hp = h["position"][under] + (h["normal"][under] * np.float32(1 / 64)) * np.float32(0.001)
    v = lts[0]["position"] - hp
    sh = port.lsvo_cast(nodes, cts.DEPTH, hp, v / np.linalg.norm(v, axis=1, keepdims=True))
    assert (sh["hit"] != 0).mean() > 0.9
    assert (got[under].astype(int).sum(1) > 0).all()


def test_light_below_the_floor_casts_nothing(vrt, port, textures):
    lts = pls.lights([[32.5, 60.5, 32.5], [10.5, 80.0, 40.5]], [[1.0, 1.0, 1.0], [2.0, 0.0, 1.0]], [np.inf, 1.0])
    nodes, h, terms, top, got = known_answer(vrt, port, textures, "floor", lts)
    assert top.sum() > 500 and top.sum() == (h["hit"] != 0).sum()
    assert not any(t["cast"].any() for t in terms)
    assert (got[top] == 0).all()


def test_range_cuts_off(vrt, port, textures):
    r = np.float32(12.0 / 64)
    lts = pls.lights([[32.5, 50.5, 30.5]], [[1.5, 1.0, 0.5]], [r])
    nodes, h, (t,), top, got = known_answer(vrt, port, textures, "floor", lts)
    v = lts[0]["position"] - (h["position"] + (h["normal"] * np.float32(1 / 64)) * np.float32(0.001))
    dist = np.sqrt((v[:, 0] * v[:, 0] + v[:, 1] * v[:, 1]) + v[:, 2] * v[:, 2])
    inside = top & (dist < r)
    assert 50 < inside.sum() < top.sum() - 50
    assert np.array_equal(t["cast"], inside) and not t["occluded"].any()
    assert (got[top & ~inside] == 0).all() and (got[inside].astype(int).sum(1) > 0).mean() > 0.9


@pytest.mark.parametrize("n", [1, 4, 16])
def test_room_lights(vrt, port, textures, n):
    """Lights in and out of range, in front of and behind the wall, below the floor: the floor is what the rule computes."""
    lts = pls.room_lights(n)
    nodes, h, terms, top, got = known_answer(vrt, port, textures, "room", lts)
    casts = sum(int(t["cast"].sum()) for t in terms)
    if n > 1:
        assert casts > 0 and any(t["occluded"].any() for t in terms)
        assert any((~t["cast"] & top).any() for t in terms)
