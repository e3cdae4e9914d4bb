"""Mirror voxels in the CPU specification (tests/cell_types_oracle.c vo_render_cell_types, DESIGN.md §2 "Mirror voxels"):

| test                                  | what it pins                                                                          |
|---------------------------------------|---------------------------------------------------------------------------------------|
| test_all_solid_table_is_vo_render_palette | no table or an all-Solid one gives vo_render_palette's frame: palette on / off, lake on / off |
| test_mirror_slab_equals_the_lake      | a complete layer painted Mirror equals the lake rule on that layer (mirror_y1)        |
| test_mirror_wall_reflects_single_face_hits | walls facing x, y and z and a cube: exactly the camera rays that hit a mirror voxel on one face reflect |
| test_facing_mirrors_bind_max_bounds   | two facing mirrors: the reflections grow with max_bounds and stop at it               |
| test_edge_and_zero_normal_hits_do_not_reflect | edge hits and a camera inside a mirror voxel shade as ordinary hits          |
"""
import numpy as np
import pytest

import cell_types_scenes as cts
from cell_types_oracle import render_cell_types
from palette_oracle import render_palette

W, H = 48, 32
DEMO_VIEW = dict(position=(256.0, 200.0, 256.0), view_angle=(0.3, -0.35))


def same_frame(a, b):
    return np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and list(a[2].rays) == list(b[2].rays) and \
        list(a[2].complexity) == list(b[2].complexity)


def painted_terrain(port):
    """T(9) with its hills painted by height band (colours 2..): some of them get Mirror in the tables below."""
    nodes = port.build_terrain(9)
    parents = np.flatnonzero(nodes["leaf_mask"])
    slots = np.concatenate([p + nodes["child_offset"][p].astype(np.int64) + s
                            for s in range(8) for p in [parents[(nodes["leaf_mask"][parents] >> s) & 1 != 0]]])
    nodes["color"][slots] = (2 + slots % 7).astype(np.uint8)
    return nodes


def test_all_solid_table_is_vo_render_palette(vrt, port, textures):
    nodes = painted_terrain(port)
    cam = vrt.Camera(aperture=0.5, focal_length=60.0, **DEMO_VIEW)
    solid = np.ones(256, np.uint8)
    for palette in (None, cts.make_palette()):
        for mirror_y1 in (0, 241):
            p = cts.port_params(vrt, cam, 64, 40, depth=9, spp=2, roughness=0.05, mirror_y1=mirror_y1)
            p.light_position[:] = [float(x) for x in cts.default_light(9)]
            want = render_palette(nodes, p, palette, *textures)
            assert want[1][..., :3].max() > 0
            for types in (None, solid):
                assert same_frame(render_cell_types(nodes, p, palette, types, *textures), want), (palette is None, mirror_y1, types is None)


@pytest.mark.parametrize("palette", [False, True])
def test_mirror_slab_equals_the_lake(vrt, port, textures, palette):
    (xyz, colours), pos, angle = cts.slab_world(layer_y=40)
    nodes = cts.host_nodes(vrt, xyz, colours)
    pal = cts.make_palette() if palette else None
    types = cts.mirror_types((9,))
    cam = vrt.Camera(position=pos, view_angle=angle, aperture=0.5, focal_length=30.0)
    for roughness, bounces in ((0.0, 1), (0.3, 2)):
        p = cts.port_params(vrt, cam, W, H, spp=3, roughness=roughness, bounces=bounces)
        got = render_cell_types(nodes, p, pal, types, *textures)
        p.mirror_y1 = 41                                      # castRay y of the layer + 1
        want = render_palette(nodes, p, pal, *textures)
        assert want[2].rays[0] > W * H * 3 + 500                # the lake reflects
        assert same_frame(got, want), roughness


@pytest.mark.parametrize("name", ["wall_x", "wall_y", "wall_z", "cube"])
def test_mirror_wall_reflects_single_face_hits(vrt, port, textures, name):
    (xyz, colours), pos, angle = cts.world(name)
    nodes = cts.host_nodes(vrt, xyz, colours)
    cam = vrt.Camera(position=pos, view_angle=angle, aperture=0.0, focal_length=60.0)
    p = cts.port_params(vrt, cam, W, H, use_gi=False, max_bounds=1)
    o, d = cts.camera_rays(port, p)
    hits = port.lsvo_cast(nodes, cts.DEPTH, o, d)
    single = np.isin(cts.hit_colours(nodes, hits), cts.MIRROR_COLOURS) & ((hits["normal"] != 0).sum(1) == 1)
    assert single.sum() > 100
    axis = {"wall_x": 0, "wall_y": 1, "wall_z": 2}.get(name)
    if axis is not None:                                        # the wall is hit on the face it shows
        assert (hits["normal"][single][:, axis] != 0).all()
    else:                                                       # the cube is hit on three faces
        assert ((hits["normal"][single] != 0).sum(0) > 0).all()
    plain = render_palette(nodes, p, None, *textures)
    got = render_cell_types(nodes, p, None, cts.mirror_types(), *textures)
    assert got[2].rays[0] == W * H + int(single.sum())        # one reflection per single-face mirror hit, none else
    assert not np.array_equal(got[1], plain[1])
    p.max_bounds = 0                                            # nothing reflects
    assert same_frame(render_cell_types(nodes, p, None, cts.mirror_types(), *textures), render_palette(nodes, p, None, *textures))


def test_facing_mirrors_bind_max_bounds(vrt, port, textures):
    (xyz, colours), pos, angle = cts.world("facing")
    nodes = cts.host_nodes(vrt, xyz, colours)
    cam = vrt.Camera(position=pos, view_angle=angle, aperture=0.0, focal_length=60.0)
    rays, frames = [], []
    for max_bounds in (0, 1, 4, 16):
        p = cts.port_params(vrt, cam, W, H, use_gi=False, max_bounds=max_bounds)
        accum, rgba, st = render_cell_types(nodes, p, None, cts.mirror_types(), *textures)
        rays.append(st.rays[0] - W * H)
        frames.append(rgba)
        assert rays[-1] <= max_bounds * W * H
    assert rays[0] == 0 and rays[1] > 0.8 * W * H and rays[1] < rays[2] < rays[3]   # rays[3] > rays[2]: bounces beyond 4
    assert all(not np.array_equal(a, b) for a, b in zip(frames, frames[1:]))


def test_edge_and_zero_normal_hits_do_not_reflect(vrt, port, textures):
    for make in (cts.edge_world, cts.inside_world):
        (xyz, colours), pos, angle = make()
        nodes = cts.host_nodes(vrt, xyz, colours)
        cam = vrt.Camera(position=pos, view_angle=angle, aperture=0.0, focal_length=60.0)
        p = cts.port_params(vrt, cam, W, H, use_gi=True, bounces=2, max_bounds=4)
        o, d = cts.camera_rays(port, p)
        hits = port.lsvo_cast(nodes, cts.DEPTH, o, d)
        mirror = np.isin(cts.hit_colours(nodes, hits), cts.MIRROR_COLOURS)
        faces = (hits["normal"] != 0).sum(1)
        other = mirror & (faces != 1)
        assert other.sum() > 10, make.__name__                  # edge hits (2 faces) or zero normals (camera inside)
        assert (faces[other] == (0 if make is cts.inside_world else 2)).all()
        got = render_cell_types(nodes, p, None, cts.mirror_types(), *textures)
        assert got[2].rays[0] == W * H + int((mirror & (faces == 1)).sum())
        if make is cts.inside_world:                            # every camera ray starts inside the mirror cube
            assert other.all()
            assert same_frame(got, render_palette(nodes, p, None, *textures))
