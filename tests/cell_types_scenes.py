"""TEST INFRASTRUCTURE ONLY: small hand-made worlds with mirror voxels (DESIGN.md §2, "Mirror voxels"), shared by
tests/test_oracle_cell_types.py (CPU) and tests/test_gpu_cell_types.py.

Worlds are written in castRay voxel coordinates (the frame cameras and the lake rule use: small y is up, where the default
light is) and handed to the builders in SVO::setCell coordinates, v -> S-1-v on every axis."""
import numpy as np

DEPTH = 6
S = 1 << DEPTH
FLOOR_Y = 56
SOLID, MIRROR = 1, 2
MIRROR_COLOURS = (9, 10)             # colours given Cell::Mirror by mirror_types()


def default_light(depth=DEPTH):
    return np.float32([-200, -1000, -300]) * np.float32(1.0 / (1 << depth)) + np.float32(1.0)


def box(x0, x1, y0, y1, z0, z1):
    """Voxels of [x0,x1) x [y0,y1) x [z0,z1), castRay coordinates."""
    g = np.mgrid[x0:x1, y0:y1, z0:z1].reshape(3, -1).T
    return g.astype(np.int64)


def to_set_cell(xyz, depth=DEPTH):
    return ((1 << depth) - 1 - np.asarray(xyz, np.int64)).astype(np.uint32)


def _world(parts):
    """parts: [(voxels, colour)], later parts win.  Returns (setCell xyz uint32 [N,3], colours uint8 [N])."""
    grid = np.zeros((S, S, S), np.int16)
    for vox, colour in parts:
        grid[vox[:, 0], vox[:, 1], vox[:, 2]] = colour
    xyz = np.argwhere(grid > 0)
    return to_set_cell(xyz), grid[xyz[:, 0], xyz[:, 1], xyz[:, 2]].astype(np.uint8)


def _floor(colour=3):
    return box(0, S, FLOOR_Y, S, 0, S), colour


def _props():
    """A pillar, a block and a step of colours 4..6 on the floor."""
    return [(box(20, 25, 30, FLOOR_Y, 30, 35), 4), (box(36, 44, 46, FLOOR_Y, 14, 22), 5), (box(8, 30, 52, FLOOR_Y, 44, 52), 6)]


# name -> (parts, camera position, view angle).  Every camera sees its mirrors; the tests check that reflections happen.
def world(name):
    if name == "wall_x":             # a mirror wall facing -x
        parts = [_floor()] + _props() + [(box(50, 53, 18, FLOOR_Y, 6, 58), 9)]
        return _world(parts), (14.0, 30.0, 8.0), (0.9, -0.3)
    if name == "wall_z":             # a mirror wall facing -z
        parts = [_floor()] + _props() + [(box(6, 58, 18, FLOOR_Y, 54, 57), 9)]
        return _world(parts), (30.0, 30.0, 6.0), (0.3, -0.3)
    if name == "wall_y":             # a mirror pool in the floor, facing up (-y)
        parts = [_floor()] + _props() + [(box(10, 50, FLOOR_Y, FLOOR_Y + 2, 24, 58), 10)]
        return _world(parts), (30.0, 24.0, 6.0), (0.1, -0.5)
    if name == "cube":               # a mirror cube on the floor, seen on three faces
        parts = [_floor()] + _props() + [(box(28, 40, 42, FLOOR_Y, 30, 42), 9)]
        return _world(parts), (10.0, 30.0, 10.0), (0.75, -0.45)
    if name == "facing":             # two facing mirror walls: rays bounce between them until max_bounds binds
        parts = [_floor()] + _props() + [(box(2, 5, 10, FLOOR_Y, 0, S), 9), (box(58, 61, 10, FLOOR_Y, 0, S), 10)]
        return _world(parts), (30.0, 36.0, 3.0), (1.25, -0.05)
    raise KeyError(name)


WORLDS = ("wall_x", "wall_y", "wall_z", "cube", "facing")


def slab_world(layer_y=40, seed=5):
    """One complete horizontal layer (castRay y = layer_y, colour 9) with hills and pillars (colours 2..8) standing on it,
    nothing below it.  Returns ((setCell xyz, colours), camera position, view angle)."""
    rng = np.random.default_rng(seed)
    parts = [(box(0, S, layer_y, layer_y + 1, 0, S), 9)]
    for _ in range(14):
        x, z = rng.integers(0, S - 8, 2)
        w, d, h = rng.integers(2, 9, 3)
        parts.append((box(x, x + w, layer_y - h, layer_y, z, z + d), int(rng.integers(2, 9))))
    parts.append((box(30, 33, layer_y - 22, layer_y, 30, 33), 7))
    return _world(parts), (32.0, 8.0, 4.0), (0.2, -0.7)


def edge_world():
    """Mirror voxels filling x < 32 and y < 32 (castRay coordinates) over all z, seen from (40.5, 40.5, 2.5) with an
    identity rotation: in a square frame the camera rays of the diagonal pixels have equal x and y components and start at
    equal x and y, so they cross each x plane with the y plane of the same index at the same parameter and hit the block on
    an edge (normal with an x and a y component).  Plus a floor at y >= 56 (colour 3)."""
    parts = [_floor(), (box(0, 32, 0, 32, 0, S), 9)]
    return _world(parts), (40.5, 40.5, 2.5), (0.0, 0.0)


def inside_world():
    """The camera sits inside a mirror cube: every camera ray starts inside a solid and hits it with a zero normal."""
    parts = [_floor(), (box(20, 40, 20, 40, 20, 40), 10)]
    return _world(parts), (30.5, 30.5, 30.5), (0.3, -0.2)


def mirror_types(colours=MIRROR_COLOURS):
    t = np.full(256, SOLID, np.uint8)
    t[list(colours)] = MIRROR
    return t


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
        live &= ((nd["child_mask"].astype(np.int64) >> slot) & 1) != 0
        child = node + nd["child_offset"].astype(np.int64) + slot
        leaf = live & (((nd["leaf_mask"].astype(np.int64) >> slot) & 1) != 0) & (out < 0)
        out[leaf] = child[leaf]
        node = np.where(live & (out < 0), child, 0)
    return out


def host_nodes(vrt, xyz, colours, depth=DEPTH):
    """The painted reference array of a world, built on the host."""
    nodes = vrt.host_build_lsvo_from_voxels(depth, xyz)
    slots = leaf_slots(nodes, depth, xyz)
    assert (slots >= 0).all()
    nodes["color"][slots] = colours
    return nodes


def hit_colours(nodes, hits, depth=DEPTH):
    """Colour of the voxel of each oracle hit record (castRay voxel -> setCell), -1 for misses."""
    slots = leaf_slots(nodes, depth, to_set_cell(np.clip(hits["voxel"], 0, (1 << depth) - 1), depth))
    out = np.where(slots >= 0, nodes["color"][np.maximum(slots, 0)].astype(np.int64), -1)
    return np.where(hits["hit"] != 0, out, -1)


def port_params(vrt, cam, W, H, depth=DEPTH, use_gi=True, bounces=2, use_samples=True, spp=1, offset=0, roughness=0.0,
                max_bounds=4, mirror_y1=0, guard=None):
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
    p.roughness, p.max_bounds, p.mirror_y1 = roughness, max_bounds, mirror_y1
    return p


def camera_rays(port, p):
    """The oracle's camera rays of sample p.sample_offset, row-major."""
    rays = [port.camera_ray(p, x, y, p.sample_offset) for y in range(p.height) for x in range(p.width)]
    return np.float32([o for o, _ in rays]), np.float32([d for _, d in rays])
