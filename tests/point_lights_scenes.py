"""TEST INFRASTRUCTURE ONLY: small hand-made worlds lit by point lights (DESIGN.md §2, "Point lights"), shared by
tests/test_oracle_point_lights.py (CPU) and tests/test_gpu_point_lights.py.

Worlds are written in castRay voxel coordinates like tests/cell_types_scenes.py (small y is up) on a floor at y >= 56.  Their
sun sits below the floor: it lights no top face, so what lights the floor is the point lights alone.  light_terms restates
the rule in numpy on the oracle's own casts, for the known-answer tests."""
import numpy as np

import cell_types_scenes as cts

S = cts.S
NIGHT_SUN = np.float32([1.5, 3.0, 1.5])           # below the floor: dot(to_sun, top-face normal) < 0


def at(v):
    """castRay voxel coordinates (may be fractional) -> the normalised castRay frame."""
    return np.float32(1.0) + np.asarray(v, np.float32) / np.float32(S)


# name -> (parts, camera position, view angle)
def world(name):
    floor = (cts.box(0, S, 56, S, 0, S), 3)
    if name == "floor":
        return cts._world([floor]), (31.0, 8.0, 4.0), (0.0, -0.9)
    if name == "wall":               # a wall across the floor at x = 30..31; the camera sees the floor on both sides
        return cts._world([floor, (cts.box(30, 32, 20, 56, 0, S), 4)]), (31.0, 8.0, 4.0), (0.0, -0.9)
    if name == "overhang":           # a slab at y = 20..23 over the floor's z < 44; the camera looks in between
        return cts._world([floor, (cts.box(0, S, 20, 24, 0, 44), 4)]), (32.0, 40.0, 60.0), (3.14159, -0.5)
    if name == "room":               # the wall world with props: lights are culled, shadowed and lit in one frame
        return cts._world([floor, (cts.box(30, 32, 20, 56, 0, S), 4)] + cts._props()), (31.0, 8.0, 4.0), (0.0, -0.9)
    raise KeyError(name)


def lights(positions, colors, ranges):
    """A LIGHT_DTYPE array from castRay voxel positions."""
    from point_lights_oracle import pack_lights
    return pack_lights(at(positions), colors, ranges)


def room_lights(n):
    """n lights (1..16) for the room world: in range, out of range (culled), below the floor (back-facing) and on both sides of
    the wall, with colours that differ per channel."""
    rng = np.random.default_rng(n)
    pos = np.column_stack([rng.uniform(2, 62, n), rng.uniform(30, 54, n), rng.uniform(2, 62, n)])
    pos[3::5, 1] = 70.0                                        # below the floor: back-facing for every top face
    col = rng.uniform(0.0, 1.5, (n, 3))
    rng_ = rng.uniform(6, 40, n) / S
    rng_[1::4] = 0.5 / S                                       # culled everywhere but right next to the light
    rng_[2::6] = np.inf
    return lights(pos, col, rng_)


def light_terms(port, nodes, p, lts, depth=cts.DEPTH):
    """The rule at the camera rays' first hits (sample p.sample_offset, one per pixel), in numpy fp32 op for op:
    returns the camera hits, and per light the cast and occluded masks and the added light [N, 3]."""
    o, d = cts.camera_rays(port, p)
    h = port.lsvo_cast(nodes, depth, o, d)
    hit = h["hit"] != 0
    n = h["normal"].astype(np.float32)
    hp = h["position"] + (n * np.float32(1.0 / (1 << depth))) * np.float32(0.001)
    out = []
    for li in lts:
        v = li["position"].astype(np.float32) - hp
        ss = (v[:, 0] * v[:, 0] + v[:, 1] * v[:, 1]) + v[:, 2] * v[:, 2]
        dist = np.sqrt(ss)
        tl = v * (np.float32(1.0) / np.sqrt(ss))[:, None]
        ndotl = (tl[:, 0] * n[:, 0] + tl[:, 1] * n[:, 1]) + tl[:, 2] * n[:, 2]
        with np.errstate(invalid="ignore"):
            cast = hit & (dist < li["range"]) & (ndotl > 0)
        occ = np.zeros(len(hit), bool)
        if cast.any():
            sh = port.lsvo_cast(nodes, depth, hp[cast], tl[cast])
            occ[cast] = (sh["hit"] != 0) & (sh["distance"] < dist[cast])
        w = np.float32(1.0) - dist / li["range"]
        add = (li["color"].astype(np.float32)[None, :] * ndotl[:, None]) * w[:, None]
        out.append(dict(cast=cast, occluded=occ, add=np.where((cast & ~occ)[:, None], add, np.float32(0))))
    return h, out


def predicted_rgb(albedo, per_light):
    """rgb of the rule with no sun, GI off and tint 1: L_c = the lights' adds in index order, f_c = min(1, max(0, L_c)),
    mult(mult(albedo_c, f_c), 1).  albedo uint8 [N, 3]."""
    L = np.zeros((len(albedo), 3), np.float32)
    for t in per_light:
        L = L + t["add"]
    f = np.minimum(np.float32(1), np.maximum(np.float32(0), L + np.float32(0)))
    mul = lambda c, x: np.minimum(np.float32(255), c.astype(np.float32) * x).astype(np.uint8)   # noqa: E731
    return mul(mul(albedo, f), np.float32(1))
