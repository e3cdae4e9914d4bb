"""Mirror voxels: what a cell-type table costs a frame.

On T(9) painted by height band with a palette, three arms of the same frame:
  - palette: the palette frame without mirrors;
  - lake:    the lake rule on the valley layer (mirror_y = 240, castRay y);
  - mirror:  no lake; the same valley layer painted with colour 250, whose cell type is Cell::Mirror.
Frames: the 1080p, 64-spp GI (2 bounces) + DOF frame (K6) and the 720p 1-spp interactive frame (K4, GI 1 bounce).  The mirror arm
descends the node array once per camera-chain hit (the palette and lake arms once per sample), and the lake and mirror arms
reflect.

Frame times are device events around the frame kernels (context option "time_frame_kernels"), with the product defaults (beam
floors, bounds exits).  Every shape is warmed up first; the arms alternate, REPEATS times each.  The node array of T(9) (84 MB)
fits the 126 MB L2: the frames are measured with it cached, as a renderer drawing frame after frame sees it.
Prints one JSON line per measurement, the first naming the card and its power limit."""
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import cpuvoxelraycaster_b200 as vrt  # noqa: E402
from probe_palette import ROOT, band_colors, card, palette, terrain_voxels  # noqa: E402

REPEATS = 7
LAKE_Y = 240                         # castRay y of the valley layer (setCell y = 511 - 240)
MIRROR_COLOUR = 250


def frames(ctx, scene, size, spp, bounces, aperture):
    tex = np.load(os.path.join(ROOT, "tests", "golden", "textures.npz"))
    scene.set_textures(tex["top"], tex["side"])
    scene.set_palette(palette())
    cam = vrt.Camera(position=(256, 200, 256), view_angle=(0.3, -0.35), aperture=aperture, focal_length=60.0)
    rc = vrt.RayCaster(scene, size)
    rc.setLightPosition(np.float32([-200, -1000, -300]) * np.float32(1 / 512.0) + np.float32(1))
    rc.use_samples, rc.use_gi, rc.gi_bounces = True, True, bounces
    types = np.ones(256, np.uint8)
    types[MIRROR_COLOUR] = 2
    ctx.set_option("time_frame_kernels", 1)
    arms = ("palette", "lake", "mirror")
    t = {a: [] for a in arms}
    rays = {}
    for k in range(2 + REPEATS):
        for arm in arms:
            rc.mirror_y = LAKE_Y if arm == "lake" else None
            scene.set_cell_types(types if arm == "mirror" else None)
            rc.resetSamples()
            rc.render(cam, spp)
            ms = sum(ctx.take_kernel_timings())
            rays[arm] = rc.last_stats["rays"][0]
            if k >= 2:
                t[arm].append(ms)
    ctx.set_option("time_frame_kernels", 0)
    scene.set_cell_types(None)
    out = dict(frame="%dx%d, %d spp, GI %d bounces, aperture %g" % (size[0], size[1], spp, bounces, aperture), repeats=REPEATS)
    for arm, v in t.items():
        v = np.asarray(v)
        out[arm] = dict(median_ms=round(float(np.median(v)), 3), min_ms=round(float(v.min()), 3), max_ms=round(float(v.max()), 3),
                        primary_rays=int(rays[arm]))
    for arm in ("lake", "mirror"):
        out[arm + "_over_palette"] = round(out[arm]["median_ms"] / out["palette"]["median_ms"], 4)
    out["mirror_over_lake"] = round(out["mirror"]["median_ms"] / out["lake"]["median_ms"], 4)
    return out


def main():
    print(json.dumps(card()), flush=True)
    ctx = vrt.Context(0)
    vox = terrain_voxels()
    colors = band_colors(vox)
    layer = vox[:, 1] == 511 - LAKE_Y
    colors[layer] = MIRROR_COLOUR
    scene = vrt.LSVO.from_terrain(ctx, 9)
    painted = scene.paint_cells(vox, colors)
    print(json.dumps(dict(scene="T(9) painted by height band, valley layer colour %d" % MIRROR_COLOUR, voxels=len(vox), painted=painted,
                          layer_voxels=int(layer.sum()))), flush=True)
    print(json.dumps(frames(ctx, scene, (1920, 1080), 64, 2, 0.5)), flush=True)
    print(json.dumps(frames(ctx, scene, (1280, 720), 1, 1, 0.0)), flush=True)
    scene.close()
    ctx.close()


if __name__ == "__main__":
    main()
