"""Per-voxel colours: what a palette costs a frame, what painting and a painted scene's edits cost.

  - the 1080p, 64-spp GI (2 bounces) + DOF frame on T(9) painted by height band (K6), palette against textures;
  - the 720p 1-spp interactive frame (K4, GI 1 bounce), palette against textures;
  - vrt_scene_paint_cells of the T(9) terrain as an 8.6 M voxel list (host list in, synchronised), voxels/s;
  - vrt_scene_set_cells of 1 000 voxels at 512^3 on a painted scene against an unpainted one.

Frame times are device events around the frame kernels (context option "time_frame_kernels"), with the product defaults (beam
floors, bounds exits).  Every shape is warmed up first; the two arms alternate, REPEATS times each.  The node array of T(9)
(84 MB) fits the 126 MB L2: the frames are measured with it cached, as a renderer drawing frame after frame sees it.
Prints one JSON line per measurement, the first naming the card and its power limit."""
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import cpuvoxelraycaster_b200 as vrt  # noqa: E402

REPEATS = 7
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return dict(device=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip())


def terrain_voxels(S=512):
    """T(9) as a plain voxel list (setCell coordinates), as tools/probe_edit.py builds it."""
    h = vrt.host_terrain_heights(S)
    hmax = np.maximum(16, np.minimum(S, h)).astype(np.int64)
    xs, zs = np.meshgrid(np.arange(S), np.arange(S), indexing="ij")
    cols = np.repeat(np.stack([xs.reshape(-1), zs.reshape(-1)], 1), hmax.reshape(-1) - 1, axis=0)
    ys = np.concatenate([np.arange(1, m) for m in hmax.reshape(-1)]) + S // 2
    return np.stack([cols[:, 0], ys, cols[:, 1]], 1).astype(np.uint32)


def band_colors(vox, S=512):
    return (2 + (vox[:, 1].astype(np.int64) - S // 2) // 8).astype(np.uint8)


def palette():
    c = np.arange(256)
    return np.stack([(c * 37) % 256, (c * 91 + 40) % 256, (c * 53 + 90) % 256], -1).astype(np.uint8)


def frame_ms(ctx, rc, cam, spp):
    rc.resetSamples()
    rc.render(cam, spp)
    return sum(ctx.take_kernel_timings())


def frames(ctx, scene, size, spp, bounces, aperture):
    tex = np.load(os.path.join(ROOT, "tests", "golden", "textures.npz"))
    scene.set_textures(tex["top"], tex["side"])
    cam = vrt.Camera(position=(256, 200, 256), view_angle=(0.3, -0.35), aperture=aperture, focal_length=60.0)
    rc = vrt.RayCaster(scene, size)
    rc.setLightPosition(np.float32([-200, -1000, -300]) * np.float32(1 / 512.0) + np.float32(1))
    rc.use_samples, rc.use_gi, rc.gi_bounces = True, True, bounces
    ctx.set_option("time_frame_kernels", 1)
    t = {"textures": [], "palette": []}
    for k in range(2 + REPEATS):
        for arm in ("textures", "palette"):
            scene.set_palette(palette() if arm == "palette" else None)
            ms = frame_ms(ctx, rc, cam, spp)
            if k >= 2:
                t[arm].append(ms)
    ctx.set_option("time_frame_kernels", 0)
    scene.set_palette(None)
    out = dict(frame="%dx%d, %d spp, GI %d bounces, aperture %g" % (size[0], size[1], spp, bounces, aperture), repeats=REPEATS)
    for arm, v in t.items():
        v = np.asarray(v)
        out[arm] = dict(median_ms=round(float(np.median(v)), 3), min_ms=round(float(v.min()), 3), max_ms=round(float(v.max()), 3))
    out["palette_over_textures"] = round(out["palette"]["median_ms"] / out["textures"]["median_ms"], 4)
    return out


def main():
    print(json.dumps(card()), flush=True)
    ctx = vrt.Context(0)
    vox = terrain_voxels()
    colors = band_colors(vox)
    scene = vrt.LSVO.from_terrain(ctx, 9)
    painted = scene.paint_cells(vox, colors)
    print(json.dumps(dict(scene="T(9) painted by height band", voxels=len(vox), painted=painted)), flush=True)
    print(json.dumps(frames(ctx, scene, (1920, 1080), 64, 2, 0.5)), flush=True)
    print(json.dumps(frames(ctx, scene, (1280, 720), 1, 1, 0.0)), flush=True)
    scene.close()

    # paint throughput: the voxel-set scene (colours also kept per resident key) and the terrain scene
    for label, make in (("voxel set (from_voxels)", lambda: vrt.LSVO.from_voxels(ctx, 9, vox, on_device=True)),
                        ("terrain (from_terrain)", lambda: vrt.LSVO.from_terrain(ctx, 9))):
        s = make()
        s.paint_cells(vox[:1000], colors[:1000])            # warm-up (first paint of a voxel set allocates its colours)
        t = []
        for k in range(REPEATS):
            t0 = time.perf_counter()
            s.paint_cells(vox, (colors + k).astype(np.uint8))
            t.append(time.perf_counter() - t0)
        med = float(np.median(t))
        print(json.dumps(dict(paint=label, voxels=len(vox), median_ms=round(med * 1e3, 2), min_ms=round(min(t) * 1e3, 2),
                              max_ms=round(max(t) * 1e3, 2), voxels_per_s=round(len(vox) / med))), flush=True)
        s.close()

    # set_cells on a painted and an unpainted voxel-set scene, alternated
    scenes = {"unpainted": vrt.LSVO.from_voxels(ctx, 9, vox, on_device=True), "painted": vrt.LSVO.from_voxels(ctx, 9, vox, on_device=True)}
    scenes["painted"].paint_cells(vox, colors)
    rng = np.random.default_rng(0)
    t = {k: [] for k in scenes}
    for k in range(4 + 2 * REPEATS):                        # the first edits size the scenes' memory pools
        edit = rng.integers(0, 512, (1000, 3)).astype(np.uint32)
        for name, s in scenes.items():
            t0 = time.perf_counter()
            s.set_cells(edit, k % 2 == 0)
            if k >= 4:
                t[name].append((time.perf_counter() - t0) * 1e3)
    same = np.array_equal(scenes["painted"].download_nodes()["child_mask"], scenes["unpainted"].download_nodes()["child_mask"])
    out = dict(set_cells="1000 voxels at 512^3, add / remove alternating", repeats=len(t["painted"]), same_structure=bool(same))
    for name, v in t.items():
        out[name] = dict(median_ms=round(float(np.median(v)), 3), min_ms=round(float(np.min(v)), 3), max_ms=round(float(np.max(v)), 3))
    print(json.dumps(out), flush=True)
    for s in scenes.values():
        s.close()
    ctx.close()


if __name__ == "__main__":
    main()
