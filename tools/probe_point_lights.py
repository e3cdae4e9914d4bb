"""Point lights: what 0, 1, 4 and 16 lights cost the bench frame, and the headline with and without the feature's code.

The bench workload (bench.py: T(11), 1920x1080, 64 spp, GI 2 bounces + DOF, camera C(11), textures) rendered through
RayCaster.render with 0, 1, 4 and 16 point lights over the terrain in front of the camera, in two arms:
  - in range: every light has range +inf, so every hit that faces a light casts one more shadow ray per light;
  - culled:   ranges of 12 voxels, so most hits are out of range of every light and pay only the cast test.
Frames with lights run on the kMirror instance of K6 (the 0-light frame on the plain instance, as bench.py does).  Frame times
are device events around the frame kernels (context option "time_frame_kernels") with the product defaults (beam floors,
bounds exits); every arm is warmed up first and the arms alternate, REPEATS times each.  Rays per class are vrt_render_stats.

Then the same frame with a palette and no lights (the kMirror instance of K6, whose chain state grew) runs from the parent checkout
and from this tree, alternating; and bench.py --gpus 1 runs from the parent checkout (--parent, built) and from this tree, alternating, BENCH_ROUNDS times each:
the headline frame never has lights, so its kernels are the parent's and its figure must not move.

  python tools/probe_point_lights.py --parent DIR [--out FILE]      (one B200; prints and writes one JSON line per measurement)"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import cpuvoxelraycaster_b200 as vrt  # noqa: E402
from probe_palette import ROOT, card  # noqa: E402

REPEATS = 5
BENCH_ROUNDS = 2
DEPTH = 11


def lights(n, culled):
    """n lights on a grid in front of camera C(11), a little above its eye height, in the normalised castRay frame."""
    if n == 0:
        return None
    S = 1 << DEPTH
    k = np.arange(n)
    pos = np.stack([S / 2.0 + (k % 4 - 1.5) * 96.0, np.full(n, S / 2.0 - 80.0), S / 2.0 + 64.0 + (k // 4) * 96.0], 1)
    pos = np.float32(pos) * np.float32(1.0 / S) + np.float32(1.0)
    col = np.float32([[1.0, 0.8, 0.6], [0.6, 0.8, 1.0], [1.0, 0.4, 0.4], [0.4, 1.0, 0.5]])[k % 4]
    rng = np.full(n, 12.0 / S if culled else np.inf, np.float32)
    return pos, col, rng


def frames(ctx, scene):
    S = 1 << DEPTH
    cam = vrt.Camera(position=(S / 2.0, S / 2.0 - 56.0, S / 2.0), view_angle=(0.0, 0.0), aperture=0.5)
    cam.autofocus(scene)                                     # as bench.py
    rc = vrt.RayCaster(scene, (1920, 1080))
    rc.setLightPosition(np.float32([-200, -1000, -300]) * np.float32(1.0 / S) + np.float32(1))
    rc.use_samples, rc.use_gi, rc.gi_bounces = True, True, 2
    arms = [(0, False)] + [(n, culled) for culled in (False, True) for n in (1, 4, 16)]
    ctx.set_option("time_frame_kernels", 1)
    t = {a: [] for a in arms}
    rays = {}
    for k in range(2 + REPEATS):
        for arm in arms:
            lt = lights(*arm)
            scene.set_point_lights(*(lt if lt is not None else (None,)))
            rc.resetSamples()
            rc.render(cam, 64)
            ms = sum(ctx.take_kernel_timings())
            rays[arm] = rc.last_stats["rays"]
            if k >= 2:
                t[arm].append(ms)
    ctx.set_option("time_frame_kernels", 0)
    scene.set_point_lights(None)
    base = float(np.median(t[(0, False)]))
    for arm in arms:
        v = np.asarray(t[arm])
        yield dict(frame="1920x1080, 64 spp, GI 2 bounces, aperture 0.5, T(11)", lights=arm[0],
                   ranges="none" if arm[0] == 0 else ("12 voxels" if arm[1] else "inf"), repeats=REPEATS,
                   median_ms=round(float(np.median(v)), 3), min_ms=round(float(v.min()), 3), max_ms=round(float(v.max()), 3),
                   over_no_lights=round(float(np.median(v)) / base, 4), rays_per_class=[int(x) for x in rays[arm]],
                   shadow_rays_per_camera_sample=round(rays[arm][1] / (1920 * 1080 * 64), 4))


# The same frame with a palette and no lights, in a process of its own from either tree: palette frames run on the kMirror
# instance of K6, whose chain state grew by the light sums (more spill traffic), so this is where the feature can cost the frames
# that do not use it.
PALETTE_FRAME = r"""
import json, os, sys
import numpy as np
sys.path.insert(0, os.getcwd())
import cpuvoxelraycaster_b200 as vrt
S = 2048
ctx = vrt.Context(0)
scene = vrt.LSVO.from_terrain(ctx, 11)
tex = np.load(os.path.join("tests", "golden", "textures.npz"))
scene.set_textures(tex["top"], tex["side"])
scene.set_palette(np.random.default_rng(7).integers(0, 256, (256, 3), dtype=np.uint8))
cam = vrt.Camera(position=(S / 2.0, S / 2.0 - 56.0, S / 2.0), view_angle=(0.0, 0.0), aperture=0.5)
cam.autofocus(scene)
rc = vrt.RayCaster(scene, (1920, 1080))
rc.setLightPosition(np.float32([-200, -1000, -300]) * np.float32(1.0 / S) + np.float32(1))
rc.use_samples, rc.use_gi, rc.gi_bounces = True, True, 2
ctx.set_option("time_frame_kernels", 1)
t = []
for k in range(2 + %d):
    rc.resetSamples()
    rc.render(cam, 64)
    ms = sum(ctx.take_kernel_timings())
    if k >= 2:
        t.append(ms)
print(json.dumps(dict(median_ms=round(float(np.median(t)), 3), min_ms=round(min(t), 3), max_ms=round(max(t), 3))))
""" % REPEATS


def palette_frame(tree):
    r = subprocess.run([sys.executable, "-c", PALETTE_FRAME], capture_output=True, text=True, cwd=tree)
    if r.returncode:
        raise RuntimeError("palette frame failed in %s: %s" % (tree, r.stderr[-2000:]))
    return json.loads(r.stdout.strip().splitlines()[-1])


def bench(tree):
    r = subprocess.run([sys.executable, os.path.join(tree, "bench.py"), "--gpus", "1", "--steps", "5", "--warmup", "2", "--no-cpu-baseline"],
                       capture_output=True, text=True, cwd=tree)
    line = [x for x in r.stdout.splitlines() if x.startswith("{")]
    if r.returncode or not line:
        raise RuntimeError("bench.py failed in %s: %s" % (tree, r.stderr[-2000:]))
    j = json.loads(line[-1])
    return dict(value=j["value"], unit=j["unit"], ms_per_step=j["ms_per_step"])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent", required=True, help="a built checkout of the parent commit")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "point_lights_probe.txt"))
    args = ap.parse_args()
    with open(args.out, "w") as out:
        def emit(d):
            print(json.dumps(d), flush=True)
            out.write(json.dumps(d) + "\n")
            out.flush()
        emit(card())
        ctx = vrt.Context(0)
        scene = vrt.LSVO.from_terrain(ctx, DEPTH)
        tex = np.load(os.path.join(ROOT, "tests", "golden", "textures.npz"))
        scene.set_textures(tex["top"], tex["side"])
        for d in frames(ctx, scene):
            emit(d)
        scene.close()
        ctx.close()
        parent = os.path.abspath(args.parent)
        pal = {"parent": [], "branch": []}
        for _ in range(BENCH_ROUNDS):
            for arm, tree in (("parent", parent), ("branch", ROOT)):
                pal[arm].append(palette_frame(tree))
        emit(dict(palette_frame="the same frame with a palette and no lights, alternating", runs=pal))
        runs = {"parent": [], "branch": []}
        for _ in range(BENCH_ROUNDS):
            for arm, tree in (("parent", parent), ("branch", ROOT)):
                runs[arm].append(bench(tree))
        emit(dict(bench="bench.py --gpus 1 --steps 5 --warmup 2 --no-cpu-baseline, alternating", runs=runs))


if __name__ == "__main__":
    main()
