"""Generates the committed golden fixtures from the REFERENCE ITSELF (needs a checkout of the reference's sources and
oracle/_ref built from it: `VRT_REFERENCE=<checkout> make -C oracle && VRT_REFERENCE=<checkout> python tests/golden/make_golden.py`).

  textures.npz        res/grass_top_16x16.bmp, res/grass_side_16x16.bmp decoded to 16x16 RGB, top-down rows
                      (what sf::Image::loadFromFile presents; raycaster.hpp:53-54)
  lsvo_kat.npz        single-voxel known answers (SURVEY.md §8c) from LSVO<9>::castRay
  lsvo_terrain9.npz   8192 seeded rays on the default terrain T(9) → reference HitPoints (coef 0 and 0.5)
  lsvo_random6.npz    random voxel scene at depth 6: voxel list, reference LNode array, rays, HitPoints
  grid_random5.npz    Grid3D<32,32,32> (patched build): occupancy, rays, HitPoints
  svo_random5.npz     intended-SVO<5> (patched build): same occupancy, rays, HitPoints
  terrain_heights.npz heights of T(8) (256x256) + sha256 of T(9), T(10) heights and of T(9) LNode array
  frame_cfg1_small.npz  RayCaster (reference, depth 9) 160x90 deterministic frame: primary+shadow colours
  frame_checker_small.npz  the reference's RayCaster driven like main.cpp:137-143 for 4 frames: alternating checkerboard
                      halves (thread-area height 18 and the odd 15) with the 0.4/0.6 temporal blend, and the
                      accumulators of two half frames in sample mode   (`make_golden.py checker` makes only this file)
  cfg1_full.json      BASELINE configs[0] at its full size: the reference's RayCaster + Camera at 1280x720, 1 sample, primary +
                      sun shadow, camera (256,200,256) view (0,0): sha256 of the image and of the integer accumulators, the
                      number of primary hits and sha256 of the packed hit/complexity arrays of the 921 600 camera rays
                      (`make_golden.py cfg1` makes only this file)
"""
import hashlib
import os
import struct
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import loader  # noqa: E402

REF = os.environ.get("VRT_REFERENCE", "")
OUT = os.path.dirname(os.path.abspath(__file__))


def read_bmp24(path):
    b = open(path, "rb").read()
    off = struct.unpack_from("<I", b, 10)[0]
    w, h = struct.unpack_from("<ii", b, 18)
    bpp = struct.unpack_from("<H", b, 28)[0]
    assert bpp == 24 and w == 16 and abs(h) == 16
    stride = (w * 3 + 3) & ~3
    img = np.zeros((16, 16, 3), np.uint8)
    for row in range(16):
        src = off + row * stride
        line = np.frombuffer(b, np.uint8, w * 3, src).reshape(w, 3)[:, ::-1]  # BGR → RGB
        y = 15 - row if h > 0 else row                                        # bottom-up when h > 0
        img[y] = line
    return img


def rays(rng, n, lo=(1, 1, 1), hi=(2, 2, 2)):
    o = rng.uniform(lo, hi, (n, 3)).astype(np.float32)
    d = rng.normal(size=(n, 3)).astype(np.float32)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    return o, d.astype(np.float32)


def make_checker_frames(R):
    T = R.scene_terrain(9)
    R.register_textures(*[read_bmp24(os.path.join(REF, "res", n)) for n in ("grass_top_16x16.bmp", "grass_side_16x16.bmp")])
    light = np.float32([-200, -1000, -300]) * np.float32(1.0 / 512.0) + np.float32(1.0)
    out = dict(cam_position=np.float32([256, 200, 256]), view_angle=np.float32([0.7, -0.4]), light=light)
    for tag, W, H, area in (("a", 128, 72, 18), ("b", 96, 60, 15)):
        p = loader.RefRenderParams()
        p.width, p.height = W, H
        p.cam_position[:] = [256.0, 200.0, 256.0]
        p.view_angle[:] = [0.7, -0.4]
        p.fov, p.aperture, p.focal_length = 1.0, 0.0, 100.0
        p.light_position[:] = [float(x) for x in light]
        p.use_gi, p.use_samples, p.spp, p.threads = 0, 0, 1, 1
        p.checker, p.checker_area_height, p.frames = 2, area, 4          # main.cpp:98,137: the first frame has offset 1
        blend = R.render(T, p)["image"]
        p.use_samples, p.checker, p.frames = 1, 1, 2
        samples = R.render(T, p)["samples"].astype(np.uint32)
        out.update({"size_" + tag: np.int32([W, H, area]), "blend4_" + tag: blend, "samples2_" + tag: samples})
    np.savez_compressed(os.path.join(OUT, "frame_checker_small.npz"), **out)
    R.scene_destroy(T)


def make_cfg1_full(R):
    import json
    T = R.scene_terrain(9)
    R.register_textures(*[read_bmp24(os.path.join(REF, "res", n)) for n in ("grass_top_16x16.bmp", "grass_side_16x16.bmp")])
    light = np.float32([-200, -1000, -300]) * np.float32(1.0 / 512.0) + np.float32(1.0)
    p = loader.RefRenderParams()
    p.width, p.height = 1280, 720
    p.cam_position[:] = [256.0, 200.0, 256.0]
    p.view_angle[:] = [0.0, 0.0]
    p.fov, p.aperture, p.focal_length = 1.0, 0.0, 100.0
    p.light_position[:] = [float(x) for x in light]
    p.use_gi, p.use_samples, p.spp, p.threads = 0, 1, 1, 8
    res = R.render(T, p)
    o, d = R.camera_rays(p)
    hits = R.lsvo_cast(T, o, d, 0.0, 0.0, threads=8)
    out = dict(width=1280, height=720, cam_position=[256.0, 200.0, 256.0], view_angle=[0.0, 0.0], focal_length=100.0,
               light=[float(x) for x in light],
               sha256_image=hashlib.sha256(res["image"].tobytes()).hexdigest(),
               sha256_samples_u32=hashlib.sha256(res["samples"].astype(np.uint32).tobytes()).hexdigest(),
               primary_hits=int((hits["hit"] != 0).sum()),
               sha256_hit_flags=hashlib.sha256((hits["hit"] != 0).astype(np.uint8).tobytes()).hexdigest(),
               sha256_complexity=hashlib.sha256(hits["complexity"].astype(np.uint32).tobytes()).hexdigest(),
               sha256_distance_of_hits=hashlib.sha256(hits["distance"][hits["hit"] != 0].astype(np.float32).tobytes()).hexdigest(),
               sum_complexity=int(hits["complexity"].astype(np.int64).sum()))
    json.dump(out, open(os.path.join(OUT, "cfg1_full.json"), "w"), indent=1)
    R.scene_destroy(T)
    print(out)


def main():
    assert REF, "set VRT_REFERENCE to a checkout of the reference (johnBuffer/CpuVoxelRaycaster)"
    if len(sys.argv) > 1 and sys.argv[1] == "checker":
        make_checker_frames(loader.ref())
        return
    if len(sys.argv) > 1 and sys.argv[1] == "cfg1":
        make_cfg1_full(loader.ref())
        return
    R = loader.ref()
    RP = loader.ref_patched()
    assert R is not None and RP is not None, "build oracle/_ref first (make -C oracle)"
    top = read_bmp24(os.path.join(REF, "res/grass_top_16x16.bmp"))
    side = read_bmp24(os.path.join(REF, "res/grass_side_16x16.bmp"))
    np.savez_compressed(os.path.join(OUT, "textures.npz"), top=top, side=side)
    R.register_textures(top, side)

    # --- single voxel KATs
    S = 512.0
    sc = R.scene_from_voxels(9, [[100, 200, 300]])
    o = np.array([[1 + 411.5 / S, 1 + 311.5 / S, 1.0], [1 + 411.5 / S, 1 + 311.5 / S, 1 + 211.5 / S],
                  [1 + 411.5 / S, 1 + 311.5 / S, 0.5], [1 + 411.5 / S, 1 + 311.5 / S, -0.5],
                  [1 + 100.5 / S, 1 + 200.5 / S, 1.0], [1.999, 1 + 311.5 / S, 1 + 211.5 / S],
                  [1 + 411.5 / S, 1.0001, 1 + 211.5 / S]], np.float32)
    d = np.array([[0, 0, 1], [0, 0, 1], [0, 0, 1], [0, 0, 1], [0, 0, 1], [-1, 0, 0], [0, 1, 0]], np.float32)
    np.savez_compressed(os.path.join(OUT, "lsvo_kat.npz"), voxels=np.array([[100, 200, 300]], np.uint32), depth=9,
                        nodes=R.nodes(sc), origin=o, dir=d, hits=R.lsvo_cast(sc, o, d))
    R.scene_destroy(sc)

    # --- terrain T(9)
    rng = np.random.default_rng(20261017)
    T = R.scene_terrain(9)
    o, d = rays(rng, 8192, (1, 1, 1), (2, 1.45, 2))
    # a quarter of the rays are camera-like (coherent, looking down at the terrain)
    o[:2048] = np.float32([1.5, 1 + 200 / 512.0, 1.5])
    np.savez_compressed(os.path.join(OUT, "lsvo_terrain9.npz"), origin=o, dir=d, hits_coef0=R.lsvo_cast(T, o, d, 0.0, 0.0),
                        hits_coef05=R.lsvo_cast(T, o, d, 0.5, 0.0), hits_bias=R.lsvo_cast(T, o, d, 0.25, 0.001))
    nodes9 = R.nodes(T)
    nodes9["pad"] = 0
    h8, h9, h10 = R.terrain_heights(256), R.terrain_heights(512), R.terrain_heights(1024)
    np.savez_compressed(os.path.join(OUT, "terrain_heights.npz"), heights8=h8,
                        sha_heights9=hashlib.sha256(h9.tobytes()).hexdigest(),
                        sha_heights10=hashlib.sha256(h10.tobytes()).hexdigest(),
                        sha_nodes9=hashlib.sha256(nodes9.tobytes()).hexdigest(), n_nodes9=len(nodes9),
                        solid_voxels9=int(np.maximum(16, np.minimum(512, h9)).astype(np.int64).sum() - h9.size))

    # --- small deterministic frame through the reference RayCaster (primary + sun shadow, no GI, aperture 0)
    p = loader.RefRenderParams()
    p.width, p.height = 160, 90
    p.cam_position[:] = [256.0, 200.0, 256.0]
    p.view_angle[:] = [0.35, -0.25]
    p.fov, p.aperture, p.focal_length = 1.0, 0.0, 100.0
    light = np.float32([-200, -1000, -300]) * np.float32(1.0 / 512.0) + np.float32(1.0)
    p.light_position[:] = [float(x) for x in light]
    p.use_gi, p.use_samples, p.spp, p.threads = 0, 1, 1, 1
    res = R.render(T, p)
    rot, cvec = R.camera_basis(np.float32([0.35, -0.25]))
    np.savez_compressed(os.path.join(OUT, "frame_cfg1_small.npz"), width=160, height=90, cam_position=np.float32([256, 200, 256]),
                        view_angle=np.float32([0.35, -0.25]), rot_mat=rot, camera_vec=cvec, light=light,
                        samples=res["samples"].astype(np.uint32), image=res["image"])
    R.scene_destroy(T)

    # --- random scene depth 6
    vox = rng.integers(0, 64, size=(6000, 3)).astype(np.uint32)
    sc = R.scene_from_voxels(6, vox)
    nodes = R.nodes(sc)
    nodes["pad"] = 0
    o, d = rays(rng, 8192, (0.8, 0.8, 0.8), (2.2, 2.2, 2.2))
    d[:64, 0] = 0.0                      # axis-parallel components exercise the |d| < 2^-23 clamp
    d[64:128, 1] = -0.0
    d[128:192] = np.float32([0, 0, 1])
    np.savez_compressed(os.path.join(OUT, "lsvo_random6.npz"), voxels=vox, nodes=nodes, origin=o, dir=d,
                        hits_coef0=R.lsvo_cast(sc, o, d, 0.0, 0.0), hits_coef05=R.lsvo_cast(sc, o, d, 0.5, 0.0))
    R.scene_destroy(sc)

    # --- Grid3D / intended SVO at 32^3
    occ = (rng.random((32, 32, 32)) < 0.03).astype(np.uint8)
    occ[:, :3, :] = 1
    g = RP.grid_create(occ)
    o = rng.uniform(0.5, 31.5, (4096, 3)).astype(np.float32)
    o[:, 1] = rng.uniform(4, 31.5, 4096)
    d = rng.normal(size=(4096, 3)).astype(np.float32)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    np.savez_compressed(os.path.join(OUT, "grid_random5.npz"), occ=occ, origin=o, dir=d, hits=RP.grid_cast(g, o, d))
    RP.grid_destroy(g)
    s = RP.svo_create(occ)
    np.savez_compressed(os.path.join(OUT, "svo_random5.npz"), occ=occ, origin=o, dir=d, hits=RP.svo_cast(s, o, d, 1 << 20),
                        hits_iter16=RP.svo_cast(s, o, d, 16))
    RP.svo_destroy(s)
    make_checker_frames(R)
    make_cfg1_full(R)
    print("golden fixtures written to", OUT)


if __name__ == "__main__":
    main()
