#!/usr/bin/env python
"""bench.py — headline benchmark of the voxel ray-traversal hot path.

  python bench.py --gpus N --steps K --warmup W            (N>1: launched under torchrun, one rank per GPU)
  python bench.py --impl reference --gpus N --steps K --warmup W

Workload (BASELINE.json configs[3], the configuration the metric "Mrays/s ... and ms/frame 1080p at
1/2/4/8 B200" is quoted on): synthetic FastNoise terrain T(11) = 2048^3 in an LSVO, 1920x1080, 64 spp,
use_samples + use_gi with 2 GI bounces + depth of field (aperture 0.5), camera C(11), rows dealt in
4-row tiles round-robin over the GPUs, frame all-gathered with NCCL.  A "step" is one such frame.
A "ray" is one distinct castRay (primary, sun shadow, GI, GI shadow, bounce-2 GI, its shadow).

value  = rays of the whole frame / device time with the scene and frame buffers resident in HBM
e2e    = the same through the user-facing FrameRenderer (libvrt's vrt_render_distributed underneath): camera/params in
         from the host and every finished RGBA frame copied back to pinned host memory inside the timed region
         (double buffered: frame i is copied on a second stream while frame i+1 renders)
The reference arm times the reference's own CPU implementation (oracle/_ref, compiled from the
reference's sources) on a bounded sample of the same frame on the host cores.

Multi-GPU (N > 1): the frame's 4-row tiles are dealt round-robin to the ranks and every rank's resolve kernel stores its
pixels straight into rank 0's frame buffer over NVLink (libvrt communicator, csrc/comm.cu); during warm-up rank 0 also
renders the frame alone and the two frames are compared by hash ("frame_identity" in the JSON line).
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark leaves the source tree as it found it (no __pycache__ of tools/, oracle/)

METRIC = "Mrays/s (primary+shadow+GI), 1080p 64-spp GI+DOF frame on LSVO 2048^3"
UNIT = "Mrays/s"


def workload(args):
    D = args.depth
    S = 1 << D
    return dict(depth=D, size=S, width=args.width, height=args.height, spp=args.spp, gi_bounces=args.gi_bounces,
                aperture=args.aperture, cam_position=[S / 2.0, S / 2.0 - 56.0, S / 2.0], view_angle=[0.0, 0.0],
                light=[-200.0, -1000.0, -300.0], seed=(0x5EED, 0))


def light_normalised(w):
    return np.float32(w["light"]) * np.float32(1.0 / w["size"]) + np.float32(1.0)      # main.cpp:124-126


def load_textures():
    t = np.load(os.path.join(ROOT, "tests", "golden", "textures.npz"))
    return t["top"], t["side"]


def config_json(w, n_gpus):
    """The same dict for both arms (the driver compares them): everything arm-specific goes into "extra"."""
    return {"workload": "cfg4: LSVO %d^3 FastNoise terrain T(%d), %dx%d, %d spp, use_samples+use_gi (%d bounces) + DOF aperture %.2f, "
                        "camera C(%d)" % (w["size"], w["depth"], w["width"], w["height"], w["spp"], w["gi_bounces"], w["aperture"], w["depth"]),
            "depth": w["depth"], "width": w["width"], "height": w["height"], "spp": w["spp"], "gi_bounces": w["gi_bounces"],
            "aperture": w["aperture"], "n_gpus": n_gpus, "rng": "Philox4x32-10 on getRand's 100-level lattice, key 0x5EED",
            "ray_definition": "distinct castRay calls of the frame (the reference's 4 identical shadow samples count once); camera rays of beam tiles with an empty frustum are answered by the beam search without a walk and are counted — primary_rays_answered_by_beam_search says how many, value_walked_rays_only leaves them out",
            "l2": "inputs larger than L2: 1.35 GB node array + 33 MB accumulator vs 126 MB L2"}


# ---- clocks sampler (B200_PROFILING.md recipe) --------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---- CPU legs (the only places that may execute oracle/) ------------------------------------------------
def cpu_port_sample(w, cores, tile_step, spp, repeat=1, single=None):
    """The oracle restatement (kind "port") on a bounded sample of the workload: every tile_step-th 4-row tile,
    `spp` of the samples, all host threads; best wall time of `repeat` runs.  single = (tile_step, spp): also one
    single-threaded run on that smaller sample (SURVEY.md 8d asks for the single-thread figure)."""
    from oracle import loader
    P = loader.port()
    nodes = P.build_terrain(w["depth"])
    top, side = load_textures()
    import cpuvoxelraycaster_b200 as vrt                     # host-only helper: camera basis (pure host code)
    cam = vrt.Camera(position=w["cam_position"], view_angle=w["view_angle"], aperture=w["aperture"], focal_length=100.0)
    p = loader.PortRenderParams()
    p.width, p.height, p.depth, p.guard = w["width"], w["height"], w["depth"], w["depth"]
    p.cam_position[:] = w["cam_position"]
    p.rot_mat[:] = [float(x) for x in cam.rot_mat]
    p.fov, p.aperture, p.focal_length = 1.0, w["aperture"], w["focal_length"]
    p.light_position[:] = [float(x) for x in light_normalised(w)]
    p.use_gi, p.gi_bounces, p.use_samples, p.spp = 1, w["gi_bounces"], 1, spp
    p.seed_lo, p.seed_hi = w["seed"]
    p.threads, p.tile_step, p.tile_index = cores, tile_step, 0
    dt = None
    for _ in range(max(1, repeat)):
        t0 = time.perf_counter()
        _, _, st = P.render(nodes, p, top, side)
        d = time.perf_counter() - t0
        dt = d if dt is None else min(dt, d)
    rays = sum(st.rays)
    if single is None:
        return rays, dt
    p.threads, p.tile_step, p.spp = 1, single[0], single[1]
    t0 = time.perf_counter()
    _, _, st1 = P.render(nodes, p, top, side)
    return rays, dt, sum(st1.rays) / (time.perf_counter() - t0)


def run_reference(args):
    """--impl reference: the reference's own CPU code (oracle/_ref, RayCaster + Camera + LSVO::castRay compiled from the
    reference's sources at the workload's depth, swarm-threaded).  A step renders WHOLE 4-row tiles of the full frame with all
    of the workload's samples per pixel — every `ref_tile_step`-th tile, spread over the frame like one GPU's share in the
    multi-GPU split — so that a step is the same kind of work as the GPU arm's, bounded to a few seconds."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import loader
    w = workload(args)
    cores = os.cpu_count() or 1
    R = loader.ref_depth(w["depth"])
    P = loader.port()
    top, side = load_textures()
    nodes = P.build_terrain(w["depth"])
    tile_step, spp = args.ref_tile_step, (args.ref_spp or w["spp"])
    sample_desc = "every %d-th 4-row tile of the frame x %d of %d spp = 1/%d of the frame per step" % (
        tile_step, spp, w["spp"], tile_step * w["spp"] // spp)
    if R is not None:
        kind = "reference"
        R.register_textures(top, side)
        scene = R.scene_from_nodes(w["depth"], nodes)
        p = loader.RefRenderParams()
        p.width, p.height = w["width"], w["height"]
        p.cam_position[:] = w["cam_position"]
        p.view_angle[:] = w["view_angle"]
        p.fov, p.aperture = 1.0, w["aperture"]
        p.light_position[:] = [float(x) for x in light_normalised(w)]
        p.focal_length = R.autofocus(scene, p)
        p.use_gi, p.use_samples, p.spp, p.threads = 1, 1, spp, cores
        p.row_begin, p.row_end, p.tile_step, p.tile_index = 0, w["height"], tile_step, 0

        def step():
            r = R.render(scene, p)
            # distinct rays: primary + shadow (4 identical invocations per hit under use_samples) + GI + GI shadow
            pixels = sum(1 for y in range(w["height"]) if (y >> 2) % tile_step == 0) * w["width"] * spp
            shadow = (r["cone0_calls"] - pixels) // 4
            return pixels + shadow + r["cone_gi_calls"], r["seconds"]
        note = ("the reference's RayCaster has ONE GI bounce (raycaster.hpp:169-207; RayContext::gi_bounce = 2 is never read): this arm "
                "renders the reference's own estimator; the GPU arm's like-for-like figure is its extra.one_bounce")
    else:
        kind = "port"
        w["focal_length"] = 100.0

        def step():
            return cpu_port_sample(w, cores, tile_step, spp)
        note = "oracle/_ref absent: timed the C restatement"
    for _ in range(args.warmup if args.ref_warmup < 0 else args.ref_warmup):
        step()
    rays, secs = 0, 0.0
    for _ in range(args.steps):
        r, s_ = step()
        rays += r
        secs += s_
    value = rays / secs / 1e6
    line = {"impl": "reference", "metric": METRIC, "value": round(value, 3), "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(1e3 * secs / args.steps, 3),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_json(w, args.gpus),
            "cpu_baseline": {"value": round(value, 3), "unit": UNIT, "cores": cores, "kind": kind, "sample": sample_desc},
            "e2e": {"value": round(value, 3), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "extra": {"note": note, "gi_bounces_rendered": 1 if kind == "reference" else w["gi_bounces"],
                                         "rays_per_step": rays // max(1, args.steps)}}
    _emit(json.dumps(line))
    return 0


# ---- our arm ----------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    import cpuvoxelraycaster_b200 as vrt
    from cpuvoxelraycaster_b200.frame import FrameRenderer

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("bench.py --gpus %d must be launched with torchrun --nproc-per-node %d" % (args.gpus, args.gpus))
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)

    w = workload(args)
    stream = torch.cuda.Stream(device)
    ctx = vrt.Context(local_rank, stream.cuda_stream)
    t0 = time.perf_counter()
    scene = vrt.LSVO.from_terrain(ctx, w["depth"])           # every rank builds its replica, on its own GPU
    ctx.synchronize()
    build_s = time.perf_counter() - t0
    n_slots = len(scene)
    scene.set_textures(*load_textures())
    cam = vrt.Camera(position=w["cam_position"], view_angle=w["view_angle"], aperture=w["aperture"])
    cam.autofocus(scene)                                     # main.cpp:115-121
    w["focal_length"] = cam.focal_length

    # the product path for every N: libvrt's communicator (vrt_render_distributed) — at N = 1 it degenerates to
    # clear + frame kernels + resolve into the double-buffered frame + host copy on the second stream
    fr = FrameRenderer(scene, w["width"], w["height"], rank, world, None, device, stream, exchange="peer", split=args.split)
    fr.use_gi, fr.gi_bounces, fr.use_samples, fr.seed = True, w["gi_bounces"], True, w["seed"]
    fr.light = light_normalised(w)

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    # ---- warm-up, and the frame-identity check: the frame assembled from all ranks == the frame rank 0 renders alone ----
    for _ in range(args.warmup):
        fr.render_device(cam, w["spp"])
    host = fr.render(cam, w["spp"])                          # collective; rank 0 gets the frame
    identity = None
    if rank == 0:
        alone = FrameRenderer(scene, w["width"], w["height"], 0, 1, None, device, stream, exchange="nccl")
        alone.use_gi, alone.gi_bounces, alone.use_samples, alone.seed, alone.light = True, w["gi_bounces"], True, w["seed"], fr.light
        single = alone.render(cam, w["spp"])
        h_multi, h_single = hashlib.sha256(host.tobytes()).hexdigest(), hashlib.sha256(single.tobytes()).hexdigest()
        identity = {"sha256": h_multi[:32], "identical_to_single_gpu_frame": h_multi == h_single, "lit_pixels": int((host[..., :3].sum(-1) > 0).sum())}
        del alone
        scene.ctx.set_stream(stream.cuda_stream)
    sync_all()

    # ---- device-resident timing -------------------------------------------------------------------------
    launches0 = ctx.launch_count
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ev_start, ev_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ctx.set_option("time_frame_kernels", 1)                  # libvrt brackets its frame kernels with CUDA events on its stream
    sync_all()
    ev_start.record(stream)
    for i in range(args.steps):
        last = fr.render_device(cam, w["spp"])
    ev_end.record(stream)
    sync_all()
    kernel_times = ctx.take_kernel_timings()                 # ms of the dominant kernel (sort + trace) per frame, this rank
    ctx.set_option("time_frame_kernels", 0)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        # the last timed frame as the caller receives it (uint8 RGBA [H, W, 4]), stored as float32: 33 MB at 1080p; larger frames
        # keep every k-th row so that the file, its .npy header (128 bytes) included, stays within 64 MB
        img = last.cpu().numpy()
        k = -(-img.size * 4 // (64_000_000 - 4096))
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "frame.npy"), img[::k].astype(np.float32))
    launches = ctx.launch_count - launches0
    ms_total = ev_start.elapsed_time(ev_end)
    kernel_ms = float(np.mean(kernel_times)) if kernel_times else float("nan")
    st = fr.stats()                                          # this rank's share, last frame
    t = torch.tensor([ms_total, kernel_ms], dtype=torch.float64, device=device)
    cnt = torch.tensor(st["rays"] + st["complexity"] + [launches, st.get("culled_primary", 0)], dtype=torch.int64, device=device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        local_cnt = cnt.clone()
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
    else:
        local_cnt = cnt
    ms_total, kernel_ms_max = float(t[0]), float(t[1])
    rays = [int(x) for x in cnt[:6].tolist()]
    cx = [int(x) for x in cnt[6:12].tolist()]
    launches = int(cnt[12])                                  # libvrt kernels launched in the timed region, all ranks
    # primary rays of samples whose 8x8-pixel beam tile has nothing in its frustum: answered (a miss) by the beam search, counted
    # in rays[0] like every castRay call the reference makes for the frame, but not walked — no node bytes, no ray / hit record
    culled = int(cnt[13])
    total_rays = sum(rays)
    ms_per_step = ms_total / args.steps
    value = total_rays / (ms_per_step * 1e-3) / 1e6

    # roofline of the dominant kernel on this rank: algorithmic bytes = sum over its rays of (8 B node per
    # iteration + 64 B ray/hit record) + 16 B accumulator write per pixel (SURVEY.md §8d, DESIGN.md)
    l_rays, l_cx = int(local_cnt[:6].sum()) - int(local_cnt[13]), int(local_cnt[6:12].sum())   # walked rays only
    if args.split == "samples":
        my_pixels = w["height"] * w["width"]
    else:
        my_pixels = sum(1 for y in range(w["height"]) if (y >> 2) % world == rank) * w["width"]
    algo_bytes = 8 * l_cx + 64 * l_rays + 16 * my_pixels
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    else:
        peak, peak_src = 6650.0, "B200_PROFILING.md fallback (of fallback)"
    achieved = algo_bytes / (kernel_ms * 1e-3) / 1e9
    ncu = {}
    tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tpath):
        try:
            ncu = json.load(open(tpath)).get("render_rounds_kernel", {})
        except Exception:
            ncu = {}
    roofline = {"bound": "hbm", "kernel": "render_rounds_kernel (K6; timed together with its sort_samples_kernel by CUDA events inside libvrt, on its stream)",
                "achieved": round(achieved, 2), "peak": peak, "unit": "GB/s",
                "frac": round(achieved / peak, 4), "traffic": ncu.get("dram_bytes_per_launch") if world == 1 else None, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": algo_bytes, "kernel_ms": round(kernel_ms, 4),
                "kernel_share_of_step": round(kernel_ms_max / ms_per_step, 4),
                # the binding resource of this kernel is instruction issue at low SIMT width, not HBM (DESIGN.md §5): the ncu
                # counters of the same launch, measured once per round (source named in the file)
                "issue_active_pct": ncu.get("issue_active_pct"), "lanes_per_instruction": ncu.get("lanes_per_instruction"),
                "alu_pipe_pct": ncu.get("alu_pipe_pct"), "warp_instructions": ncu.get("warp_instructions"),
                "l1_global_load_bytes": ncu.get("l1_global_load_bytes_per_launch"), "l2_bytes": ncu.get("l2_bytes_per_launch"),
                "ncu_source": ncu.get("source"),
                "sector_granular_GBs": round((32 * l_cx + 64 * l_rays + 16 * my_pixels) / (kernel_ms * 1e-3) / 1e9, 1),
                "note": "pointer chasing: latency/divergence bound by design, see DESIGN.md; node fetches are mostly L1/L2 hits"}

    # ---- end to end through the public API: camera + parameters in, every frame out to pinned host memory ----------
    for _ in range(2):
        fr.render(cam, w["spp"])
    sync_all()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        fr.render_pipelined(cam, w["spp"])                   # frame i's host copy overlaps frame i+1's rendering
    frame = fr.flush()                                       # all K frames are in host memory when this returns
    sync_all()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    te = torch.tensor([e2e_ms], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_ms = float(te[0])
    import ctypes as C
    h2d = C.sizeof(vrt.capi.Camera) + C.sizeof(vrt.capi.RenderParams)
    e2e = {"value": round(total_rays / (e2e_ms * 1e-3) / 1e6, 2), "unit": UNIT, "ms_per_step": round(e2e_ms, 3),
           "h2d_bytes_per_step": h2d * world, "d2h_bytes_per_step": w["width"] * w["height"] * 4,
           "note": "a renderer's per-frame input is the camera + render parameters (per rank); the scene is resident like model weights; "
                   "the finished frame is delivered to rank 0's pinned host memory every step (wall clock incl. the final flush)"}
    if rank == 0 and frame is not None and identity is not None:
        identity["e2e_last_frame_sha256_matches"] = hashlib.sha256(frame.tobytes()).hexdigest()[:32] == identity["sha256"]

    # ---- like-for-like with the reference arm: the reference's own ONE-bounce estimator on the whole frame --------------
    extra = {"focal_length": w["focal_length"], "lsvo_slots": n_slots, "scene_build_s_device": round(build_s, 3),
             "split": args.split, "exchange": "libvrt communicator: resolve kernel stores pixels into rank 0's frame over NVLink (peer-mapped, CUDA IPC)"}
    if not args.no_extra:
        fr.gi_bounces = 1
        fr.render_device(cam, w["spp"])
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(args.steps):
            fr.render_device(cam, w["spp"])
        e1.record(stream)
        sync_all()
        st1 = fr.stats()
        t1 = torch.tensor([e0.elapsed_time(e1) / args.steps], dtype=torch.float64, device=device)
        c1 = torch.tensor(st1["rays"], dtype=torch.int64, device=device)
        if world > 1:
            dist.all_reduce(t1, op=dist.ReduceOp.MAX)
            dist.all_reduce(c1, op=dist.ReduceOp.SUM)
        extra["one_bounce"] = {"what": "the same frame with the reference's own one-bounce GI (raycaster.hpp:169-207) — the workload the reference arm renders",
                               "ms_per_step": round(float(t1[0]), 4), "rays_per_frame": int(c1.sum()),
                               "value": round(int(c1.sum()) / (float(t1[0]) * 1e-3) / 1e6, 2), "unit": UNIT}
        fr.gi_bounces = w["gi_bounces"]

    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            cores = os.cpu_count() or 1
            c_rays, c_dt, c_single = cpu_port_sample(w, cores, args.cpu_tile_step, args.cpu_spp, repeat=3, single=(32, 8))
            cpu = {"value": round(c_rays / c_dt / 1e6, 3), "unit": UNIT, "cores": cores, "kind": "port",
                   "sample": "every %d-th 4-row tile x %d of %d spp = 1/%d of the frame, best of 3 runs: %.1f s wall" % (
                       args.cpu_tile_step, args.cpu_spp, w["spp"], args.cpu_tile_step * w["spp"] // args.cpu_spp, c_dt),
                   "single_thread_value": round(c_single / 1e6, 3)}
        if world == 1 and not args.no_extra:
            # the other BASELINE.json configurations, device resident (parity for each is in tests/): driver-observed numbers
            try:
                sys.path.insert(0, os.path.join(ROOT, "tools"))
                import measure_configs
                extra["configs"] = measure_configs.measure(ctx, stream, [1, 2, 3, 5], 3, args.cfg5_rays)
            except Exception as e:                           # never lose the headline line over a side measurement
                extra["configs"] = {"error": repr(e)}
        line = {"metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": round(ms_per_step, 4), "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": config_json(w, world),
                "rays_per_frame": dict(zip(["primary", "shadow", "gi", "gi_shadow", "gi2", "gi2_shadow"], rays)),
                "primary_rays_answered_by_beam_search": culled,
                "value_walked_rays_only": round((total_rays - culled) / (ms_per_step * 1e-3) / 1e6, 2),
                "mean_complexity": round(sum(cx) / max(1, total_rays), 2),
                "ms_per_frame": round(ms_per_step, 4), "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e,
                "gpu_launches": int(launches), "clocks": clocks, "frame_identity": identity, "extra": extra}
        _emit(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


_emit = print


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--depth", type=int, default=11)
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--spp", type=int, default=64)
    ap.add_argument("--gi-bounces", type=int, default=2)
    ap.add_argument("--aperture", type=float, default=0.5)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-tile-step", type=int, default=2)      # cpu_baseline sample: 1/2 of the tiles x 1/2 of the
    ap.add_argument("--cpu-spp", type=int, default=32)           # samples = 1/4 frame, ~30-40 core-seconds
    ap.add_argument("--ref-tile-step", type=int, default=16)     # reference arm: 1/16 of the frame's tiles, all samples (~1.3 s per step)
    ap.add_argument("--ref-spp", type=int, default=0)            # 0 = the workload's spp
    ap.add_argument("--ref-warmup", type=int, default=1)         # CPU code needs no 3 warm-up passes; -1 = --warmup
    ap.add_argument("--split", default="tiles", choices=["tiles", "samples"])   # multi-GPU partition of the frame
    ap.add_argument("--no-extra", action="store_true")           # skip extra.one_bounce / extra.configs
    ap.add_argument("--cfg5-rays", type=int, default=100_000_000)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None)   # writes DIR/frame.npy: the last timed frame
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the frame of --impl ours")
    if args.warmup < 3:
        args.warmup = 3
    # stdout must carry the ONE JSON line: libraries (NCCL's version banner, for one) printf to file descriptor 1, so the
    # run happens with fd 1 pointing at stderr and the line is written to the saved descriptor at the end
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    global _emit
    _emit = lambda text: os.write(real_stdout, (text + "\n").encode())
    return run_reference(args) if args.impl == "reference" else run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
