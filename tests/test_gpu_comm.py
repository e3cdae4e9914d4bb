r"""The communicator frame path (csrc/comm.cu) against oracle/port.c on ONE GPU.

bench.py renders every frame it times through FrameRenderer(..., exchange="peer"), libvrt's communicator, also on one GPU:
vrt_comm_create, vrt_render_distributed, resolve_push_kernel (a second copy of resolve_kernel's samples_to_image and 0.4/0.6
blend, with its own tile-to-row mapping), the double-buffered frame with its host copy on a second stream, render_pipelined
and flush.  tests/test_gpu_multigpu.py needs two GPUs, and compares with libvrt's own single-GPU frame only.  Here:

| test                                            | what it pins                                                                     |
|-------------------------------------------------|----------------------------------------------------------------------------------|
| test_world1_frames_as_benchmarked               | world 1, both splits: render, render_device, frame_device_ptr(1), render_pipelined + flush, stats |
| test_world1_product_defaults_and_nccl_exchange  | beam floors + bounds exits on the peer exchange; the torch exchange gives the same frames |
| test_benchmark_frame_crop_vs_oracle             | bench.py's frame itself (T(11), 1080p, 64 spp) on a 32-row crop; the three delivery paths agree |
| test_ranks_sharing_one_gpu                      | world 2-4 on one device (vrt_comm_create_local): arrival slots, the sample-split reduce, deliver_all, the double-buffer waits, per-rank stats, a temporal-blend checkerboard sequence |
| test_cpp_host_with_three_ranks_on_one_gpu       | tests/cpp/multigpu_test.cpp with every rank on device 0                          |
| test_present_device_on_the_peer_frame           | FrameRenderer.present_device on the communicator's buffer, chained over two frames |
| test_communicator_argument_checks               | the refusals of vrt_render_distributed, vrt_comm_frame_device, vrt_comm_create, vrt_comm_connect |
| test_temporal_blend_takes_one_sample_per_frame  | spp != 1 without use_samples is refused on every frame path (the blend would wrap the sums) |

Every frame is compared with the oracle: the 8-bit image exactly, and the per-class ray and loop-trip counts exactly (contexts
render without beam floors and bounds exits, tests/conftest.py, except where a test turns the product defaults on).

Ranks that share a device each get a context of their own, i.e. a non-blocking stream of their own: the spin kernels that order
the ranks must never sit on a stream another rank needs.  Host buffers are pinned (a copy into pageable memory returns only when
it is done, so rank 0 would wait for ranks not yet enqueued), and every scene renders one frame of the largest size and sample
count before its communicator starts: a scratch buffer that grows frees the old one, and cudaFree waits for the whole device.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

DEMO_VIEW = dict(position=(256, 200, 256), view_angle=(0.3, -0.35))
W1, H1, SPP1 = 330, 187, 8            # world 1: ragged, K6 (>= 8 samples per pixel), beam tiles cut at both edges
WN, HN, SPPN = 203, 77, 12            # world 2-4: 77 % (4 * world) != 0 for every world; 12 samples split over 2, 3 or 4 ranks
THREADS = min(16, os.cpu_count() or 1)


def default_light(depth=9):
    return np.float32([-200, -1000, -300]) * np.float32(1.0 / (1 << depth)) + np.float32(1.0)


def port_params(W, H, depth, cam, light, spp, offset=0, use_samples=True, rows=(0, 0), tiles=(1, 0), checker=(0, 0)):
    from oracle import loader
    p = loader.PortRenderParams()
    p.width, p.height, p.depth, p.guard = W, H, depth, depth
    p.cam_position[:] = [float(x) for x in cam.position]
    p.rot_mat[:] = [float(x) for x in cam.rot_mat]
    p.fov, p.aperture, p.focal_length = cam.fov, cam.aperture, cam.focal_length
    p.light_position[:] = [float(x) for x in light]
    p.use_gi, p.gi_bounces, p.use_samples, p.spp = 1, 2, int(use_samples), spp
    p.seed_lo, p.seed_hi, p.sample_offset = 0x5EED, 0, offset
    p.row_begin, p.row_end, p.threads = rows[0], rows[1], THREADS
    p.tile_step, p.tile_index = tiles
    p.checker, p.checker_area_height = checker
    return p


_oracle_frames = {}


def oracle_render(port, nodes, p, textures, prev=None):
    """port.render, memoised on the parameter block and the previous image (the same oracle frame serves several worlds)."""
    key = (id(nodes), C.string_at(C.addressof(p), C.sizeof(p)), None if prev is None else prev.tobytes())
    if key not in _oracle_frames:
        _oracle_frames[key] = port.render(nodes, p, *textures, prev_rgba=prev)
    return _oracle_frames[key]


def render_params(W, H, spp, offset=0, use_samples=True, checker=(0, 0), light=None):
    from cpuvoxelraycaster_b200 import capi
    p = capi.RenderParams()
    p.width, p.height, p.row_begin, p.row_end = W, H, 0, H
    p.spp, p.sample_offset = spp, offset
    p.seed_lo, p.seed_hi = 0x5EED, 0
    p.light_position[:] = [float(x) for x in (default_light() if light is None else light)]
    p.use_gi, p.gi_bounces, p.use_samples = 1, 2, int(use_samples)
    p.max_bounds = 4
    p.checker, p.checker_area_height = checker
    return p


def stats_of(st):
    return list(st.rays), list(st.complexity)


def assert_image(got, want, label):
    bad = np.flatnonzero((np.asarray(got) != want).any(-1).reshape(-1))
    assert bad.size == 0, "%s: %d pixels differ, first at (x, y) = %s" % (label, bad.size, [(int(i % want.shape[1]), int(i // want.shape[1])) for i in bad[:6]])


def pinned(H, W, fill=0x5A):
    import torch
    return torch.full((H * W * 4,), fill, dtype=torch.uint8).pin_memory()


def device_image(addr, H, W):
    """A host copy of the uint8 [H, W, 4] frame at device address `addr` (the caller has synchronised its stream)."""
    import torch

    class _Alias:
        __cuda_array_interface__ = {"shape": (H, W, 4), "typestr": "|u1", "data": (addr, False), "version": 2}
    return torch.as_tensor(_Alias(), device="cuda:0").cpu().numpy()


def lsvo_scene(vrt, ctx, nodes, textures):
    s = vrt.LSVO(ctx, nodes, 9)
    s.set_textures(*textures)
    return s


def frame_renderer(vrt, scene, W, H, exchange="peer", split="tiles", light=None):
    import torch
    from cpuvoxelraycaster_b200.frame import FrameRenderer
    dev = torch.device("cuda", 0)
    fr = FrameRenderer(scene, W, H, 0, 1, None, dev, torch.cuda.Stream(dev), exchange=exchange, split=split)
    fr.use_gi, fr.gi_bounces, fr.use_samples = True, 2, True
    fr.light = default_light() if light is None else light
    return fr


def close_renderer(fr):
    if fr is not None and fr.peer is not None:
        fr.stream.synchronize()
        fr.peer.close()


# ---- world 1, as benchmarked ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("split", ["tiles", "samples"])
def test_world1_frames_as_benchmarked(vrt, port, terrain9_nodes, textures, split):
    """The world-1 peer FrameRenderer that bench.py times: three frames of consecutive sample batches through render(), two
    through render_device() (and frame_device_ptr(1) still holding the earlier one), four through render_pipelined() + flush()
    (the host frames then hold the last two), every one u8-exact with exact stats."""
    cam = vrt.Camera(aperture=0.5, focal_length=60.0, **DEMO_VIEW)
    want = [oracle_render(port, terrain9_nodes, port_params(W1, H1, 9, cam, default_light(), SPP1, k * SPP1), textures) for k in range(4)]
    assert want[0][1][..., :3].max() > 0
    c = vrt.Context(0)
    fr = None
    try:
        s = lsvo_scene(vrt, c, terrain9_nodes, textures)
        fr = frame_renderer(vrt, s, W1, H1, split=split)
        for k in range(3):
            img = fr.render(cam, SPP1, k * SPP1)
            assert_image(img, want[k][1], "%s render() frame %d" % (split, k))
            st = fr.stats()
            assert (st["rays"], st["complexity"]) == stats_of(want[k][2]), (split, k)
        a = fr.render_device(cam, SPP1, 0)
        fr.stream.synchronize()
        assert_image(a.cpu().numpy(), want[0][1], split + " render_device() frame 0")
        b = fr.render_device(cam, SPP1, SPP1)
        fr.stream.synchronize()
        assert_image(b.cpu().numpy(), want[1][1], split + " render_device() frame 1")
        assert_image(device_image(fr.peer.frame_device_ptr(1), H1, W1), want[0][1], split + " frame_device_ptr(1)")
        assert_image(device_image(fr.peer.frame_device_ptr(0), H1, W1), want[1][1], split + " frame_device_ptr(0)")
        i0, K = fr.frames_done, 4
        for k in range(K):
            assert fr.render_pipelined(cam, SPP1, k * SPP1) is None
        last = fr.flush()
        assert_image(last, want[K - 1][1], split + " flush()")
        assert_image(fr.host_frames[(i0 + K - 1) & 1].view(H1, W1, 4).numpy(), want[K - 1][1], split + " host frame K-1")
        assert_image(fr.host_frames[(i0 + K - 2) & 1].view(H1, W1, 4).numpy(), want[K - 2][1], split + " host frame K-2")
        st = fr.stats()
        assert (st["rays"], st["complexity"]) == stats_of(want[K - 1][2]), split
    finally:
        close_renderer(fr)
        c.close()


def test_world1_product_defaults_and_nccl_exchange(vrt, port, terrain9_nodes, textures):
    """With beam floors (beam_tile 8) and bounds exits on, the peer frames keep their pixels and ray counts and walk no more;
    the torch exchange (vrt_render_accumulate_device + resolve_kernel) gives the same frames."""
    cam = vrt.Camera(aperture=0.5, focal_length=60.0, **DEMO_VIEW)
    want = [oracle_render(port, terrain9_nodes, port_params(W1, H1, 9, cam, default_light(), SPP1, k * SPP1), textures) for k in range(2)]
    c = vrt.Context(0)
    try:
        s = lsvo_scene(vrt, c, terrain9_nodes, textures)
        for beam in (0, 1):
            c.set_option("beam_tile", 8 * beam)
            c.set_option("bounds_exit", beam)
            for exchange in ("peer", "nccl"):
                fr = frame_renderer(vrt, s, W1, H1, exchange=exchange)
                try:
                    for k in range(2):
                        img = fr.render(cam, SPP1, k * SPP1)
                        label = "%s exchange, product defaults %d, frame %d" % (exchange, beam, k)
                        assert_image(img, want[k][1], label)
                        st = fr.stats()
                        assert st["rays"] == list(want[k][2].rays), label
                        if beam:
                            assert all(x <= y for x, y in zip(st["complexity"], want[k][2].complexity)), label
                            assert st["complexity"][0] < want[k][2].complexity[0], label
                        else:
                            assert st["complexity"] == list(want[k][2].complexity), label
                finally:
                    close_renderer(fr)
    finally:
        c.close()


def test_benchmark_frame_crop_vs_oracle(vrt, port, textures):
    """bench.py's frame, restated from its workload(): T(11) = 2048^3, 1920x1080, 64 spp, GI with 2 bounces, aperture 0.5, camera
    C(11) with Camera.autofocus, seed (0x5EED, 0), the product defaults, through the world-1 peer renderer.  Rows 536-568 (the
    horizon band) u8-exact against the oracle; render_device(), render() and render_pipelined() + flush() give the same bytes."""
    S, W, H, spp = 2048, 1920, 1080, 64
    rows = (536, 568)
    c = vrt.Context(0)
    c.set_option("beam_tile", 8)
    c.set_option("bounds_exit", 1)
    fr = None
    try:
        s = vrt.LSVO.from_terrain(c, 11)
        s.set_textures(*textures)
        cam = vrt.Camera(position=(S / 2.0, S / 2.0 - 56.0, S / 2.0), view_angle=(0.0, 0.0), aperture=0.5)
        cam.autofocus(s)
        light = np.float32([-200, -1000, -300]) * np.float32(1.0 / S) + np.float32(1.0)
        fr = frame_renderer(vrt, s, W, H, light=light)
        fr.seed = (0x5EED, 0)
        host = fr.render(cam, spp).copy()
        dev = fr.render_device(cam, spp)
        fr.stream.synchronize()
        assert np.array_equal(dev.cpu().numpy(), host)
        for _ in range(2):
            fr.render_pipelined(cam, spp)
        assert np.array_equal(fr.flush(), host)
        _, want, _ = port.render(port.build_terrain(11), port_params(W, H, 11, cam, light, spp, rows=rows), *textures)
        assert_image(host[rows[0]:rows[1]], want[rows[0]:rows[1]], "benchmark frame, rows %d-%d" % rows)
        assert host[rows[0]:rows[1], :, :3].max() > 0
    finally:
        close_renderer(fr)
        c.close()


# ---- several ranks on one device ----------------------------------------------------------------------------------------------
class LocalComm:
    """`world` contexts on device 0, one T(9) scene each, joined by vrt_comm_create_local."""

    def __init__(self, vrt, nodes, textures, world, W, H, warm_spp):
        from cpuvoxelraycaster_b200 import capi
        self.capi, self.world, self.W, self.H = capi, world, W, H
        self.ctxs = [vrt.Context(0) for _ in range(world)]
        self.scenes = [lsvo_scene(vrt, c, nodes, textures) for c in self.ctxs]
        warm = render_params(W, H, warm_spp)
        cam = vrt.Camera(aperture=0.5, focal_length=60.0, **DEMO_VIEW).as_struct()
        rgba = np.zeros((H, W, 4), np.uint8)
        for s in self.scenes:                   # scratch buffers at their largest before any spin kernel is enqueued
            capi.check(capi.lib().vrt_render(s.handle, C.byref(cam), C.byref(warm), capi.ptr(rgba), None, None))
        ctxs = (C.c_void_p * world)(*[c.handle.value for c in self.ctxs])
        out = (C.c_void_p * world)()
        capi.check(capi.lib().vrt_comm_create_local(ctxs, world, W, H, out))
        self.comm = [C.c_void_p(out[r]) for r in range(world)]

    def render(self, rank, cam, p, split, deliver_all=False, host=None, scene=None):
        sc = self.scenes[rank] if scene is None else scene
        self.capi.check(self.capi.lib().vrt_render_distributed(self.comm[rank], sc.handle, C.byref(cam), C.byref(p), split,
                                                               int(deliver_all), self.capi.ptr(host)))

    def wait_all(self):
        for r in range(self.world):
            self.capi.check(self.capi.lib().vrt_comm_frame_wait(self.comm[r]))

    def frame_device(self, rank, frames_ago):
        p = C.c_void_p()
        self.capi.check(self.capi.lib().vrt_comm_frame_device(self.comm[rank], frames_ago, C.byref(p)))
        return p.value

    def stats(self, rank):
        st = self.capi.RenderStats()
        self.capi.check(self.capi.lib().vrt_scene_last_render_stats(self.scenes[rank].handle, C.byref(st)))
        return stats_of(st)

    def close(self):
        for h in self.comm:
            self.capi.lib().vrt_comm_destroy(h)
        self.comm = []
        for c in self.ctxs:
            c.close()


@pytest.mark.parametrize("world", [2, 3, 4])
def test_ranks_sharing_one_gpu(vrt, port, terrain9_nodes, textures, world):
    """world ranks on one B200.  For the tile and the sample split, each enqueued in rank order and in reverse order, delivered
    to rank 0's host buffer and (deliver_all) to every rank's: three back-to-back frames, each equal to the oracle frame; after the
    last one every rank's stats equal the oracle's for that rank's share of the frame.  Then a 4-frame temporal-blend
    checkerboard sequence (tile split, one sample per frame) continues from the last delivered frame, against the oracle's blend."""
    from cpuvoxelraycaster_b200 import capi
    cam = vrt.Camera(aperture=0.5, focal_length=60.0, **DEMO_VIEW)
    cs, light = cam.as_struct(), default_light()
    want = [oracle_render(port, terrain9_nodes, port_params(WN, HN, 9, cam, light, SPPN, k * SPPN), textures) for k in range(3)]
    share = {capi.SPLIT_TILES: [port_params(WN, HN, 9, cam, light, SPPN, 2 * SPPN, tiles=(world, r)) for r in range(world)],
             capi.SPLIT_SAMPLES: [port_params(WN, HN, 9, cam, light, SPPN // world, 2 * SPPN + r * (SPPN // world)) for r in range(world)]}
    lc = LocalComm(vrt, terrain9_nodes, textures, world, WN, HN, SPPN)
    try:
        runs = [(split, order, deliver_all) for split in (capi.SPLIT_TILES, capi.SPLIT_SAMPLES)
                for order in ("rank order", "reverse order") for deliver_all in (False, True)]
        runs.append(runs[0])                    # a tile-split frame right after sample-split ones
        for split, order, deliver_all in runs:
            ranks = list(range(world)) if order == "rank order" else list(range(world))[::-1]
            receivers = list(range(world)) if deliver_all else [0]
            hosts = [{r: pinned(HN, WN) for r in receivers} for _ in range(3)]
            for k in range(3):
                p = render_params(WN, HN, SPPN, k * SPPN)
                for r in ranks:
                    lc.render(r, cs, p, split, deliver_all, hosts[k].get(r))
            lc.wait_all()
            label = "world %d, %s split, %s, deliver_all %d" % (world, "tile" if split == capi.SPLIT_TILES else "sample", order, deliver_all)
            for k in range(3):
                for r in receivers:
                    assert_image(hosts[k][r].view(HN, WN, 4).numpy(), want[k][1], "%s: frame %d on rank %d" % (label, k, r))
            for r in receivers:
                assert_image(device_image(lc.frame_device(r, 0), HN, WN), want[2][1], "%s: device frame on rank %d" % (label, r))
            rays, cx = np.zeros(6, np.uint64), np.zeros(6, np.uint64)
            for r in range(world):
                got = lc.stats(r)
                assert got == stats_of(oracle_render(port, terrain9_nodes, share[split][r], textures)[2]), "%s: stats of rank %d" % (label, r)
                rays += np.uint64(got[0])
                cx += np.uint64(got[1])
            assert (rays.tolist(), cx.tolist()) == stats_of(want[2][2]), label
        # temporal blend: every rank blends into its own tiles of the previous frame, unrendered checkerboard pixels keep theirs
        prev = want[2][1]
        for k in range(4):
            checker = (1 + (k & 1), 15)
            p = render_params(WN, HN, 1, k, use_samples=False, checker=checker)
            host = pinned(HN, WN)
            for r in range(world):
                lc.render(r, cs, p, capi.SPLIT_TILES, False, host if r == 0 else None)
            lc.wait_all()
            expect = oracle_render(port, terrain9_nodes, port_params(WN, HN, 9, cam, light, 1, k, use_samples=False, checker=checker),
                                   textures, prev=prev)
            assert_image(host.view(HN, WN, 4).numpy(), expect[1], "world %d, blend frame %d" % (world, k))
            assert sum(np.uint64(lc.stats(r)[0][0]) for r in range(world)) == expect[2].rays[0]
            prev = expect[1]
    finally:
        lc.close()


def test_cpp_host_with_three_ranks_on_one_gpu(tmp_path):
    """tests/cpp/multigpu_test.cpp with every rank on device 0: tile and sample splits, and deliver_all into every rank's
    host buffer, byte for byte against vrt_render."""
    from test_gpu_multigpu import build_multigpu_test
    exe, tex = build_multigpu_test(tmp_path)
    r = subprocess.run([exe, tex, "3", "1"], capture_output=True, text=True, timeout=300)
    out = r.stdout[-3000:] + r.stderr[-2000:]
    assert r.returncode == 0 and "multigpu_test: OK" in r.stdout and "MISMATCH" not in r.stdout, out
    assert r.stdout.count("identical") == 3 + 3 + 3, out


# ---- presentation on the device -------------------------------------------------------------------------------------------------
def test_present_device_on_the_peer_frame(vrt, port, terrain9_nodes, textures):
    """main.cpp:159-177 on the communicator's frame buffer: median 0 / 3 / 5, persistence 0.1 / 0.7, two frames chained."""
    cam = vrt.Camera(aperture=0.5, focal_length=60.0, **DEMO_VIEW)
    want = [oracle_render(port, terrain9_nodes, port_params(W1, H1, 9, cam, default_light(), SPP1, k * SPP1), textures)[1] for k in range(2)]
    c = vrt.Context(0)
    fr = None
    try:
        s = lsvo_scene(vrt, c, terrain9_nodes, textures)
        fr = frame_renderer(vrt, s, W1, H1)
        for median in (0, 3, 5):
            for conservation in (0.1, 0.7):
                fr.display = None
                expect = np.zeros((H1, W1, 4), np.uint8)
                for k in range(2):
                    shown = fr.present_device(fr.render_device(cam, SPP1, k * SPP1), median, conservation)
                    expect = port.present(want[k], expect, median, conservation)
                fr.stream.synchronize()
                assert_image(shown.cpu().numpy(), expect, "median %d, conservation %.1f" % (median, conservation))
    finally:
        close_renderer(fr)
        c.close()


# ---- argument checks ------------------------------------------------------------------------------------------------------------
def test_communicator_argument_checks(vrt, terrain9_nodes, textures):
    from cpuvoxelraycaster_b200 import capi
    L = capi.lib()
    cs = vrt.Camera(aperture=0.5, focal_length=60.0, **DEMO_VIEW).as_struct()
    lc = LocalComm(vrt, terrain9_nodes, textures, 2, WN, HN, 4)
    try:
        def refused(rank, p, split, scene=None):
            with pytest.raises(capi.VrtError) as e:
                lc.render(rank, cs, p, split, scene=scene)
            assert e.value.code == -1                                          # VRT_ERR_INVALID
        refused(0, render_params(WN, HN, 3), capi.SPLIT_SAMPLES)               # spp % world != 0
        refused(0, render_params(WN, HN, 4, checker=(1, 0)), capi.SPLIT_SAMPLES)
        refused(0, render_params(WN, HN, 4, use_samples=False), capi.SPLIT_SAMPLES)
        refused(0, render_params(WN + 1, HN, 4), capi.SPLIT_TILES)
        refused(0, render_params(WN, HN - 1, 4), capi.SPLIT_TILES)
        refused(0, render_params(WN, HN, 4), capi.SPLIT_TILES, scene=lc.scenes[1])
        refused(0, render_params(WN, HN, 1, use_samples=False), 2)             # no such split
        with pytest.raises(capi.VrtError):
            lc.frame_device(0, 0)                                              # before any frame
        for k in range(2):
            for r in range(2):
                lc.render(r, cs, render_params(WN, HN, 4, 4 * k), capi.SPLIT_TILES)
            lc.wait_all()
            with pytest.raises(capi.VrtError):
                lc.frame_device(0, k + 1)
            assert lc.frame_device(0, 0)
        assert lc.frame_device(0, 1) != lc.frame_device(0, 0)
        with pytest.raises(capi.VrtError):
            lc.frame_device(0, -1)
        h = C.c_void_p()
        for rank, world in ((2, 2), (-1, 2), (0, 0), (0, 17)):
            with pytest.raises(capi.VrtError):
                capi.check(L.vrt_comm_create(lc.ctxs[0].handle, rank, world, WN, HN, C.byref(h)))
        # two members of one process exported for the IPC path: vrt_comm_connect refuses before opening any handle
        members = []
        try:
            for r in range(2):
                m = C.c_void_p()
                capi.check(L.vrt_comm_create(lc.ctxs[r].handle, r, 2, WN, HN, C.byref(m)))
                members.append(m)
            blobs = [(C.c_uint8 * capi.COMM_HANDLE_BYTES)() for _ in range(2)]
            for m, b in zip(members, blobs):
                capi.check(L.vrt_comm_export(m, b))
            with pytest.raises(capi.VrtError, match="lives in this process"):
                capi.check(L.vrt_comm_connect(members[0], b"".join(bytes(b) for b in blobs)))
        finally:
            for m in members:
                L.vrt_comm_destroy(m)
    finally:
        lc.close()


def test_temporal_blend_takes_one_sample_per_frame(vrt, port, terrain9_nodes, textures):
    """The blend resolves the accumulated colour as one 8-bit sample, so spp != 1 without use_samples would wrap the sums:
    vrt_render, vrt_render_accumulate_device and vrt_render_distributed (both FrameRenderer exchanges) refuse it.  A refused frame
    leaves no trace: the 1-sample blend frames that follow equal the oracle's."""
    import torch
    from cpuvoxelraycaster_b200 import capi
    L = capi.lib()
    cam = vrt.Camera(aperture=0.5, focal_length=60.0, **DEMO_VIEW)
    cs = cam.as_struct()
    c = vrt.Context(0)
    try:
        s = lsvo_scene(vrt, c, terrain9_nodes, textures)
        bad = render_params(WN, HN, 2, use_samples=False)
        accum = torch.zeros(HN * WN * 4, dtype=torch.int32, device="cuda:0")
        with pytest.raises(capi.VrtError, match="one sample per frame"):
            capi.check(L.vrt_render_accumulate_device(s.handle, C.byref(cs), C.byref(bad), capi.ptr(accum)))
        with pytest.raises(capi.VrtError, match="one sample per frame"):
            capi.check(L.vrt_render(s.handle, C.byref(cs), C.byref(bad), capi.ptr(np.zeros((HN, WN, 4), np.uint8)), None, None))
        for exchange in ("peer", "nccl"):
            fr = frame_renderer(vrt, s, WN, HN, exchange=exchange)
            try:
                fr.use_samples = False
                prev = None
                for k in range(3):
                    with pytest.raises(capi.VrtError, match="one sample per frame"):
                        fr.render(cam, 2, k)
                    img = fr.render(cam, 1, k)
                    _, want, _ = oracle_render(port, terrain9_nodes, port_params(WN, HN, 9, cam, default_light(), 1, k, use_samples=False),
                                               textures, prev=prev)
                    assert_image(img, want, "%s exchange, blend frame %d" % (exchange, k))
                    prev = want
            finally:
                close_renderer(fr)
    finally:
        c.close()
