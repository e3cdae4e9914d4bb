"""Whole-frame rendering on 1..N GPUs of one box — the replacement of the reference's per-frame driver,
the swarm lambda src/main.cpp:139-154 (16 CPU threads in 4x4 screen tiles) + samples_to_image (:156-158).

One process per GPU.  The voxel scene is replicated; a frame is split over the ranks either by 4-row tiles dealt
round-robin (sky and terrain rows cost very differently, so contiguous slabs would be unbalanced) or by samples
(every rank renders all pixels for spp / world of the samples; the integer accumulators add up exactly).  Because the
RNG is counter based (pixel, sample, dimension) the assembled frame is bit-identical for every world size and both splits.

Two exchange paths:
  * `PeerFrame` (default on GPUs): libvrt's own communicator (include/vrt.h "multi-GPU frames", csrc/comm.cu) — the
    resolve kernel stores finished pixels straight into rank 0's frame buffer over NVLink (peer-mapped memory, CUDA IPC
    between the processes), frames are double buffered and copied to the host on a second stream.  torch.distributed is
    used once, to all-gather the 256-byte IPC handles.
  * `TileExchange`: one all-gather of RGBA tiles through torch.distributed (NCCL on GPUs; gloo in the CPU tests).

torch is used for device buffers, the stream and torch.distributed only.
"""
import ctypes as C

import numpy as np
import torch

from . import capi
from .capi import check, lib, ptr


class TileExchange:
    """Round-robin 4-row-tile partition of a W x H RGBA frame over `world` ranks and its all-gather.
    Pure torch (any device / backend): NCCL on the GPUs, gloo in the CPU tests."""

    def __init__(self, width, height, rank, world, device, group=None):
        self.W, self.H, self.rank, self.world, self.group = int(width), int(height), int(rank), int(world), group
        unit = 4 * self.world
        self.H_pad = (self.H + unit - 1) // unit * unit
        self.tiles_local = self.H_pad // unit
        self.row_bytes = self.W * 4
        self.tile_bytes = 4 * self.row_bytes
        if self.world > 1:
            self.slab = torch.empty(self.tiles_local * self.tile_bytes, dtype=torch.uint8, device=device)
            self.gathered = torch.empty(self.world * self.slab.numel(), dtype=torch.uint8, device=device)
            self.frame = torch.empty(self.H_pad * self.row_bytes, dtype=torch.uint8, device=device)

    def owned_rows(self):
        """Rows this rank renders: 4-row tile t belongs to rank t % world."""
        return [y for y in range(self.H) if (y >> 2) % self.world == self.rank]

    def gather(self, rgba):
        """rgba: flat uint8 [H_pad*W*4] with this rank's rows filled → the assembled frame on every rank."""
        if self.world == 1:
            return rgba
        import torch.distributed as dist
        tiles = rgba.view(self.tiles_local, self.world, self.tile_bytes)                # [local tile, owner, bytes]
        self.slab.view(self.tiles_local, self.tile_bytes).copy_(tiles[:, self.rank, :])
        dist.all_gather_into_tensor(self.gathered, self.slab, group=self.group)
        g = self.gathered.view(self.world, self.tiles_local, self.tile_bytes)
        self.frame.view(self.tiles_local, self.world, self.tile_bytes).copy_(g.permute(1, 0, 2))
        return self.frame


class PeerFrame:
    """libvrt's multi-GPU communicator for one process per GPU (vrt_comm_create / export / connect).
    `bootstrap(blob: bytes) -> list[bytes]` all-gathers the ranks' export blobs in rank order; the default uses
    torch.distributed (any backend)."""

    def __init__(self, ctx, width, height, rank, world, group=None, bootstrap=None):
        self.ctx, self.rank, self.world = ctx, int(rank), int(world)
        h = C.c_void_p()
        check(lib().vrt_comm_create(ctx.handle, self.rank, self.world, int(width), int(height), C.byref(h)))
        self.handle = h
        if self.world > 1:
            blob = (C.c_uint8 * capi.COMM_HANDLE_BYTES)()
            check(lib().vrt_comm_export(self.handle, blob))
            blobs = (bootstrap or self._torch_bootstrap(group))(bytes(blob))
            joined = b"".join(blobs)
            assert len(joined) == self.world * capi.COMM_HANDLE_BYTES
            check(lib().vrt_comm_connect(self.handle, joined))

    @staticmethod
    def _torch_bootstrap(group):
        def gather(blob):
            import torch.distributed as dist
            out = [None] * dist.get_world_size(group)
            dist.all_gather_object(out, blob, group=group)
            return out
        return gather

    def render(self, scene, cam_struct, p, split=capi.SPLIT_TILES, deliver_all=False, host_rgba=None):
        """Enqueues one frame on every rank (vrt_render_distributed)."""
        check(lib().vrt_render_distributed(self.handle, scene.handle, C.byref(cam_struct), C.byref(p), int(split), int(bool(deliver_all)),
                                           ptr(host_rgba)))

    def wait(self):
        check(lib().vrt_comm_frame_wait(self.handle))

    def frame_device_ptr(self, frames_ago=0):
        p = C.c_void_p()
        check(lib().vrt_comm_frame_device(self.handle, int(frames_ago), C.byref(p)))
        return p.value

    def close(self):
        if self.handle:
            check(lib().vrt_comm_destroy(self.handle))
            self.handle = None


class FrameRenderer:
    def __init__(self, scene, width, height, rank=0, world=1, group=None, device=None, stream=None, exchange="auto", split="tiles"):
        self.scene, self.W, self.H = scene, int(width), int(height)
        self.rank, self.world, self.group = int(rank), int(world), group
        self.device = device if device is not None else torch.device("cuda", scene.ctx.device)
        # libvrt's launches and torch's copies/collectives must share one stream
        self.stream = stream if stream is not None else torch.cuda.Stream(self.device)
        scene.ctx.set_stream(self.stream.cuda_stream)      # libvrt re-applies an installed L2 access-policy window to it
        scene.ctx.torch_stream = self.stream               # keeps the cudaStream_t alive as long as the context uses it
        # Device buffers are created ON the render stream: their zero fills are then ordered before the first frame (on torch's
        # current stream — the default one, behind whatever collective is still pending there — a fill could land between a frame's
        # trace and its resolve and wipe the accumulator: seen as all-zero tiles of one rank in the first frame on 4 GPUs), and the
        # caching allocator ties the blocks to the stream that uses them.
        with torch.cuda.stream(self.stream):
            self.exchange = TileExchange(self.W, self.H, self.rank, self.world, self.device, group)
            self.H_pad, self.row_bytes = self.exchange.H_pad, self.exchange.row_bytes
            self.accum = torch.zeros(self.H_pad * self.W * 4, dtype=torch.int32, device=self.device)   # r,g,b,count sums
            self.rgba = torch.zeros(self.H_pad * self.W * 4, dtype=torch.uint8, device=self.device)
        # two pinned host frames: frame i is copied out while frame i+1 renders (render_pipelined)
        self.host_frames = [torch.empty(self.H * self.row_bytes, dtype=torch.uint8).pin_memory() for _ in range(2)]
        self.host_frame = self.host_frames[0]
        self.frames_done = 0
        self.use_gi, self.gi_bounces, self.use_samples = False, 1, True
        self.roughness, self.max_bounds = 0.0, 4
        self.mirror_y = None                                              # LSVO frames: mirror layer (vrt_render_params::mirror_y1 - 1)
        self.checker_board_offset, self.checker_area_height = None, 0     # main.cpp:137,143 / :132
        self.display = None                                               # denoised_tex of main.cpp:159-177
        self.autofocus = False                                            # device-side centre-ray focus, main.cpp:114-121
        self.seed = (0x5EED, 0)
        self.light = np.zeros(3, np.float32)
        # multi-GPU exchange: "peer" = libvrt communicator (NVLink peer stores), "nccl" = torch.distributed all-gather
        if exchange == "auto":
            import torch.distributed as dist
            live = dist.is_available() and dist.is_initialized()     # probes simulate "rank r of N" in one process: no peers there
            exchange = "peer" if (self.world > 1 and self.device.type == "cuda" and live) else "nccl"
        self.exchange_kind = exchange
        self.split = capi.SPLIT_SAMPLES if split == "samples" else capi.SPLIT_TILES
        self.peer = PeerFrame(scene.ctx, self.W, self.H, self.rank, self.world, group) if exchange == "peer" else None

    def params(self, spp, sample_offset=0):
        p = capi.RenderParams()
        p.width, p.height, p.row_begin, p.row_end = self.W, self.H, 0, self.H
        p.spp, p.sample_offset = int(spp), int(sample_offset)
        p.seed_lo, p.seed_hi = self.seed
        p.light_position[:] = [float(x) for x in self.light]
        p.use_gi, p.gi_bounces, p.use_samples = int(self.use_gi), int(self.gi_bounces), int(self.use_samples)
        p.tile_step, p.tile_index = self.world, self.rank
        p.roughness, p.max_bounds = float(self.roughness), int(self.max_bounds)
        p.checker = 0 if self.checker_board_offset is None else 1 + (int(self.checker_board_offset) & 1)
        p.checker_area_height = int(self.checker_area_height)
        p.mirror_y1 = 0 if self.mirror_y is None else int(self.mirror_y) + 1
        p.autofocus = int(bool(self.autofocus))
        return p

    # -- device-resident frame: enqueue only (the caller owns stream/synchronisation) --
    def accumulate(self, cam_struct, p):
        check(lib().vrt_render_accumulate_device(self.scene.handle, C.byref(cam_struct), C.byref(p), ptr(self.accum)))

    def resolve(self, p):
        check(lib().vrt_render_resolve_device(self.scene.handle, C.byref(p), ptr(self.accum), ptr(self.rgba)))

    def gather(self):
        """All-gather of the ranks' RGBA tiles (the torch.distributed exchange path).  No-op on one GPU."""
        return self.exchange.gather(self.rgba)

    def render_device(self, camera, spp, sample_offset=0, clear=True):
        """One frame, device resident: clear, accumulate, resolve, exchange.  Returns a uint8 view [H, W, 4] of the
        assembled frame — on every rank with the all-gather exchange, on rank 0 with the peer exchange (None elsewhere)."""
        p = self.params(spp, sample_offset)
        if self.peer is not None:
            with torch.cuda.stream(self.stream):
                self.peer.render(self.scene, camera.as_struct(), p, self.split)
            self.frames_done += 1
            return self._peer_frame_view() if self.rank == 0 else None
        with torch.cuda.stream(self.stream):
            if clear:
                self.accum.zero_()
            self.accumulate(camera.as_struct(), p)
            self.resolve(p)
            frame = self.gather()
        return frame.view(self.H_pad, self.W, 4)[: self.H]

    def _peer_frame_view(self):
        """uint8 [H, W, 4] tensor aliasing the communicator's most recent frame buffer (valid for two frames)."""
        addr = self.peer.frame_device_ptr(0)

        class _Alias:
            __cuda_array_interface__ = {"shape": (self.H, self.W, 4), "typestr": "|u1", "data": (addr, False), "version": 2}
        return torch.as_tensor(_Alias(), device=self.device)

    def present_device(self, frame, median=0, old_value_conservation=0.1):
        """main.cpp:159-177 on the device: optional median, then the persistence blend of `frame` (a device uint8
        [H, W, 4] view such as render_device returns) into the display surface, which is returned."""
        if self.display is None:
            with torch.cuda.stream(self.stream):             # fill ordered before the first use (see __init__)
                self.display = torch.zeros(self.H * self.W * 4, dtype=torch.uint8, device=self.device)
        p = capi.PresentParams(self.W, self.H, int(median), float(old_value_conservation))
        with torch.cuda.stream(self.stream):
            check(lib().vrt_present_device(self.scene.ctx.handle, ptr(frame), ptr(self.display), C.byref(p)))
        return self.display.view(self.H, self.W, 4)

    def render(self, camera, spp, sample_offset=0):
        """The user-facing call: a finished frame in host memory (pinned), as numpy [H, W, 4] uint8 — on rank 0 with the
        peer exchange (other ranks return None), on every rank otherwise."""
        if self.peer is not None:
            p = self.params(spp, sample_offset)
            host = self.host_frame if self.rank == 0 else None
            with torch.cuda.stream(self.stream):
                self.peer.render(self.scene, camera.as_struct(), p, self.split, False, host)
            self.frames_done += 1
            self.peer.wait()
            return self.host_frame.view(self.H, self.W, 4).numpy() if self.rank == 0 else None
        frame = self.render_device(camera, spp, sample_offset)
        with torch.cuda.stream(self.stream):
            self.host_frame.view(self.H, self.W, 4).copy_(frame, non_blocking=True)
        self.stream.synchronize()
        return self.host_frame.view(self.H, self.W, 4).numpy()

    def render_pipelined(self, camera, spp, sample_offset=0):
        """Streaming form of render() for the peer exchange: enqueues this frame (its host copy runs on a second stream
        while the next frame renders) and returns None.  K calls + flush() deliver K frames: frame i (counted by
        frames_done) is copied to host_frames[i & 1], so after flush() the last two frames are in host memory."""
        assert self.peer is not None, "render_pipelined needs the peer exchange"
        p = self.params(spp, sample_offset)
        i = self.frames_done
        host = self.host_frames[i & 1] if self.rank == 0 else None
        with torch.cuda.stream(self.stream):
            self.peer.render(self.scene, camera.as_struct(), p, self.split, False, host)
        self.frames_done += 1
        # vrt_render_distributed makes frame i wait for the host copy of frame i-2 (same buffers), so host_frames[(i-1)&1]
        # is complete once the copy stream has passed frame i-1: that is guaranteed after the NEXT call's wait, or flush()
        return None

    def flush(self):
        """Completes all frames in flight; returns the last frame's host image on rank 0."""
        if self.peer is None:
            self.stream.synchronize()
            return None
        self.peer.wait()
        if self.rank != 0 or self.frames_done == 0:
            return None
        return self.host_frames[(self.frames_done - 1) & 1].view(self.H, self.W, 4).numpy()

    def stats(self):
        st = capi.RenderStats()
        check(lib().vrt_scene_last_render_stats(self.scene.handle, C.byref(st)))
        culled = C.c_uint64(0)                      # primary rays answered by the beam search (counted in rays[0], no walk)
        check(lib().vrt_scene_last_render_culled(self.scene.handle, C.byref(culled)))
        return dict(rays=list(st.rays), complexity=list(st.complexity), culled_primary=int(culled.value))
