// Multi-GPU frames behind the C ABI (include/vrt.h, "multi-GPU frames").
//
// Replaces the reference's only parallel decomposition — 16 CPU threads, one 4x4 screen area each, src/main.cpp:139-143 —
// across the GPUs of one box.  The voxel scene is replicated; a frame is split either by 4-row TILES dealt round-robin to
// the ranks, or by SAMPLES (every rank renders all pixels for spp/world of the samples; the integer accumulators add up
// exactly, so both splits give the byte-identical frame).  There is no collective library in the data path:
//
//   * every rank owns one "window" allocation: [flags | 2 RGBA frame buffers | accumulator], exported with
//     cudaIpcGetMemHandle (one process per GPU) or used directly with peer access (one process driving several GPUs);
//   * resolve_push_kernel turns a rank's accumulators into RGBA and STORES the pixels straight into the frame buffer of
//     the delivery rank(s) over NVLink (plain st.global on peer-mapped addresses) — resolve and gather are one kernel;
//   * in the sample split reduce_push_kernel first LOADS the other ranks' accumulators for the rank's own tiles over
//     NVLink and adds them (a reduce-scatter by peer loads), then resolves and pushes as above;
//   * ordering between ranks uses monotonically increasing counters in the delivery rank's window: a 1-thread kernel
//     adds to them after a rank's stores (stream order makes the stores visible first), a 1-thread kernel spins on them
//     where a rank has to wait.  Frame buffers are double buffered: frame i+1 is rendered and pushed while frame i is
//     copied to the host on a second stream.
//
// Spin kernels give up after ~4 s (a peer died) and record an error instead of hanging the GPU.
#include <cstdio>
#include <cstring>
#include <new>
#include <string>
#include <vector>
#include <unistd.h>

#include "capi_internal.h"

using vrt::cuda_fail;
using vrt::fail;
using vrt::use_device;

namespace {

constexpr uint32_t kMagic = 0x56525443u;   // "VRTC"
constexpr int kMaxWorld = 16;

// Counters at the start of every window; only the ones in the ROOT's window (and, for deliver_all, in each window) are used.
struct Flags {
    unsigned long long unused0;
    unsigned long long consumed;   // frames of this window's buffers that have been handed to the consumer (host copy done)
    unsigned long long acc_done;   // sample split: += 1 per rank and frame when its accumulator is complete
    unsigned long long reduced;    // sample split: += 1 per rank and frame when it has finished reading the peers' accumulators
    unsigned long long error;      // != 0: a wait timed out
    unsigned long long pad[3];
    // arrived_from[r] = 1 + ordinal of the latest frame whose tiles rank r has stored into this window's frame buffer.  One slot
    // per SOURCE: a shared arrival count cannot tell a fast rank's next frame from a slow rank's current one (with three or more
    // ranks the consumer then takes a frame before its last tiles are in — found by tests/multigpu_frame_check.py on 4 GPUs).
    unsigned long long arrived_from[kMaxWorld];
};
static_assert(sizeof(Flags) == 64 + 8 * kMaxWorld && sizeof(Flags) <= 256, "Flags layout (the window header is 256 bytes)");

struct Blob {                      // what vrt_comm_export writes: VRT_COMM_HANDLE_BYTES
    uint32_t magic, rank, world, device;
    uint64_t pid, bytes;
    int32_t width, height;
    cudaIpcMemHandle_t handle;
    char pad[VRT_COMM_HANDLE_BYTES - 40 - sizeof(cudaIpcMemHandle_t)];
};
static_assert(sizeof(Blob) == VRT_COMM_HANDLE_BYTES, "Blob layout");

}  // namespace

struct vrt_comm {
    vrt_context* ctx = nullptr;
    int rank = 0, world = 1, root = 0;
    int width = 0, height = 0, h_pad = 0;
    size_t frame_bytes = 0, accum_bytes = 0, window_bytes = 0;
    char* window = nullptr;                 // this rank's allocation
    char* peer[kMaxWorld] = {};             // every rank's window as seen from this device (peer[rank] == window)
    bool opened[kMaxWorld] = {};            // peer[r] came from cudaIpcOpenMemHandle
    bool connected = false;
    uint64_t frame_no = 0;                  // frames started
    uint64_t sample_frames = 0;             // frames rendered with the sample split so far (orders acc_done / reduced)
    long long last_in_buf[kMaxWorld][2];    // frame ordinal last delivered into buffer b of rank t's window (-1: none); identical on all ranks
    cudaStream_t copy_stream = nullptr;     // root: device-to-host copies overlap the next frame
    cudaEvent_t frame_ready = nullptr, copy_done[2] = {nullptr, nullptr};
    bool copy_pending[2] = {false, false};
    uint8_t* local_rgba = nullptr;          // this rank's own resolved pixels (previous frame of the temporal blend)

    Flags* flags(int r) const { return reinterpret_cast<Flags*>(peer[r]); }
    uint8_t* frame(int r, int buf) const { return reinterpret_cast<uint8_t*>(peer[r] + 256 + size_t(buf) * frame_bytes); }
    uint32_t* accum(int r) const { return reinterpret_cast<uint32_t*>(peer[r] + 256 + 2 * frame_bytes); }
};

namespace {

__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

// += 1 on a (possibly remote) counter.  Launched after the kernel whose stores it publishes: stream order completes
// those stores first; the fence orders them before the counter update for observers on other devices.
__global__ void signal_kernel(unsigned long long* counter, unsigned long long add) {
    __threadfence_system();
    atomicAdd_system(counter, add);
}
__global__ void set_kernel(unsigned long long* counter, unsigned long long value) {
    __threadfence_system();
    atomicMax_system(counter, value);
}
// spins until counter[0..n) are all >= want
__global__ void wait_all_kernel(const unsigned long long* counter, int n, unsigned long long want, unsigned long long* err) {
    unsigned long long t0, t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    for (int r = 0; r < n; ++r)
        while (ld_acquire_sys(counter + r) < want) {
            __nanosleep(200);
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
            if (t - t0 > 4000000000ull) {
                atomicAdd_system(err, 1ull);
                return;
            }
        }
}
// spins until *counter >= want (at most ~4 s of globaltimer), else records an error in `err`
__global__ void wait_kernel(const unsigned long long* counter, unsigned long long want, unsigned long long* err) {
    unsigned long long t0, t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    while (ld_acquire_sys(counter) < want) {
        __nanosleep(200);
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        if (t - t0 > 4000000000ull) {
            atomicAdd_system(err, 1ull);
            return;
        }
    }
}

struct Targets {
    uint8_t* frame[kMaxWorld];
    int n;
};
struct Sources {
    const uint32_t* accum[kMaxWorld];
    int n;
};

// samples_to_image (raycaster.hpp:94-103) or the 0.4/0.6 temporal blend (:79-85) for this rank's 4-row tiles, stored into
// the frame buffer of every delivery target.  kReduce: the pixel's sums are first added up over all ranks' accumulators.
template <bool kReduce>
__global__ void __launch_bounds__(256) resolve_push_kernel(Sources src, Targets dst, uint8_t* __restrict__ local_rgba, int width, int height,
                                                           int use_samples, int tile_step, int tile_index) {
    const uint64_t j = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    const int x = int(j % uint64_t(width));
    const int row = int(j / uint64_t(width));
    const int y = ((row >> 2) * tile_step + tile_index) * 4 + (row & 3);
    if (y >= height) return;
    const uint64_t i = uint64_t(y) * width + x;
    uint4 a = reinterpret_cast<const uint4*>(src.accum[0])[i];
    if (kReduce) {
        for (int r = 1; r < src.n; ++r) {
            const uint4 b = reinterpret_cast<const uint4*>(src.accum[r])[i];     // peer load over NVLink
            a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
        }
    }
    uchar4 out;
    if (use_samples) {
        const uint32_t n = a.w ? a.w : 1u;
        out = make_uchar4(uint8_t(a.x / n), uint8_t(a.y / n), uint8_t(a.z / n), 255);
    } else {
        const uchar4 old = reinterpret_cast<const uchar4*>(local_rgba)[i];
        if (a.w == 0u) {
            out = old;                                                             // not rendered this frame (checkerboard)
        } else {
            auto mul = [](uint8_t c, float f) { return uint8_t(fminf(255.0f, float(c) * f)); };   // utils.cpp:43-48
            const int r = min(255, int(mul(old.x, 0.4f)) + int(mul(uint8_t(a.x), 1.0f - 0.4f)));
            const int g = min(255, int(mul(old.y, 0.4f)) + int(mul(uint8_t(a.y), 1.0f - 0.4f)));
            const int b = min(255, int(mul(old.z, 0.4f)) + int(mul(uint8_t(a.z), 1.0f - 0.4f)));
            out = make_uchar4(uint8_t(r), uint8_t(g), uint8_t(b), 255);
        }
    }
    reinterpret_cast<uchar4*>(local_rgba)[i] = out;
    for (int t = 0; t < dst.n; ++t) reinterpret_cast<uchar4*>(dst.frame[t])[i] = out;   // peer store over NVLink
}

// Loads the communicator's kernels into the current context.  With lazy module loading (the CUDA 12 default) a kernel is loaded
// at its first launch, and loading may synchronise the context: a first launch queued behind a spin kernel then blocks the host
// until the spin ends — which, with one thread driving several ranks, waits for ranks that thread has not enqueued yet (seen on
// one GPU: the first sample-split frame timed out in resolve_push_kernel<true>).
cudaError_t load_comm_kernels() {
    const void* kernels[] = {reinterpret_cast<const void*>(signal_kernel), reinterpret_cast<const void*>(set_kernel),
                             reinterpret_cast<const void*>(wait_all_kernel), reinterpret_cast<const void*>(wait_kernel),
                             reinterpret_cast<const void*>(resolve_push_kernel<false>), reinterpret_cast<const void*>(resolve_push_kernel<true>)};
    cudaFuncAttributes a;
    for (const void* k : kernels)
        if (cudaError_t e = cudaFuncGetAttributes(&a, k)) return e;
    return cudaSuccess;
}

int check_comm(const vrt_comm* c, const char* who) {
    if (!c) return fail(VRT_ERR_INVALID, std::string(who) + ": comm is NULL");
    if (!c->connected) return fail(VRT_ERR_INVALID, std::string(who) + ": call vrt_comm_connect first");
    return VRT_OK;
}

int comm_alloc(vrt_context* ctx, int rank, int world, int width, int height, vrt_comm** out, const char* who) {
    if (!ctx || !out) return fail(VRT_ERR_INVALID, std::string(who) + ": NULL argument");
    if (world < 1 || world > kMaxWorld || rank < 0 || rank >= world) return fail(VRT_ERR_INVALID, std::string(who) + ": need 0 <= rank < world <= 16");
    if (width <= 0 || height <= 0 || width > 65536 || height > 65536) return fail(VRT_ERR_INVALID, std::string(who) + ": bad frame size");
    if (int s = use_device(ctx)) return s;
    if (cudaError_t e = load_comm_kernels()) return cuda_fail(e, who);
    vrt_comm* c = new (std::nothrow) vrt_comm();
    if (!c) return fail(VRT_ERR_OOM, std::string(who) + ": host allocation failed");
    c->ctx = ctx; c->rank = rank; c->world = world; c->width = width; c->height = height;
    const int unit = 4 * world;
    c->h_pad = (height + unit - 1) / unit * unit;
    c->frame_bytes = (size_t(c->h_pad) * width * 4 + 255) & ~size_t(255);
    c->accum_bytes = (size_t(c->h_pad) * width * 16 + 255) & ~size_t(255);
    c->window_bytes = 256 + 2 * c->frame_bytes + c->accum_bytes;
    cudaError_t e = cudaMalloc(&c->window, c->window_bytes);
    if (e == cudaSuccess) e = cudaMalloc(&c->local_rgba, c->frame_bytes);
    if (e == cudaSuccess) e = cudaMemsetAsync(c->window, 0, c->window_bytes, ctx->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(c->local_rgba, 0, c->frame_bytes, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->frame_ready, cudaEventDisableTiming);
    for (int b = 0; b < 2 && e == cudaSuccess; ++b) e = cudaEventCreateWithFlags(&c->copy_done[b], cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
        vrt_comm_destroy(c);
        return e == cudaErrorMemoryAllocation ? fail(VRT_ERR_OOM, std::string(who) + ": device allocation failed") : cuda_fail(e, who);
    }
    for (int t = 0; t < kMaxWorld; ++t) c->last_in_buf[t][0] = c->last_in_buf[t][1] = -1;
    c->peer[rank] = c->window;
    c->connected = world == 1;
    *out = c;
    return VRT_OK;
}

}  // namespace

extern "C" {

int vrt_comm_create(vrt_context* ctx, int rank, int world, int width, int height, vrt_comm** out) {
    return comm_alloc(ctx, rank, world, width, height, out, "vrt_comm_create");
}

int vrt_comm_export(vrt_comm* c, void* blob) {
    if (!c || !blob) return fail(VRT_ERR_INVALID, "vrt_comm_export: NULL argument");
    if (int s = use_device(c->ctx)) return s;
    Blob b;
    std::memset(&b, 0, sizeof(b));
    b.magic = kMagic; b.rank = uint32_t(c->rank); b.world = uint32_t(c->world); b.device = uint32_t(c->ctx->device);
    b.pid = uint64_t(getpid()); b.bytes = c->window_bytes; b.width = c->width; b.height = c->height;
    VRT_CUDA(cudaIpcGetMemHandle(&b.handle, c->window));
    std::memcpy(blob, &b, sizeof(b));
    return VRT_OK;
}

int vrt_comm_connect(vrt_comm* c, const void* blobs) {
    if (!c || !blobs) return fail(VRT_ERR_INVALID, "vrt_comm_connect: NULL argument");
    if (c->connected) return VRT_OK;
    if (int s = use_device(c->ctx)) return s;
    const Blob* B = static_cast<const Blob*>(blobs);
    for (int r = 0; r < c->world; ++r) {
        Blob b;
        std::memcpy(&b, B + r, sizeof(b));
        if (b.magic != kMagic || int(b.rank) != r || int(b.world) != c->world || b.width != c->width || b.height != c->height ||
            b.bytes != c->window_bytes)
            return fail(VRT_ERR_INVALID, "vrt_comm_connect: blob " + std::to_string(r) + " does not describe rank " + std::to_string(r) +
                                             " of this frame geometry (gather the exports in rank order)");
        if (r == c->rank) continue;
        if (b.pid == uint64_t(getpid()))
            return fail(VRT_ERR_INVALID, "vrt_comm_connect: rank " + std::to_string(r) + " lives in this process — use vrt_comm_create_local");
        void* p = nullptr;
        VRT_CUDA(cudaIpcOpenMemHandle(&p, b.handle, cudaIpcMemLazyEnablePeerAccess));
        c->peer[r] = static_cast<char*>(p);
        c->opened[r] = true;
    }
    c->connected = true;
    return VRT_OK;
}

int vrt_comm_create_local(vrt_context* const* ctxs, int world, int width, int height, vrt_comm** out) {
    if (!ctxs || !out) return fail(VRT_ERR_INVALID, "vrt_comm_create_local: NULL argument");
    if (world < 1 || world > kMaxWorld) return fail(VRT_ERR_INVALID, "vrt_comm_create_local: world must be 1..16");
    for (int r = 0; r < world; ++r) out[r] = nullptr;
    for (int r = 0; r < world; ++r)
        if (int s = comm_alloc(ctxs[r], r, world, width, height, &out[r], "vrt_comm_create_local")) {
            for (int q = 0; q < r; ++q) { vrt_comm_destroy(out[q]); out[q] = nullptr; }
            return s;
        }
    for (int r = 0; r < world; ++r) {
        cudaSetDevice(ctxs[r]->device);
        for (int q = 0; q < world; ++q) {
            out[r]->peer[q] = out[q]->window;
            if (q == r || ctxs[q]->device == ctxs[r]->device) continue;
            int can = 0;
            cudaDeviceCanAccessPeer(&can, ctxs[r]->device, ctxs[q]->device);
            cudaError_t e = can ? cudaDeviceEnablePeerAccess(ctxs[q]->device, 0) : cudaErrorPeerAccessUnsupported;
            if (e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); e = cudaSuccess; }
            if (e != cudaSuccess) {
                for (int k = 0; k < world; ++k) { vrt_comm_destroy(out[k]); out[k] = nullptr; }
                return cuda_fail(e, "vrt_comm_create_local: peer access between the devices");
            }
        }
        out[r]->connected = true;
    }
    return VRT_OK;
}

int vrt_comm_destroy(vrt_comm* c) {
    if (!c) return VRT_OK;
    cudaSetDevice(c->ctx->device);
    cudaStreamSynchronize(c->ctx->stream);
    if (c->copy_stream) { cudaStreamSynchronize(c->copy_stream); cudaStreamDestroy(c->copy_stream); }
    for (int r = 0; r < c->world; ++r)
        if (c->opened[r]) cudaIpcCloseMemHandle(c->peer[r]);
    if (c->frame_ready) cudaEventDestroy(c->frame_ready);
    for (int b = 0; b < 2; ++b)
        if (c->copy_done[b]) cudaEventDestroy(c->copy_done[b]);
    if (c->window) cudaFree(c->window);
    if (c->local_rgba) cudaFree(c->local_rgba);
    delete c;
    return VRT_OK;
}

int vrt_comm_info(const vrt_comm* c, int* rank, int* world, uint64_t* frames) {
    if (!c) return fail(VRT_ERR_INVALID, "vrt_comm_info: comm is NULL");
    if (rank) *rank = c->rank;
    if (world) *world = c->world;
    if (frames) *frames = c->frame_no;
    return VRT_OK;
}

// One frame.  Every rank of the communicator calls this with the same camera and parameters (width/height as at creation;
// row_begin/row_end/tile_step/tile_index/sample_offset are chosen here).  Enqueues only; see vrt_comm_frame_wait.
int vrt_render_distributed(vrt_comm* c, vrt_scene* sc, const vrt_camera* cam, const vrt_render_params* p_in, int split, int deliver_all,
                           uint8_t* host_rgba) {
    if (int s = check_comm(c, "vrt_render_distributed")) return s;
    if (!sc || !cam || !p_in) return fail(VRT_ERR_INVALID, "vrt_render_distributed: NULL argument");
    if (sc->ctx != c->ctx) return fail(VRT_ERR_INVALID, "vrt_render_distributed: the scene lives on another context than the communicator");
    if (p_in->width != c->width || p_in->height != c->height) return fail(VRT_ERR_INVALID, "vrt_render_distributed: frame size differs from the communicator's");
    if (split != VRT_SPLIT_TILES && split != VRT_SPLIT_SAMPLES) return fail(VRT_ERR_INVALID, "vrt_render_distributed: split must be VRT_SPLIT_TILES or VRT_SPLIT_SAMPLES");
    if (split == VRT_SPLIT_SAMPLES && (!p_in->use_samples || p_in->checker || p_in->spp % c->world))
        return fail(VRT_ERR_INVALID, "vrt_render_distributed: the sample split needs use_samples, no checkerboard and spp divisible by the number of GPUs");
    vrt_context* ctx = c->ctx;
    if (int s = use_device(ctx)) return s;
    cudaStream_t st = ctx->stream;
    const int W = c->world, root = c->root;
    const uint64_t f = c->frame_no;                 // this frame's ordinal
    const int buf = int(f & 1);
    vrt_render_params p = *p_in;
    p.row_begin = 0; p.row_end = c->height; p.accum_in = 0;
    uint32_t* accum = c->accum(c->rank);
    Flags* rf = c->flags(root);

    // the peers read this accumulator during their reduce of the latest sample-split frame — wait for all of them before it is
    // cleared, whichever split this frame uses
    if (W > 1 && c->sample_frames > 0) {
        wait_kernel<<<1, 1, 0, st>>>(&rf->reduced, c->sample_frames * uint64_t(W), &c->flags(c->rank)->error);
        ctx->launches += 1;
    }
    VRT_CUDA(cudaMemsetAsync(accum, 0, size_t(c->h_pad) * c->width * 16, st));
    if (split == VRT_SPLIT_TILES) {
        p.tile_step = W; p.tile_index = c->rank;
    } else {
        p.tile_step = 1; p.tile_index = 0;
        p.spp = p_in->spp / W;
        p.sample_offset = p_in->sample_offset + c->rank * p.spp;
    }
    if (int s = vrt_render_accumulate_device(sc, cam, &p, accum)) return s;

    // the buffer this frame is pushed into may still hold an earlier frame of the target that its consumer has not taken yet
    for (int t = 0; t < W; ++t) {
        if (!deliver_all && t != root) continue;
        const long long last = c->last_in_buf[t][buf];
        c->last_in_buf[t][buf] = (long long)f;
        if (last < 0) continue;
        if (t == c->rank) {                                  // own window: ordered by the copy's event
            if (c->copy_pending[buf]) {
                VRT_CUDA(cudaStreamWaitEvent(st, c->copy_done[buf], 0));
                c->copy_pending[buf] = false;
            }
            continue;
        }
        wait_kernel<<<1, 1, 0, st>>>(&c->flags(t)->consumed, (unsigned long long)(last + 1), &c->flags(c->rank)->error);
        ctx->launches += 1;
    }

    Targets dst;
    dst.n = 0;
    for (int t = 0; t < W; ++t)
        if (deliver_all || t == root) dst.frame[dst.n++] = c->frame(t, buf);
    Sources src;
    src.n = 1;
    src.accum[0] = accum;
    const int tiles = (c->h_pad / 4) / W;
    const uint64_t n = uint64_t(tiles) * 4 * c->width;
    const unsigned grid = unsigned((n + 255) / 256);
    if (split == VRT_SPLIT_SAMPLES && W > 1) {
        signal_kernel<<<1, 1, 0, st>>>(&rf->acc_done, 1ull);
        wait_kernel<<<1, 1, 0, st>>>(&rf->acc_done, (c->sample_frames + 1) * uint64_t(W), &c->flags(c->rank)->error);
        for (int r = 0; r < W; ++r)
            if (r != c->rank) src.accum[src.n++] = c->accum(r);
        resolve_push_kernel<true><<<grid, 256, 0, st>>>(src, dst, c->local_rgba, c->width, c->height, p_in->use_samples, W, c->rank);
        signal_kernel<<<1, 1, 0, st>>>(&rf->reduced, 1ull);
        ctx->launches += 4;
    } else {
        resolve_push_kernel<false><<<grid, 256, 0, st>>>(src, dst, c->local_rgba, c->width, c->height, p_in->use_samples, W, c->rank);
        ctx->launches += 1;
    }
    VRT_CUDA(cudaGetLastError());
    // publish: this rank's tiles are in the targets' buffers
    for (int t = 0; t < W; ++t)
        if (deliver_all || t == root) {
            set_kernel<<<1, 1, 0, st>>>(&c->flags(t)->arrived_from[c->rank], f + 1);
            ctx->launches += 1;
        }
    // consumer side: wait for everybody's tiles, then hand the frame over
    if (deliver_all || c->rank == root) {
        Flags* mine = c->flags(c->rank);
        if (W > 1) {
            wait_all_kernel<<<1, 1, 0, st>>>(mine->arrived_from, W, f + 1, &mine->error);
            ctx->launches += 1;
        }
        if (host_rgba) {
            VRT_CUDA(cudaEventRecord(c->frame_ready, st));
            VRT_CUDA(cudaStreamWaitEvent(c->copy_stream, c->frame_ready, 0));
            VRT_CUDA(cudaMemcpyAsync(host_rgba, c->frame(c->rank, buf), size_t(c->height) * c->width * 4, cudaMemcpyDeviceToHost, c->copy_stream));
            set_kernel<<<1, 1, 0, c->copy_stream>>>(&mine->consumed, f + 1);
            VRT_CUDA(cudaEventRecord(c->copy_done[buf], c->copy_stream));
            c->copy_pending[buf] = true;
        } else {
            set_kernel<<<1, 1, 0, st>>>(&mine->consumed, f + 1);   // device-resident consumer: valid until frame f + 2 is pushed
        }
        ctx->launches += 1;
    }
    VRT_CUDA(cudaGetLastError());
    c->frame_no = f + 1;
    if (split == VRT_SPLIT_SAMPLES) c->sample_frames += 1;
    return VRT_OK;
}

// Blocks until the most recent frame (and its host copy, if one was requested) is complete on this rank.
int vrt_comm_frame_wait(vrt_comm* c) {
    if (int s = check_comm(c, "vrt_comm_frame_wait")) return s;
    if (int s = use_device(c->ctx)) return s;
    VRT_CUDA(cudaStreamSynchronize(c->ctx->stream));
    VRT_CUDA(cudaStreamSynchronize(c->copy_stream));
    c->copy_pending[0] = c->copy_pending[1] = false;
    unsigned long long err = 0;
    VRT_CUDA(cudaMemcpy(&err, &c->flags(c->rank)->error, sizeof(err), cudaMemcpyDeviceToHost));
    if (err) return fail(VRT_ERR_CUDA, "vrt_comm_frame_wait: a peer GPU did not reach the frame's synchronisation point within 4 s");
    return VRT_OK;
}

// Device address of the assembled frame `frames_ago` frames back (0 = the most recent one) on a rank that receives frames
// (the root, or every rank with deliver_all).  Valid until two more frames have been rendered.
int vrt_comm_frame_device(vrt_comm* c, int frames_ago, uint8_t** d_rgba) {
    if (int s = check_comm(c, "vrt_comm_frame_device")) return s;
    if (!d_rgba || frames_ago < 0 || frames_ago > 1 || uint64_t(frames_ago) >= c->frame_no)
        return fail(VRT_ERR_INVALID, "vrt_comm_frame_device: no such frame");
    *d_rgba = c->frame(c->rank, int((c->frame_no - 1 - uint64_t(frames_ago)) & 1));
    return VRT_OK;
}

}  // extern "C"
