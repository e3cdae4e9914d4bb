// Private to libvrt: the opaque handle types of include/vrt.h and the error helpers, shared by capi.cu and comm.cu.
#pragma once
#include <string>
#include <utility>
#include <vector>

#include "kernels.h"

namespace vrt {
int fail(int code, const std::string& msg);          // records the text for vrt_last_error() and returns `code`
int cuda_fail(cudaError_t e, const char* what);
}  // namespace vrt
#define VRT_CUDA(call)                                           \
    do {                                                         \
        cudaError_t e_ = (call);                                 \
        if (e_ != cudaSuccess) return vrt::cuda_fail(e_, #call); \
    } while (0)

// grow-only device scratch buffer
struct DeviceBuffer {
    void* ptr = nullptr;
    size_t bytes = 0;
    cudaError_t reserve(size_t want) {
        if (want <= bytes) return cudaSuccess;
        if (ptr) cudaFree(ptr);
        ptr = nullptr;
        bytes = 0;
        cudaError_t e = cudaMalloc(&ptr, want);
        if (e == cudaSuccess) bytes = want;
        return e;
    }
    void release() {
        if (ptr) cudaFree(ptr);
        ptr = nullptr;
        bytes = 0;
    }
};

struct vrt_context {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool owns_stream = false;
    uint64_t launches = 0;
    int sm_count = 0;
    // 1 = persistent threads with per-lane ray regeneration; 0 = one thread per ray / pixel.
    // Defaults follow the measurements in profiles/r01_summary.md: batched casts regenerate (warp-adaptive),
    // frames keep one lane per pixel (coherent primary/shadow rays lose more from de-phasing than GI rays gain).
    int cast_variant = 3, render_variant = 0;
    int help_window = 64;                       // K6: see RenderLaunch::help_window (0/8/32/64/256: 5.53/5.41/5.36/5.35/5.34 ms on a 1/8 slice)
    int sort_bins1 = 0, sort_bins2 = 0;         // K5: angle bins of the two GI bounces (0 = automatic)
    int spp_chunks = 0;                        // K4: 0 = automatic
    int trav_policy = -1;                      // K6: traversal loop variant (kernels.h RenderLaunch::trav_policy)
    int samples_per_warp = 0;                  // K4: lanes sharing a pixel (power of two), 0 = automatic
    int refill_cast = 0, refill_render = 16;   // parked lanes that trigger a refill (1..32); cast: 0 = warp-adaptive
    DeviceBuffer scratch_in, scratch_out;   // host-variant staging
    int bounds_exit = 1;                    // LSVO frames: walks end when the ray leaves the scene's bounds (1) or the root cube (0, the reference)
    int beam_tile = 8;                      // LSVO frames: edge of the screen tiles that get a beam floor (beam_kernels.cu); 0 = off
    int grid_variant = 0;                   // 0 = bordered-grid DDA, 1 = generic loop (flat / fetch-skipping pyramid)
    bool time_frame_kernels = false;        // "time_frame_kernels": bracket the frame kernels of every accumulate call with events
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> frame_events;   // recorded, not yet taken (vrt_context_take_timings)
    cudaAccessPolicyWindow l2_window{};     // installed by vrt_scene_set_layout(.., l2_persist); follows the stream (set_stream)
};

constexpr int kCounterSlots = 24;    // length of vrt_scene::d_counters

struct vrt_scene {
    vrt_context* ctx = nullptr;
    int kind = 0;
    uint32_t depth = 0;
    int32_t guard = 0;
    // LSVO
    uint2* d_nodes = nullptr;
    uint64_t n_nodes = 0;
    uint64_t device_bytes = 0;
    unsigned long long* d_counters = nullptr;   // kCounterSlots: [0] Σ complexity of the last cast; [2..13] render rays/complexity per class; [14] gate / K4p work; [15] focal; [16] culled primaries
    vrt::SceneBounds bounds{{1.0f, 1.0f, 1.0f}, {2.0f, 2.0f, 2.0f}};   // LSVO: bounds of the solid voxels (scene_device.cu), castRay coordinates
    uint2* d_compact = nullptr;                 // optional compact breadth-first copy (vrt_scene_set_layout)
    uint64_t n_compact = 0;
    bool use_compact = false;
    int32_t* d_heights = nullptr;               // heightfield scenes: column heights [S*S], resident for edits
    vrt::BuildPool build_pool;                  // heightfield scenes: work arrays + spare node array kept between edits
    uint64_t nodes_capacity = 0;                // slots d_nodes can hold (>= n_nodes once an edit has built it from the pool)
    DeviceBuffer edit_old, bounds_work;         // staged rectangle of an edit; work memory of the scene-bounds sweep
    uint64_t* d_voxel_keys = nullptr;           // voxel-set scenes: sorted distinct path keys, resident for edits
    uint32_t n_voxel_keys = 0;
    // voxel-set scenes once painted: the colour of each resident key (it survives set_cells); an edit gathers the colours of the
    // new key set into the second buffer and swaps the two, so that edits of a painted scene allocate nothing in the steady state
    DeviceBuffer voxel_colors, voxel_colors_next;
    uint8_t* d_tex = nullptr;                   // kTextureBlockBytes: top (768 B), side (768 B), palette (768 B), cell types (256 B),
                                                // point lights (count + 16 x 7 floats)
    bool has_tex = false;
    bool has_palette = false;                   // LSVO: frames take the albedo from the palette (vrt_scene_set_palette)
    bool has_cell_types = false;                // LSVO: the cell-type table has a Cell::Mirror entry (vrt_scene_set_cell_types)
    bool has_lights = false;                    // LSVO: one or more point lights (vrt_scene_set_point_lights)
    DeviceBuffer frame_accum, frame_rgba;       // vrt_render staging
    DeviceBuffer frame_lists;                   // K6: sorted sample lists of the frame in flight
    DeviceBuffer beam_floor;                    // per-tile start distances of the camera rays of the frame in flight
    // Grid3D / MipmapGrid3D / SVO: bit-packed occupancy pyramid
    vrt::GridLevels grid{};
    uint32_t* d_grid_bits = nullptr;
    bool use_mip = false;
};


namespace vrt {
inline int use_device(const vrt_context* ctx) {
    cudaError_t e = cudaSetDevice(ctx->device);
    return e == cudaSuccess ? VRT_OK : cuda_fail(e, "cudaSetDevice");
}
}  // namespace vrt
