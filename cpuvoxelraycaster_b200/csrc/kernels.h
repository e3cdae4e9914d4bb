// Kernel launchers of libvrt (implemented in the .cu files, called by capi.cu).
#pragma once
#include <cstdint>
#include <vector>
#include <cuda_runtime.h>
#include "../../include/vrt.h"

namespace vrt {

// K1: LSVO<D>::castRay over a ray buffer, reference node layout (lsvo_kernels.cu)
cudaError_t launch_lsvo_cast_ref(const uint2* nodes, bool compact, int depth, int guard, const float* d_origin, const float* d_dir,
                                 float coef, float bias, uint64_t n, vrt_hit* d_out, unsigned long long* d_complexity,
                                 cudaStream_t stream);
// K1b: the same on Trav2 (lsvo_step.cuh), reference layout.  d_gate != NULL: the kernel runs only if *d_gate == want.
cudaError_t launch_lsvo_cast2(const uint2* nodes, int depth, int guard, const float* d_origin, const float* d_dir, float coef, float bias,
                              uint64_t n, vrt_hit* d_out, unsigned long long* d_complexity, cudaStream_t stream,
                              const unsigned long long* d_gate = nullptr, unsigned long long want = 0);
// *d_gate = 1 if the batch's rays are coherent in groups of 32 consecutive rays (n >= 1024), else 0
cudaError_t launch_classify_rays(const float* d_origin, const float* d_dir, uint64_t n, unsigned long long* d_gate, cudaStream_t stream);

// Bit-packed occupancy pyramid of a dense grid: level l holds cubes of edge 2^l, z-contiguous like
// Grid3D::m_cells[x][y][z] (grid_3d.hpp:26); bit i of the level = word i>>5, bit i&31.
struct GridLevel {
    const uint32_t* bits;
    int nx, ny, nz;
};
struct GridLevels {
    GridLevel level[13];
    int n_levels;
    int X, Y, Z;
    const uint32_t* mirror;   // level-0 bit plane: Cell::type == Mirror (cell.hpp:8); may be null
    // Level 0 once more with a one-cell border: (X+2) x (Y+2) x (Z+2) bits, cell (x,y,z) at ((x+1) * pad_y + (y+1)) * pad_z + (z+1),
    // every border cell set.  A ray that leaves the grid lands on a border cell, so the DDA needs no bounds test per step
    // (grid_kernels.cu, grid_dda_fast).  Null when the padded grid has 2^32 bits or more (the generic loop is used then).
    const uint32_t* pad_bits;
    uint32_t pad_y, pad_z;
};

// K2 / K2m: Grid3D::castRay, flat or with the fetch-skipping pyramid (grid_kernels.cu)
// variant: 0 = the bordered-grid DDA when the scene has one (default), 1 = the generic loop (flat, or with the fetch-skipping pyramid)
cudaError_t launch_grid_cast(const GridLevels& g, bool use_mip, int variant, const float* d_origin, const float* d_dir, uint64_t n,
                             vrt_hit* d_out, unsigned long long* d_counters, cudaStream_t stream);
// K3: SVO<N>::castRay with the hit fill restored (grid_kernels.cu)
cudaError_t launch_svo_cast(const GridLevels& g, int depth, const float* d_origin, const float* d_dir, uint32_t max_iter,
                            uint64_t n, vrt_hit* d_out, unsigned long long* d_counters, cudaStream_t stream);

// Bounds of everything solid in an LSVO scene, castRay coordinates (see lsvo_step.cuh, Trav2 kBounds)
struct SceneBounds {
    float lo[3], hi[3];
};

// Everything one render launch needs, passed by value (constant bank).
struct RenderLaunch {
    int width, height, row_begin, row_end;
    int spp, sample_offset;
    int depth, guard;
    int use_gi, gi_bounces;
    int tile_step, tile_index;   // 4-row tiles t with t % tile_step == tile_index are rendered
    int spp_chunks;              // K4: runs the samples are cut into (0 = chosen by the launcher)
    int samples_per_warp;        // K4: lanes sharing a pixel, power of two 1..32 (0 = chosen by the launcher)
    int sort_bins1, sort_bins2;  // K5: angle bins per GI bounce (0 = chosen by the launcher; product <= 256)
    int help_window;             // K6: groups of 32 blocks, counted from the last started, over which helping CTAs spread (0 = all start at the last)
    void* scratch;               // K6: device scratch for the sorted sample lists (render_scratch_bytes)
    size_t scratch_bytes;
    int mapping;                 // 0 = automatic (K5 for many-sample GI frames, else K4), 2 = K4, 3 = K5
    SceneBounds bounds;          // LSVO frames: walks end when the ray leaves this box (the whole cube [1,2]^3 = the reference's walk)
    const float* beam_floor;     // LSVO frames: per-tile start distance of the camera rays (beam_kernels.cu), or null
    int beam_shift, beam_tiles_x;  // tile edge = 1 << beam_shift pixels; tiles per row
    int grid_variant;            // grid frames: 0 = bordered-grid DDA (default), 1 = generic loop
    int trav_policy;             // K6 traversal loop: 0 = Trav, 1 = Trav2, 2 = Trav2 without the cone test on coef-0 rays (default)
    uint32_t seed_lo, seed_hi;
    float light[3];
    vrt_camera cam;
    const uint8_t* tex_top;    // 16x16 RGB, device
    const uint8_t* tex_side;
    float roughness;           // grid frames: blur of mirror reflections
    int max_bounds;            // reflection depth (RayCaster::max_bounds, raycaster.hpp:277)
    int mirror_y1;             // LSVO frames: 1 + y of the voxel layer whose top faces are Cell::Mirror; 0 = none
    // LSVO frames (kMirror kernels) and shade rays: 1 = albedo = palette[colour of the hit voxel's leaf slot], the 256 RGB entries
    // at tex_top + kPaletteOffset; 0 = the textures.  A flag in the alignment gap before `focal` rather than a pointer at the
    // end: the struct keeps its 272 bytes, so no kernel parameter behind it moves.
    int palette;
    const float* focal;       // device: focal length computed by the autofocus kernel, or null = cam.focal_length
    int checker;               // 0 = every pixel, 1 / 2 = checkerboard with offset 0 / 1 (main.cpp:137,143)
    int checker_area_height;   // thread-area height the checkerboard phase restarts at (0 = never)
};

// A scene's texture block on the device: top texture, side texture (16x16 RGB each), then the 256-entry RGB palette.
constexpr size_t kPaletteOffset = 1536;
constexpr size_t kTextureBlockBytes = kPaletteOffset + 768;

// main.cpp:143: inside a thread area, rows start at area_start + (x + offset) % 2 and step by 2.
// Returns the parity x must have for pixel (x, y) to be rendered this frame.
__host__ __device__ inline int checker_x_parity(int checker, int area_height, int y) {
    const int rel = area_height > 0 ? y % area_height : y;
    return (rel + (checker - 1)) & 1;
}

// K0+K4: ray generation, traversal, shading and accumulation for rows [row_begin,row_end) (render_kernels.cu)
// d_counters of the frame launchers: [0..5] rays per class, [6..11] loop trips per class, [12] K4p's work counter,
// [kCulledCounter] primary rays answered by the beam search without a walk (K6: sort_samples_kernel)
constexpr int kCulledCounter = 14;
// device scratch launch_render_accumulate_ref needs for this launch (0 unless the K6 mapping is selected)
size_t render_scratch_bytes(const RenderLaunch& L);
cudaError_t launch_render_accumulate_ref(const uint2* nodes, bool compact, const RenderLaunch& L, uint32_t* d_accum,
                                         unsigned long long* d_counters, cudaStream_t stream);
// bounds of the solid voxels of an LSVO in the reference layout, enlarged by `margin_voxels`, into d_bounds (6 floats: lo xyz, hi xyz);
// d_work: scratch of bounds_work_bytes() bytes (scene_device.cu)
size_t bounds_work_bytes();
cudaError_t device_scene_bounds(const uint2* d_nodes, int depth, float margin_voxels, float* d_bounds, void* d_work, cudaStream_t stream);
// per-tile conservative start distances of the camera rays of rows [row_begin, row_end) (beam_kernels.cu); tile = 4, 8, 16 ...
cudaError_t launch_beam_floor(const uint2* nodes, const RenderLaunch& L, int tile, float* d_floor, cudaStream_t stream);
// RayCaster::castRay for explicit rays (vrt_shade_rays)
cudaError_t launch_shade_rays(const uint2* nodes, bool compact, const RenderLaunch& L, uint64_t n, const vrt_shade_job* d_jobs,
                              vrt_shade_result* d_out, cudaStream_t stream);
// Camera::getClosestPoint + main.cpp:114-121 on the device: *d_focal = hit ? distance * 2^depth : 100
cudaError_t launch_autofocus(const uint2* nodes, bool compact, int depth, int guard, const vrt_camera& cam, float* d_focal,
                             cudaStream_t stream);
cudaError_t launch_resolve(const uint32_t* d_accum, uint8_t* d_rgba, int width, int row_begin, int row_end, int use_samples,
                           int tile_step, int tile_index, cudaStream_t stream);
// median filter + persistence blend of main.cpp:159-177 (present_kernels.cu)
cudaError_t launch_present(const uint8_t* d_frame, uint8_t* d_display, int width, int height, int median, uint32_t c1, uint32_t c2,
                           cudaStream_t stream);

}  // namespace vrt

namespace vrt {
// K1p / K4p: persistent-thread variants with per-lane ray regeneration (persistent_kernels.cu).
// `refill` = number of parked lanes that makes a warp leave the traversal loop (1..32).
// d_counters: cast: [0] Σ complexity, [1] work counter; render: [0..11] stats, [12] work counter — zeroed by the caller.
cudaError_t launch_lsvo_cast_persistent(const uint2* nodes, bool compact, int depth, int guard, const float* d_origin, const float* d_dir,
                                        float coef, float bias, uint64_t n, vrt_hit* d_out, unsigned long long* d_counters,
                                        int refill, cudaStream_t stream, const unsigned long long* d_gate = nullptr,
                                        unsigned long long want = 0);
cudaError_t launch_render_persistent(const uint2* nodes, const RenderLaunch& L, uint32_t* d_accum, unsigned long long* d_counters,
                                     int refill, cudaStream_t stream);
// Grid frames: camera rays, DDA, mirror reflections, texture + sun shadow, accumulation (grid_kernels.cu)
cudaError_t launch_grid_render(const GridLevels& g, bool use_mip, const RenderLaunch& L, uint32_t* d_accum,
                               unsigned long long* d_counters, cudaStream_t stream);
// Scene construction on the device (scene_device.cu): T(depth) in the reference's LNode layout, nothing crosses PCIe.
// *d_slots is cudaMalloc'ed (the caller frees it); d_heights_out may be null.
// d_heights_in (device, [S*S] int32, index x*S+z): build from these column heights instead of the FastNoise terrain.
// Device memory a scene keeps between rebuilds (edits re-flatten the world: without this every edit pays cudaMalloc / cudaFree of the
// node array and of ~40 work arrays — most of the 11-14 ms an edit took at 2048^3).  Work arrays are handed out in call order and
// grow on demand; the node array that an edit replaces becomes the spare the next edit builds into.
struct BuildPool {
    std::vector<void*> ptr;
    std::vector<size_t> bytes;
    size_t next = 0;               // next work array to hand out (reset per build)
    uint2* spare = nullptr;        // a node array of spare_slots slots, free to build into
    uint64_t spare_slots = 0;
    void release() {
        for (void* p : ptr) cudaFree(p);
        ptr.clear(); bytes.clear(); next = 0;
        if (spare) cudaFree(spare);
        spare = nullptr; spare_slots = 0;
    }
};
// Work arrays of one build: from the pool (call order, grown on demand, kept) or cudaMalloc'ed and freed on destruction.
struct PoolScratch {
    BuildPool* pool;
    std::vector<void*> owned;
    explicit PoolScratch(BuildPool* p) : pool(p) { if (pool) pool->next = 0; }
    ~PoolScratch() { for (void* q : owned) cudaFree(q); }
    template <typename T> cudaError_t alloc(T** q, size_t n) {
        const size_t want = (n ? n : 1) * sizeof(T);
        if (!pool) {
            cudaError_t e = cudaMalloc(reinterpret_cast<void**>(q), want);
            if (e == cudaSuccess) owned.push_back(*q);
            return e;
        }
        const size_t i = pool->next++;
        if (i >= pool->ptr.size()) { pool->ptr.push_back(nullptr); pool->bytes.push_back(0); }
        if (pool->bytes[i] < want) {                       // grow with some slack: edits change the counts a little
            if (pool->ptr[i]) cudaFree(pool->ptr[i]);
            pool->ptr[i] = nullptr; pool->bytes[i] = 0;
            const size_t cap = want + want / 8 + 256;
            cudaError_t e = cudaMalloc(&pool->ptr[i], cap);
            if (e != cudaSuccess) return e;
            pool->bytes[i] = cap;
        }
        *q = static_cast<T*>(pool->ptr[i]);
        return cudaSuccess;
    }
};
// pool != NULL: work arrays and the node array come from the pool (the array may be larger than *n_slots: *capacity_slots), and the
// call returns without waiting for the device (the caller keeps the replaced array alive as the pool's spare instead of freeing it).
cudaError_t device_build_terrain_lsvo(int depth, uint2** d_slots, uint64_t* n_slots, int32_t* d_heights_out, cudaStream_t stream,
                                      const int32_t* d_heights_in = nullptr, BuildPool* pool = nullptr, uint64_t* capacity_slots = nullptr);
// Reference layout → compact breadth-first array of live nodes, on the device (scene_device.cu); caller frees *d_out.
// voxel_build.cu: arbitrary voxel sets on the device (sorted path keys → LNode array) and voxel edits
// pool (optional): work arrays — and, for the node array, the spare — are taken from / kept in the scene's BuildPool (edits)
cudaError_t device_voxel_keys(const uint32_t* d_xyz, uint64_t n, int depth, uint64_t** d_keys, uint32_t* n_keys, cudaStream_t stream,
                              BuildPool* pool = nullptr);
cudaError_t device_edit_voxel_keys(const uint64_t* d_keys, uint32_t n_keys, const uint64_t* d_edit, uint32_t n_edit, int add, int depth,
                                   uint64_t** d_out, uint32_t* n_out, cudaStream_t stream, BuildPool* pool = nullptr);
cudaError_t device_build_lsvo_from_keys(int depth, const uint64_t* d_keys, uint32_t n_keys, uint2** d_slots, uint64_t* n_slots,
                                        cudaStream_t stream, BuildPool* pool = nullptr, uint64_t* capacity_slots = nullptr);
cudaError_t device_compact_lsvo(const uint2* d_ref, uint64_t n_ref, int depth, uint2** d_out, uint64_t* n_out, cudaStream_t stream);
// Per-voxel colours (voxel_build.cu), the `color` byte of each solid voxel's leaf slot in the reference layout.
// Paints d_colors[i] into voxel d_xyz[i] (setCell coordinates); empty voxels are skipped, the last occurrence of a voxel wins.
// d_keys / d_key_colors (optional, voxel-set scenes): the resident sorted keys and their colours, updated alongside.
// *painted = distinct solid voxels painted.  Synchronises the stream.
cudaError_t device_paint_cells(uint2* d_nodes, int depth, const uint32_t* d_xyz, const uint8_t* d_colors, uint64_t n,
                               const uint64_t* d_keys, uint32_t n_keys, uint8_t* d_key_colors, uint64_t* painted, cudaStream_t stream);
// d_out[i] = colour of voxel d_xyz[i], or -1 when it is empty
cudaError_t launch_cell_colors(const uint2* d_nodes, int depth, const uint32_t* d_xyz, uint64_t n, int16_t* d_out, cudaStream_t stream);
// Colours of a new sorted key set: the colour of the same key in the old set, else 1 (LNode())
cudaError_t launch_gather_key_colors(const uint64_t* d_old_keys, const uint8_t* d_old_colors, uint32_t n_old, const uint64_t* d_new_keys,
                                     uint32_t n_new, uint8_t* d_new_colors, cudaStream_t stream);
// Writes the colour of every key into its leaf slot of a node array built from those keys
cudaError_t launch_stamp_key_colors(uint2* d_nodes, int depth, const uint64_t* d_keys, const uint8_t* d_colors, uint32_t n_keys,
                                    cudaStream_t stream);
}  // namespace vrt
