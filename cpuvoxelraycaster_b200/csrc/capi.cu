// C ABI of libvrt (include/vrt.h).  Thin: argument checks, device memory, kernel launches.
// There is no CPU fallback — every compute entry point needs a CUDA device.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <new>
#include <string>
#include <utility>
#include <vector>

#include "capi_internal.h"
#include "host_util.h"

namespace {
thread_local std::string g_last_error;
}  // namespace
namespace vrt {
int fail(int code, const std::string& msg) {
    g_last_error = msg;
    return code;
}
int cuda_fail(cudaError_t e, const char* what) {
    return fail(VRT_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}
}  // namespace vrt
using vrt::cuda_fail;
using vrt::fail;
using vrt::use_device;


namespace {
// (re)computes the bounds of the solid voxels of an LSVO scene from its node array (reference layout) — after creation and
// after every edit.  Synchronises the stream.
int update_bounds(vrt_scene* sc, const char* who) {
    vrt_context* ctx = sc->ctx;
    // work memory + 6 result floats, kept with the scene (an edit must not pay for cudaMalloc / cudaFree)
    cudaError_t e = sc->bounds_work.reserve(vrt::bounds_work_bytes() + 256);
    float* d_bounds = e == cudaSuccess ? reinterpret_cast<float*>(static_cast<char*>(sc->bounds_work.ptr) + vrt::bounds_work_bytes()) : nullptr;
    if (e == cudaSuccess) e = vrt::device_scene_bounds(sc->d_nodes, int(sc->depth), 2.0f, d_bounds, sc->bounds_work.ptr, ctx->stream);
    float host[6];
    if (e == cudaSuccess) e = cudaMemcpyAsync(host, d_bounds, sizeof(host), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    ctx->launches += 2 * sc->depth + 1;
    if (e != cudaSuccess) return e == cudaErrorMemoryAllocation ? fail(VRT_ERR_OOM, std::string(who) + ": device allocation failed (scene bounds)") : cuda_fail(e, who);
    for (int a = 0; a < 3; ++a) { sc->bounds.lo[a] = host[a]; sc->bounds.hi[a] = host[3 + a]; }
    return VRT_OK;
}

}  // namespace

extern "C" {

int vrt_abi_version(void) { return VRT_ABI_VERSION; }
const char* vrt_last_error(void) { return g_last_error.c_str(); }
const char* vrt_build_info(void) {
    return "libvrt sm_100a --fmad=false -prec-div=true -prec-sqrt=true -ftz=false; kernels: lsvo_cast_kernel (K1), lsvo_cast2_kernel (K1b), "
           "lsvo_cast_persistent_kernel (K1p), classify_rays_kernel (default: gates K1b / K1p per batch), render_accumulate_kernel (K4, "
           "interactive frames), render_sorted_kernel (K5), beam_floor_kernel + sort_samples_kernel + render_rounds_kernel (K6, default for "
           ">= 8 samples per pixel), render_persistent_kernel (K4p), shade_rays_kernel, autofocus_kernel, resolve_kernel, "
           "resolve_push_kernel (multi-GPU), present_kernel, grid_cast_fast_kernel (K2f, default), grid_cast_kernel<mip> (K2/K2m), "
           "svo_cast_kernel (K3), grid_render_kernel<mode>, terrain / heightfield / voxel-set builders";
}

int vrt_context_create(int device, void* stream, vrt_context** out) {
    if (!out) return fail(VRT_ERR_INVALID, "vrt_context_create: out is NULL");
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess) return cuda_fail(e, "cudaGetDeviceCount");
    if (device < 0 || device >= count) return fail(VRT_ERR_INVALID, "vrt_context_create: no such device");
    vrt_context* ctx = new (std::nothrow) vrt_context();
    if (!ctx) return fail(VRT_ERR_OOM, "vrt_context_create: host allocation failed");
    ctx->device = device;
    if ((e = cudaSetDevice(device)) != cudaSuccess) { delete ctx; return cuda_fail(e, "cudaSetDevice"); }
    cudaDeviceGetAttribute(&ctx->sm_count, cudaDevAttrMultiProcessorCount, device);
    if (stream) {
        ctx->stream = static_cast<cudaStream_t>(stream);
    } else {
        if ((e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess) {
            delete ctx;
            return cuda_fail(e, "cudaStreamCreate");
        }
        ctx->owns_stream = true;
    }
    *out = ctx;
    return VRT_OK;
}

int vrt_context_destroy(vrt_context* ctx) {
    if (!ctx) return VRT_OK;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    ctx->scratch_in.release();
    ctx->scratch_out.release();
    for (auto& ev : ctx->frame_events) { cudaEventDestroy(ev.first); cudaEventDestroy(ev.second); }
    if (ctx->owns_stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return VRT_OK;
}

int vrt_context_synchronize(vrt_context* ctx) {
    if (!ctx) return fail(VRT_ERR_INVALID, "vrt_context_synchronize: ctx is NULL");
    if (int s = use_device(ctx)) return s;
    VRT_CUDA(cudaStreamSynchronize(ctx->stream));
    return VRT_OK;
}

int vrt_context_set_stream(vrt_context* ctx, void* stream) {
    if (!ctx) return fail(VRT_ERR_INVALID, "vrt_context_set_stream: ctx is NULL");
    if (ctx->owns_stream) {
        cudaStreamSynchronize(ctx->stream);
        cudaStreamDestroy(ctx->stream);
        ctx->owns_stream = false;
    }
    ctx->stream = static_cast<cudaStream_t>(stream);
    if (ctx->l2_window.num_bytes) {                       // the access-policy window is a stream attribute: carry it over
        if (int s = use_device(ctx)) return s;
        cudaStreamAttrValue attr;
        std::memset(&attr, 0, sizeof(attr));
        attr.accessPolicyWindow = ctx->l2_window;
        VRT_CUDA(cudaStreamSetAttribute(ctx->stream, cudaStreamAttributeAccessPolicyWindow, &attr));
    }
    return VRT_OK;
}

uint64_t vrt_context_launch_count(const vrt_context* ctx) { return ctx ? ctx->launches : 0; }

int vrt_context_take_timings(vrt_context* ctx, float* ms, int32_t cap, int32_t* count) {
    if (!ctx || !count) return fail(VRT_ERR_INVALID, "vrt_context_take_timings: NULL argument");
    if (int s = use_device(ctx)) return s;
    VRT_CUDA(cudaStreamSynchronize(ctx->stream));
    const int32_t n = int32_t(ctx->frame_events.size());
    *count = n;
    for (int32_t i = 0; i < n; ++i) {
        float t = 0.0f;
        cudaError_t e = cudaEventElapsedTime(&t, ctx->frame_events[i].first, ctx->frame_events[i].second);
        if (ms && i < cap) ms[i] = e == cudaSuccess ? t : -1.0f;
        cudaEventDestroy(ctx->frame_events[i].first);
        cudaEventDestroy(ctx->frame_events[i].second);
    }
    ctx->frame_events.clear();
    return VRT_OK;
}

int vrt_context_set_option(vrt_context* ctx, const char* key, int value) {
    if (!ctx || !key) return fail(VRT_ERR_INVALID, "vrt_context_set_option: NULL argument");
    const std::string k(key);
    if (k == "cast_variant" && value >= 0 && value <= 3) ctx->cast_variant = value;
    else if (k == "render_variant" && value >= 0 && value <= 4) ctx->render_variant = value;
    else if (k == "help_window" && value >= 0 && value <= 4096) ctx->help_window = value;
    else if (k == "sort_bins1" && value >= 0 && value <= 256) ctx->sort_bins1 = value;
    else if (k == "sort_bins2" && value >= 0 && value <= 256) ctx->sort_bins2 = value;
    else if (k == "spp_chunks" && value >= 0 && value <= 4096) ctx->spp_chunks = value;
    else if (k == "trav_policy" && value >= 0 && value <= 2) ctx->trav_policy = value;
    else if (k == "samples_per_warp" && value >= 0 && value <= 32 && (value & (value - 1)) == 0) ctx->samples_per_warp = value;
    else if (k == "time_frame_kernels" && (value == 0 || value == 1)) ctx->time_frame_kernels = value != 0;
    else if (k == "grid_variant" && (value == 0 || value == 1)) ctx->grid_variant = value;
    else if (k == "beam_tile" && value >= 0 && value <= 64) ctx->beam_tile = value;
    else if (k == "bounds_exit" && (value == 0 || value == 1)) ctx->bounds_exit = value;
    else if (k == "refill_cast" && value >= 0 && value <= 32) ctx->refill_cast = value;
    else if (k == "refill_render" && value >= 1 && value <= 32) ctx->refill_render = value;
    else return fail(VRT_ERR_INVALID, "vrt_context_set_option: unknown key or value out of range: " + k);
    return VRT_OK;
}

// ---- host builders ---------------------------------------------------------------------------------
int vrt_host_terrain_heights(int32_t size, int32_t* out) {
    if (size <= 0 || !out) return fail(VRT_ERR_INVALID, "vrt_host_terrain_heights: bad arguments");
    vrt::host_terrain_heights(size, out);
    return VRT_OK;
}

float vrt_host_noise2d(float x, float y) { return vrt::host_noise2d(x, y); }

int vrt_host_build_terrain_lsvo(uint32_t depth, const int32_t* heights, vrt_lnode* out, uint64_t cap, uint64_t* count) {
    // the fill writes y + S/2 with y up to max(16, height): needs S/2 + 80 < S like the reference scene
    if (depth < 8 || depth > 12 || !heights || !count)
        return fail(VRT_ERR_INVALID, "vrt_host_build_terrain_lsvo: depth must be 8..12, heights/count non-NULL");
    *count = vrt::host_build_terrain_lsvo(depth, heights, out, cap);
    if (out && *count > cap) return fail(VRT_ERR_INVALID, "vrt_host_build_terrain_lsvo: buffer too small");
    return VRT_OK;
}

int vrt_host_build_lsvo_from_voxels(uint32_t depth, const uint32_t* xyz, uint64_t n_voxels, vrt_lnode* out, uint64_t cap,
                                    uint64_t* count) {
    if (depth < 1 || depth > 12 || (!xyz && n_voxels) || !count)
        return fail(VRT_ERR_INVALID, "vrt_host_build_lsvo_from_voxels: bad arguments");
    const uint32_t S = 1u << depth;
    for (uint64_t i = 0; i < 3 * n_voxels; ++i)
        if (xyz[i] >= S) return fail(VRT_ERR_INVALID, "vrt_host_build_lsvo_from_voxels: voxel out of range");
    *count = vrt::host_build_lsvo_from_voxels(depth, xyz, n_voxels, out, cap);
    if (out && *count > cap) return fail(VRT_ERR_INVALID, "vrt_host_build_lsvo_from_voxels: buffer too small");
    return VRT_OK;
}

int vrt_host_camera_rotation(const float view_angle[2], float rot_mat[9], float camera_vec[3]) {
    if (!view_angle || !rot_mat || !camera_vec) return fail(VRT_ERR_INVALID, "vrt_host_camera_rotation: NULL argument");
    vrt::host_camera_rotation(view_angle, rot_mat, camera_vec);
    return VRT_OK;
}

// ---- scenes ----------------------------------------------------------------------------------------
int vrt_lsvo_create(vrt_context* ctx, const vrt_lnode* nodes, uint64_t n_nodes, uint32_t depth, int32_t guard, vrt_scene** out) {
    if (!ctx || !nodes || !n_nodes || !out) return fail(VRT_ERR_INVALID, "vrt_lsvo_create: NULL argument");
    if (depth < 1 || depth > 12) return fail(VRT_ERR_INVALID, "vrt_lsvo_create: depth must be 1..12");
    if (n_nodes > 0xffffffffull) return fail(VRT_ERR_UNSUPPORTED, "vrt_lsvo_create: more than 2^32 slots");
    // The traversal follows child_offset blindly and indexes its stack by level; a malformed array would fault (or spin)
    // on the device, so the structure is checked once here by walking it from the root with each node's level:
    // every referenced child block lies inside the array and behind its parent (compileSVO emits children after their
    // parent, lsvo_utils.cpp:7-10: indices grow along every path, so the walk terminates), leaves have no block, the
    // children of a node on level depth-1 are voxels (all leaves), and nothing is interior below that level — a tree
    // deeper than `depth` would drive the stack index scale - (23 - depth) negative (lsvo.hpp:97-100).
    {
        std::vector<std::pair<uint64_t, uint32_t>> todo;
        todo.emplace_back(0, 0u);
        while (!todo.empty()) {
            const uint64_t i = todo.back().first;
            const uint32_t level = todo.back().second;
            todo.pop_back();
            const vrt_lnode& nd = nodes[i];
            if (!nd.child_mask) {
                if (nd.leaf_mask) return fail(VRT_ERR_INVALID, "vrt_lsvo_create: malformed node array at slot " + std::to_string(i));
                continue;
            }
            if ((nd.leaf_mask & ~nd.child_mask) || nd.child_offset == 0 || i + nd.child_offset + 8 > n_nodes)
                return fail(VRT_ERR_INVALID, "vrt_lsvo_create: malformed node array at slot " + std::to_string(i));
            if (level + 1 >= depth && nd.leaf_mask != nd.child_mask)
                return fail(VRT_ERR_INVALID, "vrt_lsvo_create: the tree is deeper than the declared depth " + std::to_string(depth) +
                                                 " (interior child below slot " + std::to_string(i) + ")");
            const uint32_t interior = nd.child_mask & ~nd.leaf_mask;
            for (uint32_t c = 0; c < 8; ++c)
                if (interior & (1u << c)) todo.emplace_back(i + nd.child_offset + c, level + 1);
        }
    }
    if (int s = use_device(ctx)) return s;
    vrt_scene* sc = new (std::nothrow) vrt_scene();
    if (!sc) return fail(VRT_ERR_OOM, "vrt_lsvo_create: host allocation failed");
    sc->ctx = ctx;
    sc->kind = VRT_SCENE_LSVO;
    sc->depth = depth;
    sc->guard = guard > 0 ? guard : (guard < 0 ? 0 : int32_t(depth));   // 0 = reference, <0 = lifted
    sc->n_nodes = n_nodes;
    cudaError_t e = cudaMalloc(&sc->d_nodes, n_nodes * sizeof(uint2));
    if (e == cudaSuccess) e = cudaMalloc(&sc->d_counters, kCounterSlots * sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMemcpyAsync(sc->d_nodes, nodes, n_nodes * sizeof(uint2), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(sc->d_counters, 0, kCounterSlots * sizeof(unsigned long long), ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
        vrt_scene_destroy(sc);
        return e == cudaErrorMemoryAllocation ? fail(VRT_ERR_OOM, "vrt_lsvo_create: device allocation failed")
                                              : cuda_fail(e, "vrt_lsvo_create");
    }
    sc->device_bytes = n_nodes * sizeof(uint2);
    if (int s = update_bounds(sc, "vrt_lsvo_create")) { vrt_scene_destroy(sc); return s; }
    *out = sc;
    return VRT_OK;
}

int vrt_lsvo_create_terrain(vrt_context* ctx, uint32_t depth, int32_t guard, vrt_scene** out) {
    if (!ctx || !out) return fail(VRT_ERR_INVALID, "vrt_lsvo_create_terrain: NULL argument");
    if (depth < 8 || depth > 12) return fail(VRT_ERR_INVALID, "vrt_lsvo_create_terrain: depth must be 8..12");
    if (int s = use_device(ctx)) return s;
    vrt_scene* sc = new (std::nothrow) vrt_scene();
    if (!sc) return fail(VRT_ERR_OOM, "vrt_lsvo_create_terrain: host allocation failed");
    sc->ctx = ctx;
    sc->kind = VRT_SCENE_LSVO;
    sc->depth = depth;
    sc->guard = guard > 0 ? guard : (guard < 0 ? 0 : int32_t(depth));
    cudaError_t e = vrt::device_build_terrain_lsvo(int(depth), &sc->d_nodes, &sc->n_nodes, nullptr, ctx->stream);
    ctx->launches += 7 + 9 * depth;      // heights, pyramid, count/scan (4 per level), size/place/emit per level, fill, root
    if (e == cudaSuccess) e = cudaMalloc(&sc->d_counters, kCounterSlots * sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMemsetAsync(sc->d_counters, 0, kCounterSlots * sizeof(unsigned long long), ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
        vrt_scene_destroy(sc);
        return e == cudaErrorMemoryAllocation ? fail(VRT_ERR_OOM, "vrt_lsvo_create_terrain: device allocation failed")
                                              : cuda_fail(e, "vrt_lsvo_create_terrain");
    }
    sc->device_bytes = sc->n_nodes * sizeof(uint2);
    if (int s = update_bounds(sc, "vrt_lsvo_create_terrain")) { vrt_scene_destroy(sc); return s; }
    *out = sc;
    return VRT_OK;
}

int vrt_lsvo_create_heightfield(vrt_context* ctx, uint32_t depth, const int32_t* heights, int32_t guard, vrt_scene** out) {
    if (!ctx || !out) return fail(VRT_ERR_INVALID, "vrt_lsvo_create_heightfield: NULL argument");
    if (depth < 5 || depth > 12) return fail(VRT_ERR_INVALID, "vrt_lsvo_create_heightfield: depth must be 5..12");
    if (!heights && depth < 8) return fail(VRT_ERR_INVALID, "vrt_lsvo_create_heightfield: the demo terrain needs depth 8..12");
    if (int s = use_device(ctx)) return s;
    vrt_scene* sc = new (std::nothrow) vrt_scene();
    if (!sc) return fail(VRT_ERR_OOM, "vrt_lsvo_create_heightfield: host allocation failed");
    sc->ctx = ctx;
    sc->kind = VRT_SCENE_LSVO;
    sc->depth = depth;
    sc->guard = guard > 0 ? guard : (guard < 0 ? 0 : int32_t(depth));
    const size_t columns = size_t(1) << (2 * depth);
    cudaError_t e = cudaMalloc(&sc->d_heights, columns * sizeof(int32_t));
    if (e == cudaSuccess && heights) e = cudaMemcpyAsync(sc->d_heights, heights, columns * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream);
    // heights == NULL: the demo terrain (FastNoise heights, main.cpp:61-68), kept resident so that it can be edited
    if (e == cudaSuccess)
        e = vrt::device_build_terrain_lsvo(int(depth), &sc->d_nodes, &sc->n_nodes, heights ? nullptr : sc->d_heights, ctx->stream,
                                           heights ? sc->d_heights : nullptr);
    ctx->launches += 7 + 9 * depth;
    if (e == cudaSuccess) e = cudaMalloc(&sc->d_counters, kCounterSlots * sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMemsetAsync(sc->d_counters, 0, kCounterSlots * sizeof(unsigned long long), ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
        vrt_scene_destroy(sc);
        return e == cudaErrorMemoryAllocation ? fail(VRT_ERR_OOM, "vrt_lsvo_create_heightfield: device allocation failed")
                                              : cuda_fail(e, "vrt_lsvo_create_heightfield");
    }
    sc->device_bytes = sc->n_nodes * sizeof(uint2) + columns * sizeof(int32_t);
    if (int s = update_bounds(sc, "vrt_lsvo_create_heightfield")) { vrt_scene_destroy(sc); return s; }
    *out = sc;
    return VRT_OK;
}

int vrt_scene_edit_heights(vrt_scene* sc, uint32_t x0, uint32_t z0, uint32_t nx, uint32_t nz, const int32_t* heights) {
    if (!sc || !heights) return fail(VRT_ERR_INVALID, "vrt_scene_edit_heights: NULL argument");
    if (sc->kind != VRT_SCENE_LSVO || !sc->d_heights)
        return fail(VRT_ERR_UNSUPPORTED, "vrt_scene_edit_heights: the scene was not created by vrt_lsvo_create_heightfield");
    const uint64_t S = uint64_t(1) << sc->depth;
    if (nx == 0 || nz == 0 || uint64_t(x0) + nx > S || uint64_t(z0) + nz > S) return fail(VRT_ERR_INVALID, "vrt_scene_edit_heights: rectangle out of range");
    vrt_context* ctx = sc->ctx;
    if (int s = use_device(ctx)) return s;
    // the edit is staged: the old rectangle is kept until the new node array exists, and put back if the rebuild fails,
    // so that the resident heights always describe the world that is being rendered.  All device memory involved is kept with
    // the scene (work arrays, the staged rectangle, and the node array this edit replaces: the next edit builds into it).
    if (sc->edit_old.reserve(size_t(nx) * nz * sizeof(int32_t)) != cudaSuccess) return fail(VRT_ERR_OOM, "vrt_scene_edit_heights: device allocation failed (scene unchanged)");
    int32_t* d_old = static_cast<int32_t*>(sc->edit_old.ptr);
    cudaError_t e = cudaMemcpy2DAsync(d_old, size_t(nz) * sizeof(int32_t), sc->d_heights + size_t(x0) * S + z0, S * sizeof(int32_t),
                                      size_t(nz) * sizeof(int32_t), nx, cudaMemcpyDeviceToDevice, ctx->stream);
    if (e == cudaSuccess)
        e = cudaMemcpy2DAsync(sc->d_heights + size_t(x0) * S + z0, S * sizeof(int32_t), heights, size_t(nz) * sizeof(int32_t),
                              size_t(nz) * sizeof(int32_t), nx, cudaMemcpyHostToDevice, ctx->stream);
    uint2* d_new = nullptr;
    uint64_t n_new = 0, cap_new = 0;
    if (e == cudaSuccess) e = vrt::device_build_terrain_lsvo(int(sc->depth), &d_new, &n_new, nullptr, ctx->stream, sc->d_heights, &sc->build_pool, &cap_new);
    ctx->launches += 7 + 9 * sc->depth;
    if (e != cudaSuccess) {
        cudaGetLastError();
        cudaMemcpy2DAsync(sc->d_heights + size_t(x0) * S + z0, S * sizeof(int32_t), d_old, size_t(nz) * sizeof(int32_t),
                          size_t(nz) * sizeof(int32_t), nx, cudaMemcpyDeviceToDevice, ctx->stream);
        cudaStreamSynchronize(ctx->stream);
        return e == cudaErrorMemoryAllocation ? fail(VRT_ERR_OOM, "vrt_scene_edit_heights: device allocation failed (scene unchanged)")
                                              : cuda_fail(e, "vrt_scene_edit_heights (scene unchanged)");
    }
    // the replaced array stays alive as the pool's spare: frames already enqueued on the stream still read it, and the next edit —
    // enqueued behind them on the same stream — builds into it
    if (sc->build_pool.spare) cudaFree(sc->build_pool.spare);
    sc->build_pool.spare = sc->d_nodes;
    sc->build_pool.spare_slots = sc->nodes_capacity ? sc->nodes_capacity : sc->n_nodes;
    sc->device_bytes += n_new * sizeof(uint2);
    sc->device_bytes -= sc->n_nodes * sizeof(uint2);
    sc->d_nodes = d_new;
    sc->n_nodes = n_new;
    sc->nodes_capacity = cap_new;
    if (int s = update_bounds(sc, "vrt_scene_edit_heights")) return s;
    if (sc->d_compact) {                                    // the compact copy is rebuilt from the new array
        cudaFree(sc->d_compact);
        sc->device_bytes -= sc->n_compact * sizeof(uint2);
        sc->d_compact = nullptr;
        sc->n_compact = 0;
        if (sc->use_compact) {
            sc->use_compact = false;
            return vrt_scene_set_layout(sc, 1, 0);
        }
    }
    return VRT_OK;
}

namespace {
// uploads a host voxel list and turns it into sorted distinct path keys on the device
int upload_voxel_keys(vrt_context* ctx, uint32_t depth, const uint32_t* xyz, uint64_t n, uint64_t** d_keys, uint32_t* n_keys, const char* who,
                      vrt::BuildPool* pool = nullptr) {
    if (n && !xyz) return fail(VRT_ERR_INVALID, std::string(who) + ": NULL voxel list");
    if (n > 0xffffffffull) return fail(VRT_ERR_INVALID, std::string(who) + ": too many voxels");
    const uint32_t S = 1u << depth;
    for (uint64_t i = 0; i < 3 * n; ++i)
        if (xyz[i] >= S) return fail(VRT_ERR_INVALID, std::string(who) + ": voxel out of range (UB in the reference, svo.hpp:72)");
    uint32_t* d_xyz = nullptr;
    cudaError_t e = cudaMalloc(&d_xyz, (n ? n : 1) * 3 * sizeof(uint32_t));
    if (e == cudaSuccess && n) e = cudaMemcpyAsync(d_xyz, xyz, n * 3 * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = vrt::device_voxel_keys(d_xyz, n, int(depth), d_keys, n_keys, ctx->stream, pool);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (d_xyz) cudaFree(d_xyz);
    ctx->launches += 4;
    if (e != cudaSuccess) return e == cudaErrorMemoryAllocation ? fail(VRT_ERR_OOM, std::string(who) + ": device allocation failed") : cuda_fail(e, who);
    return VRT_OK;
}

// re-flattens a voxel-set scene from its resident keys and swaps the node array in
// pooled: an edit (the scene keeps work arrays and the replaced node array for the next one); else the arrays are freed
int rebuild_from_keys(vrt_scene* sc, const uint64_t* d_keys, uint32_t n_keys, const char* who, bool pooled = false) {
    vrt_context* ctx = sc->ctx;
    uint2* d_new = nullptr;
    uint64_t n_new = 0, cap_new = 0;
    cudaError_t e = vrt::device_build_lsvo_from_keys(int(sc->depth), d_keys, n_keys, &d_new, &n_new, ctx->stream, pooled ? &sc->build_pool : nullptr, &cap_new);
    ctx->launches += 2 + 4 * sc->depth;
    if (e != cudaSuccess) return e == cudaErrorMemoryAllocation ? fail(VRT_ERR_OOM, std::string(who) + ": device allocation failed") : cuda_fail(e, who);
    if (sc->d_nodes) {                                      // the builder synchronised the stream: nothing reads the old array any more
        if (pooled) {
            if (sc->build_pool.spare) cudaFree(sc->build_pool.spare);
            sc->build_pool.spare = sc->d_nodes;
            sc->build_pool.spare_slots = sc->nodes_capacity ? sc->nodes_capacity : sc->n_nodes;
        } else {
            cudaFree(sc->d_nodes);
        }
    }
    sc->device_bytes += n_new * sizeof(uint2);
    sc->device_bytes -= sc->n_nodes * sizeof(uint2);
    sc->d_nodes = d_new;
    sc->n_nodes = n_new;
    sc->nodes_capacity = cap_new;
    if (int s = update_bounds(sc, who)) return s;
    if (sc->d_compact) {
        cudaFree(sc->d_compact);
        sc->device_bytes -= sc->n_compact * sizeof(uint2);
        sc->d_compact = nullptr;
        sc->n_compact = 0;
        if (sc->use_compact) {
            sc->use_compact = false;
            return vrt_scene_set_layout(sc, 1, 0);
        }
    }
    return VRT_OK;
}
}  // namespace

int vrt_lsvo_create_from_voxels(vrt_context* ctx, uint32_t depth, const uint32_t* xyz, uint64_t n, int32_t guard, vrt_scene** out) {
    if (!ctx || !out) return fail(VRT_ERR_INVALID, "vrt_lsvo_create_from_voxels: NULL argument");
    if (depth < 1 || depth > 12) return fail(VRT_ERR_INVALID, "vrt_lsvo_create_from_voxels: depth must be 1..12");
    if (int s = use_device(ctx)) return s;
    vrt_scene* sc = new (std::nothrow) vrt_scene();
    if (!sc) return fail(VRT_ERR_OOM, "vrt_lsvo_create_from_voxels: host allocation failed");
    sc->ctx = ctx;
    sc->kind = VRT_SCENE_LSVO;
    sc->depth = depth;
    sc->guard = guard > 0 ? guard : (guard < 0 ? 0 : int32_t(depth));
    int s = upload_voxel_keys(ctx, depth, xyz, n, &sc->d_voxel_keys, &sc->n_voxel_keys, "vrt_lsvo_create_from_voxels");
    if (s == VRT_OK) s = rebuild_from_keys(sc, sc->d_voxel_keys, sc->n_voxel_keys, "vrt_lsvo_create_from_voxels");
    if (s == VRT_OK) {
        cudaError_t e = cudaMalloc(&sc->d_counters, kCounterSlots * sizeof(unsigned long long));
        if (e == cudaSuccess) e = cudaMemsetAsync(sc->d_counters, 0, kCounterSlots * sizeof(unsigned long long), ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) s = cuda_fail(e, "vrt_lsvo_create_from_voxels");
    }
    if (s != VRT_OK) {
        vrt_scene_destroy(sc);
        return s;
    }
    sc->device_bytes += uint64_t(sc->n_voxel_keys) * sizeof(uint64_t);
    *out = sc;
    return VRT_OK;
}

int vrt_scene_set_cells(vrt_scene* sc, const uint32_t* xyz, uint64_t n, int32_t solid) {
    if (!sc) return fail(VRT_ERR_INVALID, "vrt_scene_set_cells: scene is NULL");
    if (sc->kind != VRT_SCENE_LSVO || !sc->d_voxel_keys)
        return fail(VRT_ERR_UNSUPPORTED, "vrt_scene_set_cells: the scene was not created by vrt_lsvo_create_from_voxels");
    if (n == 0) return VRT_OK;
    vrt_context* ctx = sc->ctx;
    if (int s = use_device(ctx)) return s;
    VRT_CUDA(cudaStreamSynchronize(ctx->stream));           // nothing in flight may still read the arrays replaced below
    uint64_t* d_edit = nullptr;
    uint32_t n_edit = 0;
    if (int s = upload_voxel_keys(ctx, sc->depth, xyz, n, &d_edit, &n_edit, "vrt_scene_set_cells", &sc->build_pool)) return s;
    uint64_t* d_merged = nullptr;
    uint32_t n_merged = 0;
    cudaError_t e = vrt::device_edit_voxel_keys(sc->d_voxel_keys, sc->n_voxel_keys, d_edit, n_edit, solid != 0, int(sc->depth), &d_merged,
                                                &n_merged, ctx->stream, &sc->build_pool);
    cudaFree(d_edit);
    ctx->launches += 3;
    if (e != cudaSuccess) return e == cudaErrorMemoryAllocation ? fail(VRT_ERR_OOM, "vrt_scene_set_cells: device allocation failed")
                                                                : cuda_fail(e, "vrt_scene_set_cells");
    // a painted scene: surviving voxels keep their colour, added ones get 1
    const bool painted = sc->voxel_colors.ptr != nullptr;
    if (painted) {
        e = sc->voxel_colors_next.reserve(size_t(n_merged) + n_merged / 16 + 4096);    // slack: edits change the count a little
        if (e == cudaSuccess)
            e = vrt::launch_gather_key_colors(sc->d_voxel_keys, static_cast<const uint8_t*>(sc->voxel_colors.ptr), sc->n_voxel_keys, d_merged,
                                              n_merged, static_cast<uint8_t*>(sc->voxel_colors_next.ptr), ctx->stream);
        ctx->launches += 1;
        if (e != cudaSuccess) {
            cudaFree(d_merged);
            return e == cudaErrorMemoryAllocation ? fail(VRT_ERR_OOM, "vrt_scene_set_cells: device allocation failed") : cuda_fail(e, "vrt_scene_set_cells");
        }
    }
    // staged: the node array is rebuilt from the candidate key set first; the resident keys are replaced only when that worked
    if (int s = rebuild_from_keys(sc, d_merged, n_merged, "vrt_scene_set_cells", true)) {
        cudaFree(d_merged);
        return s;
    }
    cudaFree(sc->d_voxel_keys);
    sc->device_bytes += uint64_t(n_merged) * sizeof(uint64_t);
    sc->device_bytes -= uint64_t(sc->n_voxel_keys) * sizeof(uint64_t);
    if (painted) {
        std::swap(sc->voxel_colors, sc->voxel_colors_next);
        sc->device_bytes += n_merged;
        sc->device_bytes -= sc->n_voxel_keys;
    }
    sc->d_voxel_keys = d_merged;
    sc->n_voxel_keys = n_merged;
    if (painted) {                                          // the new leaf slots carry LNode()'s colour 1 until stamped
        VRT_CUDA(vrt::launch_stamp_key_colors(sc->d_nodes, int(sc->depth), sc->d_voxel_keys, static_cast<const uint8_t*>(sc->voxel_colors.ptr),
                                              sc->n_voxel_keys, ctx->stream));
        ctx->launches += 1;
        VRT_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    return VRT_OK;
}

namespace {
// checks a voxel list (setCell coordinates) and copies it into a device buffer with `tail_bytes` more behind it, filled from
// `tail` unless that is NULL (caller frees)
int upload_cells(vrt_scene* sc, const uint32_t* xyz, uint64_t n, const void* tail, size_t tail_bytes, uint32_t** d_xyz, const char* who) {
    *d_xyz = nullptr;
    if (n > 0x7fffffffull) return fail(VRT_ERR_INVALID, std::string(who) + ": too many voxels");
    const uint32_t S = 1u << sc->depth;
    for (uint64_t i = 0; i < 3 * n; ++i)
        if (xyz[i] >= S) return fail(VRT_ERR_INVALID, std::string(who) + ": voxel out of range (UB in the reference, svo.hpp:72)");
    if (int s = use_device(sc->ctx)) return s;
    const size_t bytes = size_t(n) * 3 * sizeof(uint32_t);
    cudaError_t e = cudaMalloc(d_xyz, bytes + tail_bytes);
    if (e == cudaSuccess) e = cudaMemcpyAsync(*d_xyz, xyz, bytes, cudaMemcpyHostToDevice, sc->ctx->stream);
    if (e == cudaSuccess && tail) e = cudaMemcpyAsync(reinterpret_cast<char*>(*d_xyz) + bytes, tail, tail_bytes, cudaMemcpyHostToDevice, sc->ctx->stream);
    if (e != cudaSuccess) {
        if (*d_xyz) cudaFree(*d_xyz);
        *d_xyz = nullptr;
        return e == cudaErrorMemoryAllocation ? fail(VRT_ERR_OOM, std::string(who) + ": device allocation failed") : cuda_fail(e, who);
    }
    return VRT_OK;
}
}  // namespace

int vrt_scene_paint_cells(vrt_scene* sc, const uint32_t* xyz, const uint8_t* colors, uint64_t n, uint64_t* painted) {
    if (!sc) return fail(VRT_ERR_INVALID, "vrt_scene_paint_cells: scene is NULL");
    if (sc->kind != VRT_SCENE_LSVO || sc->d_heights)
        return fail(VRT_ERR_UNSUPPORTED, "vrt_scene_paint_cells: needs an LSVO scene that is not a heightfield (every height edit re-flattens it)");
    if (n && (!xyz || !colors)) return fail(VRT_ERR_INVALID, "vrt_scene_paint_cells: NULL voxel or colour list");
    if (painted) *painted = 0;
    if (n == 0) return VRT_OK;
    uint32_t* d_xyz = nullptr;
    if (int s = upload_cells(sc, xyz, n, colors, size_t(n), &d_xyz, "vrt_scene_paint_cells")) return s;
    vrt_context* ctx = sc->ctx;
    cudaError_t e = cudaSuccess;
    if (sc->d_voxel_keys && !sc->voxel_colors.ptr) {         // first paint of a voxel-set scene: every voxel has LNode()'s colour 1
        e = sc->voxel_colors.reserve(size_t(sc->n_voxel_keys) + sc->n_voxel_keys / 16 + 4096);
        if (e == cudaSuccess) e = cudaMemsetAsync(sc->voxel_colors.ptr, 1, sc->n_voxel_keys, ctx->stream);
        if (e == cudaSuccess) sc->device_bytes += sc->n_voxel_keys;
        else sc->voxel_colors.release();
    }
    uint64_t count = 0;
    if (e == cudaSuccess)
        e = vrt::device_paint_cells(sc->d_nodes, int(sc->depth), d_xyz, reinterpret_cast<const uint8_t*>(d_xyz + 3 * n), n, sc->d_voxel_keys,
                                    sc->n_voxel_keys, static_cast<uint8_t*>(sc->voxel_colors.ptr), &count, ctx->stream);
    ctx->launches += 3;                                       // leaf slots, sort, write
    cudaFree(d_xyz);
    if (e != cudaSuccess) return e == cudaErrorMemoryAllocation ? fail(VRT_ERR_OOM, "vrt_scene_paint_cells: device allocation failed")
                                                                : cuda_fail(e, "vrt_scene_paint_cells");
    if (painted) *painted = count;
    return VRT_OK;
}

int vrt_scene_cell_colors(vrt_scene* sc, const uint32_t* xyz, uint64_t n, int16_t* out) {
    if (!sc) return fail(VRT_ERR_INVALID, "vrt_scene_cell_colors: scene is NULL");
    if (sc->kind != VRT_SCENE_LSVO) return fail(VRT_ERR_UNSUPPORTED, "vrt_scene_cell_colors: needs an LSVO scene");
    if (n && (!xyz || !out)) return fail(VRT_ERR_INVALID, "vrt_scene_cell_colors: NULL buffer");
    if (n == 0) return VRT_OK;
    uint32_t* d_xyz = nullptr;
    if (int s = upload_cells(sc, xyz, n, nullptr, size_t(n) * sizeof(int16_t), &d_xyz, "vrt_scene_cell_colors")) return s;
    vrt_context* ctx = sc->ctx;
    int16_t* d_out = reinterpret_cast<int16_t*>(d_xyz + 3 * n);
    cudaError_t e = vrt::launch_cell_colors(sc->d_nodes, int(sc->depth), d_xyz, n, d_out, ctx->stream);
    ctx->launches += 1;
    if (e == cudaSuccess) e = cudaMemcpyAsync(out, d_out, size_t(n) * sizeof(int16_t), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    cudaFree(d_xyz);
    if (e != cudaSuccess) return cuda_fail(e, "vrt_scene_cell_colors");
    return VRT_OK;
}

int vrt_scene_voxel_count(const vrt_scene* sc, uint64_t* count) {
    if (!sc || !count) return fail(VRT_ERR_INVALID, "vrt_scene_voxel_count: NULL argument");
    if (!sc->d_voxel_keys) return fail(VRT_ERR_UNSUPPORTED, "vrt_scene_voxel_count: not a voxel-set scene");
    *count = sc->n_voxel_keys;
    return VRT_OK;
}

int vrt_scene_download_heights(vrt_scene* sc, int32_t* heights) {
    if (!sc || !heights) return fail(VRT_ERR_INVALID, "vrt_scene_download_heights: NULL argument");
    if (!sc->d_heights) return fail(VRT_ERR_UNSUPPORTED, "vrt_scene_download_heights: not a heightfield scene");
    if (int s = use_device(sc->ctx)) return s;
    const size_t columns = size_t(1) << (2 * sc->depth);
    VRT_CUDA(cudaMemcpyAsync(heights, sc->d_heights, columns * sizeof(int32_t), cudaMemcpyDeviceToHost, sc->ctx->stream));
    VRT_CUDA(cudaStreamSynchronize(sc->ctx->stream));
    return VRT_OK;
}

int vrt_scene_set_layout(vrt_scene* sc, int32_t layout, int32_t l2_persist) {
    if (!sc) return fail(VRT_ERR_INVALID, "vrt_scene_set_layout: scene is NULL");
    if (sc->kind != VRT_SCENE_LSVO) return fail(VRT_ERR_INVALID, "vrt_scene_set_layout: not an LSVO scene");
    if (layout != 0 && layout != 1) return fail(VRT_ERR_INVALID, "vrt_scene_set_layout: layout must be 0 (reference) or 1 (compact)");
    vrt_context* ctx = sc->ctx;
    if (int s = use_device(ctx)) return s;
    if (layout == 1 && !sc->d_compact) {
        cudaError_t e = vrt::device_compact_lsvo(sc->d_nodes, sc->n_nodes, int(sc->depth), &sc->d_compact, &sc->n_compact, ctx->stream);
        ctx->launches += 5 * (sc->depth + 1);
        if (e != cudaSuccess) return e == cudaErrorMemoryAllocation ? fail(VRT_ERR_OOM, "vrt_scene_set_layout: device allocation failed")
                                                                    : cuda_fail(e, "vrt_scene_set_layout");
        sc->device_bytes += sc->n_compact * sizeof(uint2);
    }
    sc->use_compact = layout == 1;
    // L2 access-policy window over the front of the node array (compact layout = top octree levels first)
    cudaStreamAttrValue attr;
    std::memset(&attr, 0, sizeof(attr));
    if (l2_persist && sc->use_compact) {
        int max_window = 0, max_persist = 0;
        cudaDeviceGetAttribute(&max_window, cudaDevAttrMaxAccessPolicyWindowSize, ctx->device);
        cudaDeviceGetAttribute(&max_persist, cudaDevAttrMaxPersistingL2CacheSize, ctx->device);
        size_t bytes = sc->n_compact * sizeof(uint2);
        if (bytes > size_t(max_window)) bytes = size_t(max_window);
        if (bytes > size_t(max_persist)) bytes = size_t(max_persist);
        if (bytes) {
            VRT_CUDA(cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, bytes));
            attr.accessPolicyWindow.base_ptr = sc->d_compact;
            attr.accessPolicyWindow.num_bytes = bytes;
            attr.accessPolicyWindow.hitRatio = 1.0f;
            attr.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
            attr.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
        }
    }
    VRT_CUDA(cudaStreamSetAttribute(ctx->stream, cudaStreamAttributeAccessPolicyWindow, &attr));
    ctx->l2_window = attr.accessPolicyWindow;
    return VRT_OK;
}

int vrt_scene_download_nodes(vrt_scene* sc, vrt_lnode* out, uint64_t cap, uint64_t* count) {
    if (!sc || !count) return fail(VRT_ERR_INVALID, "vrt_scene_download_nodes: NULL argument");
    if (sc->kind != VRT_SCENE_LSVO) return fail(VRT_ERR_INVALID, "vrt_scene_download_nodes: not an LSVO scene");
    *count = sc->n_nodes;
    if (!out) return VRT_OK;
    if (cap < sc->n_nodes) return fail(VRT_ERR_INVALID, "vrt_scene_download_nodes: buffer too small");
    if (int s = use_device(sc->ctx)) return s;
    VRT_CUDA(cudaMemcpyAsync(out, sc->d_nodes, sc->n_nodes * sizeof(uint2), cudaMemcpyDeviceToHost, sc->ctx->stream));
    VRT_CUDA(cudaStreamSynchronize(sc->ctx->stream));
    return VRT_OK;
}

int vrt_scene_destroy(vrt_scene* sc) {
    if (!sc) return VRT_OK;
    cudaSetDevice(sc->ctx->device);
    cudaStreamSynchronize(sc->ctx->stream);
    if (sc->d_nodes) cudaFree(sc->d_nodes);
    if (sc->d_counters) cudaFree(sc->d_counters);
    if (sc->d_compact) cudaFree(sc->d_compact);
    if (sc->d_heights) cudaFree(sc->d_heights);
    if (sc->d_voxel_keys) cudaFree(sc->d_voxel_keys);
    if (sc->d_tex) cudaFree(sc->d_tex);
    if (sc->d_grid_bits) cudaFree(sc->d_grid_bits);
    sc->frame_accum.release();
    sc->frame_rgba.release();
    sc->frame_lists.release();
    sc->beam_floor.release();
    sc->build_pool.release();
    sc->edit_old.release();
    sc->voxel_colors.release();
    sc->voxel_colors_next.release();
    sc->bounds_work.release();
    delete sc;
    return VRT_OK;
}

int vrt_scene_info(const vrt_scene* sc, int32_t* kind, uint32_t* depth, uint64_t* device_bytes) {
    if (!sc) return fail(VRT_ERR_INVALID, "vrt_scene_info: scene is NULL");
    if (kind) *kind = sc->kind;
    if (depth) *depth = sc->depth;
    if (device_bytes) *device_bytes = sc->device_bytes;
    return VRT_OK;
}

// ---- batched traversal -----------------------------------------------------------------------------
constexpr int kGateSlot = 14;        // d_counters[14]: verdict of the ray classifier (automatic cast variant)
int vrt_cast_rays_device(vrt_scene* sc, const float* d_origin, const float* d_dir, float coef, float bias, uint64_t n,
                         vrt_hit* d_out) {
    if (!sc) return fail(VRT_ERR_INVALID, "vrt_cast_rays_device: scene is NULL");
    if (n && (!d_origin || !d_dir || !d_out)) return fail(VRT_ERR_INVALID, "vrt_cast_rays_device: NULL buffer");
    if (n > ((1ull << 31) - 1ull) * 128ull) return fail(VRT_ERR_UNSUPPORTED, "vrt_cast_rays_device: too many rays for one launch (gridDim.x <= 2^31 - 1)");
    vrt_context* ctx = sc->ctx;
    if (int s = use_device(ctx)) return s;
    VRT_CUDA(cudaMemsetAsync(sc->d_counters, 0, 2 * sizeof(unsigned long long), ctx->stream));
    if (n == 0) return VRT_OK;
    switch (sc->kind) {
        case VRT_SCENE_LSVO:
            if (ctx->cast_variant == 3 && !sc->use_compact) {
                // automatic: cone rays are short — one thread per ray wins whatever their order; small batches are not worth a
                // look; otherwise a classifier kernel decides on the device and both kernels are enqueued, gated on its verdict
                // (no host round trip: the call stays asynchronous)
                if (fabsf(coef) >= 0.05f || n < 65536) {
                    VRT_CUDA(vrt::launch_lsvo_cast2(sc->d_nodes, int(sc->depth), sc->guard, d_origin, d_dir, coef, bias, n, d_out, sc->d_counters, ctx->stream));
                } else {
                    unsigned long long* gate = sc->d_counters + kGateSlot;
                    VRT_CUDA(vrt::launch_classify_rays(d_origin, d_dir, n, gate, ctx->stream));
                    VRT_CUDA(vrt::launch_lsvo_cast2(sc->d_nodes, int(sc->depth), sc->guard, d_origin, d_dir, coef, bias, n, d_out, sc->d_counters, ctx->stream, gate, 1ull));
                    VRT_CUDA(vrt::launch_lsvo_cast_persistent(sc->d_nodes, false, int(sc->depth), sc->guard, d_origin, d_dir, coef, bias, n, d_out, sc->d_counters,
                                                              ctx->refill_cast, ctx->stream, gate, 0ull));
                    ctx->launches += 2;
                }
            } else if ((ctx->cast_variant == 2 || ctx->cast_variant == 3) && !sc->use_compact)
                VRT_CUDA(vrt::launch_lsvo_cast2(sc->d_nodes, int(sc->depth), sc->guard, d_origin, d_dir, coef, bias, n, d_out, sc->d_counters, ctx->stream));
            else if (ctx->cast_variant == 0 || ctx->cast_variant == 2)
                VRT_CUDA(vrt::launch_lsvo_cast_ref(sc->use_compact ? sc->d_compact : sc->d_nodes, sc->use_compact, int(sc->depth), sc->guard, d_origin, d_dir, coef, bias, n, d_out,
                                                   sc->d_counters, ctx->stream));
            else
                VRT_CUDA(vrt::launch_lsvo_cast_persistent(sc->use_compact ? sc->d_compact : sc->d_nodes, sc->use_compact, int(sc->depth), sc->guard, d_origin, d_dir, coef, bias, n,
                                                          d_out, sc->d_counters, ctx->refill_cast, ctx->stream));
            ctx->launches += 1;
            return VRT_OK;
        case VRT_SCENE_GRID:
        case VRT_SCENE_MIPGRID:
            VRT_CUDA(cudaMemsetAsync(sc->d_counters, 0, 2 * sizeof(unsigned long long), ctx->stream));
            VRT_CUDA(vrt::launch_grid_cast(sc->grid, sc->use_mip, ctx->grid_variant, d_origin, d_dir, n, d_out, sc->d_counters, ctx->stream));
            ctx->launches += 1;
            return VRT_OK;
        default:
            return fail(VRT_ERR_UNSUPPORTED, "vrt_cast_rays_device: scene kind not supported (SVO scenes use vrt_cast_rays_svo)");
    }
}

int vrt_cast_rays(vrt_scene* sc, const float* origin, const float* dir, float coef, float bias, uint64_t n, vrt_hit* out) {
    if (!sc) return fail(VRT_ERR_INVALID, "vrt_cast_rays: scene is NULL");
    if (n == 0) return VRT_OK;
    if (!origin || !dir || !out) return fail(VRT_ERR_INVALID, "vrt_cast_rays: NULL buffer");
    vrt_context* ctx = sc->ctx;
    if (int s = use_device(ctx)) return s;
    const size_t ray_bytes = size_t(n) * 3 * sizeof(float);
    if (ctx->scratch_in.reserve(2 * ray_bytes) != cudaSuccess || ctx->scratch_out.reserve(size_t(n) * sizeof(vrt_hit)) != cudaSuccess)
        return fail(VRT_ERR_OOM, "vrt_cast_rays: device staging allocation failed");
    float* d_o = static_cast<float*>(ctx->scratch_in.ptr);
    float* d_d = d_o + size_t(n) * 3;
    vrt_hit* d_h = static_cast<vrt_hit*>(ctx->scratch_out.ptr);
    VRT_CUDA(cudaMemcpyAsync(d_o, origin, ray_bytes, cudaMemcpyHostToDevice, ctx->stream));
    VRT_CUDA(cudaMemcpyAsync(d_d, dir, ray_bytes, cudaMemcpyHostToDevice, ctx->stream));
    if (int s = vrt_cast_rays_device(sc, d_o, d_d, coef, bias, n, d_h)) return s;
    VRT_CUDA(cudaMemcpyAsync(out, d_h, size_t(n) * sizeof(vrt_hit), cudaMemcpyDeviceToHost, ctx->stream));
    VRT_CUDA(cudaStreamSynchronize(ctx->stream));
    return VRT_OK;
}

int vrt_scene_last_complexity(vrt_scene* sc, uint64_t* total) {
    if (!sc || !total) return fail(VRT_ERR_INVALID, "vrt_scene_last_complexity: NULL argument");
    if (int s = use_device(sc->ctx)) return s;
    unsigned long long v = 0;
    VRT_CUDA(cudaMemcpyAsync(&v, sc->d_counters, sizeof(v), cudaMemcpyDeviceToHost, sc->ctx->stream));
    VRT_CUDA(cudaStreamSynchronize(sc->ctx->stream));
    *total = v;
    return VRT_OK;
}

// ---- rendering -------------------------------------------------------------------------------------
namespace {
constexpr int kRenderCounters = 2;   // offset of the 12 render counters inside d_counters (+ kernels.h kCulledCounter = slot 16)
constexpr int kFocalSlot = 15;       // d_counters[15] holds the float focal length of vrt_render_params::autofocus

int check_render_args(const vrt_scene* sc, const vrt_camera* cam, const vrt_render_params* p, const char* who) {
    if (!sc || !p) return fail(VRT_ERR_INVALID, std::string(who) + ": NULL argument");
    if (sc->kind != VRT_SCENE_LSVO && sc->kind != VRT_SCENE_GRID && sc->kind != VRT_SCENE_MIPGRID)
        return fail(VRT_ERR_UNSUPPORTED, std::string(who) + ": rendering needs an LSVO or grid scene");
    if (cam && sc->kind != VRT_SCENE_LSVO && (p->use_gi || p->max_bounds < 0 || p->max_bounds > 16))
        return fail(VRT_ERR_INVALID, std::string(who) + ": grid frames have no GI pass; max_bounds must be 0..16");
    if (p->width <= 0 || p->height <= 0 || p->width > 65536 || p->height > 65536) return fail(VRT_ERR_INVALID, std::string(who) + ": bad frame size");
    if (p->row_begin < 0 || p->row_end > p->height || p->row_begin > p->row_end) return fail(VRT_ERR_INVALID, std::string(who) + ": bad row range");
    if (cam && (p->spp <= 0 || p->gi_bounces < 0 || p->gi_bounces > 2)) return fail(VRT_ERR_INVALID, std::string(who) + ": spp must be > 0 and gi_bounces in 0..2");
    // the resolve blends the accumulated colour as ONE 8-bit sample: spp sums would wrap around
    if (cam && !p->use_samples && p->spp != 1)
        return fail(VRT_ERR_INVALID, std::string(who) + ": the temporal-blend mode renders one sample per frame (raycaster.hpp:77-85)");
    if (p->tile_step > 1 && (p->tile_index < 0 || p->tile_index >= p->tile_step)) return fail(VRT_ERR_INVALID, std::string(who) + ": tile_index must be in [0, tile_step)");
    if (cam && !sc->has_tex && !sc->has_palette) return fail(VRT_ERR_INVALID, std::string(who) + ": call vrt_scene_set_textures first (raycaster.hpp:53-54)");
    if (cam)    // a rotation (camera_controller.hpp:27-32): the frame kernels rely on |ray direction| staying near 1 (Trav2, kUnit)
        for (int i = 0; i < 9; ++i)
            if (!(std::fabs(cam->rot_mat[i]) <= 1024.0f)) return fail(VRT_ERR_INVALID, std::string(who) + ": rot_mat is not a rotation matrix");
    if (p->checker < 0 || p->checker > 2 || p->checker_area_height < 0) return fail(VRT_ERR_INVALID, std::string(who) + ": checker must be 0, 1 or 2 and checker_area_height >= 0");
    if (cam && sc->kind == VRT_SCENE_LSVO && p->mirror_y1 != 0) {
        if (p->mirror_y1 < 0 || p->mirror_y1 > (1 << sc->depth) || p->max_bounds < 0 || p->max_bounds > 16)
            return fail(VRT_ERR_INVALID, std::string(who) + ": mirror_y1 must be 0..2^depth and max_bounds 0..16");
        if (sc->use_compact || sc->ctx->render_variant == 1 || sc->ctx->render_variant == 3)
            return fail(VRT_ERR_UNSUPPORTED, std::string(who) + ": mirror reflections need the reference node layout and render_variant 0, 2 or 4");
    }
    if (cam && sc->has_cell_types) {
        if (p->max_bounds < 0 || p->max_bounds > 16) return fail(VRT_ERR_INVALID, std::string(who) + ": max_bounds must be 0..16");
        if (sc->use_compact || sc->ctx->render_variant == 1 || sc->ctx->render_variant == 3)
            return fail(VRT_ERR_UNSUPPORTED, std::string(who) + ": mirror voxels need the reference node layout and render_variant 0, 2 or 4");
    }
    if (cam && sc->has_palette && (sc->use_compact || sc->ctx->render_variant == 1 || sc->ctx->render_variant == 3))
        return fail(VRT_ERR_UNSUPPORTED, std::string(who) + ": palette frames need the reference node layout and render_variant 0, 2 or 4");
    if (cam && sc->has_lights && (sc->use_compact || sc->ctx->render_variant == 1 || sc->ctx->render_variant == 3))
        return fail(VRT_ERR_UNSUPPORTED, std::string(who) + ": point lights need the reference node layout and render_variant 0, 2 or 4");
    if (cam && p->autofocus && sc->kind != VRT_SCENE_LSVO) return fail(VRT_ERR_UNSUPPORTED, std::string(who) + ": autofocus needs an LSVO scene");
    if (cam && p->checker && sc->kind == VRT_SCENE_LSVO && (sc->ctx->render_variant == 1 || sc->ctx->render_variant >= 3))
        return fail(VRT_ERR_UNSUPPORTED, std::string(who) + ": the checkerboard needs render_variant 0 or 2");
    return VRT_OK;
}

vrt::RenderLaunch make_launch(const vrt_scene* sc, const vrt_camera* cam, const vrt_render_params* p) {
    vrt::RenderLaunch L;
    L.width = p->width; L.height = p->height; L.row_begin = p->row_begin; L.row_end = p->row_end;
    L.spp = p->spp; L.sample_offset = p->sample_offset;
    L.depth = int(sc->depth); L.guard = sc->guard;
    L.use_gi = p->use_gi; L.gi_bounces = p->gi_bounces < 1 ? 1 : p->gi_bounces;
    L.seed_lo = p->seed_lo; L.seed_hi = p->seed_hi;
    for (int i = 0; i < 3; ++i) L.light[i] = p->light_position[i];
    L.cam = *cam;
    L.spp_chunks = sc->ctx->spp_chunks;
    L.samples_per_warp = sc->ctx->samples_per_warp;
    L.mapping = sc->ctx->render_variant == 1 ? 0 : sc->ctx->render_variant;
    L.scratch = nullptr; L.scratch_bytes = 0;
    L.beam_floor = nullptr; L.beam_shift = 0; L.beam_tiles_x = 0;
    if (sc->kind == VRT_SCENE_LSVO && sc->ctx->bounds_exit) L.bounds = sc->bounds;
    else L.bounds = vrt::SceneBounds{{1.0f, 1.0f, 1.0f}, {2.0f, 2.0f, 2.0f}};
    L.trav_policy = sc->ctx->trav_policy;
    L.grid_variant = sc->ctx->grid_variant;
    L.sort_bins1 = sc->ctx->sort_bins1; L.sort_bins2 = sc->ctx->sort_bins2;
    L.help_window = sc->ctx->help_window;
    L.roughness = p->roughness;
    L.max_bounds = p->max_bounds;
    L.mirror_y1 = sc->kind == VRT_SCENE_LSVO ? p->mirror_y1 : 0;
    L.palette = (sc->has_palette ? vrt::kPaletteAlbedo : 0) | (sc->has_cell_types ? vrt::kCellTypes : 0) |
                (sc->has_lights ? vrt::kPointLights : 0);
    L.checker = p->checker; L.checker_area_height = p->checker_area_height;
    L.focal = p->autofocus ? reinterpret_cast<const float*>(sc->d_counters + kFocalSlot) : nullptr;
    L.tile_step = p->tile_step > 1 ? p->tile_step : 1;
    L.tile_index = p->tile_step > 1 ? p->tile_index : 0;
    L.tex_top = sc->d_tex; L.tex_side = sc->d_tex + 768;
    return L;
}
}  // namespace

int vrt_scene_set_textures(vrt_scene* sc, const uint8_t* top_rgb, const uint8_t* side_rgb) {
    if (!sc || !top_rgb || !side_rgb) return fail(VRT_ERR_INVALID, "vrt_scene_set_textures: NULL argument");
    if (int s = use_device(sc->ctx)) return s;
    if (!sc->d_tex) VRT_CUDA(cudaMalloc(&sc->d_tex, vrt::kTextureBlockBytes));
    VRT_CUDA(cudaMemcpyAsync(sc->d_tex, top_rgb, 768, cudaMemcpyHostToDevice, sc->ctx->stream));
    VRT_CUDA(cudaMemcpyAsync(sc->d_tex + 768, side_rgb, 768, cudaMemcpyHostToDevice, sc->ctx->stream));
    VRT_CUDA(cudaStreamSynchronize(sc->ctx->stream));
    sc->has_tex = true;
    return VRT_OK;
}

int vrt_scene_set_palette(vrt_scene* sc, const uint8_t* rgb) {
    if (!sc) return fail(VRT_ERR_INVALID, "vrt_scene_set_palette: scene is NULL");
    if (sc->kind != VRT_SCENE_LSVO) return fail(VRT_ERR_UNSUPPORTED, "vrt_scene_set_palette: needs an LSVO scene");
    if (!rgb) {
        sc->has_palette = false;
        return VRT_OK;
    }
    if (int s = use_device(sc->ctx)) return s;
    if (!sc->d_tex) VRT_CUDA(cudaMalloc(&sc->d_tex, vrt::kTextureBlockBytes));
    VRT_CUDA(cudaMemcpyAsync(sc->d_tex + vrt::kPaletteOffset, rgb, 768, cudaMemcpyHostToDevice, sc->ctx->stream));
    VRT_CUDA(cudaStreamSynchronize(sc->ctx->stream));
    sc->has_palette = true;
    return VRT_OK;
}

int vrt_scene_set_cell_types(vrt_scene* sc, const uint8_t* types) {
    if (!sc) return fail(VRT_ERR_INVALID, "vrt_scene_set_cell_types: scene is NULL");
    if (sc->kind != VRT_SCENE_LSVO)
        return fail(VRT_ERR_UNSUPPORTED, "vrt_scene_set_cell_types: needs an LSVO scene (grid and SVO scenes have cell types of their own)");
    bool mirror = false;
    if (types)
        for (int i = 0; i < 256; ++i) {
            if (types[i] != 1 && types[i] != 2)
                return fail(VRT_ERR_INVALID, "vrt_scene_set_cell_types: every entry must be 1 (Cell::Solid) or 2 (Cell::Mirror)");
            mirror |= types[i] == 2;
        }
    if (!mirror) {                                            // all Solid: the frames of a scene without a table
        sc->has_cell_types = false;
        return VRT_OK;
    }
    if (int s = use_device(sc->ctx)) return s;
    if (!sc->d_tex) VRT_CUDA(cudaMalloc(&sc->d_tex, vrt::kTextureBlockBytes));
    VRT_CUDA(cudaMemcpyAsync(sc->d_tex + vrt::kCellTypesOffset, types, 256, cudaMemcpyHostToDevice, sc->ctx->stream));
    VRT_CUDA(cudaStreamSynchronize(sc->ctx->stream));
    sc->has_cell_types = true;
    return VRT_OK;
}

int vrt_scene_set_point_lights(vrt_scene* sc, const vrt_point_light* lights, uint32_t n) {
    if (!sc) return fail(VRT_ERR_INVALID, "vrt_scene_set_point_lights: scene is NULL");
    if (sc->kind != VRT_SCENE_LSVO) return fail(VRT_ERR_UNSUPPORTED, "vrt_scene_set_point_lights: needs an LSVO scene");
    if (n > uint32_t(vrt::kMaxPointLights)) return fail(VRT_ERR_INVALID, "vrt_scene_set_point_lights: at most 16 lights");
    if (n && !lights) return fail(VRT_ERR_INVALID, "vrt_scene_set_point_lights: lights is NULL");
    float block[1 + vrt::kMaxPointLights * vrt::kPointLightFloats];
    const uint32_t count = n;
    std::memcpy(block, &count, 4);
    for (uint32_t i = 0; i < n; ++i) {
        const vrt_point_light& l = lights[i];
        for (int a = 0; a < 3; ++a) {
            if (!std::isfinite(l.position[a])) return fail(VRT_ERR_INVALID, "vrt_scene_set_point_lights: positions must be finite");
            if (!std::isfinite(l.color[a]) || l.color[a] < 0.0f)
                return fail(VRT_ERR_INVALID, "vrt_scene_set_point_lights: colours must be finite and >= 0");
        }
        if (!(l.range > 0.0f)) return fail(VRT_ERR_INVALID, "vrt_scene_set_point_lights: ranges must be > 0 (+inf allowed)");
        float* r = block + 1 + vrt::kPointLightFloats * i;
        r[0] = l.position[0]; r[1] = l.position[1]; r[2] = l.position[2];
        r[3] = l.color[0]; r[4] = l.color[1]; r[5] = l.color[2];
        r[6] = l.range;
    }
    if (!n) {                                                 // no lights: the frames of a scene that never had any
        sc->has_lights = false;
        return VRT_OK;
    }
    if (int s = use_device(sc->ctx)) return s;
    if (!sc->d_tex) VRT_CUDA(cudaMalloc(&sc->d_tex, vrt::kTextureBlockBytes));
    VRT_CUDA(cudaMemcpyAsync(sc->d_tex + vrt::kLightsOffset, block, 4 * (1 + vrt::kPointLightFloats * size_t(n)), cudaMemcpyHostToDevice,
                             sc->ctx->stream));
    VRT_CUDA(cudaStreamSynchronize(sc->ctx->stream));
    sc->has_lights = true;
    return VRT_OK;
}

int vrt_render_accumulate_device(vrt_scene* sc, const vrt_camera* cam, const vrt_render_params* p, uint32_t* d_accum) {
    if (!cam || !d_accum) return fail(VRT_ERR_INVALID, "vrt_render_accumulate_device: NULL argument");
    if (int s = check_render_args(sc, cam, p, "vrt_render_accumulate_device")) return s;
    vrt_context* ctx = sc->ctx;
    if (int s = use_device(ctx)) return s;
    VRT_CUDA(cudaMemsetAsync(sc->d_counters + kRenderCounters, 0, 13 * sizeof(unsigned long long), ctx->stream));
    VRT_CUDA(cudaMemsetAsync(sc->d_counters + kRenderCounters + vrt::kCulledCounter, 0, sizeof(unsigned long long), ctx->stream));
    if (p->row_end == p->row_begin) return VRT_OK;
    cudaEvent_t ev_begin = nullptr, ev_end = nullptr;
    if (ctx->time_frame_kernels) {                           // device time of this call's frame kernels, on the launching stream
        VRT_CUDA(cudaEventCreate(&ev_begin));
        VRT_CUDA(cudaEventCreate(&ev_end));
        VRT_CUDA(cudaEventRecord(ev_begin, ctx->stream));
        ctx->frame_events.emplace_back(ev_begin, ev_end);
    }
    struct RecordEnd {                                       // records ev_end on every exit path of the function
        cudaEvent_t ev; cudaStream_t st;
        ~RecordEnd() { if (ev) cudaEventRecord(ev, st); }
    } record_end{ev_end, ctx->stream};
    if (p->autofocus) {
        VRT_CUDA(vrt::launch_autofocus(sc->use_compact ? sc->d_compact : sc->d_nodes, sc->use_compact, int(sc->depth), sc->guard, *cam,
                                       reinterpret_cast<float*>(sc->d_counters + kFocalSlot), ctx->stream));
        ctx->launches += 1;
    }
    if (sc->kind != VRT_SCENE_LSVO)
        VRT_CUDA(vrt::launch_grid_render(sc->grid, sc->use_mip, make_launch(sc, cam, p), d_accum, sc->d_counters + kRenderCounters,
                                         ctx->stream));
    else if (ctx->render_variant != 1) {
        vrt::RenderLaunch L = make_launch(sc, cam, p);
        // beam floors (beam_kernels.cu): conservative start distances of the camera rays, per screen tile.  Frames are
        // identical with and without them; only the trip counts of the primary rays shrink.
        // Worth its own launch (a latency-bound tree search, eight lanes per tile) only when every floor is used by many
        // rays: frames with >= 8 samples per pixel.  The interactive 1-sample frames (0.2 ms in all) go without.
        if (ctx->beam_tile > 0 && p->spp >= 8 && !sc->use_compact && (ctx->render_variant == 0 || ctx->render_variant == 2 || ctx->render_variant == 4)) {
            int shift = 0;
            while ((1 << (shift + 1)) <= ctx->beam_tile) ++shift;
            const int tile = 1 << shift, tiles_x = (p->width + tile - 1) / tile, tiles_y = (p->height + tile - 1) / tile;
            const size_t bytes = size_t(tiles_x) * tiles_y * sizeof(float);
            if (bytes > sc->beam_floor.bytes) VRT_CUDA(cudaStreamSynchronize(ctx->stream));
            if (sc->beam_floor.reserve(bytes) != cudaSuccess) return fail(VRT_ERR_OOM, "vrt_render_accumulate_device: beam floor allocation failed");
            VRT_CUDA(vrt::launch_beam_floor(sc->d_nodes, L, tile, static_cast<float*>(sc->beam_floor.ptr), ctx->stream));
            ctx->launches += 1;
            L.beam_floor = static_cast<const float*>(sc->beam_floor.ptr);
            L.beam_shift = shift;
            L.beam_tiles_x = tiles_x;
        }
        const size_t need = vrt::render_scratch_bytes(L);
        if (need) {
            if (need > sc->frame_lists.bytes) VRT_CUDA(cudaStreamSynchronize(ctx->stream));     // an earlier frame may still read the old buffer
            if (sc->frame_lists.reserve(need) != cudaSuccess) return fail(VRT_ERR_OOM, "vrt_render_accumulate_device: scratch allocation failed");
            L.scratch = sc->frame_lists.ptr;
            L.scratch_bytes = sc->frame_lists.bytes;
            ctx->launches += 1;                                                                  // the sort kernel
        }
        VRT_CUDA(vrt::launch_render_accumulate_ref(sc->use_compact ? sc->d_compact : sc->d_nodes, sc->use_compact, L, d_accum, sc->d_counters + kRenderCounters,
                                                   ctx->stream));
    }
    else
        VRT_CUDA(vrt::launch_render_persistent(sc->d_nodes, make_launch(sc, cam, p), d_accum, sc->d_counters + kRenderCounters,
                                               ctx->refill_render, ctx->stream));
    ctx->launches += 1;
    return VRT_OK;
}

int vrt_render_resolve_device(vrt_scene* sc, const vrt_render_params* p, const uint32_t* d_accum, uint8_t* d_rgba) {
    if (!d_accum || !d_rgba) return fail(VRT_ERR_INVALID, "vrt_render_resolve_device: NULL argument");
    if (int s = check_render_args(sc, nullptr, p, "vrt_render_resolve_device")) return s;
    vrt_context* ctx = sc->ctx;
    if (int s = use_device(ctx)) return s;
    if (p->row_end == p->row_begin) return VRT_OK;
    VRT_CUDA(vrt::launch_resolve(d_accum, d_rgba, p->width, p->row_begin, p->row_end, p->use_samples,
                                 p->tile_step > 1 ? p->tile_step : 1, p->tile_step > 1 ? p->tile_index : 0, ctx->stream));
    ctx->launches += 1;
    return VRT_OK;
}

int vrt_shade_rays(vrt_scene* sc, const vrt_render_params* p, uint64_t n, const vrt_shade_job* jobs, vrt_shade_result* out) {
    if (!sc || !p) return fail(VRT_ERR_INVALID, "vrt_shade_rays: NULL argument");
    if (sc->kind != VRT_SCENE_LSVO) return fail(VRT_ERR_UNSUPPORTED, "vrt_shade_rays: needs an LSVO scene");
    if (!sc->has_tex && !sc->has_palette) return fail(VRT_ERR_INVALID, "vrt_shade_rays: call vrt_scene_set_textures first (raycaster.hpp:53-54)");
    if (p->gi_bounces < 0 || p->gi_bounces > 2) return fail(VRT_ERR_INVALID, "vrt_shade_rays: gi_bounces must be 0..2");
    if (sc->has_cell_types && (p->max_bounds < 0 || p->max_bounds > 16)) return fail(VRT_ERR_INVALID, "vrt_shade_rays: max_bounds must be 0..16");
    if (n == 0) return VRT_OK;
    if (!jobs || !out) return fail(VRT_ERR_INVALID, "vrt_shade_rays: NULL buffer");
    if (n > (1ull << 31)) return fail(VRT_ERR_UNSUPPORTED, "vrt_shade_rays: too many rays for one call");
    vrt_context* ctx = sc->ctx;
    if (int s = use_device(ctx)) return s;
    if (ctx->scratch_in.reserve(size_t(n) * sizeof(vrt_shade_job)) != cudaSuccess || ctx->scratch_out.reserve(size_t(n) * sizeof(vrt_shade_result)) != cudaSuccess)
        return fail(VRT_ERR_OOM, "vrt_shade_rays: device staging allocation failed");
    vrt_shade_job* d_jobs = static_cast<vrt_shade_job*>(ctx->scratch_in.ptr);
    vrt_shade_result* d_out = static_cast<vrt_shade_result*>(ctx->scratch_out.ptr);
    VRT_CUDA(cudaMemcpyAsync(d_jobs, jobs, size_t(n) * sizeof(vrt_shade_job), cudaMemcpyHostToDevice, ctx->stream));
    vrt_camera cam;
    std::memset(&cam, 0, sizeof(cam));
    vrt_render_params q = *p;
    if (q.width <= 0) q.width = 1;
    if (q.height <= 0) q.height = 1;
    // the palette instance (palette, cell types, point lights) reads the reference array
    const bool compact = sc->use_compact && !sc->has_palette && !sc->has_cell_types && !sc->has_lights;
    VRT_CUDA(vrt::launch_shade_rays(compact ? sc->d_compact : sc->d_nodes, compact, make_launch(sc, &cam, &q), n, d_jobs, d_out, ctx->stream));
    ctx->launches += 1;
    VRT_CUDA(cudaMemcpyAsync(out, d_out, size_t(n) * sizeof(vrt_shade_result), cudaMemcpyDeviceToHost, ctx->stream));
    VRT_CUDA(cudaStreamSynchronize(ctx->stream));
    return VRT_OK;
}

int vrt_beam_floors(vrt_scene* sc, const vrt_camera* cam, const vrt_render_params* p, int32_t tile, float* out) {
    if (!sc || !cam || !p || !out) return fail(VRT_ERR_INVALID, "vrt_beam_floors: NULL argument");
    if (sc->kind != VRT_SCENE_LSVO || sc->use_compact) return fail(VRT_ERR_UNSUPPORTED, "vrt_beam_floors: needs an LSVO scene in the reference layout");
    if (tile < 1 || tile > 64 || (tile & (tile - 1))) return fail(VRT_ERR_INVALID, "vrt_beam_floors: tile must be a power of two, 1..64");
    if (p->width <= 0 || p->height <= 0 || p->width > 65536 || p->height > 65536) return fail(VRT_ERR_INVALID, "vrt_beam_floors: bad frame size");
    vrt_context* ctx = sc->ctx;
    if (int s = use_device(ctx)) return s;
    const int tiles_x = (p->width + tile - 1) / tile, tiles_y = (p->height + tile - 1) / tile;
    const size_t bytes = size_t(tiles_x) * tiles_y * sizeof(float);
    if (bytes > sc->beam_floor.bytes) VRT_CUDA(cudaStreamSynchronize(ctx->stream));
    if (sc->beam_floor.reserve(bytes) != cudaSuccess) return fail(VRT_ERR_OOM, "vrt_beam_floors: device allocation failed");
    vrt_render_params q = *p;
    q.row_begin = 0; q.row_end = p->height; q.autofocus = 0;
    VRT_CUDA(vrt::launch_beam_floor(sc->d_nodes, make_launch(sc, cam, &q), tile, static_cast<float*>(sc->beam_floor.ptr), ctx->stream));
    ctx->launches += 1;
    VRT_CUDA(cudaMemcpyAsync(out, sc->beam_floor.ptr, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    VRT_CUDA(cudaStreamSynchronize(ctx->stream));
    return VRT_OK;
}

int vrt_scene_last_render_stats(vrt_scene* sc, vrt_render_stats* stats) {
    if (!sc || !stats) return fail(VRT_ERR_INVALID, "vrt_scene_last_render_stats: NULL argument");
    if (int s = use_device(sc->ctx)) return s;
    unsigned long long v[12];
    VRT_CUDA(cudaMemcpyAsync(v, sc->d_counters + kRenderCounters, sizeof(v), cudaMemcpyDeviceToHost, sc->ctx->stream));
    VRT_CUDA(cudaStreamSynchronize(sc->ctx->stream));
    for (int k = 0; k < 6; ++k) { stats->rays[k] = v[k]; stats->complexity[k] = v[6 + k]; }
    return VRT_OK;
}

int vrt_scene_last_render_culled(vrt_scene* sc, uint64_t* primary_rays) {
    if (!sc || !primary_rays) return fail(VRT_ERR_INVALID, "vrt_scene_last_render_culled: NULL argument");
    if (int s = use_device(sc->ctx)) return s;
    unsigned long long v = 0;
    VRT_CUDA(cudaMemcpyAsync(&v, sc->d_counters + kRenderCounters + vrt::kCulledCounter, sizeof(v), cudaMemcpyDeviceToHost, sc->ctx->stream));
    VRT_CUDA(cudaStreamSynchronize(sc->ctx->stream));
    *primary_rays = v;
    return VRT_OK;
}

int vrt_render(vrt_scene* sc, const vrt_camera* cam, const vrt_render_params* p, uint8_t* rgba, uint32_t* accum,
               vrt_render_stats* stats) {
    if (!cam || !rgba) return fail(VRT_ERR_INVALID, "vrt_render: NULL argument");
    if (int s = check_render_args(sc, cam, p, "vrt_render")) return s;
    vrt_context* ctx = sc->ctx;
    if (int s = use_device(ctx)) return s;
    const size_t px = size_t(p->width) * p->height;
    if (sc->frame_accum.reserve(px * 16) != cudaSuccess || sc->frame_rgba.reserve(px * 4) != cudaSuccess)
        return fail(VRT_ERR_OOM, "vrt_render: device frame allocation failed");
    uint32_t* d_accum = static_cast<uint32_t*>(sc->frame_accum.ptr);
    uint8_t* d_rgba = static_cast<uint8_t*>(sc->frame_rgba.ptr);
    const size_t row0 = size_t(p->row_begin) * p->width, nrow = size_t(p->row_end - p->row_begin) * p->width;
    if (p->accum_in && accum)
        VRT_CUDA(cudaMemcpyAsync(d_accum + row0 * 4, accum + row0 * 4, nrow * 16, cudaMemcpyHostToDevice, ctx->stream));
    else
        VRT_CUDA(cudaMemsetAsync(d_accum + row0 * 4, 0, nrow * 16, ctx->stream));
    if (!p->use_samples)   // the blend reads the previous frame
        VRT_CUDA(cudaMemcpyAsync(d_rgba + row0 * 4, rgba + row0 * 4, nrow * 4, cudaMemcpyHostToDevice, ctx->stream));
    if (int s = vrt_render_accumulate_device(sc, cam, p, d_accum)) return s;
    if (int s = vrt_render_resolve_device(sc, p, d_accum, d_rgba)) return s;
    VRT_CUDA(cudaMemcpyAsync(rgba + row0 * 4, d_rgba + row0 * 4, nrow * 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (accum) VRT_CUDA(cudaMemcpyAsync(accum + row0 * 4, d_accum + row0 * 4, nrow * 16, cudaMemcpyDeviceToHost, ctx->stream));
    VRT_CUDA(cudaStreamSynchronize(ctx->stream));
    if (stats) return vrt_scene_last_render_stats(sc, stats);
    return VRT_OK;
}

namespace {
int check_present_args(const vrt_context* ctx, const void* frame, const void* display, const vrt_present_params* p, const char* who) {
    if (!ctx || !frame || !display || !p) return fail(VRT_ERR_INVALID, std::string(who) + ": NULL argument");
    if (p->width <= 0 || p->height <= 0 || p->width > 65536 || p->height > 65536) return fail(VRT_ERR_INVALID, std::string(who) + ": bad frame size");
    if (p->median != 0 && p->median != 3 && p->median != 5) return fail(VRT_ERR_INVALID, std::string(who) + ": median must be 0, 3 or 5");
    if (!(p->old_value_conservation >= 0.0f && p->old_value_conservation <= 1.0f))
        return fail(VRT_ERR_INVALID, std::string(who) + ": old_value_conservation must be in [0, 1]");
    return VRT_OK;
}
}  // namespace

int vrt_present_device(vrt_context* ctx, const uint8_t* d_frame, uint8_t* d_display, const vrt_present_params* p) {
    if (int s = check_present_args(ctx, d_frame, d_display, p, "vrt_present_device")) return s;
    if (int s = use_device(ctx)) return s;
    // sf::Color(255 * old_value_conservation, ...) and c2 = 255 * (1.0f - old_value_conservation): float → Uint8 (main.cpp:160-165)
    const uint32_t c1 = uint8_t(255 * p->old_value_conservation), c2 = uint8_t(255 * (1.0f - p->old_value_conservation));
    VRT_CUDA(vrt::launch_present(d_frame, d_display, p->width, p->height, p->median, c1, c2, ctx->stream));
    ctx->launches += 1;
    return VRT_OK;
}

int vrt_present(vrt_context* ctx, const uint8_t* frame, uint8_t* display, const vrt_present_params* p) {
    if (int s = check_present_args(ctx, frame, display, p, "vrt_present")) return s;
    if (int s = use_device(ctx)) return s;
    const size_t bytes = size_t(p->width) * p->height * 4;
    if (ctx->scratch_in.reserve(bytes) != cudaSuccess || ctx->scratch_out.reserve(bytes) != cudaSuccess)
        return fail(VRT_ERR_OOM, "vrt_present: device allocation failed");
    uint8_t* d_frame = static_cast<uint8_t*>(ctx->scratch_in.ptr);
    uint8_t* d_display = static_cast<uint8_t*>(ctx->scratch_out.ptr);
    VRT_CUDA(cudaMemcpyAsync(d_frame, frame, bytes, cudaMemcpyHostToDevice, ctx->stream));
    VRT_CUDA(cudaMemcpyAsync(d_display, display, bytes, cudaMemcpyHostToDevice, ctx->stream));
    if (int s = vrt_present_device(ctx, d_frame, d_display, p)) return s;
    VRT_CUDA(cudaMemcpyAsync(display, d_display, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    VRT_CUDA(cudaStreamSynchronize(ctx->stream));
    return VRT_OK;
}

int vrt_autofocus(vrt_scene* sc, const vrt_camera* cam, float* focal_length) {
    if (!sc || !cam || !focal_length) return fail(VRT_ERR_INVALID, "vrt_autofocus: NULL argument");
    if (sc->kind != VRT_SCENE_LSVO) return fail(VRT_ERR_UNSUPPORTED, "vrt_autofocus: needs an LSVO scene");
    // Camera::getClosestPoint (camera_controller.hpp:56-60): position*scale + 1 along camera_vec = (0,0,1)*rot_mat
    const float scale = 1.0f / float(1u << sc->depth);
    float o[3], d[3];
    for (int i = 0; i < 3; ++i) {
        o[i] = cam->position[i] * scale + 1.0f;
        d[i] = (cam->rot_mat[3 * i + 0] * 0.0f + cam->rot_mat[3 * i + 1] * 0.0f) + cam->rot_mat[3 * i + 2] * 1.0f;
    }
    vrt_hit h;
    if (int s = vrt_cast_rays(sc, o, d, 0.0f, 0.0f, 1, &h)) return s;
    *focal_length = (h.flags & VRT_HIT_FLAG_HIT) ? h.distance * float(1u << sc->depth) : 100.0f;   // main.cpp:116-121
    return VRT_OK;
}

// ---- dense grids: Grid3D / MipmapGrid3D / SVO ---------------------------------------------------------
namespace {
// Packs occupancy (cells != 0) into bits and builds the OR-pyramid up to `levels` levels (level l = cubes of
// edge 2^l; dims rounded up).  Returns the host words and fills `g` with word offsets in place of pointers.
std::vector<uint32_t> build_grid_pyramid(const uint8_t* cells, int X, int Y, int Z, int levels, vrt::GridLevels& g,
                                         std::vector<size_t>& offsets) {
    std::vector<uint32_t> words;
    g.X = X; g.Y = Y; g.Z = Z; g.n_levels = levels;
    std::vector<uint8_t> cur(cells, cells + size_t(X) * Y * Z), next;
    int nx = X, ny = Y, nz = Z;
    for (int l = 0; l < levels; ++l) {
        g.level[l].nx = nx; g.level[l].ny = ny; g.level[l].nz = nz;
        const size_t nbits = size_t(nx) * ny * nz, nwords = (nbits + 31) / 32;
        offsets.push_back(words.size());
        words.resize(words.size() + nwords, 0u);
        uint32_t* w = words.data() + offsets.back();
        for (size_t i = 0; i < nbits; ++i)
            if (cur[i]) w[i >> 5] |= 1u << (i & 31);
        if (l + 1 < levels) {
            const int mx = (nx + 1) / 2, my = (ny + 1) / 2, mz = (nz + 1) / 2;
            next.assign(size_t(mx) * my * mz, 0);
            for (int x = 0; x < nx; ++x)
                for (int y = 0; y < ny; ++y)
                    for (int z = 0; z < nz; ++z)
                        if (cur[(size_t(x) * ny + y) * nz + z]) next[(size_t(x >> 1) * my + (y >> 1)) * mz + (z >> 1)] = 1;
            cur.swap(next);
            nx = mx; ny = my; nz = mz;
        }
    }
    return words;
}

int create_grid_scene(vrt_context* ctx, const uint8_t* cells, int X, int Y, int Z, int levels, int kind, uint32_t depth,
                      vrt_scene** out) {
    if (int s = use_device(ctx)) return s;
    vrt_scene* sc = new (std::nothrow) vrt_scene();
    if (!sc) return fail(VRT_ERR_OOM, "grid scene: host allocation failed");
    sc->ctx = ctx; sc->kind = kind; sc->depth = depth;
    std::vector<size_t> offsets;
    std::vector<uint32_t> words = build_grid_pyramid(cells, X, Y, Z, levels, sc->grid, offsets);
    // Cell::Mirror (= 2, cell.hpp:8) bit plane for the reflection pass, only if the grid has mirrors
    const size_t ncell = size_t(X) * Y * Z;
    size_t mirror_off = 0;
    bool any_mirror = false;
    for (size_t i = 0; i < ncell && !any_mirror; ++i) any_mirror = cells[i] == 2;
    if (any_mirror) {
        mirror_off = words.size();
        words.resize(words.size() + (ncell + 31) / 32, 0u);
        for (size_t i = 0; i < ncell; ++i)
            if (cells[i] == 2) words[mirror_off + (i >> 5)] |= 1u << (i & 31);
    }
    // level 0 with a solid one-cell border (kernels.h GridLevels::pad_bits): rows are copied with their z bits shifted by one
    size_t pad_off = 0;
    const uint64_t PX = uint64_t(X) + 2, PY = uint64_t(Y) + 2, PZ = uint64_t(Z) + 2;
    const bool padded = kind != VRT_SCENE_SVO && PX * PY * PZ < (1ull << 32);
    if (padded) {
        pad_off = words.size();
        const uint64_t nbits = PX * PY * PZ;
        words.resize(words.size() + size_t((nbits + 31) / 32), 0u);
        uint32_t* w = words.data() + pad_off;
        auto set_bit = [&](uint64_t i) { w[i >> 5] |= 1u << (i & 31); };
        for (uint64_t x = 0; x < PX; ++x)
            for (uint64_t y = 0; y < PY; ++y) {
                const uint64_t row = (x * PY + y) * PZ;
                if (x == 0 || x == PX - 1 || y == 0 || y == PY - 1) {
                    for (uint64_t z = 0; z < PZ; ++z) set_bit(row + z);
                    continue;
                }
                set_bit(row);
                set_bit(row + PZ - 1);
                const uint8_t* src = cells + ((x - 1) * uint64_t(Y) + (y - 1)) * uint64_t(Z);
                for (uint64_t z = 0; z < uint64_t(Z); ++z)
                    if (src[z]) set_bit(row + 1 + z);
            }
    }
    cudaError_t e = cudaMalloc(&sc->d_grid_bits, words.size() * sizeof(uint32_t));
    if (e == cudaSuccess) e = cudaMalloc(&sc->d_counters, kCounterSlots * sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMemcpyAsync(sc->d_grid_bits, words.data(), words.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(sc->d_counters, 0, kCounterSlots * sizeof(unsigned long long), ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) { vrt_scene_destroy(sc); return cuda_fail(e, "grid scene upload"); }
    for (int l = 0; l < levels; ++l) sc->grid.level[l].bits = sc->d_grid_bits + offsets[l];
    sc->grid.mirror = any_mirror ? sc->d_grid_bits + mirror_off : nullptr;
    sc->grid.pad_bits = padded ? sc->d_grid_bits + pad_off : nullptr;
    sc->grid.pad_y = uint32_t(PY);
    sc->grid.pad_z = uint32_t(PZ);
    sc->device_bytes = words.size() * sizeof(uint32_t);
    *out = sc;
    return VRT_OK;
}
}  // namespace

int vrt_grid_create(vrt_context* ctx, const uint8_t* cell_types, int32_t X, int32_t Y, int32_t Z, int32_t mip_levels,
                    vrt_scene** out) {
    if (!ctx || !cell_types || !out) return fail(VRT_ERR_INVALID, "vrt_grid_create: NULL argument");
    if (X <= 0 || Y <= 0 || Z <= 0 || X > 4096 || Y > 4096 || Z > 4096) return fail(VRT_ERR_INVALID, "vrt_grid_create: dimensions must be 1..4096");
    if (mip_levels < 0 || mip_levels > 11) return fail(VRT_ERR_INVALID, "vrt_grid_create: mip_levels must be 0..11");
    int s = create_grid_scene(ctx, cell_types, X, Y, Z, 1 + mip_levels, mip_levels > 0 ? VRT_SCENE_MIPGRID : VRT_SCENE_GRID, 0, out);
    if (s == VRT_OK) (*out)->use_mip = mip_levels > 0;
    return s;
}

int vrt_svo_create(vrt_context* ctx, const uint8_t* occ, uint32_t depth, vrt_scene** out) {
    if (!ctx || !occ || !out) return fail(VRT_ERR_INVALID, "vrt_svo_create: NULL argument");
    if (depth < 1 || depth > 10) return fail(VRT_ERR_INVALID, "vrt_svo_create: depth must be 1..10 (dense occupancy input)");
    const int S = 1 << depth;
    return create_grid_scene(ctx, occ, S, S, S, int(depth) + 1, VRT_SCENE_SVO, depth, out);
}

int vrt_cast_rays_svo(vrt_scene* sc, const float* origin, const float* dir, uint32_t max_iter, uint64_t n, vrt_hit* out) {
    if (!sc) return fail(VRT_ERR_INVALID, "vrt_cast_rays_svo: scene is NULL");
    if (sc->kind != VRT_SCENE_SVO) return fail(VRT_ERR_INVALID, "vrt_cast_rays_svo: not an SVO scene");
    if (n == 0) return VRT_OK;
    if (!origin || !dir || !out) return fail(VRT_ERR_INVALID, "vrt_cast_rays_svo: NULL buffer");
    vrt_context* ctx = sc->ctx;
    if (int s = use_device(ctx)) return s;
    const size_t ray_bytes = size_t(n) * 3 * sizeof(float);
    if (ctx->scratch_in.reserve(2 * ray_bytes) != cudaSuccess || ctx->scratch_out.reserve(size_t(n) * sizeof(vrt_hit)) != cudaSuccess)
        return fail(VRT_ERR_OOM, "vrt_cast_rays_svo: device staging allocation failed");
    float* d_o = static_cast<float*>(ctx->scratch_in.ptr);
    float* d_d = d_o + size_t(n) * 3;
    vrt_hit* d_h = static_cast<vrt_hit*>(ctx->scratch_out.ptr);
    VRT_CUDA(cudaMemcpyAsync(d_o, origin, ray_bytes, cudaMemcpyHostToDevice, ctx->stream));
    VRT_CUDA(cudaMemcpyAsync(d_d, dir, ray_bytes, cudaMemcpyHostToDevice, ctx->stream));
    VRT_CUDA(cudaMemsetAsync(sc->d_counters, 0, 2 * sizeof(unsigned long long), ctx->stream));
    VRT_CUDA(vrt::launch_svo_cast(sc->grid, int(sc->depth), d_o, d_d, max_iter, n, d_h, sc->d_counters, ctx->stream));
    ctx->launches += 1;
    VRT_CUDA(cudaMemcpyAsync(out, d_h, size_t(n) * sizeof(vrt_hit), cudaMemcpyDeviceToHost, ctx->stream));
    VRT_CUDA(cudaStreamSynchronize(ctx->stream));
    return VRT_OK;
}

}  // extern "C"
