// Scene construction on the GPU for ARBITRARY voxel sets, and voxel edits (dynamic scenes).
//
// Replaces, with byte-identical output (tests compare against the host flattener, which is pinned to compileSVO):
//   include/svo.hpp:72-114               SVO::setCell / rec_setCell (one 80-byte node per level and voxel — never built)
//   include/lsvo_utils.hpp:45-55,
//   src/lsvo_utils.cpp:4-49              compileSVO / compileSVO_rec: DFS pre-order, 8 slots per interior node,
//                                        children visited x outer / y / z inner, slot = z*4 + y*2 + x
// and gives LSVO::setCell (a no-op in the reference, lsvo.hpp:26) a meaning: the scene keeps its sorted voxel keys on
// the device; adding or removing voxels merges / filters that list and re-flattens.
//
// DFS numbering without a DFS, for any voxel set.  A voxel's key is its path from the root, three bits per level in
// VISIT order (x, y, z — most significant first), so sorting the keys sorts the voxels in compileSVO_rec's pre-order.
// The interior nodes of level l are the distinct key prefixes of 3*l bits (P_l, sorted).  compileSVO_rec appends a node's
// 8-slot child block when it visits the node, so
//     child_pos(N) = 1 + 8 * #{interior nodes visited before N}
// and a node M is visited before N (level l, prefix p) iff
//     M is shallower (level l' < l) and   prefix(M) <= p >> 3(l - l')          (an ancestor, or left of one)
//     M is on N's level            and   prefix(M) <  p
//     M is deeper  (level l' > l) and   prefix(M) >> 3(l' - l) <  p            (below something left of N)
// — one binary search per level.  The node's own slot is child_pos(parent) + slot, its masks come from the range of
// P_{l+1} that shares its prefix.  Sorting / unique / select are CUB device primitives (scene construction is not the hot
// path); keys, ranks and slots are the kernels below.
#include <cub/cub.cuh>

#include <vector>

#include "kernels.h"
#include "lsvo_traverse.cuh"

namespace vrt {

namespace {

constexpr int kMaxLevels = 14;

struct PrefixLevels {
    const uint64_t* p[kMaxLevels];    // p[l]: sorted distinct prefixes of level l (p[depth] = the voxel keys)
    uint32_t n[kMaxLevels];
    int depth;
};

using Scratch = PoolScratch;

#define VRT_TRY(call)                          \
    do {                                       \
        cudaError_t e_ = (call);               \
        if (e_ != cudaSuccess) return e_;      \
    } while (0)

// path key of a voxel in SVO::setCell coordinates: per level (top first) the visit-order digit x*4 + y*2 + z
__global__ void voxel_keys_kernel(const uint32_t* __restrict__ xyz, uint64_t n, int depth, uint64_t* __restrict__ keys) {
    const uint64_t i = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t x = xyz[3 * i], y = xyz[3 * i + 1], z = xyz[3 * i + 2];
    uint64_t key = 0;
    for (int b = depth - 1; b >= 0; --b)
        key = (key << 3) | uint64_t((((x >> b) & 1u) << 2) | (((y >> b) & 1u) << 1) | ((z >> b) & 1u));
    keys[i] = key;
}

__global__ void shift3_kernel(const uint64_t* __restrict__ in, uint32_t n, uint64_t* __restrict__ out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = in[i] >> 3;
}

__device__ __forceinline__ uint32_t lower_bound_u64(const uint64_t* __restrict__ a, uint32_t n, uint64_t v) {   // first a[i] >= v
    uint32_t lo = 0, hi = n;
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (a[mid] < v) lo = mid + 1; else hi = mid;
    }
    return lo;
}
__device__ __forceinline__ uint32_t upper_bound_u64(const uint64_t* __restrict__ a, uint32_t n, uint64_t v) {   // first a[i] > v
    uint32_t lo = 0, hi = n;
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (a[mid] <= v) lo = mid + 1; else hi = mid;
    }
    return lo;
}
__device__ __forceinline__ uint32_t slot_of_digit(uint64_t digit) {        // visit digit x*4+y*2+z → sub-index z*4+y*2+x
    const uint32_t d = uint32_t(digit) & 7u;
    return ((d & 1u) << 2) | (d & 2u) | (d >> 2);
}

// child_pos of every interior node of level l
__global__ void rank_kernel(PrefixLevels P, int l, uint32_t* __restrict__ cpos) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P.n[l]) return;
    const uint64_t p = P.p[l][i];
    uint64_t before = i;                                                    // same level: distinct and sorted
    for (int m = 0; m < l; ++m) before += upper_bound_u64(P.p[m], P.n[m], p >> (3 * (l - m)));
    for (int m = l + 1; m < P.depth; ++m) before += lower_bound_u64(P.p[m], P.n[m], p << (3 * (m - l)));
    cpos[i] = uint32_t(1u + 8u * before);
}

// the LNode of every interior node of level l (lsvo_utils.hpp:5-18): color 1, child mask, leaf mask, child_offset
__global__ void emit_nodes_kernel(PrefixLevels P, int l, const uint32_t* __restrict__ cpos, const uint32_t* __restrict__ cpos_parent,
                                  uint2* __restrict__ slots) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P.n[l]) return;
    const uint64_t p = P.p[l][i];
    uint32_t self = 0u;                                                      // the root is slot 0
    if (l > 0) self = cpos_parent[lower_bound_u64(P.p[l - 1], P.n[l - 1], p >> 3)] + slot_of_digit(p);
    const uint64_t* kids = P.p[l + 1];
    const uint32_t lo = lower_bound_u64(kids, P.n[l + 1], p << 3), hi = lower_bound_u64(kids, P.n[l + 1], (p + 1) << 3);
    uint32_t mask = 0u;
    for (uint32_t k = lo; k < hi; ++k) mask |= 1u << slot_of_digit(kids[k]);
    const uint32_t leaf = (l == P.depth - 1) ? mask : 0u;                   // children of the last interior level are voxels
    slots[self] = make_uint2(1u | (mask << 8) | (leaf << 16), cpos[i] - self);
}

__global__ void fill_default_slots_kernel(uint2* __restrict__ slots, uint64_t n) {
    for (uint64_t i = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += uint64_t(gridDim.x) * blockDim.x)
        slots[i] = make_uint2(1u, 0u);                                       // LNode(): color 1, masks 0, offset 0
}

// flags[i] = 1 iff keys[i] is NOT in the sorted list `gone`
__global__ void keep_flags_kernel(const uint64_t* __restrict__ keys, uint32_t n, const uint64_t* __restrict__ gone, uint32_t n_gone,
                                  uint8_t* __restrict__ flags) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t j = lower_bound_u64(gone, n_gone, keys[i]);
    flags[i] = (j < n_gone && gone[j] == keys[i]) ? 0 : 1;
}

cudaError_t sort_unique(uint64_t* d_in, uint32_t n, int bits, uint64_t* d_sorted, uint64_t* d_unique, uint32_t* n_unique, Scratch& sc,
                        cudaStream_t stream) {
    *n_unique = 0;
    if (n == 0) return cudaSuccess;
    size_t t1 = 0, t2 = 0;
    uint32_t* d_count = nullptr;
    VRT_TRY(sc.alloc(&d_count, 1));
    VRT_TRY(cub::DeviceRadixSort::SortKeys(nullptr, t1, d_in, d_sorted, n, 0, bits, stream));
    VRT_TRY(cub::DeviceSelect::Unique(nullptr, t2, d_sorted, d_unique, d_count, n, stream));
    uint8_t* d_temp = nullptr;
    VRT_TRY(sc.alloc(&d_temp, t1 > t2 ? t1 : t2));
    VRT_TRY(cub::DeviceRadixSort::SortKeys(d_temp, t1, d_in, d_sorted, n, 0, bits, stream));
    VRT_TRY(cub::DeviceSelect::Unique(d_temp, t2, d_sorted, d_unique, d_count, n, stream));
    VRT_TRY(cudaMemcpyAsync(n_unique, d_count, sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
    return cudaStreamSynchronize(stream);
}

// ---- per-voxel colours: the `color` byte of a solid voxel's leaf slot (DESIGN.md §2) ----------------------------------------
__device__ __forceinline__ uint64_t voxel_key(uint32_t x, uint32_t y, uint32_t z, int depth) {     // as voxel_keys_kernel
    uint64_t key = 0;
    for (int b = depth - 1; b >= 0; --b)
        key = (key << 3) | uint64_t((((x >> b) & 1u) << 2) | (((y >> b) & 1u) << 1) | ((z >> b) & 1u));
    return key;
}

// slot[i] = leaf slot of voxel i (kNoLeafSlot when empty), index[i] = i
__global__ void paint_slots_kernel(const uint2* __restrict__ nodes, int depth, const uint32_t* __restrict__ xyz, uint32_t n,
                                   uint32_t* __restrict__ slot, uint32_t* __restrict__ index) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    slot[i] = lsvo_leaf_slot(nodes, depth, xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2]);
    index[i] = i;
}

// (slot, index) pairs sorted by slot, stably: the last entry of a run of equal slots is the voxel's last occurrence in the list
__global__ void paint_write_kernel(uint2* __restrict__ nodes, int depth, const uint32_t* __restrict__ xyz, const uint8_t* __restrict__ colors,
                                   const uint32_t* __restrict__ slot, const uint32_t* __restrict__ index, uint32_t n,
                                   const uint64_t* __restrict__ keys, uint32_t n_keys, uint8_t* __restrict__ key_colors,
                                   unsigned long long* __restrict__ painted) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const uint32_t s = slot[j];
    if (s == kNoLeafSlot || (j + 1 < n && slot[j + 1] == s)) return;
    const uint32_t i = index[j];
    const uint8_t c = colors[i];
    reinterpret_cast<uint8_t*>(nodes + s)[0] = c;                           // LNode::color, lsvo_utils.hpp:14
    if (key_colors) {
        const uint64_t key = voxel_key(xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2], depth);
        key_colors[lower_bound_u64(keys, n_keys, key)] = c;                  // solid: the key is resident
    }
    atomicAdd(painted, 1ull);
}

__global__ void cell_colors_kernel(const uint2* __restrict__ nodes, int depth, const uint32_t* __restrict__ xyz, uint64_t n,
                                   int16_t* __restrict__ out) {
    const uint64_t i = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t s = lsvo_leaf_slot(nodes, depth, xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2]);
    out[i] = s == kNoLeafSlot ? int16_t(-1) : int16_t(__ldg(nodes + s).x & 0xffu);
}

__global__ void gather_key_colors_kernel(const uint64_t* __restrict__ old_keys, const uint8_t* __restrict__ old_colors, uint32_t n_old,
                                         const uint64_t* __restrict__ new_keys, uint32_t n_new, uint8_t* __restrict__ new_colors) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_new) return;
    const uint64_t key = new_keys[j];
    const uint32_t k = lower_bound_u64(old_keys, n_old, key);
    new_colors[j] = (k < n_old && old_keys[k] == key) ? old_colors[k] : uint8_t(1);    // added voxels: LNode() colour
}

__global__ void stamp_key_colors_kernel(uint2* __restrict__ nodes, int depth, const uint64_t* __restrict__ keys,
                                        const uint8_t* __restrict__ colors, uint32_t n_keys) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_keys) return;
    const uint64_t key = keys[j];
    uint32_t x = 0, y = 0, z = 0;
    for (int b = depth - 1; b >= 0; --b) {
        const uint32_t d = uint32_t(key >> (3 * b)) & 7u;
        x |= (d >> 2) << b; y |= ((d >> 1) & 1u) << b; z |= (d & 1u) << b;
    }
    const uint32_t s = lsvo_leaf_slot(nodes, depth, x, y, z);
    if (s != kNoLeafSlot) reinterpret_cast<uint8_t*>(nodes + s)[0] = colors[j];
}

}  // namespace

cudaError_t device_paint_cells(uint2* d_nodes, int depth, const uint32_t* d_xyz, const uint8_t* d_colors, uint64_t n,
                               const uint64_t* d_keys, uint32_t n_keys, uint8_t* d_key_colors, uint64_t* painted, cudaStream_t stream) {
    *painted = 0;
    if (n == 0) return cudaSuccess;
    if (n > 0x7fffffffull) return cudaErrorInvalidValue;
    const uint32_t m = uint32_t(n);
    Scratch sc(nullptr);
    uint32_t *slot = nullptr, *index = nullptr, *slot_sorted = nullptr, *index_sorted = nullptr;
    unsigned long long* d_count = nullptr;
    VRT_TRY(sc.alloc(&slot, m));
    VRT_TRY(sc.alloc(&index, m));
    VRT_TRY(sc.alloc(&slot_sorted, m));
    VRT_TRY(sc.alloc(&index_sorted, m));
    VRT_TRY(sc.alloc(&d_count, 1));
    size_t t = 0;
    VRT_TRY(cub::DeviceRadixSort::SortPairs(nullptr, t, slot, slot_sorted, index, index_sorted, m, 0, 32, stream));
    uint8_t* d_temp = nullptr;
    VRT_TRY(sc.alloc(&d_temp, t));
    VRT_TRY(cudaMemsetAsync(d_count, 0, sizeof(unsigned long long), stream));
    const unsigned blocks = (m + 255) / 256;
    paint_slots_kernel<<<blocks, 256, 0, stream>>>(d_nodes, depth, d_xyz, m, slot, index);
    VRT_TRY(cudaGetLastError());
    VRT_TRY(cub::DeviceRadixSort::SortPairs(d_temp, t, slot, slot_sorted, index, index_sorted, m, 0, 32, stream));   // LSD radix: stable
    paint_write_kernel<<<blocks, 256, 0, stream>>>(d_nodes, depth, d_xyz, d_colors, slot_sorted, index_sorted, m, d_keys, n_keys,
                                                   d_key_colors, d_count);
    VRT_TRY(cudaGetLastError());
    unsigned long long count = 0;
    VRT_TRY(cudaMemcpyAsync(&count, d_count, sizeof(count), cudaMemcpyDeviceToHost, stream));
    VRT_TRY(cudaStreamSynchronize(stream));
    *painted = count;
    return cudaSuccess;
}

cudaError_t launch_cell_colors(const uint2* d_nodes, int depth, const uint32_t* d_xyz, uint64_t n, int16_t* d_out, cudaStream_t stream) {
    if (n == 0) return cudaSuccess;
    cell_colors_kernel<<<unsigned((n + 255) / 256), 256, 0, stream>>>(d_nodes, depth, d_xyz, n, d_out);
    return cudaGetLastError();
}

cudaError_t launch_gather_key_colors(const uint64_t* d_old_keys, const uint8_t* d_old_colors, uint32_t n_old, const uint64_t* d_new_keys,
                                     uint32_t n_new, uint8_t* d_new_colors, cudaStream_t stream) {
    if (n_new == 0) return cudaSuccess;
    gather_key_colors_kernel<<<(n_new + 255) / 256, 256, 0, stream>>>(d_old_keys, d_old_colors, n_old, d_new_keys, n_new, d_new_colors);
    return cudaGetLastError();
}

cudaError_t launch_stamp_key_colors(uint2* d_nodes, int depth, const uint64_t* d_keys, const uint8_t* d_colors, uint32_t n_keys,
                                    cudaStream_t stream) {
    if (n_keys == 0) return cudaSuccess;
    stamp_key_colors_kernel<<<(n_keys + 255) / 256, 256, 0, stream>>>(d_nodes, depth, d_keys, d_colors, n_keys);
    return cudaGetLastError();
}

// xyz (device, n triples, coordinates < 2^depth) → sorted distinct voxel keys.  *d_keys is cudaMalloc'ed (caller frees).
cudaError_t device_voxel_keys(const uint32_t* d_xyz, uint64_t n, int depth, uint64_t** d_keys, uint32_t* n_keys, cudaStream_t stream,
                              BuildPool* pool) {
    *d_keys = nullptr;
    *n_keys = 0;
    if (n > 0xffffffffull) return cudaErrorInvalidValue;
    Scratch sc(pool);
    uint64_t *raw = nullptr, *sorted = nullptr, *uniq = nullptr;
    VRT_TRY(sc.alloc(&raw, n));
    VRT_TRY(sc.alloc(&sorted, n));
    VRT_TRY(cudaMalloc(&uniq, (n ? n : 1) * sizeof(uint64_t)));
    cudaError_t e = cudaSuccess;
    if (n) {
        voxel_keys_kernel<<<unsigned((n + 255) / 256), 256, 0, stream>>>(d_xyz, n, depth, raw);
        e = cudaGetLastError();
        if (e == cudaSuccess) e = sort_unique(raw, uint32_t(n), 3 * depth, sorted, uniq, n_keys, sc, stream);
    }
    if (e != cudaSuccess) { cudaFree(uniq); return e; }
    *d_keys = uniq;
    return cudaSuccess;
}

// Merges (add != 0) or removes the keys of `d_edit` (n_edit sorted distinct keys) into / from the scene's list.
// *d_out is cudaMalloc'ed (caller frees).
cudaError_t device_edit_voxel_keys(const uint64_t* d_keys, uint32_t n_keys, const uint64_t* d_edit, uint32_t n_edit, int add, int depth,
                                   uint64_t** d_out, uint32_t* n_out, cudaStream_t stream, BuildPool* pool) {
    *d_out = nullptr;
    *n_out = 0;
    Scratch sc(pool);
    const uint64_t total = uint64_t(n_keys) + (add ? n_edit : 0);
    if (total > 0xffffffffull) return cudaErrorInvalidValue;
    uint64_t* result = nullptr;
    VRT_TRY(cudaMalloc(&result, (total ? total : 1) * sizeof(uint64_t)));
    cudaError_t e = cudaSuccess;
    if (add) {
        uint64_t *both = nullptr, *sorted = nullptr;
        e = sc.alloc(&both, total);
        if (e == cudaSuccess) e = sc.alloc(&sorted, total);
        if (e == cudaSuccess && n_keys) e = cudaMemcpyAsync(both, d_keys, size_t(n_keys) * 8, cudaMemcpyDeviceToDevice, stream);
        if (e == cudaSuccess && n_edit) e = cudaMemcpyAsync(both + n_keys, d_edit, size_t(n_edit) * 8, cudaMemcpyDeviceToDevice, stream);
        if (e == cudaSuccess) e = sort_unique(both, uint32_t(total), 3 * depth, sorted, result, n_out, sc, stream);
    } else if (n_keys) {
        uint8_t* flags = nullptr;
        uint32_t* d_count = nullptr;
        e = sc.alloc(&flags, n_keys);
        if (e == cudaSuccess) e = sc.alloc(&d_count, 1);
        if (e == cudaSuccess) {
            keep_flags_kernel<<<(n_keys + 255) / 256, 256, 0, stream>>>(d_keys, n_keys, d_edit, n_edit, flags);
            e = cudaGetLastError();
        }
        size_t t = 0;
        uint8_t* d_temp = nullptr;
        if (e == cudaSuccess) e = cub::DeviceSelect::Flagged(nullptr, t, d_keys, flags, result, d_count, n_keys, stream);
        if (e == cudaSuccess) e = sc.alloc(&d_temp, t);
        if (e == cudaSuccess) e = cub::DeviceSelect::Flagged(d_temp, t, d_keys, flags, result, d_count, n_keys, stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(n_out, d_count, sizeof(uint32_t), cudaMemcpyDeviceToHost, stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
    }
    if (e != cudaSuccess) { cudaFree(result); return e; }
    *d_out = result;
    return cudaSuccess;
}

// Sorted distinct voxel keys → the reference's LNode array.  *d_slots is cudaMalloc'ed (caller frees).
cudaError_t device_build_lsvo_from_keys(int depth, const uint64_t* d_keys, uint32_t n_keys, uint2** d_slots, uint64_t* n_slots,
                                        cudaStream_t stream, BuildPool* pool, uint64_t* capacity_slots) {
    *d_slots = nullptr;
    *n_slots = 0;
    if (capacity_slots) *capacity_slots = 0;
    if (depth < 1 || depth + 1 > kMaxLevels) return cudaErrorInvalidValue;
    Scratch sc(pool);
    uint2* slots = nullptr;
    if (n_keys == 0) {                                                       // LSVO of an empty SVO: the root alone, child_offset 1
        VRT_TRY(cudaMalloc(&slots, sizeof(uint2)));
        const uint2 root = make_uint2(1u, 1u);
        cudaError_t e = cudaMemcpyAsync(slots, &root, sizeof(root), cudaMemcpyHostToDevice, stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
        if (e != cudaSuccess) { cudaFree(slots); return e; }
        *d_slots = slots;
        *n_slots = 1;
        return cudaSuccess;
    }
    // distinct prefixes per level, bottom up
    PrefixLevels P;
    P.depth = depth;
    P.p[depth] = d_keys;
    P.n[depth] = n_keys;
    uint32_t* d_count = nullptr;
    VRT_TRY(sc.alloc(&d_count, 1));
    uint64_t* shifted = nullptr;
    VRT_TRY(sc.alloc(&shifted, n_keys));
    size_t temp_bytes = 0;
    VRT_TRY(cub::DeviceSelect::Unique(nullptr, temp_bytes, shifted, shifted, d_count, n_keys, stream));
    uint8_t* d_temp = nullptr;
    VRT_TRY(sc.alloc(&d_temp, temp_bytes));
    uint64_t interior = 0;
    for (int l = depth - 1; l >= 0; --l) {
        const uint32_t n_below = P.n[l + 1];
        uint64_t* level = nullptr;
        VRT_TRY(sc.alloc(&level, n_below));
        shift3_kernel<<<(n_below + 255) / 256, 256, 0, stream>>>(P.p[l + 1], n_below, shifted);
        size_t t = temp_bytes;
        VRT_TRY(cub::DeviceSelect::Unique(d_temp, t, shifted, level, d_count, n_below, stream));
        uint32_t count = 0;
        VRT_TRY(cudaMemcpyAsync(&count, d_count, sizeof(count), cudaMemcpyDeviceToHost, stream));
        VRT_TRY(cudaStreamSynchronize(stream));
        P.p[l] = level;
        P.n[l] = count;
        interior += count;
    }
    const uint64_t n = 1 + 8 * interior;                                     // root slot + one 8-slot block per interior node
    if (n > 0xffffffffull) return cudaErrorInvalidValue;
    uint64_t capacity = n;
    if (pool && pool->spare && pool->spare_slots >= n) {                     // build into the array the previous edit replaced
        slots = pool->spare;
        capacity = pool->spare_slots;
        pool->spare = nullptr;
        pool->spare_slots = 0;
    } else {
        if (pool) capacity = n + n / 16 + 4096;
        VRT_TRY(cudaMalloc(&slots, capacity * sizeof(uint2)));
    }
    if (capacity_slots) *capacity_slots = capacity;
    fill_default_slots_kernel<<<148 * 8, 256, 0, stream>>>(slots, n);
    std::vector<uint32_t*> cpos(depth, nullptr);
    cudaError_t e = cudaSuccess;
    for (int l = 0; l < depth && e == cudaSuccess; ++l) {
        e = sc.alloc(&cpos[l], P.n[l]);
        if (e == cudaSuccess) rank_kernel<<<(P.n[l] + 127) / 128, 128, 0, stream>>>(P, l, cpos[l]);
    }
    for (int l = 0; l < depth && e == cudaSuccess; ++l)
        emit_nodes_kernel<<<(P.n[l] + 127) / 128, 128, 0, stream>>>(P, l, cpos[l], l > 0 ? cpos[l - 1] : nullptr, slots);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
    if (e != cudaSuccess) {
        if (pool) { if (pool->spare) cudaFree(pool->spare); pool->spare = slots; pool->spare_slots = capacity; }
        else cudaFree(slots);
        return e;
    }
    *d_slots = slots;
    *n_slots = n;
    return cudaSuccess;
}

}  // namespace vrt
