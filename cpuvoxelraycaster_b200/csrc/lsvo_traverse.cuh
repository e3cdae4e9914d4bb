// LSVO traversal on the device: node access and the hit epilogue of LSVO<D>::castRay
// (reference include/lsvo.hpp:148-169).  The loop itself is in lsvo_step.cuh.
// fp32 without contraction, op for op, so that the hit record is bit-identical to the CPU reference.
#pragma once
#include "vrt_device.cuh"

namespace vrt {

// One octree node as the traversal sees it, whatever the memory format.
struct NodeView {
    uint32_t raw;          // first word of the slot: color | child_mask << 8 | leaf_mask << 16 (lsvo_utils.hpp:14-17)
    uint32_t child_base;   // index such that child slot s lives at child_base + s
};

// Reference layout (lsvo_utils.hpp:5-18): 8-byte slots, children at parent + child_offset + slot.
struct RefNodes {
    const uint2* __restrict__ slots;
    __device__ __forceinline__ NodeView fetch(uint32_t id) const {
        const uint2 w = __ldg(slots + id);                 // one 8-byte load per loop trip (lsvo.hpp:74)
        NodeView v;
        v.raw = w.x;
        v.child_base = id + w.y;
        return v;
    }
    __device__ __forceinline__ uint32_t child(const NodeView& v, uint32_t slot) const { return v.child_base + slot; }
    // the same in two halves, for a walk that keeps the node's two words across trips (Trav2): nothing is computed from the
    // loaded words until a descent needs the child's index, so no instruction waits for the load at the end of a trip
    __device__ __forceinline__ uint2 load(uint32_t id) const { return __ldg(slots + id); }
    __device__ __forceinline__ uint32_t child_of(uint32_t id, const uint2& w, uint32_t slot) const { return id + w.y + slot; }
};

// Compact layout (built on the device by scene_device.cu): only nodes that own a child block are stored, level by
// level (breadth first), 8 bytes each: the reference's mask word and the index of the first INTERIOR child; interior
// children of a node are contiguous in slot order, so child s sits at first + popc(interior mask below s).
// 8x smaller than the reference layout (which reserves 8 slots per node, 87.5 % of them dead), top levels first.
struct CompactNodes {
    const uint2* __restrict__ slots;
    __device__ __forceinline__ NodeView fetch(uint32_t id) const {
        const uint2 w = __ldg(slots + id);
        NodeView v;
        v.raw = w.x;
        v.child_base = w.y;
        return v;
    }
    __device__ __forceinline__ uint32_t child(const NodeView& v, uint32_t slot) const {
        const uint32_t interior = (v.raw >> 8) & ~(v.raw >> 16) & 0xffu;       // child_mask & ~leaf_mask
        return v.child_base + __popc(interior & ((1u << slot) - 1u));
    }
    __device__ __forceinline__ uint2 load(uint32_t id) const { return __ldg(slots + id); }
    __device__ __forceinline__ uint32_t child_of(uint32_t, const uint2& w, uint32_t slot) const {
        const uint32_t interior = (w.x >> 8) & ~(w.x >> 16) & 0xffu;
        return w.y + __popc(interior & ((1u << slot) - 1u));
    }
};

// Leaf slot of voxel (x, y, z) in SVO::setCell coordinates (svo.hpp:72) in the reference layout: the root-to-leaf descent of
// LSVO::getAtRayHit (lsvo.hpp:174-285), which returns node N and child slot s of the leaf; the leaf's own slot is
// N + child_offset + s.  A voxel that castRay reports at v lies at S-1-v in these coordinates (SURVEY.md §0 item 2), so
// the child slot is built from the coordinate bits directly.  kNoLeafSlot when a child bit on the way is missing (empty).
// Only interior slots are loaded.
constexpr uint32_t kNoLeafSlot = 0xffffffffu;
__device__ __forceinline__ uint32_t lsvo_leaf_slot(const uint2* __restrict__ nodes, int depth, uint32_t x, uint32_t y, uint32_t z) {
    uint32_t node = 0u;
    for (int b = depth - 1; b >= 0; --b) {
        const uint32_t slot = ((x >> b) & 1u) | (((y >> b) & 1u) << 1) | (((z >> b) & 1u) << 2);
        const uint2 w = __ldg(nodes + node);
        if (!((w.x >> (8 + slot)) & 1u)) return kNoLeafSlot;
        node += w.y + slot;
        if ((w.x >> (16 + slot)) & 1u) return node;
    }
    return kNoLeafSlot;
}

// Traversal state at termination (what the epilogue needs).
struct LsvoResult {
    float px, py, pz;      // cell low corner in the mirrored frame (un-mirrored by lsvo_finish)
    float t_min;
    float scale_f;
    int scale;
    uint32_t face;         // step mask that entered the cell (`normal` in lsvo.hpp:69,122)
    uint32_t mirror;
    uint32_t complexity;
    bool hit;
    float dx, dy, dz;      // direction after the |d| >= 2^-23 clamp (lsvo.hpp:44-46)
};

// Hit epilogue, lsvo.hpp:148-169.  Only valid when r.hit.
struct LsvoHit {
    float pos[3];
    float normal[3];
    float uv[2];
    float distance;
    float corner[3];   // un-mirrored low corner of the hit cell
};

__device__ __forceinline__ float glm_sign(float x) { return float(0.0f < x) - float(x < 0.0f); }

__device__ __forceinline__ void lsvo_finish(const LsvoResult& r, float ox, float oy, float oz, int depth, LsvoHit& h) {
    h.normal[0] = (-glm_sign(r.dx)) * float(r.face & 1u);                // :149
    h.normal[1] = (-glm_sign(r.dy)) * float(r.face & 2u);
    h.normal[2] = (-glm_sign(r.dz)) * float(r.face & 4u);
    float px = r.px, py = r.py, pz = r.pz;
    if ((r.mirror & 1u) == 0u) px = 3.0f - r.scale_f - px;               // :151-153
    if ((r.mirror & 2u) == 0u) py = 3.0f - r.scale_f - py;
    if ((r.mirror & 4u) == 0u) pz = 3.0f - r.scale_f - pz;
    h.corner[0] = px; h.corner[1] = py; h.corner[2] = pz;
    h.distance = r.t_min;                                                // :155
    h.pos[0] = fminf(fmaxf(ox + r.t_min * r.dx, px + kEps), px + r.scale_f - kEps);   // :156-158
    h.pos[1] = fminf(fmaxf(oy + r.t_min * r.dy, py + kEps), py + r.scale_f - kEps);
    h.pos[2] = fminf(fmaxf(oz + r.t_min * r.dz, pz + kEps), pz + r.scale_f - kEps);
    const float S = float(1 << depth);                                   // :39
    if (h.normal[0] != 0.0f) { h.uv[0] = fracf(h.pos[2] * S); h.uv[1] = fracf(h.pos[1] * S); }        // :160-168
    else if (h.normal[1] != 0.0f) { h.uv[0] = fracf(h.pos[0] * S); h.uv[1] = fracf(h.pos[2] * S); }
    else if (h.normal[2] != 0.0f) { h.uv[0] = fracf(h.pos[0] * S); h.uv[1] = fracf(h.pos[1] * S); }
    else { h.uv[0] = 0.0f; h.uv[1] = 0.0f; }   // uninitialised in the reference (start inside a solid cell)
}

}  // namespace vrt
