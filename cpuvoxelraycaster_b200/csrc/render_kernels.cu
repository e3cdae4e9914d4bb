// Frame rendering: ray generation (K0), traversal, shading and accumulation fused into one kernel per frame; resolve.
//
// Replaces the swarm lambda src/main.cpp:139-154, Camera::getRay (camera_controller.hpp:34-54),
// RayCaster::renderRay/castRay/getGlobalIllumination and the texture lookup (raycaster.hpp:67-240),
// samples_to_image (raycaster.hpp:94-103).  The per-sample arithmetic is in render_chain.cuh: a sample is a chain of up
// to six rays, a small state machine around ONE inlined copy of the traversal loop, so lanes at different chain stages
// still execute the traversal converged.  Three ways of giving samples to lanes, all with bit-identical results
// (integer sums), measured against each other in profiles/r01_summary.md:
//   K4  render_accumulate_kernel   a lane walks samples of one pixel (8x4 pixel tile per warp, Q lanes per pixel);
//                                  the interactive loop (1 sample, checkerboard, device-side autofocus)
//   K5  render_sorted_kernel       the samples of a 32x4-pixel block are counting-sorted by GI direction in shared
//                                  memory and traced 32 neighbours at a time
//   K6  sort_samples_kernel + render_rounds_kernel   the same lists in global memory, traced by persistent CTAs that
//                                  help each other finish; the default for frames with >= 8 samples per pixel
#include "lsvo_step.cuh"
#include "render_chain.cuh"

namespace vrt {

// Can the loop guard `scale > guard` (lsvo.hpp:72) ever stop a walk?  Not when the voxels' own scale passes it (Trav2, kGuard).
static bool guard_binds(const RenderLaunch& L) { return L.guard >= kSvoMaxDepth - L.depth; }

// 8 CTAs per SM (64 registers).  Round 1 ran K4 at 4 (128 registers: more warps at fewer registers spilled into the loop and
// measured slower); with the Trav2 loop and its invariants held in registers (lsvo_step.cuh) the loops compile spill-free at 64
// registers (~200 bytes of spills in the chain code) and the extra warps pay: 4 / 6 / 8 CTAs per SM = 0.201 / 0.180 / 0.172 ms on
// the 720p 1-sample frame, 4.19 / 3.72 / 3.62 ms on a 1080p 4-sample GI frame, 1.38 / 1.20 / 1.15 ms on the 4K interactive frame
// (profiles/r02_ab_k4.txt).
#ifndef VRT_K4_MIN_CTAS
#define VRT_K4_MIN_CTAS 8
#endif
// kLive: the interactive-loop extras (checkerboard pixel mapping, focal length read from the autofocus kernel's output).
// Compiled out of the plain instantiation so that they cost the many-sample frames nothing (register allocation of the
// traversal loop is sensitive to every extra live value: 73.9 vs 75.6 ms on cfg 4).
// kGuard = false: the loop guard cannot bind for this scene and is compiled out (lsvo_step.cuh, Trav2).
template <typename Nodes, bool kLive, bool kMirror = false, bool kGuard = true>
__global__ void __launch_bounds__(128, VRT_K4_MIN_CTAS) render_accumulate_kernel(Nodes nodes, RenderLaunch L, uint32_t* __restrict__ accum,
                                                                unsigned long long* __restrict__ counters) {
    extern __shared__ uint2 smem[];
    nodes.slots = pin(nodes.slots);
    const int guard = keep_in_register(L.guard, smem + threadIdx.x);
    Stack64s<128> stack = Stack64s<128>::make(smem + threadIdx.x, kSvoMaxDepth - L.depth);
    const float guard_sf = keep_in_register(guard_scale_f(L.guard), smem + threadIdx.x);

    // 8x4 pixel tile per warp, 4 tiles side by side per block: coherent primary rays share nodes
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // checkerboard frames (main.cpp:137,143) render every other pixel of a row: the tile's columns are then the
    // indices of the rendered pixels, so that no lane idles
    const int checker = kLive ? L.checker : 0;
    const int columns = checker ? (L.width + 1) / 2 : L.width;
    const int tiles_x = (columns + 31) / 32;
    // blockIdx.x = chunk * tiles + tile: the pixel's samples are cut into L.spp_chunks runs handled by different CTAs
    // (more, shorter CTAs: keeps the tail short when a GPU owns only a slice of the frame; sums stay exact — integers)
    const int tiles_y = int(gridDim.x) / (tiles_x * L.spp_chunks);
    const int chunk = int(blockIdx.x) / (tiles_x * tiles_y), tile = int(blockIdx.x) - chunk * tiles_x * tiles_y;
    const int bx = tile % tiles_x, by = tile / tiles_x;
    const int s_begin = (chunk * L.spp) / L.spp_chunks, s_end = ((chunk + 1) * L.spp) / L.spp_chunks;
    // Lane → (pixel, sample) mapping inside the warp's 8x4 pixel tile.  Q = L.samples_per_warp lanes share a pixel and
    // take consecutive samples; the tile's 32 pixels are walked in Q groups of P = 32/Q pixels.  Q = 1 is the plain
    // one-lane-per-pixel mapping.  With many samples per pixel, lanes of one pixel cast nearly identical primary and
    // shadow rays (they differ by the lens jitter only), which keeps the warp converged far better than 32 neighbouring
    // pixels do.  Sums are integers, so the mapping cannot change the frame.
    const int Q = L.samples_per_warp, P = 32 / Q;
    const int sub = lane & (Q - 1);                        // which of the pixel's Q concurrent samples
    const int runs = (s_end - s_begin) / Q;                // launcher guarantees divisibility

    // ray statistics per class: private shared-memory pairs behind the stack (12 registers less across the traversal loop)
#pragma unroll
    for (int k = 0; k < 6; ++k) stack.stat_zero(k);
    const float SCALE = 1.0f / float(1 << L.depth);                           // raycaster.hpp:123-124 / main.cpp:82
    const float n_norm = SCALE * 0.0078125f * 2.0f;                           // raycaster.hpp:171-172
    const float aspect = float(L.width) / float(L.height);                    // main.cpp:133
    const float focal_length = (kLive && L.focal) ? __ldg(L.focal) : L.cam.focal_length;   // main.cpp:114-121 on the device

    for (int g = 0; g < Q; ++g) {
        const int j = g * P + lane / Q;                    // pixel index inside the 8x4 tile
        // 4-row tiles are dealt round-robin to tile_step owners (multi-GPU row partition, balanced sky/terrain)
        const int y = L.row_begin + (by * L.tile_step + L.tile_index) * 4 + (j >> 3);
        int x = bx * 32 + warp * 8 + (j & 7);
        if (checker) x = 2 * x + checker_x_parity(checker, L.checker_area_height, y);
        const bool active = x < L.width && y < L.row_end;
        const uint32_t pixel = uint32_t(y) * uint32_t(L.width) + uint32_t(x);
        uint32_t sum_r = 0, sum_g = 0, sum_b = 0;
        if (active) {
            const float lens_x = float(x) / float(L.height) - aspect * 0.5f;  // main.cpp:145
            const float lens_y = float(y) / float(L.height) - 0.5f;           // main.cpp:146
            for (int k = 0; k < runs; ++k) {
                const uint32_t sample = uint32_t(L.sample_offset + s_begin + k * Q + sub);
                ChainState c;
                NextRay nr;
                chain_begin(L, c, pixel, sample, lens_x, lens_y, SCALE, focal_length, nr);
                nr.t_floor = beam_floor_of(L, x, y, nr.dx, nr.dy, nr.dz);
                int stage = kPrimary;
                while (stage != kDone) {
                    LsvoResult r;
                    if (stage < kGi0) lsvo_cast_ray2<false, true, kGuard, true>(nodes, stack, guard, guard_sf, nr.ox, nr.oy, nr.oz, nr.dx, nr.dy, nr.dz, 0.0f, 0.0f, r, nr.t_floor, &L.bounds);
                    else lsvo_cast_ray2<true, false, kGuard, true>(nodes, stack, guard, guard_sf, nr.ox, nr.oy, nr.oz, nr.dx, nr.dy, nr.dz, nr.coef, 0.0f, r);
                    stack.stat_add(stage, 1u, r.complexity);
                    LsvoHit h;
                    if (r.hit) lsvo_finish(r, nr.ox, nr.oy, nr.oz, L.depth, h);
                    stage = chain_advance<kMirror>(L, c, stage, r, h, pixel, sample, SCALE, n_norm, nr, nodes.slots);
                }
                chain_colour<kMirror>(L, c, sum_r, sum_g, sum_b);
            }
        }
        // the Q lanes of a pixel add up their sums; lane sub == 0 commits them
        for (int o = Q >> 1; o > 0; o >>= 1) {
            sum_r += __shfl_xor_sync(0xffffffffu, sum_r, o);
            sum_g += __shfl_xor_sync(0xffffffffu, sum_g, o);
            sum_b += __shfl_xor_sync(0xffffffffu, sum_b, o);
        }
        if (active && sub == 0) {
            uint4* a = reinterpret_cast<uint4*>(accum) + pixel;               // Sample, raycaster.hpp:18-24,87-90
            if (L.spp_chunks == 1) {
                uint4 v = *a;
                v.x += sum_r; v.y += sum_g; v.z += sum_b; v.w += uint32_t(L.spp);
                *a = v;
            } else {
                uint32_t* w = reinterpret_cast<uint32_t*>(a);
                atomicAdd(w, sum_r); atomicAdd(w + 1, sum_g); atomicAdd(w + 2, sum_b); atomicAdd(w + 3, uint32_t(s_end - s_begin));
            }
        }
    }

    // statistics: rays and Σ complexity per ray class (warp reduce, one atomic per warp and class)
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        uint32_t a, b;
        stack.stat_get(k, a, b);
        for (int o = 16; o > 0; o >>= 1) {
            a += __shfl_xor_sync(0xffffffffu, a, o);
            b += __shfl_xor_sync(0xffffffffu, b, o);
        }
        if (lane == 0 && a) {
            atomicAdd(counters + k, (unsigned long long)a);
            atomicAdd(counters + 6 + k, (unsigned long long)b);
        }
    }
}

// ---- K5: the same frame with the samples of a CTA's pixel block regrouped by GI direction -----------------------------
//
// In K4 the four GI ray classes take 69 % of the many-sample frame at 10.8 of 32 lanes (profiles/r01_summary.md): the GI
// rays of a warp leave in unrelated directions (raycaster.hpp:178-192 draws them from a 100x100 lattice), so after the
// common initial descent every loop trip executes all three branch paths and the warp waits for its longest ray.
// Which lane runs which (pixel, sample) is free — the sums are integers — and the sample's random numbers are a pure
// function of (pixel, sample) (Philox), so they can be evaluated BEFORE tracing anything: the CTA computes, for every
// sample of its 32x4-pixel block, the angles of the first- and second-bounce GI noise, counting-sorts the samples by
// (angle 1 bin, angle 2 bin) in shared memory and hands them out to its warps 32 at a time.  A warp then traces GI rays
// that are nearly parallel and start within a few voxels of each other — as coherent as primary rays.
// tools/probe_gi_sorting.py measured the effect on the traversal alone: 192 -> 300 G loop trips/s on first-bounce rays,
// 219 -> 299 on their shadow rays.  Results cannot change: same samples, same numbers, integer sums.

// pseudo-angle of the tangent-plane noise (c1, c2) = 20 * (i - 50, j - 50): 0 <= a < 4 around the circle ("diamond angle")
__device__ __forceinline__ float noise_angle(uint32_t w1, uint32_t w2) {
    const float x = float(int(w1 % 100u) - 50), y = float(int(w2 % 100u) - 50);
    const float s = fabsf(x) + fabsf(y);
    if (s == 0.0f) return 0.0f;
    const float t = __fdividef(y, s);                                          // -1..1; a sort key only: no need for the IEEE quotient
    return x >= 0.0f ? (y >= 0.0f ? t : 4.0f + t) : 2.0f - t;
}

// 5 CTAs per SM: K5 needs 95 registers without spilling (K4 does not fit: 12 B of spills and slower).  Measured on cfg 4:
// 67.8 ms at 4 CTAs, 63.9 ms at 5, 74.4 ms at 6 (80 registers, spills).
#ifndef VRT_K5_MIN_CTAS
#define VRT_K5_MIN_CTAS 5
#endif
struct SortPlan {
    int bins1, bins2;      // angle bins of bounce 1 and 2 (bins1 * bins2 <= 256)
};

template <typename Nodes>
__global__ void __launch_bounds__(128, VRT_K5_MIN_CTAS) render_sorted_kernel(Nodes nodes, RenderLaunch L, SortPlan plan,
                                                                            uint32_t* __restrict__ accum,
                                                                            unsigned long long* __restrict__ counters) {
    extern __shared__ uint2 smem[];
    Stack64<128> stack{smem + threadIdx.x};
    nodes.slots = pin(nodes.slots);
    const int guard = pin(L.guard);
    const int depth_offset = pin(kSvoMaxDepth - L.depth);
    const int lane = threadIdx.x & 31;

    // blockIdx.x = chunk * tiles + tile, a tile = 32x4 pixels, a chunk = one run of the pixels' samples (as in K4)
    const int tiles_x = (L.width + 31) / 32;
    const int tiles_y = int(gridDim.x) / (tiles_x * L.spp_chunks);
    const int chunk = int(blockIdx.x) / (tiles_x * tiles_y), tile = int(blockIdx.x) - chunk * tiles_x * tiles_y;
    const int bx = tile % tiles_x, by = tile / tiles_x;
    const int s_begin = (chunk * L.spp) / L.spp_chunks, s_end = ((chunk + 1) * L.spp) / L.spp_chunks;
    const int n_s = s_end - s_begin;
    const int n_chains = 128 * n_s;                                            // launcher: <= 8192
    const int x0 = bx * 32, y0 = L.row_begin + (by * L.tile_step + L.tile_index) * 4;
    // sample c of the block: pixel c / n_s (walked 8x4 sub-tile by sub-tile), sample c % n_s.  The scatter below runs in
    // ascending c and is nearly stable, so inside one direction bin consecutive list entries are samples of the same or of
    // neighbouring pixels: their primary and sun-shadow rays stay coherent too.
    auto pixel_of = [&](int j, int& x, int& y) { x = x0 + (j >> 5) * 8 + (j & 7); y = y0 + ((j >> 3) & 3); };

    // shared memory: stacks | statistics | sorted sample list | histogram / cursors | pixel sums | work counter
    uint32_t* cnt = reinterpret_cast<uint32_t*>(smem + (L.depth + 1) * 128) + threadIdx.x;
    uint32_t* base = reinterpret_cast<uint32_t*>(smem + (L.depth + 1) * 128) + 12 * 128;
    uint32_t* hist = base;                                                     // 257 words
    uint32_t* sums = base + 260;                                               // 128 pixels x (r, g, b, count)
    uint32_t* next_round = base + 260 + 512;
    uint16_t* ids = reinterpret_cast<uint16_t*>(base + 260 + 512 + 4);        // n_chains entries
#pragma unroll
    for (int k = 0; k < 12; ++k) cnt[k * 128] = 0u;
    for (int i = threadIdx.x; i < 257; i += 128) hist[i] = 0u;
    for (int i = threadIdx.x; i < 512; i += 128) sums[i] = 0u;
    if (threadIdx.x == 0) *next_round = 0u;
    __syncthreads();

    // ---- sort the block's samples by GI direction: histogram, scan, scatter (keys are recomputed, not stored) ----
    const int n_keys = plan.bins1 * plan.bins2;
    auto sample_key = [&](int c, bool& active) -> int {
        const int j = c / n_s, s = s_begin + (c - j * n_s);
        int x, y;
        pixel_of(j, x, y);
        active = x < L.width && y < L.row_end;
        const uint32_t pixel = uint32_t(y) * uint32_t(L.width) + uint32_t(x), sample = uint32_t(L.sample_offset + s);
        const uint4 r0 = philox4x32_10(pixel, sample, 0u, 0u, L.seed_lo, L.seed_hi);
        int key = min(plan.bins1 - 1, int(noise_angle(r0.z, r0.w) * (float(plan.bins1) * 0.25f)));
        if (plan.bins2 > 1) {
            const uint4 r1 = philox4x32_10(pixel, sample, 1u, 0u, L.seed_lo, L.seed_hi);
            key = key * plan.bins2 + min(plan.bins2 - 1, int(noise_angle(r1.x, r1.y) * (float(plan.bins2) * 0.25f)));
        }
        return key;
    };
    for (int c = threadIdx.x; c < n_chains; c += 128) {
        bool active;
        const int key = sample_key(c, active);
        if (active) atomicAdd(hist + key, 1u);
    }
    __syncthreads();
    if (threadIdx.x < 32) {                                                    // exclusive scan of <= 256 counters by one warp
        uint32_t v[8], run = 0u;
#pragma unroll
        for (int k = 0; k < 8; ++k) { const int i = lane * 8 + k; v[k] = i < n_keys ? hist[i] : 0u; run += v[k]; }
        uint32_t incl = run;
        for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
        uint32_t excl = incl - run;
#pragma unroll
        for (int k = 0; k < 8; ++k) { const int i = lane * 8 + k; if (i < n_keys) hist[i] = excl; excl += v[k]; }
        if (lane == 31) hist[256] = incl;                                      // number of active samples
    }
    __syncthreads();
    for (int c = threadIdx.x; c < n_chains; c += 128) {
        bool active;
        const int key = sample_key(c, active);
        if (active) ids[atomicAdd(hist + key, 1u)] = uint16_t(c);
    }
    __syncthreads();
    const uint32_t total = hist[256];

    // ---- trace: warps fetch rounds of 32 consecutive sorted samples ----
    const float SCALE = 1.0f / float(1 << L.depth);                           // raycaster.hpp:123-124 / main.cpp:82
    const float n_norm = SCALE * 0.0078125f * 2.0f;                           // raycaster.hpp:171-172
    const float aspect = float(L.width) / float(L.height);                    // main.cpp:133
    const float focal_length = L.focal ? __ldg(L.focal) : L.cam.focal_length;
    for (;;) {
        uint32_t round = 0u;
        if (lane == 0) round = atomicAdd(next_round, 1u);
        round = __shfl_sync(0xffffffffu, round, 0);
        if (round * 32u >= total) break;
        const uint32_t slot = round * 32u + uint32_t(lane);
        if (slot < total) {
            const int c = ids[slot];
            const int j = c / n_s, s = s_begin + (c - j * n_s);
            int x, y;
            pixel_of(j, x, y);
            const uint32_t pixel = uint32_t(y) * uint32_t(L.width) + uint32_t(x), sample = uint32_t(L.sample_offset + s);
            const float lens_x = float(x) / float(L.height) - aspect * 0.5f;  // main.cpp:145
            const float lens_y = float(y) / float(L.height) - 0.5f;           // main.cpp:146
            ChainState cs;
            NextRay nr;
            chain_begin(L, cs, pixel, sample, lens_x, lens_y, SCALE, focal_length, nr);
            int stage = kPrimary;
            while (stage != kDone) {
                LsvoResult r;
                lsvo_cast_ray(nodes, stack, depth_offset, guard, nr.ox, nr.oy, nr.oz, nr.dx, nr.dy, nr.dz, nr.coef, 0.0f, r);
                cnt[stage * 128] += 1u;
                cnt[(6 + stage) * 128] += r.complexity;
                LsvoHit h;
                if (r.hit) lsvo_finish(r, nr.ox, nr.oy, nr.oz, L.depth, h);
                stage = chain_advance(L, cs, stage, r, h, pixel, sample, SCALE, n_norm, nr);
            }
            uint32_t cr = 0, cg = 0, cb = 0;
            chain_colour(L, cs, cr, cg, cb);
            if (cr) atomicAdd(sums + 4 * j, cr);
            if (cg) atomicAdd(sums + 4 * j + 1, cg);
            if (cb) atomicAdd(sums + 4 * j + 2, cb);
        }
        __syncwarp();
    }
    __syncthreads();

    // ---- commit the block's pixel sums (every active pixel received s_end - s_begin samples) ----
    {
        const int j = threadIdx.x;
        int x, y;
        pixel_of(j, x, y);
        if (x < L.width && y < L.row_end) {
            uint32_t* w = accum + 4 * (size_t(y) * size_t(L.width) + size_t(x));   // Sample, raycaster.hpp:18-24,87-90
            if (L.spp_chunks == 1) {
                uint4 v = *reinterpret_cast<uint4*>(w);
                v.x += sums[4 * j]; v.y += sums[4 * j + 1]; v.z += sums[4 * j + 2]; v.w += uint32_t(L.spp);
                *reinterpret_cast<uint4*>(w) = v;
            } else {
                atomicAdd(w, sums[4 * j]); atomicAdd(w + 1, sums[4 * j + 1]); atomicAdd(w + 2, sums[4 * j + 2]);
                atomicAdd(w + 3, uint32_t(s_end - s_begin));
            }
        }
    }
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        uint32_t a = cnt[k * 128], b = cnt[(6 + k) * 128];
        for (int o = 16; o > 0; o >>= 1) {
            a += __shfl_xor_sync(0xffffffffu, a, o);
            b += __shfl_xor_sync(0xffffffffu, b, o);
        }
        if (lane == 0 && a) {
            atomicAdd(counters + k, (unsigned long long)a);
            atomicAdd(counters + 6 + k, (unsigned long long)b);
        }
    }
}

// ---- K6: K5's sorted lists in global memory + persistent CTAs that help each other finish ------------------------------
//
// K5's unit of scheduling is a CTA-sized block of samples (2.9 ms of work on the headline frame): the launch ends with SMs
// idling while the last blocks finish, and on an 8-GPU slice the blocks must be cut into short runs (less to sort) to keep
// that tail small.  K6 splits the two jobs: `sort_samples_kernel` writes every block's direction-sorted sample list to
// global memory (16 KB per block), `render_rounds_kernel` runs one persistent CTA set that takes blocks from a global
// counter — the CTA's warps pull rounds of 32 list entries from the block's own counter, so a block still has the L1 of one
// SM to itself — and, once no blocks are left, every warp looks for blocks that still have rounds and helps with them.
// A round commits its colours itself, with RED operations on the pixels' accumulators in global memory, so several CTAs can
// work on one block.  Same samples, same numbers, integer sums: the frame cannot change.

struct BlockGeometry {
    int tiles_x, tiles_y;      // 32x4-pixel blocks owned by this launch
    int runs;                  // sample runs per block (1 unless spp > 64)
    int cap;                   // list capacity per (block, run): 128 * longest run
};

__device__ __forceinline__ void block_origin(const RenderLaunch& L, const BlockGeometry& G, int work, int& x0, int& y0, int& s_begin, int& n_s) {
    const int tiles = G.tiles_x * G.tiles_y;
    const int run = work / tiles, tile = work - run * tiles;
    const int bx = tile % G.tiles_x, by = tile / G.tiles_x;
    x0 = bx * 32;
    y0 = L.row_begin + (by * L.tile_step + L.tile_index) * 4;
    s_begin = (run * L.spp) / G.runs;
    n_s = ((run + 1) * L.spp) / G.runs - s_begin;
}
// list entry c = pixel j of the block, sample s of the run: c = j * n_s + s.  Runs are powers of two except for odd sample
// counts: a shift instead of the ~25-instruction integer division (log2 < 0: divide).
__device__ __forceinline__ int run_log2(int n_s) { return (n_s & (n_s - 1)) == 0 ? 31 - __clz(n_s) : -1; }
__device__ __forceinline__ int entry_pixel(int c, int n_s, int log2) { return log2 >= 0 ? c >> log2 : c / n_s; }
__device__ __forceinline__ void block_pixel(int x0, int y0, int j, int& x, int& y) {     // 8x4 sub-tile by sub-tile
    x = x0 + (j >> 5) * 8 + (j & 7);
    y = y0 + ((j >> 3) & 3);
}

// Samples whose pixel lies in a beam tile with NOTHING in its frustum (floor 3.0, beam_kernels.cu: no non-empty node meets
// the tile's lens-widened frustum, so every camera ray of the tile misses) never enter a list: the sort counts them — one add to
// the pixel's sample count per run, one to the primary-ray statistics (complexity 0) and one to `culled` per block — and K6 only
// traces what can hit something.  Their colour is the reference's black (raycaster.hpp:38), i.e. nothing to add to the sums.
__global__ void __launch_bounds__(128) sort_samples_kernel(RenderLaunch L, SortPlan plan, BlockGeometry G, uint16_t* __restrict__ lists,
                                                           uint32_t* __restrict__ meta, uint32_t* __restrict__ accum,
                                                           unsigned long long* __restrict__ counters, unsigned long long* __restrict__ culled) {
    __shared__ uint32_t hist[260];
    __shared__ uint8_t keys[8192];                                             // one key per sample of the block (255 = not in the list)
    __shared__ uint32_t s_culled;
    const int lane = threadIdx.x & 31, work = blockIdx.x;
    int x0, y0, s_begin, n_s;
    block_origin(L, G, work, x0, y0, s_begin, n_s);
    const int n_chains = 128 * n_s, n_keys = plan.bins1 * plan.bins2, n_s_log2 = run_log2(n_s);
    uint16_t* ids = lists + size_t(work) * G.cap;
    for (int i = threadIdx.x; i < 257; i += 128) hist[i] = 0u;
    if (threadIdx.x == 0) s_culled = 0u;
    __syncthreads();
    // pass 1: keys and histogram.  Lanes of a warp holding the same key add up first (one shared-memory atomic per key
    // and warp instead of one per sample: with 16 sectors the plain version serialises 8 deep)
    const int n_padded = (n_chains + 31) & ~31;
    for (int c = threadIdx.x; c < n_padded; c += 128) {
        uint32_t key = 255u;
        if (c < n_chains) {
            const int j = entry_pixel(c, n_s, n_s_log2), s = s_begin + (c - j * n_s);
            int x, y;
            block_pixel(x0, y0, j, x, y);
            bool in_list = x < L.width && y < L.row_end;
#ifndef VRT_NO_CULL                                                            // (A/B builds: make EXTRA=-DVRT_NO_CULL)
            if (in_list && L.beam_floor && __ldg(L.beam_floor + (y >> L.beam_shift) * L.beam_tiles_x + (x >> L.beam_shift)) == 3.0f) {
                in_list = false;                                               // answered by the beam search: a miss
                if (c == j * n_s) {                                            // once per pixel and run
                    atomicAdd(accum + 4 * (size_t(y) * size_t(L.width) + size_t(x)) + 3, uint32_t(n_s));
                    atomicAdd(&s_culled, uint32_t(n_s));
                }
            }
#endif
            if (in_list) {
                key = 0u;
                if (n_keys > 1) {
                    const uint32_t pixel = uint32_t(y) * uint32_t(L.width) + uint32_t(x), sample = uint32_t(L.sample_offset + s);
                    const uint4 r0 = philox4x32_10(pixel, sample, 0u, 0u, L.seed_lo, L.seed_hi);
                    key = uint32_t(min(plan.bins1 - 1, int(noise_angle(r0.z, r0.w) * (float(plan.bins1) * 0.25f))));
                    if (plan.bins2 > 1) {
                        const uint4 r1 = philox4x32_10(pixel, sample, 1u, 0u, L.seed_lo, L.seed_hi);
                        key = key * uint32_t(plan.bins2) + uint32_t(min(plan.bins2 - 1, int(noise_angle(r1.x, r1.y) * (float(plan.bins2) * 0.25f))));
                    }
                    key = min(key, 254u);
                }
            }
            keys[c] = uint8_t(key);
        }
        const unsigned peers = __match_any_sync(0xffffffffu, key);
        if (key != 255u && lane == __ffs(peers) - 1) atomicAdd(hist + key, uint32_t(__popc(peers)));
    }
    __syncthreads();
    if (threadIdx.x < 32) {                                                    // exclusive scan of <= 256 counters by one warp
        uint32_t v[8], run = 0u;
#pragma unroll
        for (int k = 0; k < 8; ++k) { const int i = lane * 8 + k; v[k] = i < n_keys ? hist[i] : 0u; run += v[k]; }
        uint32_t incl = run;
        for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
        uint32_t excl = incl - run;
#pragma unroll
        for (int k = 0; k < 8; ++k) { const int i = lane * 8 + k; if (i < n_keys) hist[i] = excl; excl += v[k]; }
        if (lane == 31) { meta[2 * work] = incl; meta[2 * work + 1] = 0u; }  // samples in the list, next round to hand out
    }
    __syncthreads();
    // pass 2: scatter, again one atomic per key and warp; inside a warp the samples keep their order (ascending c =
    // pixel by pixel), so a sector's list stays nearly pixel-ordered
    for (int c = threadIdx.x; c < n_padded; c += 128) {
        const uint32_t key = c < n_chains ? keys[c] : 255u;
        const unsigned peers = __match_any_sync(0xffffffffu, key);
        uint32_t first = 0u;
        const int leader = __ffs(peers) - 1;
        if (key != 255u && lane == leader) first = atomicAdd(hist + key, uint32_t(__popc(peers)));
        first = __shfl_sync(0xffffffffu, first, leader);
        if (key != 255u) ids[first + uint32_t(__popc(peers & ((1u << lane) - 1u)))] = uint16_t(c);
    }
    if (threadIdx.x == 0 && s_culled) {                                        // (the barriers above order the block's adds before this read)
        atomicAdd(counters + kPrimary, (unsigned long long)s_culled);
        atomicAdd(culled, (unsigned long long)s_culled);
    }
}

// kTrav: 0 = the first traversal loop (Trav), 1 = Trav2, 2 = Trav2 with the cone test compiled out of the primary / sun-shadow
// casts (they are cast with coef = 0).  Same operations per ray, identical results.
//
// 8 CTAs per SM (64 registers): with the loop invariants held in registers (keep_in_register, lsvo_step.cuh) the four traversal
// loops compile without spills at 64 registers — the ~270 bytes of spills sit in the chain code between the casts — and the
// kernel, which was waiting on instruction latency at 20 warps per SM (issue slots 74 % busy, 1.75 eligible warps per scheduler),
// gains from every step: 5 / 6 / 7 / 8 CTAs per SM = 45.06 / 42.83 / 41.69 / 41.15 ms on the headline frame, same box
// (profiles/r02_ab_keepreg.txt).  Beyond 8 it loses again although the loops still hold at 56 / 48 / 40 registers: 9 / 10 / 12 CTAs =
// 42.1 / 42.0 / 43.8 ms against 40.3 (profiles/r02_ab_ctas2.txt; L1 shrinks and the chain code spills 260-420 bytes), and per-warp
// statistics counters (6 KB of shared memory less per CTA, redux + two shared atomics per cast) cost 0.3 ms instead of gaining.
#ifndef VRT_K6_MIN_CTAS
#define VRT_K6_MIN_CTAS 8
#endif
template <typename Nodes, int kTrav, bool kMirror = false, bool kGuard = true>
__global__ void __launch_bounds__(128, VRT_K6_MIN_CTAS) render_rounds_kernel(Nodes nodes, RenderLaunch L, BlockGeometry G,
                                                                            const uint16_t* __restrict__ lists, uint32_t* meta,
                                                                            uint32_t* __restrict__ accum,
                                                                            unsigned long long* __restrict__ counters) {
    extern __shared__ uint2 smem[];
    __shared__ int s_block;
    Stack64<128> stack{smem + threadIdx.x};
    nodes.slots = pin(nodes.slots);
    // kTrav 0 keeps the first loop's recipe (blockIdx.y sums); the Trav2 loops hold their invariants in registers
    const int guard = kTrav == 0 ? pin(L.guard) : keep_in_register(L.guard, smem + threadIdx.x);
    const int depth_offset = pin(kSvoMaxDepth - L.depth);
    Stack64s<128> stack2 = Stack64s<128>::make(smem + threadIdx.x, kSvoMaxDepth - L.depth);
    const float guard_sf = keep_in_register(guard_scale_f(L.guard), smem + threadIdx.x);
    (void)stack; (void)stack2; (void)guard_sf;
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int k = 0; k < 6; ++k) stack2.stat_zero(k);                          // rays and loop trips per ray class, behind the stack
    const float SCALE = 1.0f / float(1 << L.depth);                           // raycaster.hpp:123-124 / main.cpp:82
    const float n_norm = SCALE * 0.0078125f * 2.0f;                           // raycaster.hpp:171-172
    const float aspect = float(L.width) / float(L.height);                    // main.cpp:133
    const float focal_length = L.focal ? __ldg(L.focal) : L.cam.focal_length;
    const int n_blocks = G.tiles_x * G.tiles_y * G.runs;
    // the next block to start: a counter behind the blocks' (samples, next round) pairs, addressed from `meta` on the spot (a pointer
    // of its own would be one more value alive across the traversal loops)

    // all rounds this warp can get of block `work`
    auto trace_block = [&](int work) {
        int x0, y0, s_begin, n_s;
        block_origin(L, G, work, x0, y0, s_begin, n_s);
        const uint32_t total = meta[2 * work];
        for (;;) {
            uint32_t round = 0u;
            if (lane == 0) round = atomicAdd(meta + 2 * work + 1, 1u);
            round = __shfl_sync(0xffffffffu, round, 0);
            if (round * 32u >= total) break;
            const uint32_t slot = round * 32u + uint32_t(lane);
            uint32_t cr = 0, cg = 0, cb = 0, key = 0xffffffffu;
            if (slot < total) {
                const int c = lists[size_t(work) * G.cap + slot];
                const int j = c / n_s, s = s_begin + (c - j * n_s);
                int x, y;
                block_pixel(x0, y0, j, x, y);
                const uint32_t pixel = uint32_t(y) * uint32_t(L.width) + uint32_t(x);
                key = uint32_t(j);
                const uint32_t sample = uint32_t(L.sample_offset + s);
                const float lens_x = float(x) / float(L.height) - aspect * 0.5f;  // main.cpp:145
                const float lens_y = float(y) / float(L.height) - 0.5f;           // main.cpp:146
                ChainState cs;
                NextRay nr;
                chain_begin(L, cs, pixel, sample, lens_x, lens_y, SCALE, focal_length, nr);
                if constexpr (kTrav == 2) nr.t_floor = beam_floor_of(L, x, y, nr.dx, nr.dy, nr.dz);
                int stage = kPrimary;
                while (stage != kDone) {
                    LsvoResult r;
                    if constexpr (kTrav == 0) {
                        lsvo_cast_ray(nodes, stack, depth_offset, guard, nr.ox, nr.oy, nr.oz, nr.dx, nr.dy, nr.dz, nr.coef, 0.0f, r);
                    } else if constexpr (kTrav == 1) {
                        lsvo_cast_ray2<true>(nodes, stack2, guard, guard_sf, nr.ox, nr.oy, nr.oz, nr.dx, nr.dy, nr.dz, nr.coef, 0.0f, r);
                    } else {
                        if (stage < kGi0) lsvo_cast_ray2<false, true, kGuard, true>(nodes, stack2, guard, guard_sf, nr.ox, nr.oy, nr.oz, nr.dx, nr.dy, nr.dz, 0.0f, 0.0f, r, nr.t_floor, &L.bounds);
                        else lsvo_cast_ray2<true, false, kGuard, true>(nodes, stack2, guard, guard_sf, nr.ox, nr.oy, nr.oz, nr.dx, nr.dy, nr.dz, nr.coef, 0.0f, r);
                    }
                    stack2.stat_add(stage, 1u, r.complexity);
                    LsvoHit h;
                    if (r.hit) lsvo_finish(r, nr.ox, nr.oy, nr.oz, L.depth, h);
                    stage = chain_advance<kMirror>(L, cs, stage, r, h, pixel, sample, SCALE, n_norm, nr, nodes.slots);
                }
                chain_colour<kMirror>(L, cs, cr, cg, cb);
            }
            __syncwarp();
            // Every lane adds its own sample to the pixel's accumulator (Sample, raycaster.hpp:18-24,87-90) with RED operations —
            // no return value, the L2 merges the adds of a pixel.  Several CTAs may work on one block, so the sums live in
            // global memory.  (Adding up the lanes of a pixel first — match_any + three reduce_add, one atomic per pixel and
            // channel — costs ~170 instructions per round for the loops ptxas makes of a reduction over a partial mask:
            // 36.74 vs 36.0 ms on the headline frame, profiles/r02_ab_commit.txt.)
            if (key != 0xffffffffu) {
                int x, y;
                block_pixel(x0, y0, int(key), x, y);
                uint32_t* w = accum + 4 * (size_t(y) * size_t(L.width) + size_t(x));
                if (cr) atomicAdd(w, cr);
                if (cg) atomicAdd(w + 1, cg);
                if (cb) atomicAdd(w + 2, cb);
                atomicAdd(w + 3, 1u);
            }
        }
    };

    // One call site for trace_block (it holds four inlined traversal loops: two copies of it do not fit the instruction cache).
    // Phase 0 — own blocks: the CTA takes a block, its warps share the block's rounds (`work >= n_blocks` is CTA-uniform, so all
    // warps leave the phase together and the barriers stay matched).  Phase 1 — help: blocks are started in order, so unfinished
    // ones are among the last started; every warp scans backwards, 32 blocks per look, and joins whatever still has rounds.
    // Helping CTAs spread out (L.help_window = W > 0): CTA c starts its scan at group (last - c mod W) of the W highest groups of 32
    // blocks and, inside a group, at a block picked by c / W; it goes round the window until a whole turn finds nothing open, then
    // continues below it as before.  Its four warps make the same choices, so they join the same block and share its nodes in L1.
    // W = 0: every warp starts at the last block (all helpers work their way down through the same blocks together).
    bool helping = false, below = false;
    const int groups = (n_blocks + 31) >> 5;
    const int W = L.help_window > groups ? groups : L.help_window;
    const int rot = W > 0 ? int(blockIdx.x / unsigned(W)) & 31 : 0;
    int g = groups - 1, looked = 0, cur = 0;
    unsigned open_mask = 0u;
    for (;;) {
        int work;
        if (!helping) {
            if (threadIdx.x == 0) s_block = int(atomicAdd(meta + 2 * n_blocks, 1u));
            __syncthreads();
            work = s_block;
            __syncthreads();
            if (work >= n_blocks) {
                helping = true;
                below = W == 0;
                g = W > 0 ? groups - 1 - int(blockIdx.x % unsigned(W)) : groups - 1;
                continue;
            }
        } else {
            if (!open_mask) {
                // (a global count of the blocks handed out completely, read here to leave at once when nothing is left, measured
                // slower: 40.85 vs 40.51 ms on the headline frame, profiles/r02_ab_exh.txt)
                if (!below && looked == W) { below = true; g = groups - 1 - W; }
                if (below && (g < 0 || g < groups - 1 - 256)) break;                  // far behind the frontier: everything is done
                cur = g * 32 + 31;
                const int w = cur - lane;
                bool open = false;
                if (w < n_blocks) open = *reinterpret_cast<volatile uint32_t*>(meta + 2 * w + 1) * 32u < meta[2 * w];
                open_mask = __ballot_sync(0xffffffffu, open);
                if (below) --g;
                else {
                    looked = open_mask ? 0 : looked + 1;
                    g = g == groups - W ? groups - 1 : g - 1;
                }
                if (!open_mask) continue;
            }
            const unsigned turned = __funnelshift_r(open_mask, open_mask, rot);
            const int bit = (__ffs(turned) - 1 + rot) & 31;
            open_mask &= ~(1u << bit);
            work = cur - bit;
        }
        trace_block(work);
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        uint32_t a, b;
        stack2.stat_get(k, a, b);
        for (int o = 16; o > 0; o >>= 1) {
            a += __shfl_xor_sync(0xffffffffu, a, o);
            b += __shfl_xor_sync(0xffffffffu, b, o);
        }
        if (lane == 0 && a) {
            atomicAdd(counters + k, (unsigned long long)a);
            atomicAdd(counters + 6 + k, (unsigned long long)b);
        }
    }
}

// RayCaster::castRay (raycaster.hpp:118-167) for explicit rays: the caller supplies start and direction — what the
// reference's renderRay receives from Camera::getRay (main.cpp:147-149) — and gets the sample's colour back.  One thread per
// ray, the same sample chain as the frame kernels (sun shadow, GI with the Philox numbers of (pixel, sample)), so a ray
// that equals the frame kernels' primary ray of (pixel, sample) gives exactly that sample's colour.
// kPalette: the colour bits of L.palette (palette albedo, mirror voxels); `nodes` is then the reference layout.  With mirror
// voxels the chain reflects like the frame kernels' (the lake rule, mirror_y1, is a frame parameter and not read here), and
// distance and complexity are those of the camera ray.
template <typename Nodes, bool kGuard, bool kPalette = false>
__global__ void __launch_bounds__(128, 8) shade_rays_kernel(Nodes nodes, RenderLaunch L, uint64_t n, const vrt_shade_job* __restrict__ jobs,
                                                         vrt_shade_result* __restrict__ out) {
    extern __shared__ uint2 smem[];
    nodes.slots = pin(nodes.slots);
    const int guard = keep_in_register(L.guard, smem + threadIdx.x);
    Stack64s<128> stack = Stack64s<128>::make(smem + threadIdx.x, kSvoMaxDepth - L.depth);
    const float guard_sf = keep_in_register(guard_scale_f(L.guard), smem + threadIdx.x);
    const uint64_t i = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const vrt_shade_job job = jobs[i];
    const float SCALE = 1.0f / float(1 << L.depth);
    const float n_norm = SCALE * 0.0078125f * 2.0f;
    ChainState c;
    const uint4 rnd0 = philox4x32_10(job.pixel, job.sample, 0u, 0u, L.seed_lo, L.seed_hi);
    c.rnd_z = rnd0.z; c.rnd_w = rnd0.w;
    c.light = 0.f; c.irr0 = 0.f; c.irr1 = 0.f;
    c.have_hit = false; c.gi0_hit = false; c.gi1_hit = false;
    if (kPalette) { c.tint = 1.0f; c.bounds = 0; }
    NextRay nr;
    nr.ox = job.start[0]; nr.oy = job.start[1]; nr.oz = job.start[2];
    nr.dx = job.direction[0]; nr.dy = job.direction[1]; nr.dz = job.direction[2];
    nr.coef = 0.0f;
    nr.t_floor = 0.0f;
    int stage = kPrimary;
    float distance = 0.0f;
    uint32_t complexity = 0u;
    while (stage != kDone) {
        LsvoResult r;
        if (stage < kGi0) lsvo_cast_ray2<false, false, kGuard>(nodes, stack, guard, guard_sf, nr.ox, nr.oy, nr.oz, nr.dx, nr.dy, nr.dz, 0.0f, 0.0f, r);
        else lsvo_cast_ray2<true, false, kGuard, true>(nodes, stack, guard, guard_sf, nr.ox, nr.oy, nr.oz, nr.dx, nr.dy, nr.dz, nr.coef, 0.0f, r);
        if (stage == kPrimary && (!kPalette || c.bounds == 0)) { complexity = r.complexity; if (r.hit) distance = r.t_min; }   // RayContext, raycaster.hpp:132-133,137
        LsvoHit h;
        if (r.hit) lsvo_finish(r, nr.ox, nr.oy, nr.oz, L.depth, h);
        stage = chain_advance<false, kPalette>(L, c, stage, r, h, job.pixel, job.sample, SCALE, n_norm, nr, nodes.slots);
    }
    uint32_t cr = 0, cg = 0, cb = 0;
    chain_colour<kPalette>(L, c, cr, cg, cb);
    vrt_shade_result res;
    res.r = uint8_t(cr); res.g = uint8_t(cg); res.b = uint8_t(cb); res.hit = c.have_hit ? 1 : 0;
    res.distance = distance;
    res.complexity = complexity;
    res.reserved = 0u;
    out[i] = res;
}

cudaError_t launch_shade_rays(const uint2* nodes, bool compact, const RenderLaunch& L, uint64_t n, const vrt_shade_job* d_jobs,
                              vrt_shade_result* d_out, cudaStream_t stream) {
    if (!n) return cudaSuccess;
    const size_t smem = size_t(L.depth + 1) * 128 * 8;
    const unsigned grid = unsigned((n + 127) / 128);
    // palette or mirror voxels: `nodes` is the reference array whatever the scene's layout (the colours live in its leaf slots)
    if (L.palette) shade_rays_kernel<RefNodes, true, true><<<grid, 128, smem, stream>>>(RefNodes{nodes}, L, n, d_jobs, d_out);
    else if (compact) shade_rays_kernel<CompactNodes, true><<<grid, 128, smem, stream>>>(CompactNodes{nodes}, L, n, d_jobs, d_out);
    else if (guard_binds(L)) shade_rays_kernel<RefNodes, true><<<grid, 128, smem, stream>>>(RefNodes{nodes}, L, n, d_jobs, d_out);
    else shade_rays_kernel<RefNodes, false><<<grid, 128, smem, stream>>>(RefNodes{nodes}, L, n, d_jobs, d_out);
    return cudaGetLastError();
}

// Camera::getClosestPoint (camera_controller.hpp:56-60) and the focal-length rule of main.cpp:114-121, one thread.
template <typename Nodes>
__global__ void __launch_bounds__(128) autofocus_kernel(Nodes nodes, int depth, int guard, vrt_camera cam, float* __restrict__ focal) {
    extern __shared__ uint2 smem[];
    if (threadIdx.x != 0) return;
    Stack64s<128> stack = Stack64s<128>::make(smem, kSvoMaxDepth - depth);
    const float scale = 1.0f / float(1 << depth);
    const float ox = cam.position[0] * scale + 1.0f, oy = cam.position[1] * scale + 1.0f, oz = cam.position[2] * scale + 1.0f;
    float dx, dy, dz;
    view_to_world(cam.rot_mat, 0.0f, 0.0f, 1.0f, dx, dy, dz);                 // camera_vec, camera_controller.hpp:31
    LsvoResult r;
    lsvo_cast_ray2<false>(nodes, stack, guard, guard_scale_f(guard), ox, oy, oz, dx, dy, dz, 0.0f, 0.0f, r);
    *focal = r.hit ? r.t_min * float(1 << depth) : 100.0f;
}

// samples_to_image (raycaster.hpp:94-103) or the 0.4/0.6 temporal blend of renderRay (:79-85).
__global__ void resolve_kernel(const uint32_t* __restrict__ accum, uint8_t* __restrict__ rgba, int width, int row_begin,
                               int row_end, int use_samples, int tile_step, int tile_index) {
    const uint64_t j = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;       // index inside the owned rows
    const int x = int(j % uint64_t(width));
    const int row = int(j / uint64_t(width));                                 // owned-row ordinal
    const int y = row_begin + ((row >> 2) * tile_step + tile_index) * 4 + (row & 3);
    if (y >= row_end) return;
    const uint64_t i = uint64_t(y) * width + x;
    const uint4 a = reinterpret_cast<const uint4*>(accum)[i];
    uchar4* out = reinterpret_cast<uchar4*>(rgba) + i;
    if (use_samples) {
        // double division then uint8 conversion == integer division for sums < 2^32 (DESIGN.md §3)
        const uint32_t n = a.w ? a.w : 1u;
        *out = make_uchar4(uint8_t(a.x / n), uint8_t(a.y / n), uint8_t(a.z / n), 255);
    } else {
        if (a.w == 0u) return;                                                // not rendered this frame (checkerboard)
        const uchar4 old = *out;
        // the accumulator holds exactly one sample in this mode
        const uint8_t nr = mul_u8(uint8_t(a.x), 1.0f - 0.4f), ng = mul_u8(uint8_t(a.y), 1.0f - 0.4f), nb = mul_u8(uint8_t(a.z), 1.0f - 0.4f);
        const int r = min(255, int(mul_u8(old.x, 0.4f)) + int(nr));          // add(sf::Color&, const sf::Color&), utils.cpp:35-40
        const int g = min(255, int(mul_u8(old.y, 0.4f)) + int(ng));
        const int b = min(255, int(mul_u8(old.z, 0.4f)) + int(nb));
        *out = make_uchar4(uint8_t(r), uint8_t(g), uint8_t(b), 255);
    }
}

namespace {
// K6's launch plan: blocks, runs, list capacity, bins — shared by the scratch-size query and the launcher
struct RoundsPlan {
    BlockGeometry G;
    SortPlan sort;
    size_t lists_bytes, meta_bytes;
};
RoundsPlan plan_rounds(const RenderLaunch& L) {
    RoundsPlan P;
    const int rows = L.row_end - L.row_begin;
    P.G.tiles_x = (L.width + 31) / 32;
    P.G.tiles_y = ((rows + 3) / 4 + L.tile_step - 1 - L.tile_index) / L.tile_step;
    if (P.G.tiles_y < 0) P.G.tiles_y = 0;
    int runs = 1;
    while ((L.spp + runs - 1) / runs > 64) runs *= 2;                               // <= 8192 samples per list (16-bit entries)
    while (runs < L.spp_chunks && runs * 2 <= L.spp) runs *= 2;                     // explicit override: more, shorter lists
    P.G.runs = runs;
    P.G.cap = 128 * ((L.spp + runs - 1) / runs);
    const int n = 128 * (L.spp / runs);
    P.sort.bins1 = !L.use_gi ? 1 : n >= 2048 ? 16 : n >= 512 ? 8 : n >= 128 ? 4 : 1;
    P.sort.bins2 = 1;
    if (L.sort_bins1 > 0) {
        P.sort.bins1 = L.sort_bins1;
        P.sort.bins2 = L.sort_bins2 > 0 ? L.sort_bins2 : 1;
        if (P.sort.bins1 * P.sort.bins2 > 256) P.sort.bins2 = 256 / P.sort.bins1;
    }
    const size_t blocks = size_t(P.G.tiles_x) * P.G.tiles_y * runs;
    P.lists_bytes = (blocks * P.G.cap * sizeof(uint16_t) + 255) & ~size_t(255);
    P.meta_bytes = ((blocks * 2 + 1) * sizeof(uint32_t) + 255) & ~size_t(255);
    return P;
}
}  // namespace

// 2 = K4, 3 = K5, 4 = K6.  Automatic: K6 for many-sample frames (with or without a GI pass: without one the lists stay
// in pixel order and K6 still wins through its even finish), K4 for the interactive loop.
static int choose_mapping(const RenderLaunch& L) {
    if (L.checker) return 2;
    if (L.mapping >= 2) return L.mapping;
    return L.spp >= 8 ? 4 : 2;
}

size_t render_scratch_bytes(const RenderLaunch& L) {
    if (choose_mapping(L) != 4 || L.row_end <= L.row_begin || L.width <= 0 || L.spp <= 0) return 0;
    const RoundsPlan P = plan_rounds(L);
    return P.lists_bytes + P.meta_bytes;
}

cudaError_t launch_render_accumulate_ref(const uint2* nodes, bool compact, const RenderLaunch& L, uint32_t* d_accum,
                                         unsigned long long* d_counters, cudaStream_t stream) {
    const int rows = L.row_end - L.row_begin;
    if (rows <= 0 || L.width <= 0 || L.spp <= 0) return cudaSuccess;
    const int block = 128;
    const int columns = L.checker ? (L.width + 1) / 2 : L.width;
    const int tiles_x = (columns + 31) / 32, tiles_y = ((rows + 3) / 4 + L.tile_step - 1 - L.tile_index) / L.tile_step;
    if (tiles_y <= 0) return cudaSuccess;
    const size_t smem = size_t(L.depth + 1) * block * 8 + 12 * block * sizeof(uint32_t);   // stacks + statistics
    const int mapping = choose_mapping(L);
    if (mapping == 4) {                                                                  // K6
        const RoundsPlan P = plan_rounds(L);
        if (!L.scratch || L.scratch_bytes < P.lists_bytes + P.meta_bytes) return cudaErrorInvalidValue;
        uint16_t* lists = static_cast<uint16_t*>(L.scratch);
        uint32_t* meta = reinterpret_cast<uint32_t*>(static_cast<char*>(L.scratch) + P.lists_bytes);
        const unsigned blocks = unsigned(P.G.tiles_x) * P.G.tiles_y * P.G.runs;
        uint32_t* next_block = meta + 2 * size_t(blocks);
        cudaError_t e = cudaMemsetAsync(next_block, 0, sizeof(uint32_t), stream);
        if (e != cudaSuccess) return e;
        sort_samples_kernel<<<blocks, 128, 0, stream>>>(L, P.sort, P.G, lists, meta, d_accum, d_counters, d_counters + kCulledCounter);
        int per_sm = 0, sms = 0, dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        auto launch6 = [&](auto kernel, auto view) {
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, block, smem);
            unsigned grid6 = unsigned(per_sm > 0 ? per_sm : 1) * unsigned(sms);
            if (grid6 > blocks) grid6 = blocks;
            kernel<<<grid6, block, smem, stream>>>(view, L, P.G, lists, meta, d_accum, d_counters);
        };
        if (compact) launch6(render_rounds_kernel<CompactNodes, 0>, CompactNodes{nodes});
        else if (L.mirror_y1 > 0 || L.palette) {
            if (guard_binds(L)) launch6(render_rounds_kernel<RefNodes, 2, true, true>, RefNodes{nodes});
            else launch6(render_rounds_kernel<RefNodes, 2, true, false>, RefNodes{nodes});
        } else switch (L.trav_policy) {
            case 0: launch6(render_rounds_kernel<RefNodes, 0>, RefNodes{nodes}); break;
            case 1: launch6(render_rounds_kernel<RefNodes, 1>, RefNodes{nodes}); break;
            default:
                if (guard_binds(L)) launch6(render_rounds_kernel<RefNodes, 2, false, true>, RefNodes{nodes});
                else launch6(render_rounds_kernel<RefNodes, 2, false, false>, RefNodes{nodes});
                break;
        }
        return cudaGetLastError();
    }
    // Sample runs: a power of two, enough for >= 28 waves of CTAs (4 CTAs x 148 SMs resident) so the last wave is a
    // small part of the launch even when a GPU owns 1/8 of the frame, but runs of >= 8 samples so that 8+ lanes can
    // share a pixel.  tools/probe_slice.py: whole frame 74.4 ms at (2 runs, 32 lanes/pixel) vs 77.7 ms at (4, 1);
    // 1/8 slice 9.60 ms at (8, 8) vs 9.92 ms at (29, 1).
    RenderLaunch Lc = L;
    const long tiles = long(tiles_x) * tiles_y;
    long chunks = 1;
    while (chunks * tiles < 28L * 4 * 148 && chunks * 2 * 8 <= L.spp) chunks *= 2;
    if (L.spp_chunks > 0) chunks = L.spp_chunks < L.spp ? L.spp_chunks : L.spp;      // explicit override
    if (mapping == 3) {                                                                  // K5 (kept selectable: render_variant 3)
        // K5 sorts better with long runs (more samples per direction bin): 12 waves of CTAs are enough here.
        // tools/probe_sorted.py, cfg 4: whole frame 67.8 ms at (1 run, 16 bins) vs 70.2 at (4, 16); the 1/8 slice of an
        // 8-GPU rank 9.07 ms at (4, 8) vs 9.69 at (1, 16).  Sorting by the second bounce's angle as well did not pay.
        if (L.spp_chunks <= 0) {
            chunks = 1;
            while (chunks * tiles < 12L * 4 * 148 && chunks * 2 * 8 <= L.spp) chunks *= 2;
        }
        while ((L.spp + chunks - 1) / chunks > 64) chunks *= 2;                     // <= 8192 samples per CTA (16-bit list)
        Lc.spp_chunks = int(chunks);
        const int n = 128 * int(L.spp / chunks);                                    // samples in the shortest run
        SortPlan plan;
        plan.bins1 = !L.use_gi ? 1 : n >= 2048 ? 16 : n >= 512 ? 8 : n >= 128 ? 4 : 1;   // 22.5 degree sectors when they fill >= 4 rounds
        plan.bins2 = 1;
        if (L.sort_bins1 > 0) {                                                     // explicit override (measurements)
            plan.bins1 = L.sort_bins1;
            plan.bins2 = L.sort_bins2 > 0 ? L.sort_bins2 : 1;
            if (plan.bins1 * plan.bins2 > 256) plan.bins2 = 256 / plan.bins1;
        }
        const int longest = int((L.spp + chunks - 1) / chunks);
        const size_t smem5 = size_t(L.depth + 1) * block * 8 + 12 * block * sizeof(uint32_t) + (260 + 512 + 4) * sizeof(uint32_t) +
                             size_t(128) * longest * sizeof(uint16_t);
        const unsigned grid5 = unsigned(tiles * chunks);
        if (compact) render_sorted_kernel<CompactNodes><<<grid5, block, smem5, stream>>>(CompactNodes{nodes}, Lc, plan, d_accum, d_counters);
        else render_sorted_kernel<RefNodes><<<grid5, block, smem5, stream>>>(RefNodes{nodes}, Lc, plan, d_accum, d_counters);
        return cudaGetLastError();
    }
    Lc.spp_chunks = int(chunks);
    // lanes per pixel: the largest power of two (<= 32) that divides every chunk's sample count
    int q = 32;
    for (long c = 0; c < chunks; ++c) {
        const long ns = ((c + 1) * L.spp) / chunks - (c * L.spp) / chunks;
        while (q > 1 && ns % q) q >>= 1;
    }
    if (L.samples_per_warp > 0 && L.samples_per_warp < q) q = L.samples_per_warp;       // explicit override (power of two)
    Lc.samples_per_warp = q;
    const unsigned grid = unsigned(tiles * chunks);
    const bool live = L.checker != 0 || L.focal != nullptr;
    auto launch4 = [&](auto kernel, auto view) { kernel<<<grid, block, smem, stream>>>(view, Lc, d_accum, d_counters); };
    const bool guarded = guard_binds(L);
    if (compact) {
        if (live) launch4(render_accumulate_kernel<CompactNodes, true>, CompactNodes{nodes});
        else launch4(render_accumulate_kernel<CompactNodes, false>, CompactNodes{nodes});
    } else if (L.mirror_y1 > 0 || L.palette) {
        if (live) { if (guarded) launch4(render_accumulate_kernel<RefNodes, true, true, true>, RefNodes{nodes}); else launch4(render_accumulate_kernel<RefNodes, true, true, false>, RefNodes{nodes}); }
        else { if (guarded) launch4(render_accumulate_kernel<RefNodes, false, true, true>, RefNodes{nodes}); else launch4(render_accumulate_kernel<RefNodes, false, true, false>, RefNodes{nodes}); }
    } else {
        if (live) { if (guarded) launch4(render_accumulate_kernel<RefNodes, true, false, true>, RefNodes{nodes}); else launch4(render_accumulate_kernel<RefNodes, true, false, false>, RefNodes{nodes}); }
        else { if (guarded) launch4(render_accumulate_kernel<RefNodes, false, false, true>, RefNodes{nodes}); else launch4(render_accumulate_kernel<RefNodes, false, false, false>, RefNodes{nodes}); }
    }
    return cudaGetLastError();
}

cudaError_t launch_autofocus(const uint2* nodes, bool compact, int depth, int guard, const vrt_camera& cam, float* d_focal,
                             cudaStream_t stream) {
    const size_t smem = size_t(depth + 1) * 128 * 8;
    if (compact) autofocus_kernel<CompactNodes><<<1, 128, smem, stream>>>(CompactNodes{nodes}, depth, guard, cam, d_focal);
    else autofocus_kernel<RefNodes><<<1, 128, smem, stream>>>(RefNodes{nodes}, depth, guard, cam, d_focal);
    return cudaGetLastError();
}

cudaError_t launch_resolve(const uint32_t* d_accum, uint8_t* d_rgba, int width, int row_begin, int row_end, int use_samples,
                           int tile_step, int tile_index, cudaStream_t stream) {
    const int tiles = ((row_end - row_begin + 3) / 4 + tile_step - 1 - tile_index) / tile_step;
    const uint64_t n = uint64_t(tiles > 0 ? tiles : 0) * 4 * width;
    if (!n) return cudaSuccess;
    resolve_kernel<<<unsigned((n + 255) / 256), 256, 0, stream>>>(d_accum, d_rgba, width, row_begin, row_end, use_samples, tile_step,
                                                                 tile_index);
    return cudaGetLastError();
}

}  // namespace vrt
