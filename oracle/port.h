/* TEST INFRASTRUCTURE ONLY (oracle/): CPU restatement of the reference's per-pixel hot path.
 *
 * Plain C, scalar, -ffp-contract=off.  Every function cites the reference file:line it follows.
 * Pinned against the reference's own compiled sources (oracle/_ref, built by oracle/Makefile) by
 * tests/test_oracle_pinned.py and against the committed fixtures under tests/golden/.
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
 * load libvrt_oracle.so — as the checker, never as the thing measured or shipped.
 */
#ifndef VRT_ORACLE_PORT_H
#define VRT_ORACLE_PORT_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* LNode, include/lsvo_utils.hpp:5-18 (8 bytes; `color` is always 1 and never read). */
typedef struct vo_lnode {
    uint8_t color, child_mask, leaf_mask, pad;
    uint32_t child_offset;
} vo_lnode;

/* HitPoint, include/volumetric.hpp:7-22, plus the traversal state a checker wants to see. */
typedef struct vo_hit {
    float position[3];
    float normal[3];
    float voxel_coord[2];
    float distance;
    uint32_t complexity;
    uint32_t hit;      /* 0 = miss (only complexity is defined, the rest is zeroed) */
    int32_t scale;     /* octree scale of the hit cell (23-depth for a leaf voxel), 0 on a miss */
    int32_t voxel[3];  /* integer cell coordinate of the hit cell's low corner, in voxel units */
    uint32_t face;     /* step mask that entered the cell: bit0 x, bit1 y, bit2 z */
} vo_hit;

/* ---- scene construction ------------------------------------------------------------------ */
/* FastNoise 0.4.1 SimplexFractal FBM heights as main.cpp:68; out[x*size+z]. */
void vo_terrain_heights(int32_t size, int32_t* out);
float vo_noise2d(float x, float y);
/* compileSVO (lsvo_utils.hpp:45-55, lsvo_utils.cpp:4-49) of the terrain fill main.cpp:63-76 with
 * 256 generalised to size/2, WITHOUT the pointer SVO.  Returns the slot count; if `out` is NULL only
 * counts.  `cap` = capacity of out in nodes. */
uint64_t vo_build_terrain_lsvo(int depth, const int32_t* heights, vo_lnode* out, uint64_t cap);
/* Same flattening for an arbitrary dense occupancy grid occ[(x*S+y)*S+z] != 0 (setCell coordinates). */
uint64_t vo_build_dense_lsvo(int depth, const uint8_t* occ, vo_lnode* out, uint64_t cap);

/* ---- traversal ---------------------------------------------------------------------------- */
/* LSVO<depth>::castRay, include/lsvo.hpp:33-172.  `guard` is the lower loop bound of lsvo.hpp:72
 * (`scale > MAX_DEPTH`): pass `depth` for the reference expression. */
void vo_lsvo_cast(const vo_lnode* nodes, int depth, int guard, const float* origin, const float* dir,
                  float coef, float bias, uint64_t n, vo_hit* out, int threads);

/* The LSVO walk restated with the structural changes of the device loop (unconditional push, one hit exit, hit read off the final
 * state, guard dropped where it cannot bind, fmaf child selection with unit != 0, node fetched when the parent changes): must
 * return exactly what vo_lsvo_cast returns — a CPU cross-check of DESIGN.md §4, not a second specification. */
void vo_lsvo_cast_restructured(const vo_lnode* nodes, int depth, int guard, const float* origin, const float* dir, float coef,
                               float bias, int unit, uint64_t n, vo_hit* out, int threads);

/* Grid3D<X,Y,Z>::castRay, include/grid_3d.hpp:35-132; cells[(x*Y+y)*Z+z] = Cell::Type. */
void vo_grid_cast(const uint8_t* cells, int X, int Y, int Z, const float* origin, const float* dir,
                  uint64_t n, vo_hit* out, uint32_t* steps, int threads);

/* Conservative miss test for Grid3D::castRay on a coarse occupancy dilated by two cubes (one byte per cube of 2^shift cells,
 * coarse[(x*CY+y)*CZ+z]): out[i] = 1 when ray i certainly misses, 0 when it has to be walked.  A prototype of what the pyramid
 * can do for dense grids without changing a record (DESIGN.md §7); pinned to vo_grid_cast by tests/test_oracle_golden.py. */
void vo_grid_miss_test(const uint8_t* coarse, int CX, int CY, int CZ, int shift, int X, int Y, int Z, const float* origin,
                       const float* dir, uint64_t n, uint8_t* out, int threads);

/* SVO<depth>::castRay with fillHitResult's commented body restored ("intended SVO"),
 * include/svo.hpp:62-70,116-194, over a dense occupancy occ[(x*S+y)*S+z]. */
void vo_svo_cast(const uint8_t* occ, int depth, const float* origin, const float* dir, uint32_t max_iter,
                 uint64_t n, vo_hit* out, int threads);

/* ---- shading ------------------------------------------------------------------------------ */
typedef struct vo_render_params {
    int32_t width, height;
    int32_t depth;            /* octree depth D; scale = 1/2^D replaces the literal 1/512 */
    int32_t guard;            /* loop guard, see vo_lsvo_cast */
    float cam_position[3];    /* voxel units (main.cpp:51) */
    float rot_mat[9];         /* Camera::rot_mat, column major (camera_controller.hpp:21) */
    float fov, aperture, focal_length;
    float light_position[3];  /* normalised: light/2^D + 1 (main.cpp:126) */
    int32_t use_gi;
    int32_t gi_bounces;       /* 1 = reference (raycaster.hpp:169-207); 2 = extension, see DESIGN.md */
    int32_t use_samples;      /* accumulate (raycaster.hpp:87-90) vs 0.4/0.6 temporal blend (:79-85) */
    int32_t spp;
    uint32_t seed_lo, seed_hi;  /* Philox4x32-10 key */
    int32_t sample_offset;      /* first sample index (spp batches) */
    int32_t row_begin, row_end; /* rows [begin,end) */
    int32_t threads;
    int32_t tile_step, tile_index; /* > 1: only 4-row tiles t (from row_begin) with t % tile_step == tile_index */
    float roughness;               /* vo_grid_render: blur of mirror reflections (0 = perfect mirror) */
    int32_t max_bounds;            /* vo_grid_render: reflection depth, RayCaster::max_bounds = 4 (raycaster.hpp:277) */
    int32_t checker;               /* 0 = all pixels; 1 / 2 = checker_board_offset 0 / 1 of main.cpp:137,143 */
    int32_t checker_area_height;   /* RENDER_HEIGHT / area_count (main.cpp:132); 0 = a single area */
    int32_t mirror_y1;             /* vo_render: 1 + y of the voxel layer whose top faces are Cell::Mirror (extension, see port.c); 0 = none */
} vo_render_params;

typedef struct vo_render_stats {
    uint64_t rays[6];        /* primary, shadow, gi, gi-shadow, gi2, gi2-shadow (distinct castRay calls) */
    uint64_t complexity[6];  /* summed HitPoint::complexity per class */
} vo_render_stats;

/* tex_top / tex_side: 16x16 RGB, top-down rows (res/grass_top_16x16.bmp, res/grass_side_16x16.bmp as
 * sf::Image presents them).  accum: [H*W*4] uint32 r,g,b,count sums (exact integer image of the
 * reference's double accumulators raycaster.hpp:87-90).  rgba: resolved image (samples_to_image
 * raycaster.hpp:94-103, or the temporal blend against `rgba` as previous frame when !use_samples). */
void vo_render(const vo_lnode* nodes, const vo_render_params* p, const uint8_t* tex_top, const uint8_t* tex_side,
               uint32_t* accum, uint8_t* rgba, vo_render_stats* stats);

/* Shading over a dense grid (Grid3D / MipmapGrid3D) with mirror reflections — an EXTENSION, "parity unpinned":
 * the reference has Cell::Mirror (cell.hpp:8), RayContext::bounds and max_bounds = 4 (raycaster.hpp:13,127,277) but no
 * code that reflects (SURVEY.md §0).  Specification (DESIGN.md §2):
 *   positions are in voxel units (Grid3D::castRay, grid_3d.hpp:35); camera ray as Camera::getRay with
 *   start = cam_position + world_rand_offset; light_position in voxel units;
 *   loop: hit = Grid3D::castRay(o, d); miss → black.  Mirror cell and bounds < max_bounds → ++bounds,
 *     o = hit + n * 0.001, d = d with the hit axis negated (reflection about the unit normal, exact),
 *     d = normalize(d + roughness * (r0, r1, r2)), r_k = getRand() of dimensions 8+3*bounce+k, tint *= 0.8, repeat.
 *   otherwise (Solid, or Mirror at max depth): albedo = texture (top iff n.y != 0; texel index min(15, uint(16*uv))),
 *     shadow ray o = hit + n * 0.001 toward the light, light = unoccluded ? max(0, dot(to_light, n)) : 0,
 *     colour = mult(mult(albedo, clamp01(light)), tint) (utils.cpp:43-48).
 * cells[(x*Y+y)*Z+z] = Cell::Type.  stats->rays: [0] primary, [1] shadow, [2] reflection rays.
 * checker / checker_area_height select pixels as in vo_render; the other pixels of accum and rgba are left alone. */
void vo_grid_render(const uint8_t* cells, int X, int Y, int Z, const vo_render_params* p, const uint8_t* tex_top,
                    const uint8_t* tex_side, uint32_t* accum, uint8_t* rgba, vo_render_stats* stats);

/* Presentation step, main.cpp:159-177 ("parity unpinned": the reference does this with OpenGL blending through SFML,
 * which is not available here; the arithmetic below is the round-to-nearest 8-bit unorm blending a GPU performs):
 *   frame' = per-channel median of the (median x median) window around each pixel, edges clamped (res/median_3.frag,
 *            res/median.frag; median = 0: frame itself);
 *   display = min(255, (display * c1 + 127) / 255 + (frame' * c2 + 127) / 255), alpha 255,
 *   c1 = (uint8)(255 * old_value_conservation), c2 = (uint8)(255 * (1 - old_value_conservation))   (main.cpp:160-165). */
void vo_present(const uint8_t* frame, uint8_t* display, int32_t width, int32_t height, int32_t median,
                float old_value_conservation);

/* Camera::getRay + main.cpp:145-149 for one pixel/sample with the Philox lattice RNG. */
void vo_camera_ray(const vo_render_params* p, int32_t x, int32_t y, int32_t sample, float origin[3], float dir[3]);

/* Philox4x32-10 (Salmon et al. 2011), exposed for the RNG parity test. */
void vo_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]);

#ifdef __cplusplus
}
#endif
#endif
