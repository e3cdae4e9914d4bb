/* vrt.h — C ABI of the B200-native voxel ray-traversal engine (libvrt.so).
 *
 * Drop-in boundary for the per-pixel hot path of johnBuffer/CpuVoxelRaycaster.  The reference has
 * no FFI; its seam is C++-source-level (SURVEY.md §8b).  Each entry point below names the reference
 * interface it replaces (file:line under the reference tree).  The C++ drop-in classes in
 * the headers under include/vrt/ (same names/signatures as the reference: Volumetric, HitPoint, LSVO<D>, SVO<N>,
 * Grid3D, MipmapGrid3D, RayCaster, Camera) and the Python mirror (cpuvoxelraycaster_b200/) are thin
 * callers of this ABI.
 *
 * Conventions
 *   - every function returns vrt_status (0 = ok, negative = error); vrt_last_error() gives the text
 *     of the last failure on the calling thread.  The reference reports no errors at all
 *     (out-of-range setCell is UB); here bad arguments are VRT_ERR_INVALID.
 *   - the caller owns every host buffer; handles are opaque; a context is bound to one CUDA device
 *     and one stream and is NOT thread-safe (one context per host thread, or external locking).
 *   - no C++ or torch types cross the ABI: plain pointers and sizes only.
 *   - "*_device" variants take device pointers and only enqueue work on the context's stream.
 *   - there is no CPU fallback: without a CUDA device every compute entry point fails with
 *     VRT_ERR_CUDA.  The vrt_host_* scene-construction helpers are pure host code by design
 *     (the reference builds its scene once on the CPU, src/main.cpp:59-86).
 */
#ifndef VRT_H
#define VRT_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VRT_ABI_VERSION 3

typedef enum vrt_status {
    VRT_OK = 0,
    VRT_ERR_INVALID = -1,   /* bad argument */
    VRT_ERR_CUDA = -2,      /* CUDA runtime failure (no device, launch error, ...) */
    VRT_ERR_OOM = -3,       /* host or device allocation failed */
    VRT_ERR_UNSUPPORTED = -4
} vrt_status;

typedef struct vrt_context vrt_context;
typedef struct vrt_scene vrt_scene;

/* LNode, include/lsvo_utils.hpp:5-18 — the reference's flattened octree slot, accepted verbatim. */
typedef struct vrt_lnode {
    uint8_t color;
    uint8_t child_mask;
    uint8_t leaf_mask;
    uint8_t pad;
    uint32_t child_offset;
} vrt_lnode;

/* Superset of HitPoint (include/volumetric.hpp:7-22), 64 bytes, so that the C++ wrapper can rebuild
 * a HitPoint exactly.  On a miss only `flags` (bit 0 clear) and `complexity` are defined — as in the
 * reference, where a miss leaves position/normal/voxel_coord/distance uninitialised — and the other
 * fields are written as zero. */
typedef struct vrt_hit {
    float position[3];    /* HitPoint::position */
    float distance;       /* HitPoint::distance */
    float normal[3];      /* HitPoint::normal (LSVO: ±1, ±2, ±4 per axis, lsvo.hpp:149) */
    uint32_t complexity;  /* HitPoint::complexity (loop iterations) */
    float voxel_coord[2]; /* HitPoint::voxel_coord */
    uint32_t flags;       /* bit 0: hit (HitPoint::cell != nullptr) */
    int32_t scale;        /* LSVO: octree scale of the hit cell (23 - depth for a leaf voxel) */
    int32_t voxel[3];     /* integer coordinate of the hit cell's low corner, voxel units */
    uint32_t face;        /* axis mask that entered the cell: bit0 x, bit1 y, bit2 z */
} vrt_hit;
#define VRT_HIT_FLAG_HIT 1u

typedef enum vrt_scene_kind {
    VRT_SCENE_LSVO = 1,   /* include/lsvo.hpp */
    VRT_SCENE_GRID = 2,   /* include/grid_3d.hpp */
    VRT_SCENE_MIPGRID = 3,/* include/mipmap_grid3D.hpp (stub in the reference; results == Grid3D) */
    VRT_SCENE_SVO = 4     /* include/svo.hpp, intended semantics (fillHitResult restored) */
} vrt_scene_kind;

/* ---- library / context --------------------------------------------------------------------- */
int vrt_abi_version(void);
const char* vrt_last_error(void);
const char* vrt_build_info(void);                   /* compile flags, arch, kernel variants */

/* Replaces swrm::Swarm(thread_count) (src/main.cpp:90-92): the execution resource. `stream` is a
 * cudaStream_t (NULL = the context creates its own non-blocking stream). */
int vrt_context_create(int device, void* stream, vrt_context** out);
/* Destroy every scene created on a context before the context itself (scenes borrow it). */
int vrt_context_destroy(vrt_context* ctx);
int vrt_context_synchronize(vrt_context* ctx);
int vrt_context_set_stream(vrt_context* ctx, void* stream);
/* Tuning knobs (no reference counterpart):
 *   "cast_variant" (default 3): 3 = automatic — a classifier kernel looks at the batch (are 32 consecutive rays neighbours, like the
 *                    reference's pixel rays?) and gates K1b (coherent) or K1p (incoherent) on the device, no host round trip;
 *                    1 = persistent threads with per-lane ray regeneration (K1p), 0 = one thread per ray (K1),
 *                    2 = one thread per ray on the Trav2 loop (K1b).  Results identical
 *   "render_variant" (default 0): 0 = automatic (K6 for frames with >= 8 samples, else K4), 1 = K4p persistent
 *                    regenerating warps, 2 = K4 one lane per pixel/sample group, 3 = K5 samples of a pixel block
 *                    regrouped by GI direction inside the CTA, 4 = K6 the same lists in global memory traced by
 *                    persistent CTAs that help each other finish
 *   "refill_cast", "refill_render"  parked lanes (1..32) that make a persistent warp regenerate rays;
 *                    refill_cast 0 = warp-adaptive (default)
 *   "spp_chunks"     frame kernel: number of runs a pixel's samples are cut into (0 = automatic)
 *   "samples_per_warp"  frame kernel: lanes of a warp sharing one pixel, power of two <= 32 (0 = automatic)
 *   "help_window" (default 64): K6 frame kernel — CTAs that have run out of blocks of their own help with unfinished ones; they spread
 *                    over the last `help_window` groups of 32 blocks instead of all starting at the last block (0).  Results identical
 *   "trav_policy" (default 2): traversal loop of the K6 frame kernel — 0 = Trav (round-1 loop), 1 = Trav2 (bookkeeping moved
 *                    off the ALU pipe), 2 = Trav2 with the cone test compiled out of the coef-0 casts; results identical
 *   "beam_tile" (default 8): LSVO frames with >= 8 samples per pixel — edge in pixels (power of two) of the screen tiles for which a conservative start
 *                    distance of the camera rays is computed in front of the frame (a front-to-back search of the octree
 *                    against each tile's frustum, cpuvoxelraycaster_b200/csrc/beam_kernels.cu).  Frames are byte-identical
 *                    with and without it; the trip counts (complexity) of the primary rays shrink.  0 = off: every ray
 *                    starts where the reference starts it (lsvo.hpp:54-57) and vrt_render_stats equals the reference's counts
 *   "bounds_exit" (default 1): LSVO frames — a walk ends as soon as its ray has left the bounding box of the solid voxels
 *                    (computed on the device when the scene is created or edited) instead of at the far side of the root cube
 *                    (lsvo.hpp:72): misses stay misses, only their trip counts shrink.  0 = the reference's walk
 *   "grid_variant" (default 0): dense grids — 0 = DDA on the bordered bit grid, 1 = the generic loop / fetch-skipping pyramid
 *   "time_frame_kernels"  see vrt_context_take_timings */
int vrt_context_set_option(vrt_context* ctx, const char* key, int value);
/* number of kernel launches this context has enqueued so far (bench.py's gpu_launches) */
uint64_t vrt_context_launch_count(const vrt_context* ctx);
/* With the option "time_frame_kernels" = 1 every vrt_render_accumulate_device call (also inside vrt_render and
 * vrt_render_distributed) is bracketed by CUDA events on the context's stream.  This synchronises the stream and returns
 * the device time of each bracketed call since the last take, oldest first (ms[i], i < min(*count, cap)). */
int vrt_context_take_timings(vrt_context* ctx, float* ms, int32_t cap, int32_t* count);

/* ---- host-side scene construction (pure host code, no GPU needed) ---------------------------- */
/* FastNoise SimplexFractal heights of the demo terrain, src/main.cpp:61-68; out[x*size+z]. */
int vrt_host_terrain_heights(int32_t size, int32_t* out);
/* FastNoise::GetNoise(x, y) of a default-constructed FastNoise set to SimplexFractal (main.cpp:61-62,68;
 * lib/fastnoise/FastNoise.cpp:1191-1333: seed 1337, frequency 0.01, 3 octaves FBM, lacunarity 2, gain 0.5), bit-exact. */
float vrt_host_noise2d(float x, float y);
/* SVO::setCell fill (main.cpp:70-76, 256 → size/2) + compileSVO (lsvo_utils.hpp:45-55,
 * lsvo_utils.cpp:4-49) in one pass, without the 80-byte pointer nodes.  Two-call protocol:
 * out == NULL → *count only. */
int vrt_host_build_terrain_lsvo(uint32_t depth, const int32_t* heights, vrt_lnode* out, uint64_t cap, uint64_t* count);
/* Same flattening for an explicit voxel list (xyz triples in SVO::setCell coordinates, svo.hpp:72). */
int vrt_host_build_lsvo_from_voxels(uint32_t depth, const uint32_t* xyz, uint64_t n_voxels, vrt_lnode* out,
                                    uint64_t cap, uint64_t* count);

/* Camera::setViewAngle (camera_controller.hpp:27-32) + generateRotationMatrix (utils.cpp:94-100,
 * glm::rotate about -y then -x): rot_mat column major, camera_vec = (0,0,1) * rot_mat. */
int vrt_host_camera_rotation(const float view_angle[2], float rot_mat[9], float camera_vec[3]);

/* ---- scenes ---------------------------------------------------------------------------------- */
/* LSVO<D>::LSVO(const SVO<D>&) (lsvo.hpp:12-24): upload a flattened octree in the reference layout.
 * `guard` = lower bound of the traversal loop `scale > MAX_DEPTH` (lsvo.hpp:72); pass 0 for the
 * reference expression (= depth). */
int vrt_lsvo_create(vrt_context* ctx, const vrt_lnode* nodes, uint64_t n_nodes, uint32_t depth, int32_t guard,
                    vrt_scene** out);
/* The demo scene T(depth), depth 8..12, built entirely on the device (FastNoise heights, the SVO::setCell fill
 * main.cpp:61-76 and compileSVO lsvo_utils.cpp:4-49 in one pass; byte-identical to vrt_host_build_terrain_lsvo and to
 * the reference's own array) — nothing crosses PCIe. */
int vrt_lsvo_create_terrain(vrt_context* ctx, uint32_t depth, int32_t guard, vrt_scene** out);
/* Dynamic scenes (SURVEY.md §8 f4; the reference's LSVO::setCell is a no-op, lsvo.hpp:26, so its world cannot change once
 * flattened).  A heightfield scene keeps its column heights resident on the device and is re-flattened there after an edit.
 *   heights[x * S + z], S = 2^depth (depth 5..12): column (x, z) is solid for y in [1, max(16, min(S/2, height))) stored
 *   at y + S/2 — the fill rule of main.cpp:70-76 (256 → S/2) wherever that rule stays inside the world (the reference's
 *   min(S, height) would write past it for height > S/2); NULL = the demo's FastNoise heights (main.cpp:61-68).
 * vrt_scene_edit_heights replaces the heights of the rectangle [x0, x0+nx) x [z0, z0+nz) (heights[i * nz + j] is column
 * (x0+i, z0+j)) and rebuilds the node array on the device: the result is byte-identical to flattening the edited world
 * from scratch (compileSVO order), so every cast and frame stays bit-exact.  Synchronises the context stream. */
/* The general form: the world is a set of voxels (SVO::setCell coordinates, svo.hpp:72), flattened on the device —
 * sorted path keys, DFS numbering by binary searches, no pointer octree (cpuvoxelraycaster_b200/csrc/voxel_build.cu); the
 * array is byte-identical to LSVO<D>(const SVO<D>&) over the same voxels.  The sorted keys stay resident:
 * vrt_scene_set_cells adds (solid != 0) or removes (solid == 0) voxels — what LSVO::setCell would do if it were not
 * a no-op (lsvo.hpp:26) — and re-flattens; duplicates and removals of absent voxels are ignored.  Both synchronise
 * the context stream. */
int vrt_lsvo_create_from_voxels(vrt_context* ctx, uint32_t depth, const uint32_t* xyz, uint64_t n_voxels, int32_t guard,
                                vrt_scene** out);
int vrt_scene_set_cells(vrt_scene* scene, const uint32_t* xyz, uint64_t n_voxels, int32_t solid);
int vrt_scene_voxel_count(const vrt_scene* scene, uint64_t* count);
int vrt_lsvo_create_heightfield(vrt_context* ctx, uint32_t depth, const int32_t* heights, int32_t guard, vrt_scene** out);
int vrt_scene_edit_heights(vrt_scene* scene, uint32_t x0, uint32_t z0, uint32_t nx, uint32_t nz, const int32_t* heights);
int vrt_scene_download_heights(vrt_scene* scene, int32_t* heights /* [S*S] */);
/* Per-voxel colours (extension, DESIGN.md §2).  A solid voxel's colour is the `color` byte of its leaf slot in the reference
 * layout (lsvo_utils.hpp:5-18): data[node + child_offset + slot] for the node and slot LSVO::getAtRayHit finds.  Unpainted
 * voxels keep LNode()'s 1.  Casts and textured frames never read it.  Accepted on scenes from vrt_lsvo_create,
 * vrt_lsvo_create_terrain and vrt_lsvo_create_from_voxels (VRT_ERR_UNSUPPORTED for heightfield, grid and SVO scenes); on a
 * voxel-set scene the colours survive vrt_scene_set_cells (added voxels get 1).
 * Sets the colour of solid voxels (xyz in SVO::setCell coordinates, svo.hpp:72).  Empty voxels are skipped; when a voxel
 * appears twice the last occurrence wins; *painted (may be NULL) = distinct solid voxels painted.  Synchronises the stream. */
int vrt_scene_paint_cells(vrt_scene* scene, const uint32_t* xyz, const uint8_t* colors, uint64_t n, uint64_t* painted);
/* out[i] = colour of voxel i, or -1 if it is empty. */
int vrt_scene_cell_colors(vrt_scene* scene, const uint32_t* xyz, uint64_t n, int16_t* out);
/* Device-side node layout of an LSVO scene (no reference counterpart; results are identical for both):
 *   0 = the reference's LNode array (default), 1 = compact breadth-first array of live nodes (8x smaller, built on the
 *   device on first use).  l2_persist != 0 additionally pins the front of the compact array (the top octree levels)
 *   in L2 through an access-policy window on the context's stream. */
int vrt_scene_set_layout(vrt_scene* scene, int32_t layout, int32_t l2_persist);
/* LSVO::data (lsvo.hpp:287): copy the scene's LNode array back to the host.  out == NULL → *count only. */
int vrt_scene_download_nodes(vrt_scene* scene, vrt_lnode* out, uint64_t cap, uint64_t* count);
/* Grid3D<X,Y,Z> (grid_3d.hpp:10-27): cell_types[(x*Y+y)*Z+z] = Cell::Type (0 = Empty).
 * mip_levels > 0 builds the MipmapGrid3D occupancy pyramid (results identical to Grid3D). */
int vrt_grid_create(vrt_context* ctx, const uint8_t* cell_types, int32_t X, int32_t Y, int32_t Z, int32_t mip_levels,
                    vrt_scene** out);
/* SVO<N> (svo.hpp:29) from a dense occupancy occ[(x*S+y)*S+z], S = 2^depth. */
int vrt_svo_create(vrt_context* ctx, const uint8_t* occ, uint32_t depth, vrt_scene** out);
int vrt_scene_destroy(vrt_scene* scene);
int vrt_scene_info(const vrt_scene* scene, int32_t* kind, uint32_t* depth, uint64_t* device_bytes);

/* ---- batched traversal ------------------------------------------------------------------------
 * Volumetric::castRay (volumetric.hpp:58) for n rays at once:
 *   LSVO<D>::castRay(position, d, ray_size_coef, ray_size_bias)  lsvo.hpp:33
 *   Grid3D::castRay(position, direction)                          grid_3d.hpp:35   (coef/bias ignored)
 *   SVO<N>::castRay(position, direction, max_iter)                svo.hpp:62       (vrt_cast_rays_svo)
 * origin/dir are xyz triples (n*3 floats).  Host variant copies in, runs, copies out, synchronises. */
int vrt_cast_rays(vrt_scene* scene, const float* origin, const float* dir, float ray_size_coef, float ray_size_bias,
                  uint64_t n, vrt_hit* out);
int vrt_cast_rays_device(vrt_scene* scene, const float* d_origin, const float* d_dir, float ray_size_coef,
                         float ray_size_bias, uint64_t n, vrt_hit* d_out);
int vrt_cast_rays_svo(vrt_scene* scene, const float* origin, const float* dir, uint32_t max_iter, uint64_t n,
                      vrt_hit* out);
/* Σ complexity over the rays of the most recent cast on this scene (valid after synchronisation). */
int vrt_scene_last_complexity(vrt_scene* scene, uint64_t* total);

/* ---- rendering ---------------------------------------------------------------------------------
 * Replaces the swarm lambda src/main.cpp:139-154 + RayCaster::renderRay (raycaster.hpp:67-92) +
 * Camera::getRay (camera_controller.hpp:34-49) + samples_to_image (raycaster.hpp:94-103). */
typedef struct vrt_camera {
    float position[3];     /* Camera::position, voxel units */
    float rot_mat[9];      /* Camera::rot_mat, column major */
    float fov;             /* Camera::fov */
    float aperture;        /* Camera::aperture */
    float focal_length;    /* Camera::focal_length */
} vrt_camera;

typedef struct vrt_render_params {
    int32_t width, height;       /* RayCaster::render_size */
    int32_t row_begin, row_end;  /* rows [begin,end) rendered by this call (multi-GPU slabs) */
    int32_t spp;                 /* renderRay passes per pixel in this call */
    int32_t sample_offset;       /* index of the first sample (spp batches) */
    uint32_t seed_lo, seed_hi;   /* Philox4x32-10 key (replaces the racy global xorshf96, utils.cpp:11-25) */
    float light_position[3];     /* RayCaster::light_position (normalised, main.cpp:126) */
    int32_t use_gi;              /* RayCaster::use_gi */
    int32_t gi_bounces;          /* 1 = reference; 2 = extension (DESIGN.md) */
    int32_t use_samples;         /* RayCaster::use_samples; 0 = the temporal blend, one sample per frame (spp must be 1) */
    int32_t accum_in;            /* vrt_render: 1 = `accum` holds earlier sums and is added to (progressive frames) */
    int32_t tile_step;           /* > 1: only 4-row tiles t (counted from row_begin) with t % tile_step == tile_index */
    int32_t tile_index;          /*      are rendered/resolved — the balanced multi-GPU row partition */
    float roughness;             /* blur of Cell::Mirror reflections (0 = perfect mirror) */
    int32_t max_bounds;          /* reflection depth, RayCaster::max_bounds = 4 (raycaster.hpp:277) */
    int32_t checker;             /* 0 = every pixel; 1 / 2 = the checkerboard of main.cpp:137,143 with
                                  * checker_board_offset 0 / 1: pixel (x,y) is rendered iff
                                  * (y - area_start(y)) % 2 == (x + offset) % 2; other pixels keep their value */
    int32_t checker_area_height; /* height of the reference's thread areas (RENDER_HEIGHT / area_count, main.cpp:132;
                                  * 135 in the demo): area_start(y) = y - y % area_height.  0 = one area (start 0) */
    int32_t mirror_y1;           /* LSVO scenes: 1 + y (castRay voxel coordinates) of the voxel layer whose TOP faces are
                                  * Cell::Mirror (cell.hpp:8) — the LSVO has one shared cell (lsvo.hpp:21-23), so mirrors are a rule:
                                  * e.g. the flat valley floors of the demo terrain.  A mirror hit reflects like on grid scenes
                                  * (roughness, max_bounds, tint 0.8 per bounce; DESIGN.md §2).  0 = no mirrors */
    int32_t autofocus;           /* 1 = LSVO scenes: focal length from the centre ray, cast on the device in front of the
                                  * frame (Camera::getClosestPoint camera_controller.hpp:56-60 + main.cpp:114-121:
                                  * distance * 2^depth, or 100 on a miss); cam->focal_length is ignored.  No host
                                  * round trip: the interactive loop stays asynchronous */
} vrt_render_params;

typedef struct vrt_render_stats {
    uint64_t rays[6];            /* primary, shadow, gi, gi-shadow, gi2, gi2-shadow */
    uint64_t complexity[6];      /* Σ HitPoint::complexity per class */
} vrt_render_stats;

/* Frames can be rendered from LSVO scenes (the reference's RayCaster: primary, sun shadow, GI, DOF) and from
 * Grid3D / MipmapGrid3D scenes (extension: primary, sun shadow, DOF and blurry mirror reflections off Cell::Mirror
 * cells; camera and light in voxel units; no GI).  See DESIGN.md §2.
 *
 * 16x16 RGB albedo textures, top-down rows: RayCaster::image_top / image_side (raycaster.hpp:53-54). */
int vrt_scene_set_textures(vrt_scene* scene, const uint8_t* top_rgb, const uint8_t* side_rgb);
/* LSVO scenes: while a palette is set, a sample's albedo is palette[colour of the voxel its camera ray hits] (the last,
 * non-mirror hit) instead of the texel; shadows, GI, mirror tint and rounding stay as they are.  Frames then need no
 * textures, the reference node layout and render_variant 0, 2 or 4 (VRT_ERR_UNSUPPORTED otherwise); vrt_shade_rays and
 * vrt_render_distributed honour it.  rgb = 256*3 bytes (entry c is the albedo of colour c); NULL = back to the textures. */
int vrt_scene_set_palette(vrt_scene* scene, const uint8_t* rgb);

/* d_accum: device uint32 [height*width*4] r,g,b,count sums (RayCaster::colors, raycaster.hpp:259; the
 * integer sums equal the reference's double accumulators exactly).  Rows outside [row_begin,row_end)
 * are not touched.  Enqueues on the context stream. */
int vrt_render_accumulate_device(vrt_scene* scene, const vrt_camera* cam, const vrt_render_params* p, uint32_t* d_accum);
/* samples_to_image (use_samples) or the 0.4/0.6 temporal blend against d_rgba's previous content. */
int vrt_render_resolve_device(vrt_scene* scene, const vrt_render_params* p, const uint32_t* d_accum, uint8_t* d_rgba);
/* Host-buffer frame (what RayCaster::render calls): uploads or clears the accumulator (accum_in),
 * renders rows, resolves, copies RGBA and — if accum != NULL — the accumulator back.
 * rgba: [height*width*4] uint8, in/out when !use_samples (previous frame of the temporal blend). */
int vrt_render(vrt_scene* scene, const vrt_camera* cam, const vrt_render_params* p, uint8_t* rgba, uint32_t* accum,
               vrt_render_stats* stats);
int vrt_scene_last_render_stats(vrt_scene* scene, vrt_render_stats* stats);
/* How many of the last frame's primary rays (they are counted in vrt_render_stats::rays[0], with complexity 0) were answered by the
 * beam search instead of a walk: samples of pixels whose beam tile has nothing in its frustum (context option "beam_tile",
 * vrt_beam_floors: floor 3.0) — such a camera ray misses whatever its lens sample, so the frame kernels do not start its chain.
 * No reference counterpart (there every castRay call walks, lsvo.hpp:72-146); 0 without beam floors. */
int vrt_scene_last_render_culled(vrt_scene* scene, uint64_t* primary_rays);
/* Diagnostic: the beam floors a frame with these parameters would use (context option "beam_tile"): out[ty * tiles_x + tx],
 * tiles_x = ceil(width / tile), for every tile of the frame — the distance (castRay units) below which no camera ray of the
 * tile (any pixel, any lens sample) can hit anything; 3.0 = nothing in the tile's frustum.  No reference counterpart. */
int vrt_beam_floors(vrt_scene* scene, const vrt_camera* cam, const vrt_render_params* p, int32_t tile, float* out);

/* RayCaster::castRay (raycaster.hpp:118-167) for explicit rays — the call the reference's per-pixel loop makes through
 * renderRay (raycaster.hpp:67-92) with the ray Camera::getRay produced (main.cpp:147-149): start and direction in the
 * normalised [1,2]^3 frame.  Returns each ray's ColorResult: the shaded 8-bit colour (texture, sun shadow, GI when
 * p->use_gi, with the Philox numbers of (pixel, sample)), hit flag, HitPoint::distance and complexity of the primary ray.
 * Only the shading fields of *p are read (light_position, use_gi, gi_bounces, seed); LSVO scenes.  This is the
 * compatibility path for hosts that keep the reference's loop structure — frames should use vrt_render. */
typedef struct vrt_shade_job {
    float start[3];
    uint32_t pixel;          /* RNG stream: y * width + x */
    float direction[3];
    uint32_t sample;         /* RNG stream: index of this sample of the pixel */
} vrt_shade_job;
typedef struct vrt_shade_result {
    uint8_t r, g, b, hit;    /* ColorResult::color; hit = the primary ray found a cell */
    float distance;          /* ColorResult::distance */
    uint32_t complexity;     /* RayContext::complexity */
    uint32_t reserved;
} vrt_shade_result;
int vrt_shade_rays(vrt_scene* scene, const vrt_render_params* p, uint64_t n, const vrt_shade_job* jobs, vrt_shade_result* out);

/* Presentation step of the main loop (main.cpp:159-177), fused into one kernel:
 *   frame'   = median filter of `frame` (median = 0: none; 3 / 5: per-channel 3x3 / 5x5 median, clamp to edge — what
 *              res/median_3.frag / res/median.frag compute; the reference ships them but never binds them)
 *   display  = min(255, mul8(display, c1) + mul8(frame', c2))       "Add some persistence to reduce the noise"
 * with c1 = uint8(255 * old_value_conservation), c2 = uint8(255 * (1 - old_value_conservation)) (main.cpp:160-165; the
 * demo uses 0.1 without samples, 0 with) and mul8(a, c) = (a * c + 127) / 255, the round-to-nearest product of two
 * 8-bit unorm values that sf::BlendMultiply / sf::BlendAdd leave in an RGBA8 render texture.  Alpha is set to 255.
 * d_frame and d_display are [height*width*4] uint8 device buffers and must not overlap. */
typedef struct vrt_present_params {
    int32_t width, height;
    int32_t median;                  /* 0, 3 or 5 */
    float old_value_conservation;    /* main.cpp:160 */
} vrt_present_params;
int vrt_present_device(vrt_context* ctx, const uint8_t* d_frame, uint8_t* d_display, const vrt_present_params* p);
/* The same with host buffers (display is in/out). */
int vrt_present(vrt_context* ctx, const uint8_t* frame, uint8_t* display, const vrt_present_params* p);
/* Camera::getClosestPoint + the focal-length rule of main.cpp:115-121. */
int vrt_autofocus(vrt_scene* scene, const vrt_camera* cam, float* focal_length);

/* ---- multi-GPU frames ----------------------------------------------------------------------------
 * Replaces the reference's only parallel decomposition of a frame — 16 swarm threads, one 4x4 screen area each
 * (src/main.cpp:139-143, swrm::Swarm src/main.cpp:90-92) — across the GPUs of one box.  The scene is replicated (one
 * vrt_scene per GPU); a frame is split over the members of a communicator either by 4-row tiles dealt round-robin
 * (VRT_SPLIT_TILES) or by samples (VRT_SPLIT_SAMPLES: every GPU renders all pixels for spp / world of the samples and the
 * integer accumulators are added up over NVLink — exact, so both splits give the byte-identical frame, identical to
 * the single-GPU frame).  No collective library is involved: the resolve kernel stores the finished RGBA pixels straight
 * into the delivery GPU's frame buffer through peer-mapped memory (cpuvoxelraycaster_b200/csrc/comm.cu).
 *
 * One member (vrt_comm) per GPU.  Two ways to form a communicator:
 *   (a) one process driving several GPUs (what the reference's main() would be): vrt_comm_create_local on an array of
 *       contexts, one per device (peer access is enabled between them);
 *   (b) one process per GPU: vrt_comm_create → vrt_comm_export (an opaque VRT_COMM_HANDLE_BYTES blob) → the caller
 *       all-gathers the blobs in rank order over whatever it has (MPI, torch.distributed, a file) → vrt_comm_connect
 *       (CUDA IPC).
 * Frames are delivered to rank 0 (or to every rank with deliver_all) into double-buffered device memory and, if
 * host_rgba is given on a receiving rank, copied to it on a second stream while the next frame renders.
 * vrt_render_distributed only enqueues; vrt_comm_frame_wait blocks until the last frame (and its host copy) is complete
 * and reports a peer that failed to show up.  Every member must call vrt_render_distributed for every frame with the
 * same camera, parameters and split; row_begin/row_end/tile_step/tile_index/accum_in of *p are ignored, sample_offset is
 * the index of the frame's first sample as in vrt_render. */
typedef struct vrt_comm vrt_comm;
#define VRT_COMM_HANDLE_BYTES 256
typedef enum vrt_split { VRT_SPLIT_TILES = 0, VRT_SPLIT_SAMPLES = 1 } vrt_split;
int vrt_comm_create_local(vrt_context* const* ctxs, int world, int width, int height, vrt_comm** out /* [world] */);
int vrt_comm_create(vrt_context* ctx, int rank, int world, int width, int height, vrt_comm** out);
int vrt_comm_export(vrt_comm* comm, void* blob /* VRT_COMM_HANDLE_BYTES */);
int vrt_comm_connect(vrt_comm* comm, const void* blobs /* world * VRT_COMM_HANDLE_BYTES, rank order */);
int vrt_comm_destroy(vrt_comm* comm);
int vrt_comm_info(const vrt_comm* comm, int* rank, int* world, uint64_t* frames);
int vrt_render_distributed(vrt_comm* comm, vrt_scene* scene, const vrt_camera* cam, const vrt_render_params* p, int split,
                           int deliver_all, uint8_t* host_rgba /* receiving ranks; may be NULL */);
int vrt_comm_frame_wait(vrt_comm* comm);
/* device address of the assembled frame (frames_ago = 0: the most recent, 1: the one before) on a receiving rank */
int vrt_comm_frame_device(vrt_comm* comm, int frames_ago, uint8_t** d_rgba);

#ifdef __cplusplus
}
#endif
#endif /* VRT_H */
