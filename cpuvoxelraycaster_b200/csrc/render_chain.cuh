// The per-sample ray chain of RayCaster — shared by the frame kernels K4 (render_kernels.cu) and K4p
// (persistent_kernels.cu).
//
//   chain_begin    Camera::getRay + the lens mapping                camera_controller.hpp:34-49, main.cpp:145-149
//   chain_advance  one ray of the chain has terminated: shade it and produce the next ray
//                  RayCaster::castRay / getGlobalIllumination         raycaster.hpp:118-207, texture lookup :209-240
//   chain_colour   the sample's 8-bit colour                          raycaster.hpp:161-163, utils.cpp:43-48
//
// A sample is a chain of up to six rays: primary, sun shadow, GI, GI shadow, second-bounce GI, its shadow.
// Arithmetic follows the cited lines op for op (fp32, no contraction); random numbers are Philox4x32-10 keyed by
// (pixel, sample, dimension) on getRand's 100-level lattice.
#pragma once
#include "kernels.h"
#include "lsvo_traverse.cuh"

namespace vrt {

enum Stage : int { kPrimary = 0, kShadow = 1, kGi0 = 2, kGi0Shadow = 3, kGi1 = 4, kGi1Shadow = 5, kDone = 6 };

struct ChainState {
    float nx, ny, nz;                // primary normal (raw ∓1/∓2/∓4, lsvo.hpp:149)
    float light;                     // light_intensity, raycaster.hpp:148,156
    float dot_gi0, dot_gi1;          // dot(gi_ray, normal) per bounce, :193
    float irr0, irr1;                // max(0, dot(gi normal, to_light)) of lit GI hits, :199-200
    float gnx, gny, gnz;             // normal of the current GI hit
    float gpx, gpy, gpz;             // hit point the next GI ray starts from (primary hit, then GI hit)
    float tlx, tly, tlz;             // unit vector to the light of the pending shadow ray
    uint32_t rnd_z, rnd_w;           // Philox words of dimensions 2,3 (GI bounce 1)
    uint8_t tex_r, tex_g, tex_b;     // albedo texel
    bool have_hit, gi0_hit, gi1_hit;
    // mirror reflections (extension, kMirror kernels only): reflections so far, and their accumulated tint
    float tint;
    int bounds;
    // point lights (extension, kPalette chains only): the light per channel, from the sun term on, and the light whose shadow
    // ray is in flight (-1: the sun's)
    float light_r, light_g, light_b;
    int light_i;
};

struct NextRay {
    float ox, oy, oz, dx, dy, dz, coef;
    float t_floor;   // conservative start distance (beam_kernels.cu): primary rays only, 0 for every other ray
};

// The beam floor of a camera ray of pixel (x, y) with direction d, or 0 when the launch has none.
// The tile's floor is lowered per ray by kPlaneSlack / min|d|: castRay computes the time at which a ray crosses a cell plane as
// p * (-1/|d|) - o * (-1/|d|) (lsvo.hpp:47-48,76) — for a direction component near zero the two products are huge and cancel, so
// which side of a plane the walk believes the ray to be on is uncertain within ~4e-7 of the plane, and a ray that runs
// nearly parallel to a plane stays inside that band for a stretch of 4e-7 / |d| in t.  Inside the band a walk that starts at
// t_floor can take the other side than the walk from 0 did, and then reports the hit cell's other face (measured on the
// oracle: ~1e-6 of the horizon rays at |d| < 1e-3, none once the start lies a band length before the hit —
// profiles/r02_summary.md).  Rays with a zero component get no floor at all.
constexpr float kPlaneSlack = 1.6e-5f;
__device__ __forceinline__ float beam_floor_of(const RenderLaunch& L, int x, int y, float dx, float dy, float dz) {
    if (!L.beam_floor) return 0.0f;
    const float tile_floor = __ldg(L.beam_floor + (y >> L.beam_shift) * L.beam_tiles_x + (x >> L.beam_shift));
    return fmaxf(0.0f, tile_floor - kPlaneSlack / fminf(fabsf(dx), fminf(fabsf(dy), fabsf(dz))));
}

__device__ __forceinline__ uint8_t mul_u8(uint8_t c, float f) {       // mult(sf::Color&, float), utils.cpp:43-48
    return uint8_t(fminf(255.0f, float(c) * f));
}

// v * rot_mat (camera_controller.hpp:51-54); m is column major
__device__ __forceinline__ void view_to_world(const float* m, float vx, float vy, float vz, float& x, float& y, float& z) {
    x = (m[0] * vx + m[1] * vy) + m[2] * vz;
    y = (m[3] * vx + m[4] * vy) + m[5] * vz;
    z = (m[6] * vx + m[7] * vy) + m[8] * vz;
}

// Starts sample `sample` of `pixel`: the primary ray.
__device__ __forceinline__ void chain_begin(const RenderLaunch& L, ChainState& c, uint32_t pixel, uint32_t sample, float lens_x,
                                            float lens_y, float SCALE, float focal_length, NextRay& nr) {
    const uint4 rnd0 = philox4x32_10(pixel, sample, 0u, 0u, L.seed_lo, L.seed_hi);
    c.rnd_z = rnd0.z; c.rnd_w = rnd0.w;
    c.light = 0.f; c.irr0 = 0.f; c.irr1 = 0.f;
    c.have_hit = false; c.gi0_hit = false; c.gi1_hit = false;
    c.tint = 1.0f; c.bounds = 0;
    const float u0 = lattice(rnd0.x, -0.5f, 0.5f), u1 = lattice(rnd0.y, -0.5f, 0.5f);    // camera_controller.hpp:40
    float fx = lens_x, fy = lens_y, fz = L.cam.fov;                                     // :37-39
    normalize3(fx, fy, fz);
    fx *= focal_length; fy *= focal_length; fz *= focal_length;
    const float rx = L.cam.aperture * u0, ry = L.cam.aperture * u1, rz = L.cam.aperture * 0.0f;
    float qx = fx - rx, qy = fy - ry, qz = fz - rz;                                     // :42
    normalize3(qx, qy, qz);
    float wx, wy, wz;
    view_to_world(L.cam.rot_mat, qx, qy, qz, nr.dx, nr.dy, nr.dz);
    view_to_world(L.cam.rot_mat, rx, ry, rz, wx, wy, wz);
    nr.ox = (L.cam.position[0] + wx) * SCALE + 1.0f;                                    // main.cpp:149
    nr.oy = (L.cam.position[1] + wy) * SCALE + 1.0f;
    nr.oz = (L.cam.position[2] + wz) * SCALE + 1.0f;
    nr.coef = 0.0f;
    nr.t_floor = 0.0f;
}

// tangent-plane noise of getGlobalIllumination (raycaster.hpp:178-190); false when the normal is all zero
// (noise_normal is uninitialised in the reference then: the ray started inside a solid cell)
__device__ __forceinline__ bool gi_noise(float nx, float ny, float nz, float c1, float c2, float& ax, float& ay, float& az) {
    if (nx != 0.0f) { ax = 0.0f; ay = c1; az = c2; return true; }
    if (ny != 0.0f) { ax = c1; ay = 0.0f; az = c2; return true; }
    if (nz != 0.0f) { ax = c1; ay = c2; az = 0.0f; return true; }
    return false;
}

// Word `dim & 3` of Philox block `dim >> 2` of the sample's stream, on getRand's lattice
__device__ __forceinline__ float lattice_dim(const RenderLaunch& L, uint32_t pixel, uint32_t sample, uint32_t dim, float lo, float hi) {
    const uint4 w = philox4x32_10(pixel, sample, dim >> 2, 0u, L.seed_lo, L.seed_hi);
    const uint32_t word = (dim & 3u) == 0u ? w.x : ((dim & 3u) == 1u ? w.y : ((dim & 3u) == 2u ? w.z : w.w));
    return lattice(word, lo, hi);
}

// Point light i as seen from the shadow origin o of a hit with raw normal n (DESIGN.md §2, "Point lights"): its distance, the
// unit vector t to it and dot(t, n).  t is glm::normalize's, and the distance shares its sum of squares.
__device__ __forceinline__ const float* point_light(const RenderLaunch& L, int i) {
    return reinterpret_cast<const float*>(L.tex_top + kLightsOffset + 4) + kPointLightFloats * i;
}
__device__ __forceinline__ float point_light_view(const float* pl, float ox, float oy, float oz, float nx, float ny, float nz,
                                                  float& tx, float& ty, float& tz, float& ndotl) {
    tx = __ldg(pl) - ox; ty = __ldg(pl + 1) - oy; tz = __ldg(pl + 2) - oz;
    const float dist = sqrtf(dot3(tx, ty, tz, tx, ty, tz));
    normalize3(tx, ty, tz);
    ndotl = dot3(tx, ty, tz, nx, ny, nz);
    return dist;
}

// The ray of stage `stage` ended with result (r, h).  Returns the next stage and, unless it is kDone, the next ray.
// kMirror: mirror reflections on LSVO frames (extension specified in oracle/port.c, shade_sample): the top faces of the voxel
// layer y = L.mirror_y1 - 1 are Cell::Mirror; a mirror hit re-enters kPrimary with the reflected, roughness-jittered ray.
// kPalette: L.palette's bits read the colour of the hit voxel from its leaf slot in `ref_nodes` (the reference layout; specified
// in tests/palette_oracle.c and tests/cell_types_oracle.c).  kPaletteAlbedo: the albedo of the final camera-chain hit is its
// palette entry.  kCellTypes: a hit on a voxel whose colour has type Cell::Mirror reflects on the face it hit (below).  The
// frame kernels have kPalette with kMirror: mirror_y1 = 0 matches no face, and without kCellTypes the tint stays 1.
// kPalette also carries the point lights (L.palette & kPointLights, specified in tests/point_lights_oracle.c): after the sun's
// shadow ray, kShadow hands out one shadow ray per light that passes its cast test, from the sun's origin, before GI starts.
template <bool kMirror = false, bool kPalette = kMirror>
__device__ __forceinline__ int chain_advance(const RenderLaunch& L, ChainState& c, int stage, const LsvoResult& r, const LsvoHit& h,
                                             uint32_t pixel, uint32_t sample, float SCALE, float n_norm, NextRay& nr,
                                             const uint2* __restrict__ ref_nodes = nullptr) {
    nr.t_floor = 0.0f;                                                     // only camera rays have a beam floor
    switch (stage) {
        case kPrimary: {                                                   // raycaster.hpp:131-145
            if (!r.hit) return kDone;
            // A camera-chain hit reflects when bounds < max_bounds and either rule holds: the lake (top faces of layer
            // mirror_y1 - 1) or, with kCellTypes, a voxel whose colour is Cell::Mirror hit on exactly one face.  Zero normals (a
            // ray that started inside a solid) and edge or corner hits do not reflect.
            const bool lake = kMirror && int((h.corner[1] - 1.0f) * float(1 << L.depth)) == L.mirror_y1 - 1 && h.normal[1] != 0.0f &&
                              h.normal[0] == 0.0f && h.normal[2] == 0.0f;
            uint32_t colour = 1u;
            // one descent per hit with cell types; without them only the final hit needs its colour (a lake hit is never final)
            if (kPalette && ((L.palette & kCellTypes) || ((L.palette & kPaletteAlbedo) && !(lake && c.bounds < L.max_bounds)))) {
                // castRay voxel v = setCell coordinate S-1-v, taken from the hit cell's corner like the lake test above
                const float S = float(1 << L.depth);
                const uint32_t S1 = (1u << L.depth) - 1u;
                const uint32_t slot = lsvo_leaf_slot(ref_nodes, L.depth, S1 - uint32_t(int((h.corner[0] - 1.0f) * S)),
                                                     S1 - uint32_t(int((h.corner[1] - 1.0f) * S)), S1 - uint32_t(int((h.corner[2] - 1.0f) * S)));
                if (slot != kNoLeafSlot) colour = __ldg(ref_nodes + slot).x & 0xffu;
            }
            if (kMirror || kPalette) {
                const int faces = int(h.normal[0] != 0.0f) + int(h.normal[1] != 0.0f) + int(h.normal[2] != 0.0f);
                const bool typed = kPalette && (L.palette & kCellTypes) && faces == 1 && __ldg(L.tex_top + kCellTypesOffset + colour) == 2;
                if (c.bounds < L.max_bounds && (lake || typed)) {
                    nr.ox = h.pos[0] + h.normal[0] * SCALE * 0.001f;
                    nr.oy = h.pos[1] + h.normal[1] * SCALE * 0.001f;
                    nr.oz = h.pos[2] + h.normal[2] * SCALE * 0.001f;
                    const uint32_t b = uint32_t(c.bounds);
                    const float r0 = lattice_dim(L, pixel, sample, 8u + 3u * b, -0.5f, 0.5f);
                    const float r1 = lattice_dim(L, pixel, sample, 9u + 3u * b, -0.5f, 0.5f);
                    const float r2 = lattice_dim(L, pixel, sample, 10u + 3u * b, -0.5f, 0.5f);
                    // the component on the normal's one axis is negated (the lake's normal lies along y)
                    nr.dx = (h.normal[0] != 0.0f ? -nr.dx : nr.dx) + L.roughness * r0;
                    nr.dy = (h.normal[1] != 0.0f ? -nr.dy : nr.dy) + L.roughness * r1;
                    nr.dz = (h.normal[2] != 0.0f ? -nr.dz : nr.dz) + L.roughness * r2;
                    normalize3(nr.dx, nr.dy, nr.dz);
                    nr.coef = 0.0f;
                    c.tint = c.tint * 0.8f;
                    ++c.bounds;
                    return kPrimary;
                }
            }
            c.have_hit = true;
            c.nx = h.normal[0]; c.ny = h.normal[1]; c.nz = h.normal[2];
            if (kPalette && (L.palette & kPaletteAlbedo)) {
                const uint8_t* entry = L.tex_top + kPaletteOffset + 3u * colour;
                c.tex_r = __ldg(entry); c.tex_g = __ldg(entry + 1); c.tex_b = __ldg(entry + 2);
            } else {
                const uint8_t* tex = (c.ny != 0.0f) ? L.tex_top : L.tex_side;  // :211-215
                const float u = fminf(fmaxf(h.uv[0], 0.0f), 1.0f), v = fminf(fmaxf(h.uv[1], 0.0f), 1.0f);   // :237-238
                const uint32_t tx = uint32_t(16.0f * u), ty = uint32_t(16.0f * v);                          // :239
                const uint8_t* texel = tex + 3u * (ty * 16u + tx);
                c.tex_r = __ldg(texel); c.tex_g = __ldg(texel + 1); c.tex_b = __ldg(texel + 2);
            }
            c.gpx = h.pos[0]; c.gpy = h.pos[1]; c.gpz = h.pos[2];         // the GI stage starts from the primary hit
            nr.ox = h.pos[0] + c.nx * SCALE * 0.001f;                      // sun shadow ray, :139
            nr.oy = h.pos[1] + c.ny * SCALE * 0.001f;
            nr.oz = h.pos[2] + c.nz * SCALE * 0.001f;
            c.tlx = L.light[0] - nr.ox; c.tly = L.light[1] - nr.oy; c.tlz = L.light[2] - nr.oz;   // :152
            normalize3(c.tlx, c.tly, c.tlz);
            nr.dx = c.tlx; nr.dy = c.tly; nr.dz = c.tlz; nr.coef = 0.0f;
            if (kPalette) c.light_i = -1;
            return kShadow;
        }
        case kShadow: {                                                    // :155-157
            if (kPalette && c.light_i >= 0) {
                // the shadow ray of point light light_i returned: it still holds the origin and direction of the light's cast
                // test, from which distance and dot(t, n) are computed again (the same operations, so the same bits).  A hit
                // beyond the light does not shadow it.
                const float* pl = point_light(L, c.light_i);
                float tx, ty, tz, ndotl;
                const float dist = point_light_view(pl, nr.ox, nr.oy, nr.oz, c.nx, c.ny, c.nz, tx, ty, tz, ndotl);
                if (!(r.hit && r.t_min < dist)) {
                    const float w = 1.0f - dist / __ldg(pl + 6);
                    c.light_r = c.light_r + (__ldg(pl + 3) * ndotl) * w;
                    c.light_g = c.light_g + (__ldg(pl + 4) * ndotl) * w;
                    c.light_b = c.light_b + (__ldg(pl + 5) * ndotl) * w;
                }
            } else if (kPalette) {                                         // the sun starts the sums (c.light stays unused)
                c.light_r = r.hit ? 0.0f : fmaxf(0.0f, dot3(c.tlx, c.tly, c.tlz, c.nx, c.ny, c.nz));
                c.light_g = c.light_r; c.light_b = c.light_r;
            } else {
                if (!r.hit) c.light = fmaxf(0.0f, dot3(c.tlx, c.tly, c.tlz, c.nx, c.ny, c.nz));
            }
            if (kPalette && (L.palette & kPointLights)) {
                // the next light in index order that passes the cast test: in range and in front of the face.  A zero normal,
                // or a light at the origin (NaN), fails it.
                const int n_lights = int(__ldg(reinterpret_cast<const uint32_t*>(L.tex_top + kLightsOffset)));
                for (int i = c.light_i + 1; i < n_lights; ++i) {
                    const float* pl = point_light(L, i);
                    float tx, ty, tz, ndotl;
                    const float dist = point_light_view(pl, nr.ox, nr.oy, nr.oz, c.nx, c.ny, c.nz, tx, ty, tz, ndotl);
                    if (dist < __ldg(pl + 6) && ndotl > 0.0f) {
                        nr.dx = tx; nr.dy = ty; nr.dz = tz;                // origin and coef 0 stay the sun shadow ray's
                        c.light_i = i;
                        return kShadow;
                    }
                }
            }
            if (!L.use_gi) return kDone;
            // getGlobalIllumination, first bounce, :169-194 — from the primary hit
            const float c1 = lattice(c.rnd_z, -1000.0f, 1000.0f), c2 = lattice(c.rnd_w, -1000.0f, 1000.0f);   // :180-181
            float ax, ay, az;
            if (!gi_noise(c.nx, c.ny, c.nz, c1, c2, ax, ay, az)) return kDone;
            nr.ox = c.gpx + c.nx * n_norm; nr.oy = c.gpy + c.ny * n_norm; nr.oz = c.gpz + c.nz * n_norm;   // :174
            nr.dx = (c.nx + ax) * n_norm; nr.dy = (c.ny + ay) * n_norm; nr.dz = (c.nz + az) * n_norm;       // :192
            normalize3(nr.dx, nr.dy, nr.dz);
            c.dot_gi0 = dot3(nr.dx, nr.dy, nr.dz, c.nx, c.ny, c.nz);      // :193
            nr.coef = 0.5f;
            return kGi0;
        }
        case kGi0:
        case kGi1: {                                                       // :194-198
            if (!r.hit) return kDone;
            if (stage == kGi0) c.gi0_hit = true; else c.gi1_hit = true;
            c.gnx = h.normal[0]; c.gny = h.normal[1]; c.gnz = h.normal[2];
            c.gpx = h.pos[0]; c.gpy = h.pos[1]; c.gpz = h.pos[2];
            nr.ox = c.gpx + c.gnx * n_norm; nr.oy = c.gpy + c.gny * n_norm; nr.oz = c.gpz + c.gnz * n_norm;   // :196
            c.tlx = L.light[0] - nr.ox; c.tly = L.light[1] - nr.oy; c.tlz = L.light[2] - nr.oz;               // :197
            normalize3(c.tlx, c.tly, c.tlz);
            nr.dx = c.tlx; nr.dy = c.tly; nr.dz = c.tlz; nr.coef = 0.5f;
            return stage + 1;
        }
        case kGi0Shadow: {                                                 // :199-200
            if (!r.hit) c.irr0 = fmaxf(0.0f, dot3(c.gnx, c.gny, c.gnz, c.tlx, c.tly, c.tlz));
            if (L.gi_bounces < 2) return kDone;
            // second bounce (extension, DESIGN.md §2): the same estimator from the GI hit, dimensions 4,5
            const uint4 rnd1 = philox4x32_10(pixel, sample, 1u, 0u, L.seed_lo, L.seed_hi);
            const float c1 = lattice(rnd1.x, -1000.0f, 1000.0f), c2 = lattice(rnd1.y, -1000.0f, 1000.0f);
            float ax, ay, az;
            if (!gi_noise(c.gnx, c.gny, c.gnz, c1, c2, ax, ay, az)) return kDone;
            nr.ox = c.gpx + c.gnx * n_norm; nr.oy = c.gpy + c.gny * n_norm; nr.oz = c.gpz + c.gnz * n_norm;
            nr.dx = (c.gnx + ax) * n_norm; nr.dy = (c.gny + ay) * n_norm; nr.dz = (c.gnz + az) * n_norm;
            normalize3(nr.dx, nr.dy, nr.dz);
            c.dot_gi1 = dot3(nr.dx, nr.dy, nr.dz, c.gnx, c.gny, c.gnz);
            nr.coef = 0.5f;
            return kGi1;
        }
        case kGi1Shadow: {
            if (!r.hit) c.irr1 = fmaxf(0.0f, dot3(c.gnx, c.gny, c.gnz, c.tlx, c.tly, c.tlz));
            return kDone;
        }
        default: return kDone;
    }
}

// Adds the finished sample's colour (raycaster.hpp:161-163) to the pixel sums (:87-90).
template <bool kMirror = false>
__device__ __forceinline__ void chain_colour(const RenderLaunch& L, const ChainState& c, uint32_t& sum_r, uint32_t& sum_g, uint32_t& sum_b) {
    if (!c.have_hit) return;                                               // ColorResult stays Black, :38
    float gi = 0.0f;
    if (L.use_gi && c.gi0_hit) {
        float irr = c.irr0;
        if (L.gi_bounces >= 2) irr = irr + (c.gi1_hit ? fminf(0.5f, c.irr1 * c.dot_gi1) : 0.0f);
        gi = fmaxf(0.0f, 1000000.0f * fminf(0.5f, irr * c.dot_gi0) / 1.0f);   // :201,:206
    }
    if (kMirror) {                                                         // :163 per channel: the point lights are coloured
        const float fr = fminf(1.0f, fmaxf(0.0f, c.light_r + gi)), fg = fminf(1.0f, fmaxf(0.0f, c.light_g + gi)),
                    fb = fminf(1.0f, fmaxf(0.0f, c.light_b + gi));
        sum_r += mul_u8(mul_u8(c.tex_r, fr), c.tint); sum_g += mul_u8(mul_u8(c.tex_g, fg), c.tint); sum_b += mul_u8(mul_u8(c.tex_b, fb), c.tint);
    } else {
        const float f = fminf(1.0f, fmaxf(0.0f, c.light + gi));            // :163
        sum_r += mul_u8(c.tex_r, f); sum_g += mul_u8(c.tex_g, f); sum_b += mul_u8(c.tex_b, f);
    }
}

}  // namespace vrt
