// vrt.hpp — C++ drop-in classes for the reference's per-pixel hot path, implemented on libvrt's C ABI.
//
// Same class names, member names and call signatures as johnBuffer/CpuVoxelRaycaster so that the
// reference's main.cpp keeps compiling with `#include <vrt/vrt.hpp>` in place of its own headers:
//
//   Cell                     include/cell.hpp:3-24
//   HitPoint, Volumetric     include/volumetric.hpp:7-22,55-61
//   SVO<N>                   include/svo.hpp:29         (setCell :72, castRay :62 — hit fill restored)
//   LSVO<D>                  include/lsvo.hpp:10        (ctor from SVO :12, castRay :33, setCell no-op :26)
//   Grid3D<X,Y,Z>            include/grid_3d.hpp:10     (castRay :16, setCell :18, getCellAt :20)
//   MipmapGrid3D<X,Y,Z,L>    include/mipmap_grid3D.hpp:14 (a stub in the reference; Grid3D results here)
//   Camera                   include/camera_controller.hpp:16-61
//   RayCaster                include/raycaster.hpp:43   (setLightPosition :62, samples_to_image :94,
//                                                        resetSamples :105, use_gi/use_samples/... :269-282)
//
// What changes for the caller: a single-ray castRay() is one tiny kernel launch, so hot loops should use
// the batched castRays(); and the swarm lambda of src/main.cpp:139-154 (one renderRay per pixel from
// 16 threads) becomes ONE call, RayCaster::render(camera).  There is no CPU fallback: every cast needs a
// CUDA device and throws vrt::Error otherwise.
//
// glm: the reference passes glm::vec3; if <glm/glm.hpp> is on the include path it is used, otherwise a
// minimal glm::vec2/vec3/mat3 with the same layout is provided so this header is self-contained.
#pragma once
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "../vrt.h"

#if defined(__has_include)
#if __has_include(<glm/glm.hpp>)
#include <glm/glm.hpp>
#define VRT_HAVE_GLM 1
#endif
#endif
#ifndef VRT_HAVE_GLM
namespace glm {
struct vec2 { float x = 0, y = 0; vec2() {} explicit vec2(float s) : x(s), y(s) {} vec2(float a, float b) : x(a), y(b) {} };
struct vec3 {
    float x = 0, y = 0, z = 0;
    vec3() {}
    explicit vec3(float s) : x(s), y(s), z(s) {}
    vec3(float a, float b, float c) : x(a), y(b), z(c) {}
    vec3(const vec2& v, float c) : x(v.x), y(v.y), z(c) {}
};
inline vec2 operator*(float s, const vec2& a) { return vec2(s * a.x, s * a.y); }
inline vec2 operator+(const vec2& a, const vec2& b) { return vec2(a.x + b.x, a.y + b.y); }
inline float dot(const vec3& a, const vec3& b);
inline vec3 normalize(const vec3& v);
inline vec3 operator+(const vec3& a, const vec3& b) { return vec3(a.x + b.x, a.y + b.y, a.z + b.z); }
inline vec3 operator-(const vec3& a, const vec3& b) { return vec3(a.x - b.x, a.y - b.y, a.z - b.z); }
inline vec3 operator*(const vec3& a, float s) { return vec3(a.x * s, a.y * s, a.z * s); }
inline vec3 operator*(float s, const vec3& a) { return vec3(s * a.x, s * a.y, s * a.z); }
struct mat3 { vec3 c[3]; vec3& operator[](int i) { return c[i]; } const vec3& operator[](int i) const { return c[i]; } };
inline float dot(const vec3& a, const vec3& b) { return (a.x * b.x + a.y * b.y) + a.z * b.z; }                  // glm: (x + y) + z
inline vec3 normalize(const vec3& v) { const float inv = 1.0f / std::sqrt(dot(v, v)); return vec3(v.x * inv, v.y * inv, v.z * inv); }
inline vec3 operator*(const vec3& v, const mat3& m) { return vec3(dot(m[0], v), dot(m[1], v), dot(m[2], v)); }   // row vector x matrix
}  // namespace glm
#endif

namespace vrt {

struct Error : std::runtime_error {
    int code;
    Error(int c, const std::string& m) : std::runtime_error("libvrt error " + std::to_string(c) + ": " + m), code(c) {}
};
inline void check(int status) {
    if (status != VRT_OK) throw Error(status, vrt_last_error());
}

// Philox4x32-10 (Salmon et al. 2011) on the host: the counter-based generator the device uses, for the host-side calls
// that draw random numbers in the reference (Camera::getRay, getGlobalIllumination through getRand, utils.cpp:77-81).
inline void philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1) {
    for (int r = 0; r < 10; ++r) {
        const uint64_t p0 = uint64_t(0xD2511F53u) * c[0], p1 = uint64_t(0xCD9E8D57u) * c[2];
        const uint32_t n0 = uint32_t(p1 >> 32) ^ c[1] ^ k0, n2 = uint32_t(p0 >> 32) ^ c[3] ^ k1;
        c[0] = n0; c[1] = uint32_t(p1); c[2] = n2; c[3] = uint32_t(p0);
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
}
struct HostRng {                       // one stream per thread; deterministic per thread, never shared (the reference's is racy)
    uint64_t counter = 0;
    uint32_t block[4] = {0, 0, 0, 0};
    int left = 0;
    uint32_t next() {
        if (!left) {
            block[0] = uint32_t(counter); block[1] = uint32_t(counter >> 32); block[2] = 0x68E31DA4u; block[3] = 0;
            philox4x32_10(block, 0x5EEDu, 0u);
            ++counter;
            left = 4;
        }
        return block[--left];
    }
};
inline HostRng& host_rng() { static thread_local HostRng r; return r; }

// One device + stream shared by every drop-in object of the process (replaces swrm::Swarm, main.cpp:90-92).
inline vrt_context* default_context(int device = 0) {
    struct Holder {
        vrt_context* ctx = nullptr;
        ~Holder() { /* scenes may outlive static destruction order: leave the context to process exit */ }
    };
    static Holder h;
    if (!h.ctx) check(vrt_context_create(device, nullptr, &h.ctx));
    return h.ctx;
}

struct SceneHandle {
    vrt_scene* s = nullptr;
    SceneHandle() {}
    SceneHandle(const SceneHandle&) = delete;
    SceneHandle& operator=(const SceneHandle&) = delete;
    ~SceneHandle() { if (s) vrt_scene_destroy(s); }
};

}  // namespace vrt

// ---- include/utils.hpp:19 / src/utils.cpp:77-81: min + (max - min) * (float(rnd % 100) / 100) -----------------------
inline float getRand(float min = -0.5f, float max = 0.5f) {
    const float rand_val = float(vrt::host_rng().next() % 100u) / 100.0f;
    return min + (max - min) * rand_val;
}

// ---- include/cell.hpp -----------------------------------------------------------------------------------
struct Cell {
    enum Type { Empty, Solid, Mirror };
    enum Texture { None, Grass, Red, White };
    Cell() : type(Type::Empty), texture(Texture::None) {}
    Type type;
    Texture texture;
};

// ---- include/volumetric.hpp ---------------------------------------------------------------------------
struct HitPoint {
    HitPoint() : cell(nullptr), distance(0.0f), complexity(0u) {}
    glm::vec3 position;
    glm::vec3 normal;
    glm::vec2 voxel_coord;
    const Cell* cell;
    float distance;
    uint32_t complexity;
};

class Volumetric {
public:
    virtual ~Volumetric() {}
    virtual HitPoint castRay(const glm::vec3& position, glm::vec3 direction, const float ray_size_coef,
                             const float ray_size_bias) const = 0;
    virtual void setCell(Cell::Type type, Cell::Texture texture, uint32_t x, uint32_t y, uint32_t z) = 0;
    // batched form (addition): n rays in, n HitPoints out, one kernel launch
    virtual std::vector<HitPoint> castRays(const std::vector<glm::vec3>& positions, const std::vector<glm::vec3>& directions,
                                           float ray_size_coef = 0.0f, float ray_size_bias = 0.0f) const = 0;
    virtual vrt_scene* scene() const = 0;
};

namespace vrt {
inline HitPoint to_hitpoint(const vrt_hit& h, const Cell* cell) {
    HitPoint p;
    p.complexity = h.complexity;
    if (h.flags & VRT_HIT_FLAG_HIT) {
        p.cell = cell;
        p.position = glm::vec3(h.position[0], h.position[1], h.position[2]);
        p.normal = glm::vec3(h.normal[0], h.normal[1], h.normal[2]);
        p.voxel_coord = glm::vec2(h.voxel_coord[0], h.voxel_coord[1]);
        p.distance = h.distance;
    }
    return p;
}
inline void flatten(const std::vector<glm::vec3>& v, std::vector<float>& out) {
    out.resize(v.size() * 3);
    for (size_t i = 0; i < v.size(); ++i) { out[3 * i] = v[i].x; out[3 * i + 1] = v[i].y; out[3 * i + 2] = v[i].z; }
}
}  // namespace vrt

// ---- include/svo.hpp --------------------------------------------------------------------------------------
// The reference grows a pointer octree voxel by voxel (80-byte nodes).  Here setCell only records the voxel;
// the octree is flattened when an LSVO is constructed from it, or packed to bits for SVO::castRay.
template <uint8_t N>
class SVO {
public:
    SVO() {}
    void setCell(Cell::Type type, Cell::Texture texture, uint32_t x, uint32_t y, uint32_t z) {
        if (x >= (1u << N) || y >= (1u << N) || z >= (1u << N)) throw vrt::Error(VRT_ERR_INVALID, "SVO::setCell: voxel out of range");
        (void)type; (void)texture;                     // every leaf of the demo is Solid/Grass (main.cpp:73)
        voxels.push_back(x); voxels.push_back(y); voxels.push_back(z);
        m_dirty = true;
    }
    // svo.hpp:62 — position in voxel units
    HitPoint castRay(const glm::vec3& position, const glm::vec3& direction, const uint32_t max_iter) const {
        static_assert(N <= 10, "SVO::castRay packs a dense occupancy: depth <= 10");
        ensure_scene();
        const float o[3] = {position.x, position.y, position.z}, d[3] = {direction.x, direction.y, direction.z};
        vrt_hit h;
        vrt::check(vrt_cast_rays_svo(m_scene->s, o, d, max_iter, 1, &h));
        return vrt::to_hitpoint(h, &m_cell);
    }
    std::vector<uint32_t> voxels;                      // xyz triples in setCell order

private:
    void ensure_scene() const {
        if (m_scene && !m_dirty) return;
        const size_t S = size_t(1) << N;
        std::vector<uint8_t> occ(S * S * S, 0);
        for (size_t i = 0; i + 2 < voxels.size(); i += 3) occ[(size_t(voxels[i]) * S + voxels[i + 1]) * S + voxels[i + 2]] = 1;
        m_scene.reset(new vrt::SceneHandle());
        vrt::check(vrt_svo_create(vrt::default_context(), occ.data(), N, &m_scene->s));
        m_dirty = false;
    }
    mutable std::unique_ptr<vrt::SceneHandle> m_scene;
    mutable bool m_dirty = true;
    Cell m_cell = solid_grass();
    static Cell solid_grass() { Cell c; c.type = Cell::Solid; c.texture = Cell::Grass; return c; }
};

// ---- include/lsvo.hpp -------------------------------------------------------------------------------------
template <uint8_t MAX_DEPTH>
struct LSVO : public Volumetric {
    LSVO(const SVO<MAX_DEPTH>& svo) { importFromSVO(svo); }
    // extension: adopt an already flattened octree (e.g. vrt_host_build_terrain_lsvo for 2048^3 and up)
    explicit LSVO(std::vector<vrt_lnode> nodes, int32_t guard = 0) : data(std::move(nodes)) { upload(guard); }

    void importFromSVO(const SVO<MAX_DEPTH>& svo) {                       // lsvo.hpp:18-24
        uint64_t n = 0;
        const uint64_t nv = svo.voxels.size() / 3;
        vrt::check(vrt_host_build_lsvo_from_voxels(MAX_DEPTH, svo.voxels.data(), nv, nullptr, 0, &n));
        data.resize(n);
        vrt::check(vrt_host_build_lsvo_from_voxels(MAX_DEPTH, svo.voxels.data(), nv, data.data(), n, &n));
        upload(0);
    }
    void setCell(Cell::Type, Cell::Texture, uint32_t, uint32_t, uint32_t) override {}   // lsvo.hpp:26

    HitPoint castRay(const glm::vec3& position, glm::vec3 d, const float ray_size_coef = 0.0f,
                     const float ray_size_bias = 0.0f) const override {          // lsvo.hpp:33
        const float o[3] = {position.x, position.y, position.z}, dir[3] = {d.x, d.y, d.z};
        vrt_hit h;
        vrt::check(vrt_cast_rays(m_scene.s, o, dir, ray_size_coef, ray_size_bias, 1, &h));
        return vrt::to_hitpoint(h, cell);
    }
    std::vector<HitPoint> castRays(const std::vector<glm::vec3>& positions, const std::vector<glm::vec3>& directions,
                                   float ray_size_coef = 0.0f, float ray_size_bias = 0.0f) const override {
        if (positions.size() != directions.size()) throw vrt::Error(VRT_ERR_INVALID, "castRays: size mismatch");
        std::vector<float> o, d;
        vrt::flatten(positions, o);
        vrt::flatten(directions, d);
        std::vector<vrt_hit> h(positions.size());
        vrt::check(vrt_cast_rays(m_scene.s, o.data(), d.data(), ray_size_coef, ray_size_bias, h.size(), h.data()));
        std::vector<HitPoint> out(h.size());
        for (size_t i = 0; i < h.size(); ++i) out[i] = vrt::to_hitpoint(h[i], cell);
        return out;
    }
    vrt_scene* scene() const override { return m_scene.s; }

    // lsvo.hpp:174-285: the node whose leaf child the ray hits (castRay without the cone), or nullptr on a miss.
    // The ray is cast on the device; the node is then found by walking `data` along the hit voxel's path.
    vrt_lnode* getAtRayHit(const glm::vec3& position, glm::vec3 d) {
        const float o[3] = {position.x, position.y, position.z}, dir[3] = {d.x, d.y, d.z};
        vrt_hit h;
        vrt::check(vrt_cast_rays(m_scene.s, o, dir, 0.0f, 0.0f, 1, &h));
        if (!(h.flags & VRT_HIT_FLAG_HIT)) return nullptr;
        const uint32_t S1 = (1u << MAX_DEPTH) - 1u;
        uint64_t node = 0;
        for (int level = int(MAX_DEPTH) - 1; level >= 0; --level) {          // child slot = bits of the mirrored coordinate (lsvo.hpp:79)
            const uint32_t slot = (((S1 - uint32_t(h.voxel[0])) >> level) & 1u) | ((((S1 - uint32_t(h.voxel[1])) >> level) & 1u) << 1) |
                                  ((((S1 - uint32_t(h.voxel[2])) >> level) & 1u) << 2);
            const vrt_lnode& n = data[node];
            if (!((n.child_mask >> slot) & 1u)) return nullptr;
            if ((n.leaf_mask >> slot) & 1u) return &data[node];
            node += n.child_offset + slot;
        }
        return nullptr;
    }

    // Per-voxel colours (extension; the reference sets LNode::color to 1 and never reads it).  xyz: SVO::setCell triples.
    // Paints the solid voxels (empty ones are skipped, the last occurrence of a voxel wins) and refreshes `data`, so that
    // data[] and getAtRayHit show the colours.  Returns the number of distinct solid voxels painted.
    uint64_t paintCells(const std::vector<uint32_t>& xyz, const std::vector<uint8_t>& colors) {
        if (xyz.size() != 3 * colors.size()) throw vrt::Error(VRT_ERR_INVALID, "paintCells: one colour per xyz triple");
        uint64_t painted = 0;
        vrt::check(vrt_scene_paint_cells(m_scene.s, xyz.data(), colors.data(), colors.size(), &painted));
        uint64_t n = data.size();
        vrt::check(vrt_scene_download_nodes(m_scene.s, data.data(), data.size(), &n));
        return painted;
    }
    // colour of each voxel, -1 where it is empty
    std::vector<int16_t> getCellColors(const std::vector<uint32_t>& xyz) const {
        std::vector<int16_t> out(xyz.size() / 3);
        vrt::check(vrt_scene_cell_colors(m_scene.s, xyz.data(), out.size(), out.data()));
        return out;
    }
    // frames take the albedo of colour c from rgb[3c..3c+2] (256 entries) instead of the textures, until clearPalette()
    void setPalette(const uint8_t rgb[768]) { vrt::check(vrt_scene_set_palette(m_scene.s, rgb)); }
    void clearPalette() { vrt::check(vrt_scene_set_palette(m_scene.s, nullptr)); }

    std::vector<vrt_lnode> data;                        // LNode[] in the reference layout (lsvo.hpp:287)
    const vrt_lnode* raw_data = nullptr;                // lsvo.hpp:288
    Cell* cell = nullptr;                               // the one shared Solid/Grass cell (lsvo.hpp:21-23,289)

private:
    void upload(int32_t guard) {
        raw_data = data.data();
        m_cell.type = Cell::Solid;
        m_cell.texture = Cell::Grass;
        cell = &m_cell;
        vrt::check(vrt_lsvo_create(vrt::default_context(), data.data(), data.size(), MAX_DEPTH, guard, &m_scene.s));
    }
    Cell m_cell;
    vrt::SceneHandle m_scene;
};

// ---- include/grid_3d.hpp / include/mipmap_grid3D.hpp ------------------------------------------------
template <int32_t X, int32_t Y, int32_t Z, int32_t MipLevels = 0>
class Grid3DBase : public Volumetric {
public:
    Grid3DBase() : m_types(size_t(X) * Y * Z, 0), m_cells(1) {}
    // grid_3d.hpp:16 (2-argument form; the 4-argument Volumetric form ignores the cone)
    HitPoint castRay(const glm::vec3& position, const glm::vec3& direction) const { return castRay(position, direction, 0.0f, 0.0f); }
    HitPoint castRay(const glm::vec3& position, glm::vec3 direction, const float, const float) const override {
        ensure_scene();
        const float o[3] = {position.x, position.y, position.z}, d[3] = {direction.x, direction.y, direction.z};
        vrt_hit h;
        vrt::check(vrt_cast_rays(m_scene->s, o, d, 0.0f, 0.0f, 1, &h));
        return hit(h);
    }
    std::vector<HitPoint> castRays(const std::vector<glm::vec3>& positions, const std::vector<glm::vec3>& directions, float = 0.0f,
                                   float = 0.0f) const override {
        ensure_scene();
        std::vector<float> o, d;
        vrt::flatten(positions, o);
        vrt::flatten(directions, d);
        std::vector<vrt_hit> h(positions.size());
        vrt::check(vrt_cast_rays(m_scene->s, o.data(), d.data(), 0.0f, 0.0f, h.size(), h.data()));
        std::vector<HitPoint> out(h.size());
        for (size_t i = 0; i < h.size(); ++i) out[i] = hit(h[i]);
        return out;
    }
    void setCell(Cell::Type type, uint32_t x, uint32_t y, uint32_t z) {   // grid_3d.hpp:18
        if (x >= uint32_t(X) || y >= uint32_t(Y) || z >= uint32_t(Z)) throw vrt::Error(VRT_ERR_INVALID, "Grid3D::setCell: out of range");
        m_types[(size_t(x) * Y + y) * Z + z] = uint8_t(type);
        m_dirty = true;
    }
    void setCell(Cell::Type type, Cell::Texture, uint32_t x, uint32_t y, uint32_t z) override { setCell(type, x, y, z); }
    Cell getCellAt(const glm::vec3& position) const {                     // grid_3d.hpp:20
        Cell c;
        c.type = Cell::Type(m_types[(size_t(int(position.x)) * Y + size_t(int(position.y))) * Z + size_t(int(position.z))]);
        return c;
    }
    vrt_scene* scene() const override { ensure_scene(); return m_scene->s; }

private:
    HitPoint hit(const vrt_hit& h) const {
        if (!(h.flags & VRT_HIT_FLAG_HIT)) return vrt::to_hitpoint(h, nullptr);
        // the reference returns a pointer into m_cells; one Cell per distinct type is enough to carry it
        const uint8_t t = m_types[(size_t(h.voxel[0]) * Y + size_t(h.voxel[1])) * Z + size_t(h.voxel[2])];
        if (m_cells.size() < 3) { m_cells.resize(3); for (int i = 0; i < 3; ++i) m_cells[i].type = Cell::Type(i); }
        return vrt::to_hitpoint(h, &m_cells[t < 3 ? t : 1]);
    }
    void ensure_scene() const {
        if (m_scene && !m_dirty) return;
        m_scene.reset(new vrt::SceneHandle());
        vrt::check(vrt_grid_create(vrt::default_context(), m_types.data(), X, Y, Z, MipLevels, &m_scene->s));
        m_dirty = false;
    }
    std::vector<uint8_t> m_types;                       // Cell::Type per cell (the reference keeps 8-byte Cells)
    mutable std::vector<Cell> m_cells;
    mutable std::unique_ptr<vrt::SceneHandle> m_scene;
    mutable bool m_dirty = true;
};
template <int32_t X, int32_t Y, int32_t Z> using Grid3D = Grid3DBase<X, Y, Z, 0>;
template <int32_t X, int32_t Y, int32_t Z, uint32_t MipmapDepth> using MipmapGrid3D = Grid3DBase<X, Y, Z, int32_t(MipmapDepth)>;

// ---- include/camera_controller.hpp ------------------------------------------------------------------
struct CameraRay {                                                         // camera_controller.hpp:10-14
    glm::vec3 ray;
    glm::vec3 world_rand_offset;
};

struct Camera {
    glm::vec3 position;
    glm::vec2 view_angle;
    glm::vec3 camera_vec;
    glm::mat3 rot_mat;
    float aperture = 0.0f;
    float focal_length = 1.0f;
    float fov = 1.0f;

    void setViewAngle(const glm::vec2& angle) {                           // camera_controller.hpp:27-32
        view_angle = angle;
        const float a[2] = {angle.x, angle.y};
        float m[9], v[3];
        vrt::check(vrt_host_camera_rotation(a, m, v));
        for (int c = 0; c < 3; ++c) rot_mat[c] = glm::vec3(m[3 * c], m[3 * c + 1], m[3 * c + 2]);
        camera_vec = glm::vec3(v[0], v[1], v[2]);
    }
    // camera_controller.hpp:34-49.  The two lens numbers come from getRand() like in the reference (host-side stream; the
    // batched RayCaster::render draws them per (pixel, sample) on the device instead).
    CameraRay getRay(const glm::vec2& lens_position) {
        const glm::vec3 screen_position = glm::vec3(lens_position.x, lens_position.y, fov);
        const glm::vec3 focal_point = glm::normalize(screen_position) * focal_length;
        const float r0 = getRand(), r1 = getRand();
        const glm::vec3 rand_vec = glm::vec3(aperture * r0, aperture * r1, aperture * 0.0f);
        const glm::vec3 ray = glm::normalize(focal_point - rand_vec);
        CameraRay result;
        result.ray = viewToWorld(ray);
        result.world_rand_offset = viewToWorld(rand_vec);
        return result;
    }
    glm::vec3 viewToWorld(const glm::vec3& v) const {                     // camera_controller.hpp:51-54: v * rot_mat
        return glm::vec3((rot_mat[0].x * v.x + rot_mat[0].y * v.y) + rot_mat[0].z * v.z,
                         (rot_mat[1].x * v.x + rot_mat[1].y * v.y) + rot_mat[1].z * v.z,
                         (rot_mat[2].x * v.x + rot_mat[2].y * v.y) + rot_mat[2].z * v.z);
    }
    // camera_controller.hpp:56-60; the literal 1/512 is 1/2^depth of the volume
    HitPoint getClosestPoint(const Volumetric& volume) const {
        uint32_t depth = 9;
        vrt::check(vrt_scene_info(volume.scene(), nullptr, &depth, nullptr));
        const float scale = 1.0f / float(1u << depth);
        return volume.castRay(glm::vec3(position.x * scale + 1.0f, position.y * scale + 1.0f, position.z * scale + 1.0f), camera_vec, 0.0f, 0.0f);
    }
    vrt_camera as_struct() const {
        vrt_camera c;
        c.position[0] = position.x; c.position[1] = position.y; c.position[2] = position.z;
        for (int k = 0; k < 3; ++k) { c.rot_mat[3 * k] = rot_mat[k].x; c.rot_mat[3 * k + 1] = rot_mat[k].y; c.rot_mat[3 * k + 2] = rot_mat[k].z; }
        c.fov = fov; c.aperture = aperture; c.focal_length = focal_length;
        return c;
    }
    // camera_controller.hpp:56-60 + main.cpp:115-121: returns the focal length the demo would use
    float autofocus(const Volumetric& volume) {
        const vrt_camera c = as_struct();
        vrt::check(vrt_autofocus(volume.scene(), &c, &focal_length));
        return focal_length;
    }
};

struct CameraController {                                                 // camera_controller.hpp:64-78
    virtual ~CameraController() {}
    virtual void updateCameraView(const glm::vec2& d_view_angle, Camera& camera) {
        glm::vec2 new_angle(camera.view_angle.x + d_view_angle.x, camera.view_angle.y + d_view_angle.y);
        const float half_pi = 3.141592653f * 0.5f;
        new_angle.y = new_angle.y < -half_pi ? -half_pi : new_angle.y > half_pi ? half_pi : new_angle.y;
        camera.setViewAngle(new_angle);
    }
    virtual void move(const glm::vec3& move_vector, Camera& camera) = 0;
    float movement_speed = 1.0f;
};
struct FlyController : CameraController {                                 // fly_controller.hpp:6-12
    void move(const glm::vec3& move_vector, Camera& camera) override {
        camera.position = glm::vec3(camera.position.x + move_vector.x, camera.position.y + move_vector.y, camera.position.z + move_vector.z);
    }
};

// ---- include/replay.hpp: a recorded camera path, `timestamp x y z view_x view_y` per tick --------------------
struct ReplayElements {
    float timestamp, x, y, z, view_x, view_y;
    static std::vector<ReplayElements> loadFromFile(const std::string& filename) {
        std::vector<ReplayElements> ticks;
        FILE* f = std::fopen(filename.c_str(), "r");
        if (!f) return ticks;
        ReplayElements e;
        while (std::fscanf(f, "%f %f %f %f %f %f", &e.timestamp, &e.x, &e.y, &e.z, &e.view_x, &e.view_y) == 6) ticks.push_back(e);
        std::fclose(f);
        return ticks;
    }
    void apply(Camera& camera) const {
        camera.position = glm::vec3(x, y, z);
        camera.setViewAngle(glm::vec2(view_x, view_y));
    }
};

// ---- include/raycaster.hpp --------------------------------------------------------------------------------
namespace vrt {
struct Vector2i { int x = 0, y = 0; Vector2i() {} Vector2i(int a, int b) : x(a), y(b) {} };   // sf::Vector2i stand-in
struct Color { uint8_t r = 0, g = 0, b = 0, a = 255; };                                       // sf::Color stand-in

// 24-bit uncompressed BMP → 16x16 RGB, top-down rows (what sf::Image::loadFromFile yields)
inline bool load_bmp16(const std::string& path, uint8_t out[768]) {
    FILE* f = std::fopen(path.c_str(), "rb");
    if (!f) return false;
    uint8_t hdr[54];
    bool ok = std::fread(hdr, 1, 54, f) == 54 && hdr[0] == 'B' && hdr[1] == 'M';
    uint32_t off = 0; int32_t w = 0, h = 0; uint16_t bpp = 0;
    if (ok) { std::memcpy(&off, hdr + 10, 4); std::memcpy(&w, hdr + 18, 4); std::memcpy(&h, hdr + 22, 4); std::memcpy(&bpp, hdr + 28, 2); }
    ok = ok && w == 16 && (h == 16 || h == -16) && bpp == 24 && std::fseek(f, long(off), SEEK_SET) == 0;
    for (int row = 0; ok && row < 16; ++row) {
        uint8_t line[48];
        ok = std::fread(line, 1, 48, f) == 48;
        const int y = h > 0 ? 15 - row : row;
        for (int x = 0; ok && x < 16; ++x) { out[3 * (y * 16 + x)] = line[3 * x + 2]; out[3 * (y * 16 + x) + 1] = line[3 * x + 1]; out[3 * (y * 16 + x) + 2] = line[3 * x]; }
    }
    std::fclose(f);
    return ok;
}
}  // namespace vrt

struct RayContext {                                       // raycaster.hpp:9-15
    float distance = 0.0f;
    uint32_t complexity = 0U;
    uint32_t bounds = 0U;
    int32_t gi_bounce = 2U;
};
struct ColorResult {                                      // raycaster.hpp:35-39
    vrt::Color color;
    float distance = 0.0f;
};

namespace vrt {
// every RayCaster with renderRay() calls waiting to be executed; swrm::WorkGroup::waitExecutionDone() flushes them
struct PendingFlush {
    virtual void flush() = 0;
    virtual ~PendingFlush() {}
};
inline std::vector<PendingFlush*>& pending_registry() { static std::vector<PendingFlush*> r; return r; }
inline void flush_all() { for (PendingFlush* p : pending_registry()) p->flush(); }
inline uint8_t mult_u8(uint8_t c, float f) { const float v = float(c) * f; return uint8_t(v < 255.0f ? v : 255.0f); }   // utils.cpp:43-48
}  // namespace vrt

template <uint8_t SVO_DEPTH_>
struct RayCasterT : vrt::PendingFlush {
    // raycaster.hpp:48 — loads res/grass_side_16x16.bmp and res/grass_top_16x16.bmp relative to the CWD like the
    // reference; pass explicit textures (16x16 RGB, top-down) to skip the files.
    RayCasterT(const LSVO<SVO_DEPTH_>& svo_, const vrt::Vector2i& render_size_, const uint8_t* top_rgb = nullptr,
               const uint8_t* side_rgb = nullptr)
        : svo(svo_), render_size(render_size_) {
        uint8_t top[768], side[768];
        if (top_rgb && side_rgb) { std::memcpy(top, top_rgb, 768); std::memcpy(side, side_rgb, 768); }
        else if (!vrt::load_bmp16("res/grass_top_16x16.bmp", top) || !vrt::load_bmp16("res/grass_side_16x16.bmp", side))
            throw vrt::Error(VRT_ERR_INVALID, "RayCaster: cannot read res/grass_{top,side}_16x16.bmp");
        vrt::check(vrt_scene_set_textures(svo.scene(), top, side));
        render_image.assign(size_t(render_size.x) * render_size.y * 4, 0);
        colors.assign(size_t(render_size.x) * render_size.y * 4, 0u);
        vrt::pending_registry().push_back(this);
    }
    ~RayCasterT() override {
        std::vector<vrt::PendingFlush*>& r = vrt::pending_registry();
        for (size_t i = 0; i < r.size(); ++i)
            if (r[i] == this) { r.erase(r.begin() + i); break; }
    }
    RayCasterT(const RayCasterT&) = delete;
    RayCasterT& operator=(const RayCasterT&) = delete;

    // ---- the reference's per-ray entry points (compatibility path; frames should call render()) --------------------------
    // raycaster.hpp:67-92.  The ray is queued; the queue is shaded in ONE launch (vrt_shade_rays) at the synchronisation point
    // the reference's loop already has — swrm::WorkGroup::waitExecutionDone() (main.cpp:156) — or by flush() / samples_to_image().
    // Pixels keep the order of the calls, so the temporal blend and the accumulators end up as in the reference.
    void renderRay(const vrt::Vector2i pixel, const glm::vec3& start, const glm::vec3& direction, float /*time*/) {
        vrt_shade_job j;
        j.start[0] = start.x; j.start[1] = start.y; j.start[2] = start.z;
        j.direction[0] = direction.x; j.direction[1] = direction.y; j.direction[2] = direction.z;
        j.pixel = uint32_t(pixel.y) * uint32_t(render_size.x) + uint32_t(pixel.x);
        j.sample = use_samples ? colors[4 * size_t(j.pixel) + 3] + pending_count(j.pixel) : frame_index;
        m_jobs.push_back(j);
    }
    void flush() override {
        if (m_jobs.empty()) return;
        std::vector<vrt_shade_result> res(m_jobs.size());
        const vrt_render_params p = shade_params();
        vrt::check(vrt_shade_rays(svo.scene(), &p, m_jobs.size(), m_jobs.data(), res.data()));
        for (size_t i = 0; i < m_jobs.size(); ++i) {
            const size_t px = m_jobs[i].pixel;
            if (!use_samples) {                                            // raycaster.hpp:79-85: 0.4 old + 0.6 new
                uint8_t* q = &render_image[4 * px];
                const uint8_t rgb[3] = {res[i].r, res[i].g, res[i].b};
                for (int c = 0; c < 3; ++c) {
                    const int v = int(vrt::mult_u8(q[c], 0.4f)) + int(vrt::mult_u8(rgb[c], 1.0f - 0.4f));   // add(), utils.cpp:35-40
                    q[c] = uint8_t(v < 255 ? v : 255);
                }
                q[3] = 255;
            } else {                                                       // raycaster.hpp:87-90
                colors[4 * px] += res[i].r; colors[4 * px + 1] += res[i].g; colors[4 * px + 2] += res[i].b; colors[4 * px + 3] += 1u;
            }
        }
        if (!use_samples) ++frame_index;
        m_jobs.clear();
        m_pending.clear();
    }
    // raycaster.hpp:118-167: one ray, shaded on the device right away (one tiny launch: not for inner loops)
    ColorResult castRay(const glm::vec3& start, const glm::vec3& direction, float /*time*/, RayContext& context) {
        ColorResult result;
        if (context.bounds > max_bounds) return result;                    // raycaster.hpp:127-129
        vrt_shade_job j;
        j.start[0] = start.x; j.start[1] = start.y; j.start[2] = start.z;
        j.direction[0] = direction.x; j.direction[1] = direction.y; j.direction[2] = direction.z;
        j.pixel = 0xffffffffu; j.sample = m_cast_counter++;
        vrt_shade_result r;
        const vrt_render_params p = shade_params();
        vrt::check(vrt_shade_rays(svo.scene(), &p, 1, &j, &r));
        context.complexity += r.complexity;                                // :132-133
        context.distance = r.distance;
        result.color.r = r.r; result.color.g = r.g; result.color.b = r.b;
        result.distance = r.distance;
        return result;
    }
    // raycaster.hpp:169-207 with the host-side getRand stream: two single-ray casts through LSVO::castRay
    float getGlobalIllumination(const HitPoint& point) {
        uint32_t depth = SVO_DEPTH_;
        const float SCALE = 1.0f / float(1u << depth);
        const float n_normalizer = SCALE * 0.0078125f * 2.0f;
        const glm::vec3& normal = point.normal;
        const glm::vec3 gi_start(point.position.x + normal.x * n_normalizer, point.position.y + normal.y * n_normalizer, point.position.z + normal.z * n_normalizer);
        const float range = 1000.0f;
        glm::vec3 noise_normal(0.0f, 0.0f, 0.0f);
        const float coord_1 = getRand(-range, range), coord_2 = getRand(-range, range);
        if (normal.x != 0.0f) noise_normal = glm::vec3(0.0f, coord_1, coord_2);
        else if (normal.y != 0.0f) noise_normal = glm::vec3(coord_1, 0.0f, coord_2);
        else if (normal.z != 0.0f) noise_normal = glm::vec3(coord_1, coord_2, 0.0f);
        else return 0.0f;                                                  // uninitialised noise_normal in the reference
        const glm::vec3 gi_ray = glm::normalize(glm::vec3((normal.x + noise_normal.x) * n_normalizer, (normal.y + noise_normal.y) * n_normalizer,
                                                          (normal.z + noise_normal.z) * n_normalizer));
        const float dot_gi = glm::dot(gi_ray, normal);
        float acc = 0.0f;
        const HitPoint gi_point = svo.castRay(gi_start, gi_ray, 0.5f, 0.0f);
        if (gi_point.cell) {
            const glm::vec3 gi_light_start(gi_point.position.x + gi_point.normal.x * n_normalizer, gi_point.position.y + gi_point.normal.y * n_normalizer,
                                           gi_point.position.z + gi_point.normal.z * n_normalizer);
            const glm::vec3 to_light = glm::normalize(glm::vec3(light_position.x - gi_light_start.x, light_position.y - gi_light_start.y,
                                                                light_position.z - gi_light_start.z));
            const HitPoint gi_light_point = svo.castRay(gi_light_start, to_light, 0.5f, 0.0f);
            if (!gi_light_point.cell) {
                const float d = glm::dot(gi_point.normal, to_light);
                acc += sun_intensity * std::min(0.5f, std::max(0.0f, d) * dot_gi);
            }
        }
        return std::max(0.0f, acc / 1.0f);
    }
    const float eps = 0.001f;                           // raycaster.hpp:45-46
    const float sun_intensity = 1000000.0f;
    const uint32_t max_bounds = 4;                      // raycaster.hpp:277

    void setLightPosition(const glm::vec3& position) { light_position = position; }          // raycaster.hpp:62

    // Replaces the swarm lambda main.cpp:139-154 (+ samples_to_image when use_samples): every pixel, `spp` passes.
    void render(const Camera& camera, int spp = 1) {
        vrt_render_params p;
        std::memset(&p, 0, sizeof(p));
        p.width = render_size.x; p.height = render_size.y; p.row_begin = 0; p.row_end = render_size.y;
        p.spp = use_samples ? spp : 1;
        flush();
        p.sample_offset = int32_t(use_samples ? sample_count : frame_index);   // blend mode: a new random stream every frame
        p.seed_lo = seed_lo; p.seed_hi = seed_hi;
        p.light_position[0] = light_position.x; p.light_position[1] = light_position.y; p.light_position[2] = light_position.z;
        p.use_gi = use_gi; p.gi_bounces = gi_bounces; p.use_samples = use_samples;
        p.accum_in = use_samples ? 1 : 0;
        p.checker = checker_board_offset < 0 ? 0 : 1 + (checker_board_offset & 1);
        p.checker_area_height = checker_area_height;
        p.mirror_y1 = mirror_y < 0 ? 0 : mirror_y + 1; p.roughness = roughness; p.max_bounds = int32_t(max_bounds);
        p.autofocus = autofocus ? 1 : 0;
        if (!use_samples) std::fill(colors.begin(), colors.end(), 0u);
        const vrt_camera c = camera.as_struct();
        vrt::check(vrt_render(svo.scene(), &c, &p, render_image.data(), colors.data(), &last_stats));
        if (use_samples) sample_count += uint32_t(p.spp);
        else ++frame_index;
    }
    // The presentation step of the main loop (main.cpp:159-177): optional 3x3 / 5x5 median (res/median_3.frag,
    // res/median.frag) and the persistence blend of render_image into `display` (denoised_tex).
    void present(int median = 0, float old_value_conservation = -1.0f) {
        if (old_value_conservation < 0.0f) old_value_conservation = use_samples ? 0.0f : 0.1f;   // main.cpp:160
        if (display.empty()) display.assign(render_image.size(), 0);
        vrt_present_params p;
        p.width = render_size.x; p.height = render_size.y; p.median = median; p.old_value_conservation = old_value_conservation;
        vrt::check(vrt_present(vrt::default_context(), render_image.data(), display.data(), &p));
    }
    // raycaster.hpp:94-103.  render() resolves on the device already; after renderRay() calls the queue is shaded first and the
    // image is resolved here (the integer sums divide exactly like the reference's doubles, DESIGN.md §3).
    void samples_to_image() {
        const bool queued = !m_jobs.empty();
        flush();
        if (!queued && !m_resolve_on_host) return;
        m_resolve_on_host = true;
        for (size_t i = 0; i < colors.size() / 4; ++i) {
            const uint32_t n = colors[4 * i + 3] ? colors[4 * i + 3] : 1u;
            render_image[4 * i] = uint8_t(colors[4 * i] / n); render_image[4 * i + 1] = uint8_t(colors[4 * i + 1] / n);
            render_image[4 * i + 2] = uint8_t(colors[4 * i + 2] / n); render_image[4 * i + 3] = 255;
        }
    }
    void resetSamples() {                               // raycaster.hpp:105-116
        flush();
        std::fill(colors.begin(), colors.end(), 0u);
        sample_count = 0;
    }
    vrt::Color getPixel(int x, int y) const {
        const uint8_t* q = &render_image[4 * (size_t(y) * render_size.x + x)];
        vrt::Color c; c.r = q[0]; c.g = q[1]; c.b = q[2]; c.a = q[3];
        return c;
    }

    std::vector<uint32_t> colors;                       // Sample accumulators r,g,b,count per pixel (raycaster.hpp:259)
    std::vector<uint8_t> render_image;                  // RGBA8, row major (sf::Image render_image, raycaster.hpp:261)
    std::vector<uint8_t> display;                       // RGBA8: denoised_tex of main.cpp:168-172, made by present()
    int checker_board_offset = -1;                      // -1 = every pixel; 0 / 1 = the checkerboard of main.cpp:137,143
    int checker_area_height = 0;                        // RENDER_HEIGHT / area_count (main.cpp:132); 0 = one area
    int mirror_y = -1;                                  // voxel layer (castRay y) whose top faces are Cell::Mirror; -1 = none (extension)
    float roughness = 0.0f;                             // blur of mirror reflections
    bool autofocus = false;                             // focal length from the centre ray on the device (main.cpp:114-121)
    const LSVO<SVO_DEPTH_>& svo;
    const vrt::Vector2i render_size;
    glm::vec3 light_position;
    bool use_ao = false;                                // toggles without effect, as in the reference (:273,:276)
    bool use_gi = false;
    bool use_samples = false;
    bool use_god_rays = false;
    int gi_bounces = 1;                                 // 2 = extension
    uint32_t seed_lo = 0x5EED, seed_hi = 0, sample_count = 0;
    uint32_t frame_index = 0;                           // frames rendered in blend mode (selects the random stream)
    vrt_render_stats last_stats{};

private:
    vrt_render_params shade_params() const {
        vrt_render_params p;
        std::memset(&p, 0, sizeof(p));
        p.width = render_size.x; p.height = render_size.y; p.row_end = render_size.y; p.spp = 1;
        p.seed_lo = seed_lo; p.seed_hi = seed_hi;
        p.light_position[0] = light_position.x; p.light_position[1] = light_position.y; p.light_position[2] = light_position.z;
        p.use_gi = use_gi; p.gi_bounces = gi_bounces; p.use_samples = use_samples;
        p.max_bounds = int32_t(max_bounds);
        return p;
    }
    uint32_t pending_count(uint32_t pixel) {            // samples of this pixel already queued in this batch
        if (m_pending.empty()) m_pending.assign(size_t(render_size.x) * render_size.y, 0);
        return m_pending[pixel]++;
    }
    std::vector<vrt_shade_job> m_jobs;
    std::vector<uint16_t> m_pending;
    uint32_t m_cast_counter = 0;
    bool m_resolve_on_host = false;
};
constexpr uint8_t SVO_DEPTH = 9u;                       // raycaster.hpp:42
using RayCaster = RayCasterT<SVO_DEPTH>;
