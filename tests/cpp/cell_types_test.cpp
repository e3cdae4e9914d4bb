// Mirror voxels through the drop-in headers: a painted LSVO<6> with LSVO::setCellTypes / clearCellTypes, frames through
// RayCaster::render.  Prints the paint count and FNV-1a hashes of the frames for tests/test_gpu_cell_types.py to compare with
// the Python API.
//   usage: cell_types_test <textures.bin (top 768 B + side 768 B)>
#include <cstdio>
#include <vector>

#include <vrt/vrt.hpp>

static uint64_t fnv1a(const uint8_t* p, size_t n) {
    uint64_t h = 1469598103934665603ull;
    for (size_t i = 0; i < n; ++i) { h ^= p[i]; h *= 1099511628211ull; }
    return h;
}

int main(int argc, char** argv) {
    if (argc < 2) { std::fprintf(stderr, "usage: %s textures.bin\n", argv[0]); return 2; }
    std::vector<uint8_t> tex(1536);
    FILE* f = std::fopen(argv[1], "rb");
    if (!f || std::fread(tex.data(), 1, 1536, f) != 1536) { std::fprintf(stderr, "cannot read textures\n"); return 2; }
    std::fclose(f);
    try {
        constexpr uint32_t S = 64;
        // boxes in castRay voxel coordinates, stored in setCell coordinates (v -> S-1-v): a floor, a mirror wall, a pillar
        std::vector<uint32_t> xyz;
        std::vector<uint8_t> colors;
        auto add = [&](uint32_t x0, uint32_t x1, uint32_t y0, uint32_t y1, uint32_t z0, uint32_t z1, uint8_t c) {
            for (uint32_t x = x0; x < x1; ++x)
                for (uint32_t y = y0; y < y1; ++y)
                    for (uint32_t z = z0; z < z1; ++z) {
                        xyz.push_back(S - 1 - x); xyz.push_back(S - 1 - y); xyz.push_back(S - 1 - z);
                        colors.push_back(c);
                    }
        };
        add(0, 64, 56, 64, 0, 64, 3);
        add(50, 53, 18, 56, 6, 58, 9);
        add(20, 25, 30, 56, 30, 35, 4);
        uint64_t n = 0;
        vrt::check(vrt_host_build_lsvo_from_voxels(6, xyz.data(), colors.size(), nullptr, 0, &n));
        std::vector<vrt_lnode> nodes(n);
        vrt::check(vrt_host_build_lsvo_from_voxels(6, xyz.data(), colors.size(), nodes.data(), n, &n));
        LSVO<6> svo(nodes);
        std::printf("paint painted=%llu\n", (unsigned long long)svo.paintCells(xyz, colors));
        Cell::Type types[256];
        for (Cell::Type& t : types) t = Cell::Solid;
        types[9] = Cell::Mirror;
        svo.setCellTypes(types);
        RayCasterT<6> rc(svo, vrt::Vector2i(96, 54), tex.data(), tex.data() + 768);
        rc.setLightPosition(glm::vec3(-200.0f / 64.0f + 1.0f, -1000.0f / 64.0f + 1.0f, -300.0f / 64.0f + 1.0f));
        rc.use_samples = true;
        rc.use_gi = true;
        rc.roughness = 0.3f;
        Camera cam;
        cam.position = glm::vec3(14.0f, 30.0f, 8.0f);
        cam.setViewAngle(glm::vec2(0.9f, -0.3f));
        cam.aperture = 0.5f;
        cam.focal_length = 30.0f;
        rc.render(cam, 2);
        std::printf("frame hash=%016llx\n", (unsigned long long)fnv1a(rc.render_image.data(), rc.render_image.size()));
        svo.clearCellTypes();
        rc.resetSamples();
        rc.render(cam, 2);
        std::printf("cleared hash=%016llx\n", (unsigned long long)fnv1a(rc.render_image.data(), rc.render_image.size()));
    } catch (const vrt::Error& e) {
        std::printf("vrt::Error %d %s\n", e.code, e.what());
        return 3;
    }
    return 0;
}
