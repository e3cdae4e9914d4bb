// Per-voxel colours through the drop-in headers: LSVO<9>::paintCells / getCellColors / setPalette, then a frame through
// RayCaster::render.  Prints the counts and an FNV-1a hash of the frame for tests/test_gpu_palette.py to compare with the Python API.
//   usage: palette_test <textures.bin (top 768 B + side 768 B)>
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
        constexpr uint32_t S = 512;
        std::vector<int32_t> heights(S * S);
        vrt::check(vrt_host_terrain_heights(int32_t(S), heights.data()));
        uint64_t n = 0;
        vrt::check(vrt_host_build_terrain_lsvo(9, heights.data(), nullptr, 0, &n));
        std::vector<vrt_lnode> nodes(n);
        vrt::check(vrt_host_build_terrain_lsvo(9, heights.data(), nodes.data(), n, &n));
        LSVO<9> svo(nodes);
        // a box of the world painted by height band (most of it empty: skipped)
        std::vector<uint32_t> xyz;
        std::vector<uint8_t> colors;
        for (uint32_t x = 160; x < 352; ++x)
            for (uint32_t y = 256; y < 352; ++y)
                for (uint32_t z = 160; z < 352; ++z) {
                    xyz.push_back(x); xyz.push_back(y); xyz.push_back(z);
                    colors.push_back(uint8_t(2 + (y - 256) / 4));
                }
        const uint64_t painted = svo.paintCells(xyz, colors);
        size_t coloured = 0;
        for (const vrt_lnode& nd : svo.data) coloured += nd.color != 1;
        const std::vector<uint32_t> probe = {200, 257, 200, 0, 511, 0};
        const std::vector<int16_t> pc = svo.getCellColors(probe);
        std::printf("paint painted=%llu coloured=%zu probe=%d,%d\n", (unsigned long long)painted, coloured, int(pc[0]), int(pc[1]));
        uint8_t palette[768];
        for (int c = 0; c < 256; ++c) {
            palette[3 * c] = uint8_t(c * 37); palette[3 * c + 1] = uint8_t(c * 91 + 40); palette[3 * c + 2] = uint8_t(c * 53 + 90);
        }
        svo.setPalette(palette);
        RayCaster rc(svo, vrt::Vector2i(96, 54), tex.data(), tex.data() + 768);
        rc.setLightPosition(glm::vec3(-200.0f / 512.0f + 1.0f, -1000.0f / 512.0f + 1.0f, -300.0f / 512.0f + 1.0f));
        rc.use_samples = true;
        rc.use_gi = true;
        Camera cam;
        cam.position = glm::vec3(256.0f, 200.0f, 256.0f);
        cam.setViewAngle(glm::vec2(0.3f, -0.35f));
        cam.aperture = 0.5f;
        cam.focal_length = 60.0f;
        rc.render(cam, 2);
        std::printf("frame hash=%016llx\n", (unsigned long long)fnv1a(rc.render_image.data(), rc.render_image.size()));
        svo.clearPalette();
        rc.resetSamples();
        rc.render(cam, 2);
        std::printf("textured hash=%016llx\n", (unsigned long long)fnv1a(rc.render_image.data(), rc.render_image.size()));
    } catch (const vrt::Error& e) {
        std::printf("vrt::Error %d %s\n", e.code, e.what());
        return 3;
    }
    return 0;
}
