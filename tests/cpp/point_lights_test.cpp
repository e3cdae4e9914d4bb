// Point lights through the drop-in headers: an LSVO<6> with LSVO::setPointLights / clearPointLights, frames through
// RayCaster::render and through the queued renderRay path (Camera::getRay per pixel and sample, samples_to_image).  Prints
// FNV-1a hashes of the frames for tests/test_gpu_point_lights.py to compare with the Python API.
//   usage: point_lights_test <textures.bin (top 768 B + side 768 B)>
#include <cmath>
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
        // boxes in castRay voxel coordinates, stored in setCell coordinates (v -> S-1-v): a floor and a wall across it
        std::vector<uint32_t> xyz;
        auto add = [&](uint32_t x0, uint32_t x1, uint32_t y0, uint32_t y1, uint32_t z0, uint32_t z1) {
            for (uint32_t x = x0; x < x1; ++x)
                for (uint32_t y = y0; y < y1; ++y)
                    for (uint32_t z = z0; z < z1; ++z) { xyz.push_back(S - 1 - x); xyz.push_back(S - 1 - y); xyz.push_back(S - 1 - z); }
        };
        add(0, 64, 56, 64, 0, 64);
        add(30, 32, 20, 56, 0, 64);
        uint64_t n = 0;
        vrt::check(vrt_host_build_lsvo_from_voxels(6, xyz.data(), xyz.size() / 3, nullptr, 0, &n));
        std::vector<vrt_lnode> nodes(n);
        vrt::check(vrt_host_build_lsvo_from_voxels(6, xyz.data(), xyz.size() / 3, nodes.data(), n, &n));
        LSVO<6> svo(nodes);
        // a warm light in front of the wall (no range limit) and a blue one behind it with a range of 20 voxels
        vrt_point_light lights[2] = {{{1.0f + 20.5f / 64.0f, 1.0f + 44.5f / 64.0f, 1.0f + 32.5f / 64.0f}, {1.0f, 0.6f, 0.3f}, INFINITY, 0u},
                                     {{1.0f + 44.5f / 64.0f, 1.0f + 40.5f / 64.0f, 1.0f + 20.5f / 64.0f}, {0.2f, 0.4f, 1.0f}, 20.0f / 64.0f, 0u}};
        svo.setPointLights(lights, 2);
        const vrt::Vector2i size(96, 54);
        RayCasterT<6> rc(svo, size, tex.data(), tex.data() + 768);
        rc.setLightPosition(glm::vec3(-200.0f / 64.0f + 1.0f, -1000.0f / 64.0f + 1.0f, -300.0f / 64.0f + 1.0f));
        rc.use_samples = true;
        rc.use_gi = true;
        Camera cam;
        cam.position = glm::vec3(31.0f, 8.0f, 4.0f);
        cam.setViewAngle(glm::vec2(0.0f, -0.9f));
        cam.aperture = 0.0f;                  // no lens sample: Camera::getRay's rays are the frame kernels' rays
        cam.focal_length = 30.0f;
        rc.render(cam, 2);
        std::printf("frame hash=%016llx\n", (unsigned long long)fnv1a(rc.render_image.data(), rc.render_image.size()));
        // the reference's loop (main.cpp:139-154): renderRay per pixel, queued and shaded at samples_to_image
        rc.resetSamples();
        const float scale = 1.0f / 64.0f, aspect = float(size.x) / float(size.y);
        for (int s = 0; s < 2; ++s)
            for (int y = 0; y < size.y; ++y)
                for (int x = 0; x < size.x; ++x) {
                    const float lens_x = float(x) / float(size.y) - aspect * 0.5f, lens_y = float(y) / float(size.y) - 0.5f;
                    const CameraRay r = cam.getRay(glm::vec2(lens_x, lens_y));
                    rc.renderRay(vrt::Vector2i(x, y), (cam.position + r.world_rand_offset) * scale + glm::vec3(1.0f), r.ray, 0.0f);
                }
        rc.samples_to_image();
        std::printf("queued hash=%016llx\n", (unsigned long long)fnv1a(rc.render_image.data(), rc.render_image.size()));
        svo.clearPointLights();
        rc.resetSamples();
        rc.render(cam, 2);
        std::printf("cleared hash=%016llx\n", (unsigned long long)fnv1a(rc.render_image.data(), rc.render_image.size()));
    } catch (const vrt::Error& e) {
        std::printf("vrt::Error %d %s\n", e.code, e.what());
        return 3;
    }
    return 0;
}
