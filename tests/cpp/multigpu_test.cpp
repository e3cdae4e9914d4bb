// One process driving several GPUs through the C ABI only (include/vrt.h): what a C++ host in the reference's style —
// main.cpp with RayCaster::render in place of the swarm lambda of src/main.cpp:139-154 — does to use a whole box.
// Builds the demo terrain T(9) on every GPU, renders GI + DOF frames with the frame split over the GPUs by tiles and by
// samples (vrt_comm_create_local + vrt_render_distributed) and compares every delivered frame byte for byte with the
// same frame rendered on GPU 0 alone (vrt_render).  usage: multigpu_test <textures.bin> [n_gpus] [one_device]
// one_device = 1: every rank is a context on device 0 with its own stream — the whole protocol (arrival counters, the
// sample-split reduce, deliver_all, the double-buffer waits) then runs on a single GPU.
// exit code 0 = identical, 3 = fewer than 2 CUDA devices (nothing to test), 1 = mismatch / error.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include <cuda_runtime.h>
#include <vrt.h>

#define CHECK(call)                                                                          \
    do {                                                                                     \
        int s_ = (call);                                                                     \
        if (s_ != VRT_OK) {                                                                  \
            std::printf("%s failed (%d): %s\n", #call, s_, vrt_last_error());                \
            return s_ == VRT_ERR_CUDA ? 3 : 1;                                               \
        }                                                                                    \
    } while (0)

int main(int argc, char** argv) {
    if (argc < 2) { std::fprintf(stderr, "usage: %s textures.bin [n_gpus]\n", argv[0]); return 2; }
    std::vector<uint8_t> tex(1536);
    FILE* f = std::fopen(argv[1], "rb");
    if (!f || std::fread(tex.data(), 1, 1536, f) != 1536) { std::fprintf(stderr, "cannot read textures\n"); return 2; }
    std::fclose(f);
    const int want = argc > 2 ? std::atoi(argv[2]) : 2;
    const bool one_device = argc > 3 && std::atoi(argv[3]) != 0;

    std::vector<vrt_context*> ctx;
    for (int d = 0; d < want; ++d) {
        vrt_context* c = nullptr;
        const int s = vrt_context_create(one_device ? 0 : d, nullptr, &c);       // a non-blocking stream of its own
        if (s != VRT_OK) break;
        ctx.push_back(c);
    }
    if (ctx.size() < 2) { std::printf("multigpu_test: %zu CUDA device(s) — needs 2: %s\n", ctx.size(), vrt_last_error()); return 3; }
    const int world = int(ctx.size());
    const int W = 330, H = 187, spp = 2 * world;
    std::vector<vrt_scene*> scene(world);
    for (int r = 0; r < world; ++r) {
        CHECK(vrt_lsvo_create_terrain(ctx[r], 9, 0, &scene[r]));
        CHECK(vrt_scene_set_textures(scene[r], tex.data(), tex.data() + 768));
    }
    vrt_camera cam;
    std::memset(&cam, 0, sizeof(cam));
    cam.position[0] = 256; cam.position[1] = 200; cam.position[2] = 256;
    const float view[2] = {0.3f, -0.35f};
    float cv[3];
    CHECK(vrt_host_camera_rotation(view, cam.rot_mat, cv));
    cam.fov = 1.0f; cam.aperture = 0.5f; cam.focal_length = 60.0f;
    vrt_render_params p;
    std::memset(&p, 0, sizeof(p));
    p.width = W; p.height = H; p.row_begin = 0; p.row_end = H; p.spp = spp;
    p.seed_lo = 0x5EED;
    const float light[3] = {-200.0f / 512 + 1, -1000.0f / 512 + 1, -300.0f / 512 + 1};
    std::memcpy(p.light_position, light, sizeof(light));
    p.use_gi = 1; p.gi_bounces = 2; p.use_samples = 1;

    // reference frames on GPU 0 alone: three consecutive sample batches
    const int n_frames = 3;
    std::vector<std::vector<uint8_t>> single(n_frames, std::vector<uint8_t>(size_t(W) * H * 4));
    for (int k = 0; k < n_frames; ++k) {
        vrt_render_params q = p;
        q.sample_offset = k * spp;
        CHECK(vrt_render(scene[0], &cam, &q, single[k].data(), nullptr, nullptr));
    }
    std::vector<vrt_comm*> comm(world);
    CHECK(vrt_comm_create_local(ctx.data(), world, W, H, comm.data()));
    int bad = 0;
    for (int split = VRT_SPLIT_TILES; split <= VRT_SPLIT_SAMPLES; ++split) {
        std::vector<std::vector<uint8_t>> got(n_frames, std::vector<uint8_t>(size_t(W) * H * 4));
        for (int k = 0; k < n_frames; ++k) {               // frames are enqueued back to back: double buffering in use
            vrt_render_params q = p;
            q.sample_offset = k * spp;
            for (int r = world - 1; r >= 0; --r)             // any order: every member only enqueues
                CHECK(vrt_render_distributed(comm[r], scene[r], &cam, &q, split, 0, r == 0 ? got[k].data() : nullptr));
        }
        for (int r = 0; r < world; ++r) CHECK(vrt_comm_frame_wait(comm[r]));
        for (int k = 0; k < n_frames; ++k) {
            const bool same = got[k] == single[k];
            std::printf("world=%d split=%s frame=%d: %s\n", world, split == VRT_SPLIT_TILES ? "tiles" : "samples", k, same ? "identical" : "MISMATCH");
            bad += !same;
        }
    }
    // deliver_all: every GPU receives the frame in its own memory and copies it to its own host buffer.  The buffers are pinned:
    // a copy into pageable memory returns only once it is done, so the first rank's call would wait for ranks not yet enqueued.
    {
        vrt_render_params q = p;
        q.sample_offset = 0;
        const size_t bytes = size_t(W) * H * 4;
        std::vector<uint8_t*> host(world, nullptr);
        for (int r = 0; r < world; ++r) {
            if (cudaHostAlloc(reinterpret_cast<void**>(&host[r]), bytes, cudaHostAllocPortable) != cudaSuccess) {
                std::printf("cudaHostAlloc failed\n");
                return 1;
            }
            std::memset(host[r], 0x5A, bytes);
        }
        for (int r = 0; r < world; ++r) CHECK(vrt_render_distributed(comm[r], scene[r], &cam, &q, VRT_SPLIT_TILES, 1, host[r]));
        for (int r = 0; r < world; ++r) CHECK(vrt_comm_frame_wait(comm[r]));
        for (int r = 0; r < world; ++r) {
            const bool same = std::memcmp(host[r], single[0].data(), bytes) == 0;
            std::printf("world=%d deliver_all rank=%d: %s\n", world, r, same ? "identical" : "MISMATCH");
            bad += !same;
            cudaFreeHost(host[r]);
        }
        uint64_t frames = 0;
        CHECK(vrt_comm_info(comm[world - 1], nullptr, nullptr, &frames));
        uint8_t* d = nullptr;
        CHECK(vrt_comm_frame_device(comm[world - 1], 0, &d));
        std::printf("deliver_all: rank %d holds frame %llu at %p\n", world - 1, (unsigned long long)frames, (void*)d);
    }
    for (int r = 0; r < world; ++r) CHECK(vrt_comm_destroy(comm[r]));
    for (int r = 0; r < world; ++r) { vrt_scene_destroy(scene[r]); }
    for (int r = 0; r < world; ++r) vrt_context_destroy(ctx[r]);
    std::printf("multigpu_test: %s\n", bad ? "FAILED" : "OK");
    return bad ? 1 : 0;
}
