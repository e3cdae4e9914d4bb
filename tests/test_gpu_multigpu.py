"""Multi-GPU frames (libvrt communicator: tile and sample splits; NCCL all-gather) are identical to single-GPU frames (needs >= 2 GPUs; skipped otherwise — the host logic
is covered on CPU by tests/test_multigpu_host.py)."""
import os
import subprocess
import sys

import pytest

from conftest import ROOT


@pytest.mark.gpu
def test_frame_identical_across_world_sizes():
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("one GPU visible")
    world = 4 if n >= 4 else 2
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
                        "--master-addr", "127.0.0.1", "--master-port", "29533", os.path.join(ROOT, "tests", "multigpu_frame_check.py")],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and r.stdout.count("OK") == 3 and "MISMATCH" not in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


@pytest.mark.gpu
def test_cpp_host_drives_several_gpus_through_the_c_abi(tmp_path):
    """tests/cpp/multigpu_test.cpp: one C++ process, vrt_comm_create_local + vrt_render_distributed on 2-4 GPUs, tile and sample
    splits, three pipelined frames each, compared byte for byte with vrt_render on one GPU."""
    import torch
    from conftest import golden
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU visible")
    exe, tex = str(tmp_path / "multigpu_test"), str(tmp_path / "textures.bin")          # outside the (possibly read-only) source tree
    lib_dir = os.path.join(ROOT, "cpuvoxelraycaster_b200")
    subprocess.run(["g++", "-O2", "-std=c++17", "-I" + os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "cpp", "multigpu_test.cpp"),
                    "-o", exe, "-L" + lib_dir, "-lvrt", "-Wl,-rpath," + lib_dir], check=True)
    t = golden("textures.npz")
    with open(tex, "wb") as fh:
        fh.write(t["top"].tobytes() + t["side"].tobytes())
    # three or more GPUs when the box has them: that is where an arrival protocol can go wrong (a fast rank overtaking a slow one)
    r = subprocess.run([exe, tex, str(min(4, torch.cuda.device_count()))], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "multigpu_test: OK" in r.stdout and "MISMATCH" not in r.stdout, r.stdout[-3000:] + r.stderr[-2000:]
