import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run with -m gpu on a B200)")
    config.addinivalue_line("markers", "slow: larger sizes")


def golden(name):
    return np.load(os.path.join(GOLDEN, name), allow_pickle=False)


def bits(a):
    """Bit pattern view for exact float comparison (distinguishes -0.0 from 0.0, NaN payloads)."""
    a = np.ascontiguousarray(a)
    return a.view(np.uint32) if a.dtype == np.float32 else a


HIT_FIELDS = ("position", "normal", "voxel_coord", "distance")


def assert_hits_equal(got, want, got_hit_flag, label="", check_uv=True):
    """Bit-exact comparison of hit records. `want` is a reference/oracle record array with a `hit` field."""
    want_hit = want["hit"] != 0
    assert np.array_equal(got_hit_flag, want_hit), "%s: hit/miss flags differ on %d rays" % (
        label, np.count_nonzero(got_hit_flag != want_hit))
    assert np.array_equal(got["complexity"], want["complexity"]), "%s: complexity differs on %d rays" % (
        label, np.count_nonzero(got["complexity"] != want["complexity"]))
    m = want_hit
    for f in HIT_FIELDS:
        if f == "voxel_coord":
            if not check_uv:
                continue
            # undefined in the reference when the ray starts inside a solid cell (all-zero normal)
            mm = m & np.any(want["normal"] != 0, axis=1)
        else:
            mm = m
        g, w = bits(got[f][mm]), bits(want[f][mm])
        assert np.array_equal(g, w), "%s: field %s differs on %d records" % (label, f, np.count_nonzero(g != w))


@pytest.fixture(scope="session")
def port():
    from oracle import loader
    loader.build()
    return loader.port()


@pytest.fixture(scope="session")
def ref():
    from oracle import loader
    r = loader.ref()
    if r is None:
        pytest.skip("oracle/_ref not built (needs the reference sources, see VRT_REFERENCE in oracle/Makefile)")
    return r


@pytest.fixture(scope="session")
def ref_patched():
    from oracle import loader
    r = loader.ref_patched()
    if r is None:
        pytest.skip("oracle/_ref not built (needs the reference sources, see VRT_REFERENCE in oracle/Makefile)")
    return r


@pytest.fixture(scope="session")
def textures():
    t = golden("textures.npz")
    return t["top"], t["side"]


@pytest.fixture(scope="session")
def vrt():
    import cpuvoxelraycaster_b200 as v
    v.capi.lib()   # raises if libvrt.so is missing: no fallback
    # Every context a test creates renders frames WITHOUT beam floors and bounds exits unless the test turns them on:
    # vrt_render_stats then carries the reference's own loop-trip counts (HitPoint::complexity) and can be compared with the
    # oracle's.  Both shortcuts (on by default in the product — the C++ test programs run with them) are tested on their own:
    # tests/test_gpu_render.py::test_beam_floors_*, tests/test_gpu_fullsize.py.
    if not getattr(v.Context, "_tests_patched", False):
        plain_init = v.Context.__init__

        def init_without_beam(self, *a, **k):
            plain_init(self, *a, **k)
            self.set_option("beam_tile", 0)
            self.set_option("bounds_exit", 0)
        v.Context.__init__ = init_without_beam
        v.Context._tests_patched = True
    return v


@pytest.fixture(scope="session")
def ctx(vrt):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    c = vrt.Context(0)          # beam floors off, see the `vrt` fixture
    yield c
    c.close()


@pytest.fixture(scope="session")
def terrain9_nodes(vrt):
    return vrt.host_build_terrain_lsvo(9)
