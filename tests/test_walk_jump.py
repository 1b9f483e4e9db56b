"""walk_jump (swift3drenderer_b200/csrc/walk.cuh) must equal n sequential binary32 additions
(render-cpp/render.cpp:374-379).  Host build of the same header, fuzzed against the loop."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def walk_lib(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("walk") / "walk_host.so")
    subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-fPIC", "-shared",
                           os.path.join(ROOT, "tests", "native", "walk_host.cpp"), "-o", out])
    lib = ctypes.CDLL(out)
    lib.walk_fuzz.argtypes = [ctypes.c_uint32, ctypes.c_uint64, ctypes.c_uint32, ctypes.c_uint64, ctypes.c_void_p]
    lib.walk_fuzz.restype = ctypes.c_uint64
    for fn in (lib.walk_jump_host, lib.walk_seq_host):
        fn.argtypes = [ctypes.c_float, ctypes.c_float, ctypes.c_uint32]
        fn.restype = ctypes.c_float
    return lib


@pytest.mark.parametrize("mode", [0, 1, 2, 3, 4])
@pytest.mark.parametrize("max_n", [8, 64, 4096, 65536])
def test_fuzz_against_sequential_adds(walk_lib, mode, max_n):
    """65536: the longest walks of frames up to 65535 pixels (fewer trials: the loop it is checked against is long)."""
    bad = np.zeros(5, np.float32)
    trials = 400000 if max_n < 4096 else 150000 if max_n == 4096 else 12000
    mism = walk_lib.walk_fuzz(mode, trials, max_n, 1000 + 10 * mode + max_n, bad.ctypes.data)
    assert mism == 0, f"first mismatch (s, d, n, jump, seq) = {bad.tolist()}"


def test_edge_cases(walk_lib):
    cases = [
        (0.0, 0.0, 100), (1.0, 0.0, 7), (0.0, 1e-3, 3840), (1.0, -1e-3, 3840), (-1.0, 1e-3, 3840),
        (2.0030441, -3.4061623e-06, 1845),  # landing exactly on a binade floor (regression)
        (1.0, 2.0 ** -24, 5000), (1.0, -(2.0 ** -25), 5000), (1.0, 1.5 * 2.0 ** -23, 5000),
        (16777216.0, 1.0, 100), (1e-38, 1e-40, 3000), (-1e-38, 1e-40, 3000), (3.0, 1e30, 10),
        (float("inf"), 1.0, 10), (0.5, 0.25, 1), (0.5, 0.25, 2),
    ]
    for s, d, n in cases:
        a, b = walk_lib.walk_jump_host(s, d, n), walk_lib.walk_seq_host(s, d, n)
        assert np.float32(a).tobytes() == np.float32(b).tobytes(), (s, d, n, a, b)


def test_split_walks_compose(walk_lib):
    rs = np.random.RandomState(5)
    for _ in range(2000):
        s, d = np.float32(rs.uniform(-2, 2)), np.float32(rs.uniform(-1, 1) / rs.randint(1, 4000))
        n1, n2 = int(rs.randint(0, 3000)), int(rs.randint(0, 3000))
        whole = walk_lib.walk_jump_host(s, d, n1 + n2)
        parts = walk_lib.walk_jump_host(walk_lib.walk_jump_host(s, d, n1), d, n2)
        assert whole == parts
