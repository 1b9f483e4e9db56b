"""tools/headless.cpp — the compiled C++ stand-in for the reference's main loop (main.swift:95-165): dlopen +
dlsym("updateAndRender"), one realloc'ed double buffer alternated per call, live resize.

CPU: driven against the UNMODIFIED reference (oracle/_ref/render_ref.so) its frame checksums must equal the
oracle port's — the harness reproduces the reference's calling pattern, stale-factor quirk included.
GPU: driven against the B200 render.so it must print the very same checksums: the oracle port's, and the
reference's where oracle/_ref is built."""
import json
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

from swift3drenderer_b200 import assets, scene as S

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FRAMES, EVERY = 60, 7
SIZE, RESIZES = (320, 180), ((20, (200, 150)), (40, (333, 187)))


def weighted_checksum(frame: np.ndarray) -> str:
    p = frame.reshape(-1).astype(np.uint64)
    with np.errstate(over="ignore"):
        return f"{int((p * np.arange(1, p.size + 1, dtype=np.uint64)).sum(dtype=np.uint64)):016x}"


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("headless") / "headless")
    subprocess.check_call(["g++", "-O2", "-std=c++17", os.path.join(ROOT, "tools", "headless.cpp"), "-o", exe, "-ldl"])
    return exe


def run_harness(exe, so_path, tmp_path, name):
    """Private copy of the library beside a data.bin (both libraries find the scene through dladdr, render.cpp:161-176)."""
    d = tmp_path / name
    d.mkdir()
    so = str(d / "render.so")
    shutil.copy(so_path, so)
    shutil.copy(assets.ensure_shipped_data_bin(), str(d / "data.bin"))
    inputs = str(d / "inputs.bin")
    S.input_script("flythrough", 600)[:FRAMES].tofile(inputs)
    cmd = [exe, "--lib", so, "--inputs", inputs, "--frames", str(FRAMES), "--every", str(EVERY), "--size", f"{SIZE[0]}x{SIZE[1]}"]
    for f, (w, h) in RESIZES:
        cmd += ["--resize", f"{f}:{w}x{h}"]
    return json.loads(subprocess.check_output(cmd, text=True))


def assert_checksums_are_the_oracles(out, oracle_port):
    assert out["frames"] == FRAMES and len(out["checksums"]) == len(range(0, FRAMES, EVERY)) + 1
    osc = oracle_port.OracleScene(path=assets.ensure_shipped_data_bin())
    mats = oracle_port.camera_path(S.input_script("flythrough", 600)[:FRAMES])
    for f, w, h, got in out["checksums"]:
        size = SIZE
        for at, s in RESIZES:
            if f >= at:
                size = s
        assert (w, h) == size
        assert got == weighted_checksum(osc.render(mats[f], w, h)["pixels"]), f"frame {f} at {w}x{h}"


def test_headless_against_the_reference_equals_the_oracle(harness, tmp_path, oracle_port):
    from oracle import refso
    if not refso.available():
        pytest.skip("oracle/_ref/render_ref.so not built")
    assert_checksums_are_the_oracles(run_harness(harness, refso.REF_SO, tmp_path, "ref"), oracle_port)


@pytest.mark.gpu
def test_headless_b200_library_is_a_drop_in(harness, tmp_path, renderer_lib, oracle_port):
    from oracle import refso
    ours = run_harness(harness, renderer_lib.LIB_PATH, tmp_path, "b200")
    assert_checksums_are_the_oracles(ours, oracle_port)
    if refso.available():
        assert ours["checksums"] == run_harness(harness, refso.REF_SO, tmp_path, "ref")["checksums"]
