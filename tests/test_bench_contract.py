"""bench.py's output contract, as far as it can be checked without a GPU: the reference arm (the unmodified render.cpp on
the host cores) prints exactly ONE JSON line on stdout with the keys the driver reads, and the product arm refuses to run
without a CUDA device instead of falling back to anything."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, timeout=300):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=timeout, cwd=ROOT)


def test_reference_arm_prints_one_contract_line():
    # a scaled-down field (2 000 solids at 640x360) keeps the CPU suite short; the line has the full-size run's shape
    p = _run(["--impl", "reference", "--steps", "2", "--warmup", "0", "--cpu-replicas", "2", "--width", "640", "--height", "360",
              "--c3-solids", "2000", "--c2-frames", "4"])
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, p.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "frames/s" and d["higher_is_better"] is True and d["scaling"] == "strong"
    assert d["value"] > 0 and d["steps"] == 2 and d["n_gpus"] == 1 and d["vs_baseline"] is None and d["gpu_launches"] == 0
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and 1 <= d["cpu_baseline"]["cores"] <= 2 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"] and d["config"]["workload"].startswith("C3")
    assert set(d["frame0_digest"]) == {"sum", "crc32"}   # compared with the product arm's digest of the same pose
    assert d["secondary"]["value"] > 0 and d["secondary"]["metric"].endswith("fly-through)")


def test_frame0_digest_of_the_reference_arm_is_the_oracles(oracle_port):
    """The digest the two arms are compared on is what it says: pose 0 of the drift path, rendered by the CPU reference."""
    sys.path.insert(0, ROOT)
    import bench
    from swift3drenderer_b200 import scene as S
    path = bench.c3_data_bin(2000)
    reps = bench.CpuReplicas(path, 640, 360, 64, gb_per_replica=0.1, cap=1)
    try:
        mats = oracle_port.camera_path(bench.drift_inputs(1))
        want = oracle_port.OracleScene(path=path).render(mats[0], 640, 360)["pixels"]
        assert reps.frame0 == bench.frame_digest(want)
        wall, busy = reps.step()
        assert 0 < busy <= wall * 1.5
    finally:
        reps.close()


def test_product_arm_needs_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present: the product arm would run")
    p = _run(["--steps", "1", "--warmup", "3", "--c3-solids", "100"])
    assert p.returncode != 0 and "no CUDA device" in (p.stderr + p.stdout)
    assert not [l for l in p.stdout.splitlines() if l.startswith("{")]   # no result line from a run that did not happen


def test_dump_outputs_writes_exact_float32_frames_and_a_fixed_sample(tmp_path, monkeypatch):
    sys.path.insert(0, ROOT)
    import bench
    rng = np.random.default_rng(5)
    frames = [rng.integers(0, 1 << 24, (90, 160), dtype=np.uint32) for _ in range(3)]
    bench.dump_outputs(str(tmp_path / "whole"), [5, 6, 7], frames)
    got = np.load(tmp_path / "whole" / "frames.npy")
    assert got.dtype == np.float32 and np.array_equal(got.astype(np.uint32), np.stack(frames).reshape(3, -1))
    assert np.load(tmp_path / "whole" / "poses.npy").tolist() == [5, 6, 7]
    monkeypatch.setattr(bench, "DUMP_BYTES", 1000 * (4 * 3 + 8))   # room for 1 000 of the 14 400 pixels of each frame
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), [5, 6, 7], frames)
    idx = np.load(tmp_path / "a" / "pixel_index.npy")
    assert idx.dtype == np.float64 and len(idx) == 1000 and np.array_equal(idx, np.load(tmp_path / "b" / "pixel_index.npy"))
    sample = np.load(tmp_path / "a" / "frames.npy")
    assert np.array_equal(sample, np.load(tmp_path / "b" / "frames.npy"))
    assert np.array_equal(sample.astype(np.uint32), np.stack(frames).reshape(3, -1)[:, idx.astype(np.int64)])


@pytest.mark.gpu
def test_dumped_outputs_are_the_oracles_frames(tmp_path, oracle_port):
    """--dump-outputs holds what the timed steps rendered: the frames of the last step still in the output ring."""
    p = _run(["--steps", "2", "--warmup", "3", "--c3-solids", "2000", "--width", "640", "--height", "360",
              "--no-cpu", "--no-e2e", "--no-secondary", "--dump-outputs", str(tmp_path)])
    assert p.returncode == 0, p.stderr[-2000:]
    assert json.loads(p.stdout.strip().splitlines()[-1])["steps"] == 2
    sys.path.insert(0, ROOT)
    import bench
    frames = np.load(tmp_path / "frames.npy")
    idx = np.load(tmp_path / "pixel_index.npy").astype(np.int64)
    poses = np.load(tmp_path / "poses.npy").astype(np.int64).tolist()
    assert frames.dtype == np.float32 and poses == [4, 5, 6, 7] and len(idx) == 640 * 360
    osc = oracle_port.OracleScene(path=bench.c3_data_bin(2000))
    mats = oracle_port.camera_path(bench.drift_inputs(bench.POSES))
    for got, pose in zip(frames, poses):
        want = osc.render(mats[pose], 640, 360)["pixels"].reshape(-1)[idx]
        assert np.array_equal(got, want.astype(np.float32)), f"pose {pose}"
