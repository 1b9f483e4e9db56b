#!/usr/bin/env python
"""ssaa_bench.py — frames/s of supersampled rendering (s3r_render_device_ssaa) against the plain render at k*W x k*H.

For each workload, output size and k in {1, 2, 4} the two calls run alternately in one process on the same poses:
  fused   s3r_render_device_ssaa(W, H, k): the k*W x k*H frame, resolved inside the write-out, W x H pixels to HBM;
  plain   s3r_render_device(k*W, k*H): the same frame unresolved, k*k times the pixels to HBM.
(k = 1: both arms are the plain call at W x H, which gives the run-to-run spread.)  Workloads, as bench.py defines them:
  C2  the demo scene (data.bin) over the recorded fly-through, --c2-views views per launch (default 24);
  C3  --c3-solids textured icosahedrons (default 1 M, 20 M triangles) over bench.py's 8-pose drift path, one pose per launch.
Times are CUDA events on the launching stream after warm-up; per-kernel times come from separate passes with option
"timing" = 1 (events after every launch), so they do not slow the timed passes.  The card's name and power limit are read
in the same run.  One JSON line per (workload, size, k); --out also writes them to a file.  Needs a GPU: there is no CPU
fallback.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card_info(torch):
    info = {"name": torch.cuda.get_device_name(0), "power_limit_w": None}
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_w"] = float(out.splitlines()[0])
    except (OSError, ValueError, IndexError, subprocess.TimeoutExpired):
        pass
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="c2,c3")
    ap.add_argument("--sizes", default="1920x1080,3840x2160")
    ap.add_argument("--ks", default="1,2,4")
    ap.add_argument("--c2-frames", type=int, default=120, help="fly-through frames per C2 step")
    ap.add_argument("--c2-views", type=int, default=24, help="C2 views per launch")
    ap.add_argument("--c3-solids", type=int, default=1_000_000)
    ap.add_argument("--rounds", type=int, default=3, help="alternating (fused, plain) timed steps")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import numpy as np
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("ssaa_bench.py: no CUDA device (the renderer has no CPU fallback)")
    from swift3drenderer_b200 import assets, renderer as R, scene as S
    from bench import c3_data_bin, drift_inputs, POSES

    card = card_info(torch)
    stream = torch.cuda.Stream()
    lines = []

    def workload(name):
        if name == "c2":
            path = assets.ensure_shipped_data_bin()
            mats = R.camera_path(S.input_script("flythrough", args.c2_frames))
            return path, mats, args.c2_views, f"C2: demo scene, {args.c2_frames}-frame fly-through, {args.c2_views} views per launch"
        path = c3_data_bin(args.c3_solids)
        mats = R.camera_path(drift_inputs(POSES))
        return path, mats, 1, f"C3: {args.c3_solids} textured icosahedrons, {POSES}-pose drift path, one pose per launch"

    for name in args.workloads.split(","):
        path, mats, vpl, desc = workload(name)
        r = R.Renderer(0)
        r.load_scene_file(path)
        for size in args.sizes.split(","):
            W, H = (int(v) for v in size.split("x"))
            for k in (int(v) for v in args.ks.split(",")):
                out_fused = torch.empty((vpl, H, W), dtype=torch.int32, device="cuda:0")
                out_plain = torch.empty((vpl, k * H, k * W), dtype=torch.int32, device="cuda:0")

                def step(arm):
                    for f0 in range(0, len(mats), vpl):
                        m = mats[f0:f0 + vpl]
                        if arm == "fused":
                            r.render_device_ssaa(m, W, H, k, out_fused.data_ptr(), stream=stream.cuda_stream)
                        else:
                            r.render_device(m, k * W, k * H, out_plain.data_ptr(), stream=stream.cuda_stream)

                for arm in ("fused", "plain"):   # warm-up, and capacities grown for both sizes
                    for _ in range(args.warmup):
                        step(arm)
                        while r.finish():
                            step(arm)
                ms = {"fused": [], "plain": []}
                for _ in range(args.rounds):
                    for arm in ("fused", "plain"):
                        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        e0.record(stream)
                        step(arm)
                        e1.record(stream)
                        assert not r.finish(), "capacity regrown inside the timed region"
                        ms[arm].append(e0.elapsed_time(e1))
                kernels = {}
                for arm in ("fused", "plain"):
                    r.set_option("timing", 1)
                    r.timing(reset=True)
                    step(arm)
                    assert not r.finish()
                    kernels[arm] = {n: round(v["ms"] / v["launches"], 4) for n, v in r.kernel_timing().items()}
                    r.timing(reset=True)
                    r.set_option("timing", 0)
                # the fused frame is the resolve of the plain one (first view of the last launch)
                a = out_fused[0].cpu().numpy().view(np.uint32)
                b = out_plain[0].cpu().numpy().view(np.uint32).reshape(H, k, W, k)
                want = np.zeros((H, W), np.uint32)
                for shift in (0, 8, 16):
                    s = ((b >> np.uint32(shift)) & np.uint32(255)).sum(axis=(1, 3), dtype=np.uint32)
                    want |= ((s + np.uint32(k * k // 2)) // np.uint32(k * k)) << np.uint32(shift)
                line = {"workload": desc, "output": f"{W}x{H}", "k": k, "rendered": f"{k * W}x{k * H}",
                        "frames_per_step": len(mats),
                        "fused_fps": [round(len(mats) / (t / 1e3), 1) for t in ms["fused"]],
                        "plain_fps": [round(len(mats) / (t / 1e3), 1) for t in ms["plain"]],
                        "fused_over_plain": round(sum(ms["plain"]) / sum(ms["fused"]), 4),
                        "kernel_ms_per_launch": kernels, "fused_equals_resolved_plain": bool(np.array_equal(a, want)),
                        "card": card}
                print(json.dumps(line), flush=True)
                lines.append(line)
                del out_fused, out_plain
                torch.cuda.empty_cache()
        r.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            for line in lines:
                fh.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
