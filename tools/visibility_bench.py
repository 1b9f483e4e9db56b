#!/usr/bin/env python
"""visibility_bench.py — frames/s of the visibility planes (s3r_render_device_visibility) against the plain render.

For each workload and frame size three arms run alternately in one process on the same poses:
  colour    s3r_render_device: the colour frame alone;
  planes    s3r_render_device_visibility with colour, triangle and depth outputs (8 more bytes per pixel to HBM);
  vis_only  s3r_render_device_visibility with the triangle and depth outputs only: nothing is shaded.
Workloads, as bench.py defines them:
  C2  the demo scene (data.bin) over the recorded fly-through, --c2-views views per launch (default 24);
  C3  --c3-solids textured icosahedrons (default 1 M, 20 M triangles) over bench.py's 8-pose drift path, one pose per launch.
Times are CUDA events on the launching stream after warm-up; per-kernel times come from separate passes with option
"timing" = 1 (events after every launch), so they do not slow the timed passes.  Each line also says whether the colour of
the planes arm equals the colour arm's and whether the planes of the two plane arms are equal (the last launch's views).
The card's name and power limit are read in the same run.  One JSON line per (workload, size); --out also writes them to
a file.  Needs a GPU: there is no CPU fallback.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

ARMS = ("colour", "planes", "vis_only")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="c2,c3")
    ap.add_argument("--sizes", default="1920x1080,3840x2160")
    ap.add_argument("--c2-frames", type=int, default=120, help="fly-through frames per C2 step")
    ap.add_argument("--c2-views", type=int, default=24, help="C2 views per launch")
    ap.add_argument("--c3-solids", type=int, default=1_000_000)
    ap.add_argument("--rounds", type=int, default=3, help="alternating (colour, planes, vis_only) timed steps")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("visibility_bench.py: no CUDA device (the renderer has no CPU fallback)")
    from swift3drenderer_b200 import assets, renderer as R, scene as S
    from bench import c3_data_bin, drift_inputs, POSES
    from ssaa_bench import card_info

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
            shape = (vpl, H, W)
            buf = {arm: {"colour": torch.empty(shape, dtype=torch.int32, device="cuda:0") if arm != "vis_only" else None,
                         "triangle": torch.empty(shape, dtype=torch.int32, device="cuda:0") if arm != "colour" else None,
                         "depth": torch.empty(shape, dtype=torch.float32, device="cuda:0") if arm != "colour" else None}
                   for arm in ARMS}

            def step(arm):
                b = buf[arm]
                for f0 in range(0, len(mats), vpl):
                    m = mats[f0:f0 + vpl]
                    if arm == "colour":
                        r.render_device(m, W, H, b["colour"].data_ptr(), stream=stream.cuda_stream)
                    else:
                        r.render_device_visibility(m, W, H, b["colour"].data_ptr() if b["colour"] is not None else 0,
                                                   b["triangle"].data_ptr(), b["depth"].data_ptr(), stream=stream.cuda_stream)

            for arm in ARMS:   # warm-up, and capacities grown
                for _ in range(args.warmup):
                    step(arm)
                    while r.finish():
                        step(arm)
            ms = {arm: [] for arm in ARMS}
            for _ in range(args.rounds):
                for arm in ARMS:
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(stream)
                    step(arm)
                    e1.record(stream)
                    assert not r.finish(), "capacity regrown inside the timed region"
                    ms[arm].append(e0.elapsed_time(e1))
            kernels = {}
            for arm in ARMS:
                r.set_option("timing", 1)
                r.timing(reset=True)
                step(arm)
                assert not r.finish()
                kernels[arm] = {n: round(v["ms"] / v["launches"], 4) for n, v in r.kernel_timing().items()}
                r.timing(reset=True)
                r.set_option("timing", 0)
            torch.cuda.synchronize()
            p, v = buf["planes"], buf["vis_only"]
            line = {"workload": desc, "size": f"{W}x{H}", "frames_per_step": len(mats),
                    **{f"{arm}_fps": [round(len(mats) / (t / 1e3), 1) for t in ms[arm]] for arm in ARMS},
                    "planes_over_colour": round(sum(ms["colour"]) / sum(ms["planes"]), 4),
                    "vis_only_over_colour": round(sum(ms["colour"]) / sum(ms["vis_only"]), 4),
                    "kernel_ms_per_launch": kernels,
                    "planes_colour_equals_colour": bool(torch.equal(p["colour"], buf["colour"]["colour"])),
                    "planes_equal_vis_only": bool(torch.equal(p["triangle"], v["triangle"])
                                                  and torch.equal(p["depth"].view(torch.int32), v["depth"].view(torch.int32))),
                    "background_px": int((p["triangle"] == -1).sum()),
                    "card": card}
            print(json.dumps(line), flush=True)
            lines.append(line)
            del buf, p, v
            torch.cuda.empty_cache()
        r.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            for line in lines:
                fh.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
