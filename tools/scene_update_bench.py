#!/usr/bin/env python
"""scene_update_bench.py — cost of animating a loaded scene in place (s3r_update_vertices) on C3.

Three arms run alternately in one process, one pose per frame over bench.py's drift path:
  render     s3r_render_device alone (whole frame);
  update     s3r_update_vertices of ALL positions from a device tensor, then the whole-frame render;
  update_b8  the same update, then the frame as 8 bands (partitioned submissions take the cluster front, which reads the
             refit copies and bounds).
The update writes the load-time positions again, so every arm's frame must equal the render arm's; the script checks that
on the last pose of each step.  Update time is CUDA events around the update call on the rendering stream (scatter +
refit kernels); bytes are what the two kernels must move at least (positions read and written, cl_src, the gathered
positions, the copies written, the triangle words and headers), over that time.  The card's name and power limit are read
in the same run.  One JSON line; needs a GPU (there is no CPU fallback).
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

ARMS = ("render", "update", "update_b8")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--solids", type=int, default=1_000_000)
    ap.add_argument("--size", default="3840x2160")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()

    import numpy as np
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("scene_update_bench.py: no CUDA device (the renderer has no CPU fallback)")
    from swift3drenderer_b200 import renderer as R, scene as S
    from bench import drift_inputs, POSES
    from ssaa_bench import card_info

    card = card_info(torch)
    W, H = (int(v) for v in args.size.split("x"))
    sc = S.c3_scene(args.solids)
    mats = R.camera_path(drift_inputs(POSES))
    r = R.Renderer(0)
    r.load_scene(sc)
    clusters = r.cluster_dump()
    n_clusters, n_cverts = len(clusters["hdr"]) - 1, clusters["pos"].shape[1]
    V, T = sc.vertices.shape[0], sc.n_triangles
    xyz = torch.from_numpy(np.ascontiguousarray(sc.vertices[:, :3], np.float32)).cuda()
    del sc, clusters
    stream = torch.cuda.Stream()
    sp = stream.cuda_stream
    frames = {arm: torch.empty((H, W), dtype=torch.int32, device="cuda:0") for arm in ARMS}
    edges = [H * k // 8 for k in range(9)]
    upd_ms = []

    def step(arm, timed_updates):
        out = frames[arm]
        for m in mats:
            if arm != "render":
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                r.update_vertices(xyz, stream=sp)
                e1.record(stream)
                if timed_updates:
                    upd_ms.append((e0, e1))
            if arm == "update_b8":
                for a, b in zip(edges[:-1], edges[1:]):
                    r.render_device(m, W, H, out.data_ptr() + 4 * a * W, y0=a, y1=b, stream=sp)
            else:
                r.render_device(m, W, H, out.data_ptr(), stream=sp)

    for arm in ARMS:
        for _ in range(args.warmup):
            step(arm, False)
            while r.finish():
                step(arm, False)
    ms = {arm: [] for arm in ARMS}
    equal = True
    for _ in range(args.rounds):
        for arm in ARMS:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            step(arm, True)
            e1.record(stream)
            assert not r.finish(), "capacity regrown inside the timed region"
            ms[arm].append(e0.elapsed_time(e1))
        torch.cuda.synchronize()
        equal = equal and all(torch.equal(frames[a], frames["render"]) for a in ARMS[1:])
    upd_us = sorted(a.elapsed_time(b) * 1e3 for a, b in upd_ms)
    bytes_min = (V * 12 * 2                     # positions read (source) and written (pos_x/y/z)
                 + n_cverts * (4 + 12 + 12)     # cl_src, gathered positions, copies written
                 + T * 4                        # triangle words
                 + n_clusters * (32 + 20))      # headers read and written
    med = upd_us[len(upd_us) // 2]
    line = {"workload": f"C3: {args.solids} textured icosahedrons, {POSES}-pose drift path", "size": f"{W}x{H}",
            "vertices": V, "clusters": n_clusters, "cluster_vertices": n_cverts,
            **{f"{arm}_fps": [round(len(mats) / (t / 1e3), 1) for t in ms[arm]] for arm in ARMS},
            "update_us_median": round(med, 1), "update_us_min": round(upd_us[0], 1), "update_us_max": round(upd_us[-1], 1),
            "update_bytes": bytes_min, "update_GBps_median": round(bytes_min / (med * 1e-6) / 1e9, 1),
            "frames_equal_render_arm": bool(equal), "card": card}
    print(json.dumps(line), flush=True)
    r.close()


if __name__ == "__main__":
    main()
