#!/usr/bin/env python
"""bench.py — frames/s at 3840x2160 of the updateAndRender() hot path on N B200s.

Primary workload (BASELINE.json configs[2], "C3", the configuration north_star's target is quoted on): 1 M textured
icosahedrons (V = 12 M, T = 20 M, A = 60 M; swift3drenderer_b200.scene.c3_scene, seed 7) at 3840x2160 over an 8-pose
drift path.  One *step* = those 8 frames, one pose per launch set.
  N = 1   the whole frame on one GPU.
  N > 1   STRONG scaling: the frame is partitioned by screen space (interleaved 32-pixel tile rows, rank = row mod N), one
          process per GPU; every rank's shading kernel stores its rows straight into the full-size frame of EVERY rank over
          NVLink peer memory (CUDA IPC) and a one-element NCCL all-reduce per frame is the ordering fence, so that every
          rank holds the assembled frame.  `--partition rows|bands` selects the NCCL all-gather assemblies instead.
  value    assembled frames/s, device-resident, CUDA-event timed on the launching stream, max over ranks.
  e2e      the same poses through the reference-facing plugin call updateAndRender(const PixelData*, const Input*)
           on a private render.so beside C3's data.bin with the caller's pageable double buffer (host camera step,
           48 B H2D, render, D2H of the frame inside the timed region).  N > 1: ONE caller (rank 0) whose updateAndRender
           drives all N GPUs from one process (S3R_DEVICES; every GPU copies its rows over its own PCIe link).
  roofline per kernel from CUDA events recorded after every launch of every fifth frame of the timed region (option
           "timing" = --timing-stride; timing every frame costs the launch overlap of the frames it measures) and for the
           frame (B_alg = 12V + 28A + 8I + 4WH, SURVEY.md 8(d)); `traffic` from the committed ncu capture.
  cpu_baseline / --impl reference: the reference's own render.cpp (oracle/_ref, compiled unmodified; falls back to the C
           port) on the host cores: one single-threaded replica process per core (bounded by memory: each replica maps
           the 4 GB scene and allocates the reference's 2x scratch), one frame per replica and step.
Secondary record (`secondary`, BASELINE.json configs[1], "C2"): the reference's data.bin demo scene, 600-frame recorded
fly-through, frame-parallel at N > 1 — last round's headline, kept for continuity (value, e2e, roofline, cpu_baseline).
"""
from __future__ import annotations

import argparse
import json
import multiprocessing as mp
import os
import subprocess
import sys
import tempfile
import time
import zlib

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "frames/s at 3840x2160 (1 M textured icosahedrons = 20 M triangles, screen-partitioned over N GPUs)"
UNIT = "frames/s"
C2_METRIC = "frames/s at 3840x2160 (data.bin scene, 600-frame fly-through)"
POSES = 8   # frames per step of the primary workload


# --------------------------------------------------------------------------------------------------
# workload definition (shared by both arms)
# --------------------------------------------------------------------------------------------------
def drift_inputs(n: int) -> np.ndarray:
    """Slow drift through the field: creep forward, pan a little (keeps the field in view)."""
    from swift3drenderer_b200 import scene as S
    inp = np.zeros(n, S.INPUT_DTYPE)
    for f in range(n):
        inp[f]["up"] = 1.0
        inp[f]["mouse"] = (0.5 * f, 0.2 * f)
    return inp


def c3_data_bin(solids: int, wait_s: float = 600.0) -> str:
    """data.bin of the C3 field, generated once per box (4 GB for 1 M solids) and shared by every rank and both arms."""
    base = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else tempfile.gettempdir()
    path = os.path.join(base, f"s3r_c3_{solids}_seed7.data.bin")
    lock = path + ".lock"
    if os.path.exists(path):
        return path
    try:
        fd = os.open(lock, os.O_CREAT | os.O_EXCL | os.O_WRONLY)
    except FileExistsError:
        t0 = time.time()
        while not os.path.exists(path):
            if time.time() - t0 > wait_s:
                raise SystemExit(f"bench.py: {path} did not appear within {wait_s:.0f} s (stale {lock}?)")
            time.sleep(0.25)
        return path
    try:
        from swift3drenderer_b200 import scene as S
        tmp = path + f".tmp{os.getpid()}"
        S.write_data_bin(tmp, S.c3_scene(solids))
        os.rename(tmp, path)
    finally:
        os.close(fd)
        os.unlink(lock)
    return path


DUMP_BYTES = 48 << 20   # bound on --dump-outputs' arrays (frames + pixel positions)


def dump_outputs(out_dir: str, poses, frames) -> None:
    """Writes frames (host 0x00RRGGBB arrays of one size) for output-for-output comparison of two builds:
    frames.npy (len(frames), S) float32, which holds every 24-bit pixel exactly; pixel_index.npy (S,) their row-major
    positions; poses.npy the drift-path pose of each frame.  S is every pixel when that fits DUMP_BYTES, else a fixed,
    seeded sample of positions, the same in every frame."""
    os.makedirs(out_dir, exist_ok=True)
    n = frames[0].size
    s = min(n, DUMP_BYTES // (4 * len(frames) + 8))
    idx = np.arange(n) if s == n else np.sort(np.random.default_rng(0).choice(n, s, replace=False))
    np.save(os.path.join(out_dir, "frames.npy"), np.stack([f.reshape(-1)[idx] for f in frames]).astype(np.float32))
    np.save(os.path.join(out_dir, "pixel_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(out_dir, "poses.npy"), np.asarray(poses, np.float64))


def frame_digest(frame: np.ndarray) -> dict:
    a = np.ascontiguousarray(frame, np.uint32)
    return {"sum": int(a.sum(dtype=np.uint64)), "crc32": int(zlib.crc32(a.tobytes()))}


def affinity_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def mem_available_gb() -> float:
    try:
        for line in open("/proc/meminfo"):
            if line.startswith("MemAvailable:"):
                return int(line.split()[1]) / 1e6
    except OSError:
        pass
    return 16.0


# --------------------------------------------------------------------------------------------------
# CPU reference arm (test infrastructure used as a *timed baseline*, never as the product)
# --------------------------------------------------------------------------------------------------
def _replica_main(conn, kind, data_bin, W, H, n_inputs):
    """One single-threaded replica of the CPU reference: loads the scene, renders pose 0 (reply: digest), then renders the
    next pose of the drift path for every 'go' it receives (reply: seconds spent inside the render call)."""
    sys.path.insert(0, ROOT)
    inp = drift_inputs(n_inputs)
    out = np.empty((H, W), np.uint32)
    if kind == "reference":
        from oracle import refso
        ref = refso.RefRenderer(data_bin)
        render = lambda f: ref.update_and_render(W, H, inp[f], out)   # noqa: E731  (camera state lives in the library)
    else:
        from oracle import port
        osc = port.OracleScene(path=data_bin)
        mats = port.camera_path(inp)
        render = lambda f: out.__setitem__(slice(None), osc.render(mats[f], W, H)["pixels"])   # noqa: E731
    t0 = time.perf_counter()
    render(0)
    conn.send(("ready", time.perf_counter() - t0, frame_digest(out)))
    f = 1
    while True:
        msg = conn.recv()
        if msg != "go":
            break
        t0 = time.perf_counter()
        render(f % n_inputs)
        conn.send(("done", time.perf_counter() - t0, f))
        f += 1
    conn.close()


class CpuReplicas:
    """`n` replica processes of the reference (memory-bounded); step() = one frame per replica, in parallel."""

    def __init__(self, data_bin: str, W: int, H: int, n_inputs: int, gb_per_replica: float, cap: int = 0):
        from oracle import refso, port
        self.kind = "reference" if refso.available() else "port"
        if self.kind == "port":
            port.build()
        n = affinity_cores()
        n = max(1, min(n, int(mem_available_gb() * 0.7 / max(gb_per_replica, 0.05))))
        if cap:
            n = min(n, cap)
        self.n = n
        ctx = mp.get_context("spawn")
        self.conns, self.procs = [], []
        t0 = time.perf_counter()
        for _ in range(n):
            a, b = ctx.Pipe()
            p = ctx.Process(target=_replica_main, args=(b, self.kind, data_bin, W, H, n_inputs), daemon=True)
            p.start()
            self.conns.append(a); self.procs.append(p)
        ready = [c.recv() for c in self.conns]
        self.load_and_first_frame_s = time.perf_counter() - t0
        self.frame0 = ready[0][2]
        assert all(r[2] == self.frame0 for r in ready), "replicas disagree on pose 0"

    def step(self):
        """-> (wall seconds of the step, summed in-call seconds)."""
        t0 = time.perf_counter()
        for c in self.conns:
            c.send("go")
        busy = [c.recv()[1] for c in self.conns]
        return time.perf_counter() - t0, sum(busy)

    def close(self):
        for c in self.conns:
            try:
                c.send("stop")
            except OSError:
                pass
        for p in self.procs:
            p.join(timeout=10)
            if p.is_alive():
                p.kill()


def _c2_cpu_worker(args):
    kind, data_bin, W, H, frames, n_inputs = args
    sys.path.insert(0, ROOT)
    from swift3drenderer_b200 import scene as S
    inp = S.input_script("flythrough", n_inputs)
    want = set(frames)
    out = np.empty((H, W), np.uint32)
    if kind == "reference":
        from oracle import refso
        ref = refso.RefRenderer(data_bin)
        # the reference's camera is internal: every Input is replayed; frames outside the sample are rendered at 16 x 9
        # AFTER the sampled frame's time has been taken (the 51-triangle loop is negligible; the depth-buffer realloc and
        # its page faults on the way back to 4K are part of the reference's own resize path and stay inside the sample)
        small = np.empty((9, 16), np.uint32)
        dt = 0.0
        for f in range(max(frames) + 1):
            if f in want:
                t0 = time.perf_counter()
                ref.update_and_render(W, H, inp[f], out)
                dt += time.perf_counter() - t0
            else:
                ref.update_and_render(16, 9, inp[f], small)
        ref.close()
    else:
        from oracle import port
        osc = port.OracleScene(path=data_bin)
        mats = port.camera_path(inp)
        t0 = time.perf_counter()
        for f in frames:
            osc.render(mats[f], W, H)
        dt = time.perf_counter() - t0
    return dt, len(frames)


def c2_cpu_reference_fps(data_bin: str, W: int, H: int, n_inputs: int, sample_frames: int, workers: int):
    """frames/s of the CPU reference over `sample_frames` evenly spaced frames of the fly-through, `workers` replicas."""
    from oracle import refso, port
    kind = "reference" if refso.available() else "port"
    if kind == "port":
        port.build()
    frames = sorted(set(np.linspace(0, n_inputs - 1, sample_frames).astype(int).tolist()))
    shards = [s for s in (frames[i::workers] for i in range(workers)) if s]
    ctx = mp.get_context("spawn")
    t0 = time.perf_counter()
    with ctx.Pool(len(shards)) as pool:
        res = pool.map(_c2_cpu_worker, [(kind, data_bin, W, H, s, n_inputs) for s in shards])
    wall = time.perf_counter() - t0
    busy = max(r[0] for r in res)
    return {"kind": kind, "cores": len(shards), "frames": len(frames), "wall_s": wall, "busy_s": busy,
            "fps": len(frames) / busy, "fps_single_core": len(frames) / sum(r[0] for r in res)}


# --------------------------------------------------------------------------------------------------
# clocks
# --------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(prefix="clocks_", suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            p = [x.strip() for x in line.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1])); mx.append(float(p[2]))
            except ValueError:
                continue
            for name, val in zip(names, p[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.path)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


# --------------------------------------------------------------------------------------------------
def measured_peak_gbs():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except (KeyError, ValueError):
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic():
    """Committed ncu figures (profiles/roofline_traffic.json): dram bytes per launch by workload and kernel, or {}."""
    path = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    try:
        return json.load(open(path))
    except (OSError, ValueError):
        return {}


# Bytes per launch the general path's kernels have to move by design (DESIGN.md section 5): the logical inputs a kernel is the
# first to need, read once, the pixels written once, and — for the two kernels whose whole job is scratch — the records /
# keys they exist to move.  (The frame-level figure, B_alg of SURVEY.md 8(d), is reported separately.)
def kernel_alg_bytes(name: str, c: dict, px: int, n: int = 1, candidates: int = 0) -> int:
    return {
        "vertex_stage": 12 * c["V"],                     # positions in
        "triangle_classify": 4 * c["I"],                 # the vertex-index stream
        "cluster_cull": 48 * c["T"] // 20,               # cluster headers (one per ~20 triangles of the benchmark field)
        "cluster_front": (12 * c["V"] + 4 * c["I"] // 3) // n,   # positions + one word per triangle of the surviving clusters (~1/N on a partition)
        "direct_walk": 40 * candidates,                  # the candidate records it reads (its key reductions stay in L2)
        "shade_tiles": 12 * px,                          # 8-byte keys read, 4-byte pixels written; attributes of visible triangles come on top
    }.get(name, 0)


_RESULT_FD = None


def claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries print there too (NCCL's version banner under NCCL_DEBUG), so
    the process's stdout is pointed at stderr for its whole life and the result line goes to the original descriptor."""
    global _RESULT_FD
    if _RESULT_FD is None:
        sys.stdout.flush()
        _RESULT_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict) -> None:
    sys.stdout.flush()
    os.write(_RESULT_FD if _RESULT_FD is not None else 1, (json.dumps(line) + "\n").encode())


def log(*a):
    print("[bench]", *a, file=sys.stderr, flush=True)


# --------------------------------------------------------------------------------------------------
def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--width", type=int, default=3840)
    ap.add_argument("--height", type=int, default=2160)
    ap.add_argument("--c3-solids", type=int, default=1_000_000, help="icosahedrons of the primary workload (20 triangles each)")
    ap.add_argument("--partition", default="fused", choices=["fused", "rows", "bands"],
                    help="N > 1: interleaved tile rows stored straight into every rank's frame over NVLink peer memory (fused), "
                         "interleaved tile rows + NCCL all-gather (rows), contiguous bands + NCCL all-gather (bands)")
    ap.add_argument("--ring", type=int, default=4, help="assembled frames kept per rank (ring slots)")
    ap.add_argument("--timing-stride", type=int, default=5, help="per-kernel CUDA events on every n-th frame of the timed region (1 = every frame)")
    ap.add_argument("--c2-frames", type=int, default=600, help="frames per step of the secondary record (the recorded fly-through)")
    ap.add_argument("--c2-views-per-launch", type=int, default=24)
    ap.add_argument("--cpu-replicas", type=int, default=0, help="cap on CPU reference replicas (0 = cores, bounded by memory)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the frames of the last step that the output still holds (N = 1: the "
                         "ring's, N > 1: the assembled last pose) to DIR as .npy, a seeded pixel sample where they exceed 48 MB")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    W, H = args.width, args.height
    assert args.warmup >= 3 or args.impl == "reference" or os.environ.get("S3R_ALLOW_SHORT_WARMUP"), "W >= 3 warm-up steps"
    solids = args.c3_solids
    counts = {"V": 12 * solids, "I": 60 * solids, "A": 60 * solids, "T": 20 * solids}
    b_alg = 12 * counts["V"] + 28 * counts["A"] + 8 * counts["I"] + 4 * W * H
    config = {
        "workload": f"C3: {solids} textured icosahedrons (V={counts['V']}, T={counts['T']}, A={counts['A']}, 2 rip-map atlases), "
                    f"seed 7, at {W}x{H}, {POSES}-pose drift path; step = {POSES} frames, one pose per launch set",
        "parallelism": ("single GPU, whole frame" if world == 1 else
                        {"fused": f"screen partition x{world}: interleaved 32-pixel tile rows, rows stored into every rank's frame over "
                                  "NVLink peer memory by the shading kernel, 1-element NCCL all-reduce per frame as the fence",
                         "rows": f"screen partition x{world}: interleaved tile rows + NCCL all-gather + de-interleave",
                         "bands": f"screen partition x{world}: contiguous bands + NCCL all-gather"}[args.partition]),
        "frames_per_step": POSES,
        "l2": f"inputs larger than L2: {b_alg / 1e6:.0f} MB of scene + frame per frame against the 126 MB L2; outputs cycle "
              f"through a ring of {args.ring} frames",
    }

    # ---------------------------------------------------------------------------------------------
    if args.impl == "reference":
        if rank != 0:
            return
        t_start = time.perf_counter()
        data_bin = c3_data_bin(solids)
        reps = CpuReplicas(data_bin, W, H, 4096, gb_per_replica=8.0 * solids / 1e6 + 0.3, cap=args.cpu_replicas)
        log(f"reference arm: {reps.n} replicas ({reps.kind}), load + pose 0 took {reps.load_and_first_frame_s:.1f} s")
        for _ in range(min(args.warmup, 1)):
            reps.step()
        walls, busys = [], []
        for _ in range(args.steps):
            w, b = reps.step()
            walls.append(w); busys.append(b)
        reps.close()
        frames = reps.n * args.steps
        fps = frames / sum(walls)
        line = {
            "impl": "reference", "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * sum(walls) / len(walls), "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
            "cpu_baseline": {"value": fps, "unit": UNIT, "cores": reps.n, "kind": reps.kind,
                             "sample": f"{reps.n} frames per step: one single-threaded replica per core (bounded by memory), each "
                                       f"rendering the next pose of the drift path at {W}x{H}; scene load and pose 0 are warm-up",
                             "single_core_fps": frames / sum(busys)},
            "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "frame0_digest": reps.frame0, "wall_s": time.perf_counter() - t_start,
        }
        if not args.no_secondary:
            from swift3drenderer_b200 import assets
            cores = affinity_cores()
            c = c2_cpu_reference_fps(assets.ensure_shipped_data_bin(), W, H, args.c2_frames, min(args.c2_frames, max(24, 3 * cores)), cores)
            line["secondary"] = {"metric": C2_METRIC, "value": c["fps"], "unit": UNIT, "cores": c["cores"], "kind": c["kind"],
                                 "sample": f"{c['frames']} evenly spaced frames of the fly-through, one replica per core",
                                 "single_core_fps": c["fps_single_core"]}
        emit(line)
        return

    # ---------------------------------------------------------------------------------------------
    import torch
    import torch.distributed as dist
    from swift3drenderer_b200 import assets, multigpu, renderer as R, scene as S

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the renderer has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    os.environ["S3R_DEVICE"] = str(local_rank)   # the drop-in (updateAndRender) of this rank renders on this rank's GPU

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(x: float) -> float:
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    R.build_library()
    if rank == 0:
        t0 = time.perf_counter()
        data_bin = c3_data_bin(solids)
        log(f"C3 data.bin ready in {time.perf_counter() - t0:.1f} s: {data_bin}")
    barrier()
    data_bin = c3_data_bin(solids)
    t0 = time.perf_counter()
    r = R.Renderer(local_rank)
    r.load_scene_file(data_bin)
    log(f"rank {rank}: scene loaded in {time.perf_counter() - t0:.1f} s")
    inputs = drift_inputs(POSES)
    mats = R.camera_path(inputs)
    stream = torch.cuda.Stream(dev)   # a real (non-default) stream: the renderer launches on it, the events time it
    torch.cuda.set_stream(stream)

    # ---- the step --------------------------------------------------------------------------------
    assembled = [None]   # callable -> this rank's assembled frame of the last pose (host array)
    pf = None
    comm = None
    if world == 1:
        ring = torch.empty((args.ring, H, W), dtype=torch.int32, device=dev)
        k = [0]

        def run_step():
            for f in range(POSES):
                r.render_device(mats[f], W, H, ring[k[0] % args.ring].data_ptr(), stream=stream.cuda_stream)
                k[0] += 1
        assembled[0] = lambda: ring[(k[0] - 1) % args.ring].cpu().numpy().view(np.uint32)
    elif args.partition == "fused":
        pf = multigpu.PeerFrames(r, H, W, rank, world, dev, ring=args.ring)
        last = [0]

        def run_step():
            for f in range(POSES):
                last[0] = pf.render(mats[f], stream=stream.cuda_stream)
                pf.fence_async()
        assembled[0] = lambda: pf.read(last[0])
        comm = {"kind": "peer stores (st.global.v4 over NVLink, CUDA IPC) from shade_tiles + 1-element NCCL all-reduce per frame",
                "bytes_per_frame_per_rank_sent": int(4 * W * H / world * (world - 1)),
                "bytes_per_frame_total": int(4 * W * H * (world - 1))}
    elif args.partition == "rows":
        asm = multigpu.InterleavedAssembler(H, W, rank, world, dev, R.tile_height())
        full = [None]

        def run_step():
            for f in range(POSES):
                r.render_device_rows(mats[f], W, H, world, rank, asm.mine.data_ptr(), stream=stream.cuda_stream)
                full[0] = asm.gather()
        assembled[0] = lambda: full[0].cpu().numpy().view(np.uint32)
        comm = {"kind": "NCCL all-gather of compacted tile rows + index_select", "bytes_per_frame_total": int(4 * W * H * (world - 1))}
    else:
        frames = torch.zeros((args.ring, H, W), dtype=torch.int32, device=dev)
        y0, y1 = multigpu.band_edges(H, world)[rank]
        assert multigpu.equal_bands(H, world), "--partition bands needs H % N == 0"
        k = [0]
        full = [None]

        def run_step():
            for f in range(POSES):
                fr = frames[k[0] % args.ring]
                r.render_device(mats[f], W, H, fr[y0:y1].data_ptr(), y0=y0, y1=y1, stream=stream.cuda_stream)
                full[0] = multigpu.gather_bands_inplace(fr, rank, world)
                k[0] += 1
        assembled[0] = lambda: full[0].cpu().numpy().view(np.uint32)
        comm = {"kind": "in-place NCCL all-gather of contiguous bands", "bytes_per_frame_total": int(4 * W * H * (world - 1))}

    def drain():
        if pf is not None:
            pf.drain()
        torch.cuda.synchronize(dev)

    for _ in range(args.warmup):
        run_step()
        drain()
        while max_over_ranks(1.0 if r.finish() else 0.0) > 0:   # capacity regrowth happens here, outside the timed region
            run_step()
            drain()
    # per-kernel CUDA events on every args.timing_stride-th frame of the timed region: an event after every launch keeps a
    # kernel from being placed while its predecessor drains (programmatic dependent launch), so timing every frame would
    # slow down what it measures; 5 is coprime to the 8 poses, every pose is sampled equally often
    r.set_option("timing", max(1, args.timing_stride))
    r.timing(reset=True)
    clocks = ClockSampler(local_rank)
    barrier()
    if rank == 0:
        clocks.start()
    launches0 = r.kernel_launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        run_step()
    if pf is not None:
        pf.join(stream)          # the timed region ends when the last frame's fence has completed
    e1.record(stream)
    barrier()
    assert not r.finish(), "capacity overflow inside the timed region"
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    launches = r.kernel_launches - launches0
    kt = r.kernel_timing()
    stage = r.timing(reset=True)
    r.set_option("timing", 0)
    clock_info = clocks.stop() if rank == 0 else None
    frames_total = args.steps * POSES
    value = frames_total / (ms_total / 1e3)

    # ---- checks (untimed): the assembled frame equals the whole frame; digest of pose 0 for the cross-arm comparison
    whole_last = r.render(mats[POSES - 1], W, H)[0]
    last_frame = assembled[0]()
    same = bool(np.array_equal(last_frame, whole_last))
    if args.dump_outputs and rank == 0:
        if world == 1:
            held = min(args.ring, POSES)
            dump_outputs(args.dump_outputs, range(POSES - held, POSES),
                         [ring[(k[0] - held + j) % args.ring].cpu().numpy().view(np.uint32) for j in range(held)])
        else:
            dump_outputs(args.dump_outputs, [POSES - 1], [last_frame])
    banded_equals_whole = bool(max_over_ranks(0.0 if same else 1.0) == 0.0)
    frame0 = frame_digest(r.render(mats[0], W, H)[0])
    stats_last = r.stats(0)

    # ---- e2e: the reference-facing plugin call with host buffers ------------------------------------------------------
    # N = 1: the drop-in on this GPU.  N > 1: ONE caller (rank 0) whose updateAndRender drives all N GPUs from one process
    # (S3R_DEVICES: interleaved tile rows, every GPU copies its rows over its own PCIe link into the caller's buffer); the
    # other ranks wait on a host-side (gloo) barrier so that nothing of theirs runs on the GPUs meanwhile.
    e2e = None
    host_group = dist.new_group(backend="gloo") if world > 1 else None
    if not args.no_e2e:
        e2e = run_e2e(R, data_bin, inputs, POSES, args.steps, W, H, rank, world, frame0, host_group, barrier)

    # ---- secondary record: C2 (data.bin demo scene, 600-frame fly-through), frame-parallel ------------------------
    secondary = None
    if not args.no_secondary:
        secondary = run_c2(args, r, rank, local_rank, world, dev, stream, barrier, max_over_ranks, host_group)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline ----------------------------------------------------------------------------------------------------
    peak, peak_src = measured_peak_gbs()
    traffic = ncu_traffic().get("c3", {})
    px_rank = W * H // world
    kernels = {}
    for name, rec in kt.items():
        n = max(rec["launches"], 1)
        us = rec["ms"] * 1e3 / n
        alg = kernel_alg_bytes(name, counts, px_rank, world, stats_last["setups"])
        # share of the timed region: the kernel's average duration x its launches in the whole region (timed frames are a sample)
        scale = frames_total / max(stage["chunks"], 1)
        kernels[name] = {"avg_launch_us": us, "launches": rec["launches"], "share_of_step": rec["ms"] * scale / ms_total if ms_total else None,
                         "algorithmic_bytes_per_launch": alg, "achieved_gbs": alg / us / 1e3 if us > 0 else None,
                         "frac": alg / us / 1e3 / peak if us > 0 else None,
                         "ncu_dram_bytes_per_launch": traffic.get(name if world == 1 else name + f"@{world}")}
    dominant = max(kernels, key=lambda n: kernels[n]["avg_launch_us"]) if kernels else None
    t_frame_s = ms_total / 1e3 / frames_total
    # a rank of the screen partition rejects the clusters that miss its rows, so what it must read is its 1/N of the frame's
    # algorithmic bytes; SURVEY.md 8(d) assumed every GPU scans all geometry (12V + 28A + 8I + 4WH/N) — reported beside it
    b_alg_rank = (12 * counts["V"] + 28 * counts["A"] + 8 * counts["I"]) // world + 4 * px_rank
    b_alg_redundant = 12 * counts["V"] + 28 * counts["A"] + 8 * counts["I"] + 4 * px_rank
    roofline = None
    if dominant:
        dk = kernels[dominant]
        roofline = {
            "bound": "hbm", "kernel": dominant, "achieved": dk["achieved_gbs"], "peak": peak, "unit": "GB/s", "frac": dk["frac"],
            "traffic": dk["ncu_dram_bytes_per_launch"], "peak_source": peak_src,
            "algorithmic_bytes_per_launch": dk["algorithmic_bytes_per_launch"], "avg_launch_us": dk["avg_launch_us"],
            "share_of_step": dk["share_of_step"],
            "frame": {"algorithmic_bytes_per_gpu": b_alg_rank, "achieved": b_alg_rank / t_frame_s / 1e9,
                      "frac": b_alg_rank / t_frame_s / 1e9 / peak,
                      "ncu_dram_bytes_per_frame": traffic.get("frame" if world == 1 else f"frame@{world}"),
                      "survey_redundant_geometry": {"algorithmic_bytes_per_gpu": b_alg_redundant, "frac": b_alg_redundant / t_frame_s / 1e9 / peak},
                      "note": "B_alg = (12V + 28A + 8I + 4WH) / N per GPU: a rank skips the clusters that miss its rows.  SURVEY.md 8(d) "
                              "assumed every GPU scans all geometry (12V + 28A + 8I + 4WH/N); that figure is given beside it and can exceed "
                              "1 because the work it counts is not done.  The kernels also read attributes of visible triangles only, so "
                              "the DRAM traffic of a frame (ncu) is below B_alg"},
            "kernels": kernels,
        }

    # ---- CPU baseline (rank 0, N = 1 only): bounded sample of the same workload ------------------------------------
    cpu_baseline = None
    if not args.no_cpu and world == 1:
        reps = CpuReplicas(data_bin, W, H, 4096, gb_per_replica=8.0 * solids / 1e6 + 0.3, cap=args.cpu_replicas)
        wall, busy = reps.step()
        reps.close()
        cpu_baseline = {"value": reps.n / wall, "unit": UNIT, "cores": reps.n, "kind": reps.kind,
                        "sample": f"{reps.n} frames: one single-threaded replica per core (bounded by memory), each rendering pose 1 of "
                                  f"the drift path at {W}x{H} once; scene load and pose 0 are warm-up ({reps.load_and_first_frame_s:.0f} s)",
                        "single_core_fps": reps.n / busy, "frame0_digest": reps.frame0,
                        "frame0_equals_b200": reps.frame0 == frame0}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": config,
        "mpixels_per_s": value * W * H / 1e6, "mtriangles_per_s": value * counts["T"] / 1e6,
        "clocks": clock_info, "e2e": e2e, "gpu_launches": int(launches),
        "roofline": roofline, "cpu_baseline": cpu_baseline,
        "banded_equals_whole": banded_equals_whole, "frame0_digest": frame0, "comm": comm,
        "stage_ms_per_frame": {"geometry": stage["geometry_ms"] / max(stage["chunks"], 1), "raster": stage["raster_ms"] / max(stage["chunks"], 1)},
        "stats_last_pose": stats_last, "secondary": secondary,
    }
    emit(line)
    if world > 1:
        dist.destroy_process_group()


def run_e2e(R, data_bin, inputs, frames, steps, W, H, rank, world, frame0, host_group, barrier, warm_frames=None):
    """frames/s through updateAndRender with the caller's pageable double buffer (main.swift:117-118), `steps` passes over
    `frames` Inputs.  Returns the e2e record on rank 0 (None elsewhere)."""
    import torch.distributed as dist
    rec = None
    barrier()
    if rank == 0:
        t0 = time.perf_counter()
        d = R.DropIn(data_bin, devices=",".join(str(k) for k in range(world)) if world > 1 else None)
        double = np.zeros((2, H, W), np.uint32)   # pageable, alternated per call
        d.update_and_render(W, H, inputs[0], out=double[0])   # scene load (on every GPU)
        first = frame_digest(double[0])
        for f in range(1, warm_frames or 2 * frames):   # warm: capacity growth, staging / registration, worker threads
            d.update_and_render(W, H, inputs[f % frames], out=double[f & 1])
        log(f"drop-in on {d.n_devices} GPU(s) ready in {time.perf_counter() - t0:.1f} s")
        t0 = time.perf_counter()
        for _ in range(steps):
            d.reset_camera()
            for f in range(frames):
                d.update_and_render(W, H, inputs[f], out=double[f & 1])
        dt = time.perf_counter() - t0
        multi = d.n_devices > 1
        rec = {"value": steps * frames / dt, "unit": UNIT, "h2d_bytes_per_step": 48 * frames,
               "d2h_bytes_per_step": (4 if multi else 3) * W * H * frames, "gpus": d.n_devices,
               "call": "updateAndRender(const PixelData*, const Input*) on a private render.so beside the scene's data.bin, caller's "
                       "pageable double buffer, synchronous per frame; " +
                       ("one process drives all GPUs (S3R_DEVICES): interleaved tile rows, one host thread per GPU, each GPU "
                        "copies its rows D2H over its own PCIe link straight into the caller's buffer (registered on first sight, "
                        "sentinel-checked)" if multi else
                        "not registered (S3R_PIN_HOST unset): the frame is rendered in row bands, each band copied D2H as 24-bit "
                        "pixels into the library's pinned staging while the next renders, copy workers expand it into the "
                        "caller's buffer"),
               "first_frame_digest": first, "first_frame_equals_device_path": (first == frame0) if frame0 else None,
               "last_frame_digest": frame_digest(double[(frames - 1) & 1])}
        d.close()
    if world > 1:
        dist.barrier(group=host_group)
    return rec


def run_c2(args, r, rank, local_rank, world, dev, stream, barrier, max_over_ranks, host_group):
    """The secondary record: BASELINE.json configs[1] — the demo scene at 4K over the recorded fly-through; every rank renders
    the full fly-through (frame-parallel replicas, no data-path collective)."""
    import torch
    from swift3drenderer_b200 import assets, renderer as R, scene as S
    W, H, F, vpl = args.width, args.height, args.c2_frames, args.c2_views_per_launch
    steps = args.steps
    data_bin = assets.ensure_shipped_data_bin()
    sc = S.read_data_bin(data_bin)
    counts = sc.counts()
    b_alg = 12 * counts["V"] + 28 * counts["A"] + 8 * counts["I"] + 4 * W * H
    r2 = R.Renderer(local_rank)
    r2.load_scene_file(data_bin)
    inp = S.input_script("flythrough", F)
    mats = R.camera_path(inp)
    ring_n = 4
    ring = torch.empty((ring_n, vpl, H, W), dtype=torch.int32, device=dev)

    def run_step():
        k = 0
        for f0 in range(0, F, vpl):
            r2.render_device(mats[f0:f0 + vpl], W, H, ring[k % ring_n].data_ptr(), stream=stream.cuda_stream)
            k += 1

    for _ in range(3):
        run_step()
        while r2.finish():
            run_step()
    r2.set_option("timing", 1)
    r2.timing(reset=True)
    barrier()
    launches0 = r2.kernel_launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        run_step()
    e1.record(stream)
    barrier()
    assert not r2.finish()
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    launches = r2.kernel_launches - launches0
    kt = r2.kernel_timing()
    r2.timing(reset=True)
    r2.set_option("timing", 0)
    value = world * steps * F / (ms_total / 1e3)

    e2e = None
    if not args.no_e2e:
        e2e = run_e2e(R, data_bin, inp, F, steps, W, H, rank, world, None, host_group, barrier, warm_frames=12)
    r2.close()
    if rank != 0:
        return None
    peak, peak_src = measured_peak_gbs()
    rec = kt.get("tile_raster", {"ms": 0.0, "launches": 0})
    launch_us = rec["ms"] * 1e3 / max(rec["launches"], 1)
    tr = ncu_traffic().get("c2", {}).get("tile_raster")
    roofline = {"bound": "hbm", "kernel": "tile_raster", "achieved": b_alg * vpl / launch_us / 1e3 if launch_us else None, "peak": peak,
                "unit": "GB/s", "frac": b_alg * vpl / launch_us / 1e3 / peak if launch_us else None,
                "traffic": int(tr["dram_bytes_per_launch"] / tr["poses_per_launch"] * vpl) if tr else None,
                "issue_slot_frac": tr.get("issue_active_frac") if tr else None, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": b_alg * vpl, "avg_launch_us": launch_us,
                "share_of_step": rec["ms"] / ms_total if ms_total else None,
                "note": "C2 is shading-bound (IEEE div/sqrt per pixel, issue slots), not HBM-bound: 33 MB per frame"}
    cpu = None
    if not args.no_cpu and world == 1:
        cores = affinity_cores()
        c = c2_cpu_reference_fps(data_bin, W, H, F, min(F, max(24, 3 * cores)), cores)
        cpu = {"value": c["fps"], "unit": UNIT, "cores": c["cores"], "kind": c["kind"],
               "sample": f"{c['frames']} evenly spaced frames of the {F}-frame fly-through, one single-threaded replica per core",
               "single_core_fps": c["fps_single_core"]}
    return {"metric": C2_METRIC, "value": value, "unit": UNIT, "scaling": "weak (frame-parallel replicas)", "steps": steps,
            "ms_per_step": ms_total / steps, "frames_per_step": F, "views_per_launch": vpl, "gpu_launches": int(launches),
            "workload": f"C2: reference data.bin scene (V={counts['V']}, T={counts['T']}) at {W}x{H}, {F}-frame recorded fly-through",
            "e2e": e2e, "roofline": roofline, "cpu_baseline": cpu}


if __name__ == "__main__":
    main()
