"""Frames beyond 4K, up to the 65535-pixel limit of the ABI, against the oracle, bit for bit, frames and statistics.

The renderer accepts any frame up to 65535 x 65535.  Several of its parts only behave differently above 4K: box bounds
packed into 16-bit fields (the top bit is set from 32768 on), exact jumps of up to 65534 steps with deltas near
1/65535, the 1 GB budget of the small-scene span tables (sized for the largest batch a renderer has submitted), the
per-view cap of the general path's row-start table, tensor-map and row-copy write-out of wide rows, 2048 tile rows
dealt to interleaved phases, and the host transport's bands and slices.  The CPU tests at the top prove from the oracle
alone that every scene and frame reaches what it exists for; the GPU tests below compare the CUDA path with the oracle.
Every GPU test uses a renderer of its own: the largest batch a renderer has seen changes its later decisions."""
import numpy as np
import pytest

from swift3drenderer_b200 import scene as S
from test_gpu_vis_edges import ROUTES, _Mesh, assert_same, assert_stats, box_sizes, render_rows, set_route, still

# wide and tall, multiples of 16 (tensor-map write-out) and not (bulk row copies), 1-pixel extremes
SIZES = [(4097, 33), (7680, 4320), (7681, 4321), (16384, 2048), (65535, 96), (96, 65535), (65535, 1), (1, 65535)]
SIZE_IDS = [f"{W}x{H}" for W, H in SIZES]
TOP_BIT = 32768
SPAN_MAX, TILE_W = 8, 64          # csrc/pipeline.cuh
ROWTAB_CAP = 8 << 20              # row-start floats per view of the general path (one view: csrc/renderer.cu)
GENERAL_SIZES = [(7680, 4320), (16384, 8192)]


def _shipped_views(renderer_lib_or_port):
    return renderer_lib_or_port.camera_path(S.input_script("flythrough", 600))


def shipped_view(mats, W, H):
    """A view of the shipped scene that sees its textured floor at this frame size.  A single row would sample the
    floor's coarsest texture level (a few colours): that frame is zoomed 300 times and tilted down instead, which any
    3 x 4 matrix may do."""
    m = mats[110]
    if H == 1:
        a = m.reshape(3, 4).astype(np.float64).copy()
        a[1] -= 0.3 * a[2]
        a[:2] *= 300.0
        m = a.reshape(12).astype(np.float32)
    return m


def general_scenes():
    return (("clip", lambda: S.clip_stress_scene(3000)),
            ("dense", lambda: S.icosahedron_field(20000, seed=9, extent=40, r_range=(0.3, 1.0))))


def general_view(mats):
    """Flythrough pose 350 looks into both general-path scenes from close by: at 16384 x 8192 the clip scene's
    tile-path triangles need more row-start floats than one view's table holds."""
    return mats[350]


# ------------------------------------------------------------------------------------------------------------------
# the probe scene: triangles placed in raster space of a W x H frame seen by the still camera
# ------------------------------------------------------------------------------------------------------------------
THRESHOLDS = (15, 16, 17, 127, 128, 129)


def probe_scene(W, H, n_filler=2100, seed=3):
    """Probes along the long axis of the frame (and along the other one when it is at least 300 px), near its far
    border: boxes that end on the last column (row) and start at 32768 or later, a triangle across the whole frame (its
    box over 60 000 px wide on the 65535 frames, well over flat_max), boxes 15/16/17 and 127/128/129 px long, two
    identical copies first and last in the list (an exact depth tie at every pixel: the first must win), slivers with
    the reference's area just above 10, then ``n_filler`` mid-size triangles behind them all (over 1920 triangles: the
    general path; a few hundred: the fused small-scene path).  Returns (scene, names): names[k] says what triangle k is."""
    rng = np.random.RandomState(seed)
    mesh = _Mesh(W, H)
    names = []
    late = []   # (name, pts, depth, rgb) added after the filler

    def colour():
        return tuple(rng.uniform(40, 255, 3))

    def axis(swap, L, Sh):
        def xy(pts):
            p = np.asarray(pts, np.float64)
            return p[:, ::-1] if swap else p

        def add(name, pts, depth):
            mesh.tri(xy(pts), depth, colour())
            names.append(name)

        tag = "y" if swap else "x"
        vc = Sh // 2 + 0.5                      # the centre row across the long axis (a pixel centre)
        hv = min(4.0, Sh / 2.0 + 2.0)           # half height of the probes across it (covers the row of 1-px frames)
        # boxes ending on the last column with their start at or beyond 32768 (the top bit of both packed fields)
        if L - 1 - 3000 >= TOP_BIT:
            for k, u0 in enumerate((TOP_BIT, TOP_BIT + 1, L - 1 - 3000, L - 1 - 200, L - 1 - 20, L - 1)):
                add(f"{tag}_top{k}", [(u0 + 0.5, vc - hv), (L + 20.0, vc - hv / 2), (u0 + 0.5, vc + hv)], 4.0 + 0.1 * k)
        # the whole long axis, behind everything: the tile kernel enters it with jumps up to L - 1 steps
        add(f"{tag}_across", [(-40.0, vc - hv - 3), (L + 40.0, vc - hv - 1), (L / 2.0, vc + hv + 40)], 13.0)
        add(f"{tag}_across_slant", [(-5.0, -3.0), (L + 5.0, vc), (-5.0, Sh + 3.0)], 13.5)
        # routing thresholds near the far border
        for k, d in enumerate(THRESHOLDS):
            u0 = L - 1 - d - 10 - 160 * k
            if u0 >= 0:
                add(f"{tag}_w{d}", [(u0 + 0.5, vc - min(hv, 3.0)), (u0 + d + 0.5, vc), (u0 + 0.5, vc + min(hv, 3.0))], 5.0)
        # exact depth tie: the same triangle first and last in the list, near the far border, two sizes
        for k, d in enumerate((40, 200)):
            u0 = L - 1 - d - 30 - 1200 * k
            if u0 >= 0:
                pts = [(u0 + 0.5, vc - hv), (u0 + d + 0.5, vc - hv / 3), (u0 + d / 3.0, vc + hv)]
                mesh.tri(xy(pts), 3.0, (250.0, 20.0, 20.0))
                names.append(f"{tag}_tie{k}_first")
                late.append((f"{tag}_tie{k}_last", xy(pts), 3.0, (20.0, 250.0, 20.0)))
        # slivers just above the area cull, along the far end
        for _ in range(40):
            c = np.array([L - 1 - rng.uniform(2, min(L - 2, 2000)), vc + rng.uniform(-hv / 2, hv / 2)])
            length, th = rng.uniform(6, 40), rng.uniform(0, np.pi)
            u = np.array([np.cos(th), np.sin(th)])
            wid = rng.uniform(10.5, 12.5) / length   # the reference's area (twice the triangle's) just above 10
            add(f"{tag}_sliver", [c - u * length / 2, c + u * length / 2, c + np.array([-u[1], u[0]]) * wid], 3.5)

    L, Sh = max(W, H), min(W, H)
    axis(H > W, L, Sh)
    if Sh >= 300:
        axis(not (H > W), Sh, L)
    for _ in range(n_filler):
        x, y = rng.uniform(-20, W), rng.uniform(-20, H)
        sx, sy = rng.uniform(4, 60), rng.uniform(4, 60)
        if W < 20:
            x = rng.uniform(-sx + 0.5, W - 0.5)
        if H < 20:
            y = rng.uniform(-sy + 0.5, H - 0.5)
        mesh.tri([(x, y), (x + sx, y + rng.uniform(0, 8)), (x + rng.uniform(0, 8), y + sy)], rng.uniform(7, 12), colour())
        names.append("filler")
    for name, pts, depth, rgb in late:
        mesh.tri(pts, depth, rgb)
        names.append(name)
    return mesh.scene(), names


def _boxes(setups):
    return {int(t): (int(setups["xmin"][k]), int(setups["xmax"][k]), int(setups["ymin"][k]), int(setups["ymax"][k]))
            for k, t in enumerate(setups["order"])}


# ------------------------------------------------------------------------------------------------------------------
# premise checks (CPU): every scene and frame reaches what it exists for
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("W,H", SIZES, ids=SIZE_IDS)
def test_shipped_scene_premise(W, H, oracle_port):
    """The small-scene path sees hundreds of distinct colours at every frame size, extreme aspect ratios included."""
    sc = S.shipped_scene(1)
    assert sc.n_triangles <= 1920
    m = shipped_view(_shipped_views(oracle_port), W, H)
    o = oracle_port.OracleScene(sc).render(m, W, H)
    assert len(np.unique(o["pixels"])) >= 300, (W, H, len(np.unique(o["pixels"])))


@pytest.mark.parametrize("W,H", SIZES, ids=SIZE_IDS)
def test_probe_scene_premise(W, H, oracle_port):
    sc, names = probe_scene(W, H)
    assert sc.n_triangles > 1920
    m = oracle_port.camera_path(still())[0]
    o = oracle_port.OracleScene(sc).render(m, W, H, want_setups=True, want_winner=True)
    box = _boxes(o["setups"])
    win = o["winner"]
    idx = {}
    for k, n in enumerate(names):
        idx.setdefault(n, []).append(k)
    tags = ["y" if H > W else "x"] + (["x" if H > W else "y"] if min(W, H) >= 300 else [])
    for tag in tags:
        L = H if tag == "y" else W
        lo, hi = (2, 3) if tag == "y" else (0, 1)
        if L - 1 - 3000 >= TOP_BIT:
            tops = [box[k] for n, ks in idx.items() if n.startswith(f"{tag}_top") for k in ks]
            assert len(tops) == 6 and all(b[hi] == L - 1 and b[lo] >= TOP_BIT for b in tops), tops
            for n in (f"{tag}_top0", f"{tag}_top3"):
                assert (win == idx[n][0]).any(), f"{n} wins no pixel"
        across = box[idx[f"{tag}_across"][0]]
        assert across[lo] == 0 and across[hi] == L - 1
        if L == 65535:
            assert across[hi] - across[lo] > 60000
        assert (win == idx[f"{tag}_across"][0]).any() and (win == idx[f"{tag}_across_slant"][0]).any()
        for d in THRESHOLDS:
            if f"{tag}_w{d}" in idx:
                b = box[idx[f"{tag}_w{d}"][0]]
                assert b[hi] - b[lo] == d and b[hi] >= L - 1 - 10 - 160 * 6 - 129, (tag, d, b)
                assert max(b[1] - b[0], b[3] - b[2]) == d   # the routing size is d
        assert all(f"{tag}_w{d}" in idx for d in (15, 16, 17)) and (L < 1000 or f"{tag}_w129" in idx)
        # exact ties: the first copy wins every pixel the two share, the last one none (their colours differ)
        for k in (0, 1):
            if f"{tag}_tie{k}_first" in idx:
                first, last = idx[f"{tag}_tie{k}_first"][0], idx[f"{tag}_tie{k}_last"][0]
                assert box[first] == box[last] and last - first > 2000   # the filler lies between them
                assert (win == first).any() and not (win == last).any()
        slivers = [box[k] for k in idx[f"{tag}_sliver"] if k in box]
        assert len(slivers) >= 20
    st = o["setups"]
    sliver_area = st["area"][np.isin(st["order"], [k for n, ks in idx.items() if n.endswith("_sliver") for k in ks])]
    assert len(sliver_area) >= 20 and (sliver_area < 13).all() and (sliver_area >= 10).all()
    # the tile kernel's jumps: some tile-path box starts more than 4096 px before the far end
    bw, bh = box_sizes(st)
    assert (np.maximum(bw, bh) >= 4096).any() or max(W, H) < 4096


@pytest.mark.parametrize("W,H", SIZES, ids=SIZE_IDS)
def test_probe_scene_small_variant_premise(W, H, oracle_port):
    """The sub-1920-triangle variant keeps every probe and takes the fused small-scene path."""
    sc, names = probe_scene(W, H, n_filler=300)
    assert sc.n_triangles <= 1920
    _, big_names = probe_scene(W, H)
    assert [n for n in names if n != "filler"] == [n for n in big_names if n != "filler"]


def test_general_path_row_start_table_overflows_at_16k(oracle_port):
    """At 16384 x 8192 the clip scene's triangles routed to the tile kernel (boxes of flat_max = 128 px or more) need
    more row-start floats (3 per box row) than one view's table holds: the table overflows by itself."""
    m = general_view(oracle_port.camera_path(S.input_script("flythrough", 600)))
    o = oracle_port.OracleScene(S.clip_stress_scene(3000)).render(m, 16384, 8192, want_setups=True)
    bw, bh = box_sizes(o["setups"])
    tile = (bw >= 128) | (bh >= 128)
    need = int((3 * (bh[tile] + 1)).sum())
    assert need > ROWTAB_CAP, (need, ROWTAB_CAP)
    assert len(np.unique(o["pixels"])) > 100000


def span_table_bytes(W, H, views):
    """Span tables of a small-scene batch (csrc/renderer.cu ensure_scratch): SPAN_MAX x tile columns x 3 x span_h."""
    return SPAN_MAX * ((W + TILE_W - 1) // TILE_W) * 3 * ((H + 31) & ~31) * views * 4


SPAN_BATCH = 22


def test_span_table_budget_premise():
    """One 7680 x 4320 view fits the 1 GB span-table budget; a batch of SPAN_BATCH does not."""
    assert span_table_bytes(7680, 4320, 1) <= 1 << 30 < span_table_bytes(7680, 4320, SPAN_BATCH)


# ------------------------------------------------------------------------------------------------------------------
# GPU: frames and statistics against the oracle
# ------------------------------------------------------------------------------------------------------------------
def _device_frame(r, torch, m, W, H, y0=0, y1=None):
    y1 = H if y1 is None else y1
    n = np.asarray(m).reshape(-1, 12).shape[0]
    out = torch.full((n, y1 - y0, W), 0x55555555, dtype=torch.int32, device="cuda:0")
    for _ in range(4):   # a fresh renderer's first general-path frame may overflow a capacity: finish() asks for a repeat
        r.render_device(m, W, H, out.data_ptr(), y0=y0, y1=y1)
        if not r.finish():
            break
    assert r.stats()["overflow"] == 0
    return out.cpu().numpy().view(np.uint32)


def _band(H):
    """A band that cuts tile rows (32 px) at both ends, or the whole frame when it is too short for one."""
    y0, y1 = H // 3 + 5, (2 * H) // 3 + 1
    return (y0, y1) if y0 < y1 else (0, H)


@pytest.mark.gpu
@pytest.mark.parametrize("W,H", SIZES, ids=SIZE_IDS)
def test_small_path_large_frames(W, H, renderer_lib, oracle_port):
    """Shipped scene (fused small-scene path, textured floor): device output, a band that cuts tile rows, interleaved
    tile rows over 3 phases and the host path."""
    import torch
    sc = S.shipped_scene(1)
    m = shipped_view(_shipped_views(renderer_lib), W, H)
    o = oracle_port.OracleScene(sc).render(m, W, H)
    r = renderer_lib.Renderer(0)
    try:
        r.load_scene(sc)
        what = f"shipped {W}x{H}"
        assert_same(_device_frame(r, torch, m, W, H)[0], o["pixels"], f"{what} device")
        assert_stats(r.stats(), o, f"{what} device")
        y0, y1 = _band(H)
        assert_same(_device_frame(r, torch, m, W, H, y0, y1)[0], o["pixels"][y0:y1], f"{what} band {y0}..{y1}")
        assert_same(render_rows(r, renderer_lib, m, W, H, 3), o["pixels"], f"{what} 3 interleaved phases")
        assert_same(r.render(m, W, H)[0], o["pixels"], f"{what} host")
        assert_stats(r.stats(), o, f"{what} host")
    finally:
        r.close()


@pytest.mark.gpu
@pytest.mark.parametrize("W,H", SIZES, ids=SIZE_IDS)
def test_probe_scene_large_frames(W, H, renderer_lib, oracle_port):
    """The probe scene on the general path under every routing, with a band and 3 interleaved phases, and its
    sub-1920-triangle variant on the fused small-scene path: the same probes through both."""
    import torch
    m = renderer_lib.camera_path(still())[0]
    y0, y1 = _band(H)
    for n_filler, fused in ((2100, 1), (300, 1), (300, 0)):
        sc, _ = probe_scene(W, H, n_filler=n_filler)
        o = oracle_port.OracleScene(sc).render(m, W, H)
        r = renderer_lib.Renderer(0)
        try:
            r.set_option("fused_small", fused)
            r.load_scene(sc)
            name = f"probes {W}x{H} T={sc.n_triangles} fused_small={fused}"
            for route in (ROUTES if sc.n_triangles > 1920 or not fused else ROUTES[:1]):
                set_route(r, route)
                what = f"{name} route {route}"
                assert_same(r.render(m, W, H)[0], o["pixels"], what)
                assert_stats(r.stats(), o, what)
            assert_same(_device_frame(r, torch, m, W, H)[0], o["pixels"], f"{name} device")
            assert_same(_device_frame(r, torch, m, W, H, y0, y1)[0], o["pixels"][y0:y1], f"{name} band {y0}..{y1}")
            assert_same(render_rows(r, renderer_lib, m, W, H, 3), o["pixels"], f"{name} 3 interleaved phases")
        finally:
            r.close()


@pytest.mark.gpu
@pytest.mark.parametrize("W,H", GENERAL_SIZES, ids=[f"{W}x{H}" for W, H in GENERAL_SIZES])
@pytest.mark.parametrize("which", [0, 1], ids=["clip", "dense"])
def test_general_path_8k_16k(which, W, H, renderer_lib, oracle_port):
    """Clip-stress scene and dense icosahedron field on the general path under every routing, 3 bands, interleaved
    rows over 2 and 8 phases.  At 16384 x 8192 the row-start table overflows by itself (see the premise)."""
    name, build = general_scenes()[which]
    sc = build()
    m = general_view(renderer_lib.camera_path(S.input_script("flythrough", 600)))
    o = oracle_port.OracleScene(sc).render(m, W, H)
    r = renderer_lib.Renderer(0)
    try:
        r.load_scene(sc)
        for route in ROUTES:
            set_route(r, route)
            what = f"{name} {W}x{H} route {route}"
            assert_same(r.render(m, W, H)[0], o["pixels"], what)
            assert_stats(r.stats(), o, what)
        set_route(r, (2, 1, 1, 128))
        edges = [0, H // 3 + 7, (2 * H) // 3 + 1, H]
        parts = [r.render(m, W, H, y0=a, y1=b)[0] for a, b in zip(edges[:-1], edges[1:])]
        assert_same(np.concatenate(parts, 0), o["pixels"], f"{name} {W}x{H} bands {edges}")
        del parts
        for world in (2, 8):
            assert_same(render_rows(r, renderer_lib, m, W, H, world), o["pixels"], f"{name} {W}x{H} {world} interleaved phases")
    finally:
        r.close()


@pytest.mark.gpu
@pytest.mark.parametrize("W,H", [(7680, 4320), (7681, 4321)], ids=["7680x4320", "7681x4321"])
def test_host_transport_8k(W, H, renderer_lib, oracle_port):
    """24- and 32-bit transport, 12 and 1 copy bands, registered and staged caller memory, on the small-scene and the
    general path: every combination gives the oracle's frame and the device frame."""
    import torch
    mats = renderer_lib.camera_path(S.input_script("flythrough", 600))
    for name, sc, m in (("shipped", S.shipped_scene(1), shipped_view(mats, W, H)),
                        ("clip", S.clip_stress_scene(3000), general_view(mats))):
        want = oracle_port.OracleScene(sc).render(m, W, H)["pixels"]
        r = renderer_lib.Renderer(0)
        try:
            r.load_scene(sc)
            assert_same(_device_frame(r, torch, m, W, H)[0], want, f"{name} {W}x{H} device")
            for pack in (1, 0):
                for bands in (12, 1):
                    for pin in (0, 1):
                        r.set_option("pack24", pack); r.set_option("host_bands", bands); r.set_option("pin_host", pin)
                        out = np.full((1, H, W), 0x55555555, np.uint32)
                        assert_same(r.render(m, W, H, out=out)[0], want, f"{name} {W}x{H} pack24={pack} host_bands={bands} pin_host={pin}")
                        del out
            r.set_option("pin_host", 0)
        finally:
            r.close()


@pytest.mark.gpu
def test_span_tables_fall_back_by_batch_size(renderer_lib, oracle_port):
    """A single 7680 x 4320 view of a small scene walks its largest survivors once per frame (span_walk: 3 launches).
    A batch whose span tables would exceed 1 GB falls back to exact jumps in every tile (2 launches); every view must
    still be the oracle's frame, and so must a single view after it."""
    import torch
    W, H = 7680, 4320
    sc = S.shipped_scene(1)
    osc = oracle_port.OracleScene(sc)
    mats = _shipped_views(renderer_lib)
    frames = list(range(40, 600, 25))[:SPAN_BATCH]
    assert len(frames) == SPAN_BATCH
    r = renderer_lib.Renderer(0)
    try:
        r.load_scene(sc)
        m = mats[110]
        want = osc.render(m, W, H)
        before = r.kernel_launches
        got = _device_frame(r, torch, m, W, H)[0]
        assert r.kernel_launches - before == 3
        assert_same(got, want["pixels"], "single view with span tables")
        assert_stats(r.stats(), want, "single view with span tables")
        before = r.kernel_launches
        got = _device_frame(r, torch, mats[frames], W, H)
        assert r.kernel_launches - before == 2
        for k, f in enumerate(frames):
            o = osc.render(mats[f], W, H)
            assert_same(got[k], o["pixels"], f"batch view {k} (frame {f})")
            assert_stats(r.stats(k), o, f"batch view {k} (frame {f})")
        del got
        # the renderer sizes its scratch for the largest batch it has submitted (views_cap only grows): the span
        # tables stay off for this renderer, and a single view keeps the exact jumps
        before = r.kernel_launches
        got = _device_frame(r, torch, m, W, H)[0]
        assert r.kernel_launches - before == 2
        assert_same(got, want["pixels"], "single view after a large batch")
    finally:
        r.close()


@pytest.mark.gpu
def test_frame_and_option_limits(renderer_lib, oracle_port):
    """W or H = 65536 is refused with S3R_E_ARG by every render entry point and writes nothing; the renderer renders
    afterwards.  views_per_chunk takes 65535 (the grid-dimension limit of its launches) and refuses 65536."""
    import ctypes
    import torch
    E_ARG = -4
    sc = S.shipped_scene(1)
    m = shipped_view(_shipped_views(renderer_lib), 640, 360)
    want = oracle_port.OracleScene(sc).render(m, 640, 360)["pixels"]
    r = renderer_lib.Renderer(0)
    lib, h = r._lib, r._h
    cams = np.ascontiguousarray(m, "<f4")
    try:
        r.load_scene(sc)
        for W, H in ((65536, 8), (8, 65536), (65536, 65536)):
            dev = torch.full((min(H, 64), min(W, 64)), 0x55555555, dtype=torch.int32, device="cuda:0")
            host = np.full((min(H, 64), min(W, 64)), 0x55555555, np.uint32)
            rcs = (lib.s3r_render_device(h, cams.ctypes.data, 1, W, H, 0, min(H, 64), ctypes.c_void_p(dev.data_ptr()), None),
                   lib.s3r_render_device_rows(h, cams.ctypes.data, 1, W, H, 1, 0, ctypes.c_void_p(dev.data_ptr()), None),
                   lib.s3r_render_host(h, cams.ctypes.data, 1, W, H, 0, min(H, 64), host.ctypes.data))
            assert rcs == (E_ARG, E_ARG, E_ARG), (W, H, rcs)
            assert r.finish() is False
            assert (dev.cpu().numpy().view(np.uint32) == 0x55555555).all() and (host == 0x55555555).all(), (W, H)
        assert_same(r.render(m, 640, 360)[0], want, "host frame after refused sizes")
        assert_same(_device_frame(r, torch, m, 640, 360)[0], want, "device frame after refused sizes")
        assert lib.s3r_set_option(h, b"views_per_chunk", 65535) == 0
        assert lib.s3r_set_option(h, b"views_per_chunk", 65536) == E_ARG
        assert lib.s3r_set_option(h, b"views_per_chunk", 0) == E_ARG
        assert_same(_device_frame(r, torch, np.stack([m, m]), 640, 360)[1], want, "batch after views_per_chunk = 65535")
    finally:
        r.close()
