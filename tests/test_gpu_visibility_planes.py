"""Visibility planes (s3r_render_device_visibility) against the oracle, bit for bit.

Per pixel the triangle plane holds the scene index of the triangle that colours it in the reference's frame (a triangle
the near-plane clip appended reports its parent; background 0xFFFFFFFF) and the depth plane the reference's depth-buffer
value, the interpolated 1/z (background +0).  Both come straight from the oracle's ``winner`` and ``depth`` outputs, and
depth is compared as uint32 bit patterns, so that -0 / +0 or a NaN cannot pass by accident.  Every output buffer carries
guard words behind it.  The CPU tests prove from the oracle alone that the scenes reach what they exist for; the GPU
tests cover the small-scene path (tile_raster writes the planes in its shading phase) under every write-out option,
the general path (shade_tiles writes them from the keys) under every routing, with and without colour, bands, view
batches, a clean key plane after visibility-only renders, capacity regrowth, frames of 4K and more, the launch count and
the rejected arguments."""
import itertools

import numpy as np
import pytest

from swift3drenderer_b200 import scene as S
from test_gpu_supersample import BANDS, general_cases
from test_gpu_vis_edges import (NO_WINNER, ROUTES, assert_same, assert_stats, box_sizes, restore_defaults, set_route,
                                still, tie_field, tie_pixels)

S3R_E_ARG = -4
GUARD = 0x55555555
PAD = 64                                                      # guard words behind every output
SUBSETS = [s for s in itertools.product((True, False), repeat=3) if any(s)]   # (colour, triangle, depth): all 7


def flythrough(lib):
    return lib.camera_path(S.input_script("flythrough", 600))


def plane_cases(lib):
    """test_gpu_supersample's general-path cases plus the clip scene seen from where near-plane clipping decides many
    pixels: there, and in the hazard scene, triangles the clipper appended win pixels."""
    cases = dict(general_cases(lib))
    cases["clip_near"] = (cases["clip"][0], lib.camera_path(S.input_script("spin", 12))[10])
    return cases


def expected(osc, n_triangles, m, W, H):
    """(colour, triangle plane, depth bits, oracle result) of the reference's W x H frame."""
    o = osc.render(m, W, H, want_depth=True, want_winner=True)
    w = o["winner"]
    tri = np.where(w == NO_WINNER, w, np.where(w >= n_triangles, w - n_triangles, w)).astype(np.uint32)
    return o["pixels"], tri, o["depth"].view(np.uint32), o


def device_planes(r, torch, m, W, H, y0=0, y1=None, subset=(True, True, True)):
    """render_device_visibility into guarded device buffers for the outputs in ``subset`` (colour, triangle, depth),
    repeated while finish() asks for it.  Returns the three (n, y1 - y0, W) uint32 arrays, None where not requested."""
    y1 = H if y1 is None else y1
    n = np.asarray(m).reshape(-1, 12).shape[0]
    px = n * (y1 - y0) * W
    bufs = [torch.full((px + PAD,), GUARD, dtype=torch.int32, device="cuda:0") if want else None for want in subset]
    ptrs = [b.data_ptr() if b is not None else 0 for b in bufs]
    for _ in range(4):
        r.render_device_visibility(m, W, H, *ptrs, y0=y0, y1=y1)
        if not r.finish():
            break
    assert r.stats()["overflow"] == 0
    out = []
    for name, b in zip(("colour", "triangle", "depth"), bufs):
        if b is None:
            out.append(None)
            continue
        host = b.cpu().numpy().view(np.uint32)
        assert (host[px:] == GUARD).all(), f"the call wrote past its {name} output"
        out.append(host[:px].reshape(n, y1 - y0, W))
    return out


def device_colour(r, torch, m, W, H, y0=0, y1=None):
    y1 = H if y1 is None else y1
    buf = torch.full(((y1 - y0) * W,), GUARD, dtype=torch.int32, device="cuda:0")
    for _ in range(4):
        r.render_device(m, W, H, buf.data_ptr(), y0=y0, y1=y1)
        if not r.finish():
            break
    return buf.cpu().numpy().view(np.uint32).reshape(y1 - y0, W)


def check(got, want, what, subset=(True, True, True)):
    """got: device_planes' result for one view; want: (colour, triangle, depth bits)."""
    for name, g, w, on in zip(("colour", "triangle", "depth"), got, want, subset):
        if on:
            assert_same(g, w, f"{what}: {name}")
        else:
            assert g is None


# ------------------------------------------------------------------------------------------------------------------
# CPU: the scenes reach what they exist for
# ------------------------------------------------------------------------------------------------------------------
def test_oracle_planes_premises(oracle_port):
    """Background pixels have depth +0 and every other pixel a positive depth; in the clip scene's near view and in the
    hazard scene triangles the clipper appended (order key T + parent) win pixels, which report their parent."""
    for name in ("clip_near", "hazard"):
        build, m = plane_cases(oracle_port)[name]
        sc = build()
        T = sc.n_triangles
        _, tri, dep, o = expected(oracle_port.OracleScene(sc), T, m, 320, 180)
        w = o["winner"]
        bg = w == NO_WINNER
        appended = (w >= T) & ~bg
        assert appended.sum() > 1000 and (w[~bg] < 2 * T).all(), name
        assert (tri[~bg] < T).all() and np.array_equal(tri[appended], w[appended] - T) and (tri[bg] == NO_WINNER).all()
        assert bg.any() and (dep[bg] == 0).all(), name
        assert (o["depth"][~bg] > 0).all(), name


def test_tie_field_has_order_decided_ties(oracle_port):
    """The tie field has pixels where two triangles reach bit-identical depth and the earlier one wins by list order."""
    sc, sites = tie_field(oracle_port)
    m = oracle_port.camera_path(still())[0]
    count, tied, o1, _ = tie_pixels(sc, sites, oracle_port.OracleScene, m, 800, 450)
    assert tied.sum() > 1000 and (count > 0).all()


def test_general_scenes_win_on_every_record_kind(oracle_port):
    """Among the winners of the general-path scenes there are boxes under 16 px (record-free when unclipped), of
    16..127 px (flat walk) and of 128 px or more (tile kernel), so every writer of the key plane is checked."""
    kinds = set()
    for name, (build, m) in plane_cases(oracle_port).items():
        sc = build()
        o = oracle_port.OracleScene(sc).render(m, 320, 180, want_setups=True, want_winner=True)
        st = o["setups"]
        bw, bh = box_sizes(st)
        big = dict(zip(st["order"].tolist(), np.maximum(bw, bh).tolist()))
        won = [big[int(t)] for t in np.unique(o["winner"]) if t != NO_WINNER]
        here = {"small" if b < 16 else "flat" if b < 128 else "tile" for b in won}
        kinds |= here
        if name == "clip":
            assert here == {"small", "flat", "tile"}, (name, here)
    assert kinds == {"small", "flat", "tile"}


# ------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------
SMALL_SIZES = [(160, 90), (101, 67), (320, 180)]


@pytest.mark.gpu
@pytest.mark.parametrize("fused_small", [1, 0])
@pytest.mark.parametrize("W,H", SMALL_SIZES, ids=[f"{W}x{H}" for W, H in SMALL_SIZES])
def test_small_scene_every_subset(W, H, fused_small, renderer_lib, oracle_port):
    """Shipped scene, several poses: all 7 non-empty output subsets, with the colour equal to s3r_render_device's and the
    oracle's, under spans, tma_store and tensor_store on and off.  fused_small = 0 moves the scene onto the general
    path."""
    import torch
    sc = S.shipped_scene(1)
    osc = oracle_port.OracleScene(sc)
    mats = flythrough(renderer_lib)
    r = renderer_lib.Renderer(0)
    try:
        r.load_scene(sc)
        r.set_option("fused_small", fused_small)
        for pose in (40, 110, 300):
            m = mats[pose]
            want = expected(osc, sc.n_triangles, m, W, H)[:3]
            for spans, tma, tensor in itertools.product((1, 0), repeat=3):
                r.set_option("spans", spans)
                r.set_option("tma_store", tma)
                r.set_option("tensor_store", tensor)
                what = f"shipped {W}x{H} fused_small={fused_small} pose {pose} spans={spans} tma={tma} tensor={tensor}"
                assert_same(device_colour(r, torch, m, W, H), want[0], f"{what}: s3r_render_device")
                for subset in SUBSETS:
                    got = [g if g is None else g[0] for g in device_planes(r, torch, m, W, H, subset=subset)]
                    check(got, want, f"{what} outputs {subset}", subset)
    finally:
        r.close()


GENERAL_CASES = [(n, W, H) for n in ("clip", "clip_near", "dense", "hazard") for W, H in ((320, 180), (1283, 721))] + [("ties", 800, 450)]


@pytest.mark.gpu
@pytest.mark.parametrize("name,W,H", GENERAL_CASES, ids=[f"{n}-{W}x{H}" for n, W, H in GENERAL_CASES])
def test_general_path_every_route(name, W, H, renderer_lib, oracle_port):
    """shade_tiles writes the planes from the keys: every routing, with and without colour, and the statistics equal the
    oracle's in both modes.  The tie field (test_gpu_vis_edges) has exact depth ties between kernels, decided by order."""
    import torch
    if name == "ties":
        sc, _ = tie_field(oracle_port)
        m = renderer_lib.camera_path(still())[0]
    else:
        build, m = plane_cases(renderer_lib)[name]
        sc = build()
    want = expected(oracle_port.OracleScene(sc), sc.n_triangles, m, W, H)
    r = renderer_lib.Renderer(0)
    try:
        r.load_scene(sc)
        for route in ROUTES:
            set_route(r, route)
            r.set_option("fused_small", 0)   # (the hazard scene has 36 triangles: the general path only on request)
            what = f"{name} {W}x{H} route {route}"
            for subset in ((True, True, True), (False, True, True)):
                got = [g if g is None else g[0] for g in device_planes(r, torch, m, W, H, subset=subset)]
                check(got, want[:3], f"{what} outputs {subset}", subset)
                assert_stats(r.stats(), want[3], f"{what} outputs {subset}")
    finally:
        restore_defaults(r)
        r.close()


def _scene(which, renderer_lib):
    if which == "shipped":
        return S.shipped_scene(1), flythrough(renderer_lib)[110]
    build, m = general_cases(renderer_lib)["dense"]
    return build(), m


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["shipped", "dense"])
def test_bands(which, renderer_lib, oracle_port):
    """Bands that start inside a tile row and inside a 4-row key column, single rows and the last row: each equals the
    same rows of the whole frame, with and without colour."""
    import torch
    W, H = 320, 180
    sc, m = _scene(which, renderer_lib)
    want = expected(oracle_port.OracleScene(sc), sc.n_triangles, m, W, H)[:3]
    r = renderer_lib.Renderer(0)
    try:
        r.load_scene(sc)
        for y0, y1 in BANDS:
            for subset in ((True, True, True), (False, True, True)):
                got = [g if g is None else g[0] for g in device_planes(r, torch, m, W, H, y0, y1, subset)]
                check(got, [w[y0:y1] for w in want], f"{which} band {y0}..{y1} outputs {subset}", subset)
    finally:
        r.close()


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["shipped", "dense"])
def test_view_batches(which, renderer_lib):
    """Five views in chunks of two: every view equals its single-view call."""
    import torch
    W, H = 320, 180
    sc, _ = _scene(which, renderer_lib)
    views = flythrough(renderer_lib)[[40, 110, 200, 300, 350]]
    r = renderer_lib.Renderer(0)
    try:
        r.load_scene(sc)
        for subset in ((True, True, True), (False, True, True)):
            single = [device_planes(r, torch, v, W, H, subset=subset) for v in views]
            r.set_option("views_per_chunk", 2)
            batch = device_planes(r, torch, views, W, H, subset=subset)
            r.set_option("views_per_chunk", 8)
            for i in range(len(views)):
                check([b if b is None else b[i] for b in batch], [s if s is None else s[0] for s in single[i]],
                      f"{which} view {i} of 5, outputs {subset}", subset)
    finally:
        r.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["dense", "clip"])
def test_key_plane_stays_clean(name, renderer_lib, oracle_port):
    """Visibility-only renders (whole frames and bands) clear the key plane as they read it: a plain render afterwards
    equals the oracle, and so do its statistics."""
    import torch
    W, H = 320, 180
    build, m = general_cases(renderer_lib)[name]
    sc = build()
    osc = oracle_port.OracleScene(sc)
    other = flythrough(renderer_lib)[300]
    r = renderer_lib.Renderer(0)
    try:
        r.load_scene(sc)
        for y0, y1 in ((0, H), (3, 91), (17, 33)):
            device_planes(r, torch, m, W, H, y0, y1, (False, True, False))
            device_planes(r, torch, other, W, H, y0, y1, (False, False, True))
        for mm in (other, m):
            plain = osc.render(mm, W, H)
            assert_same(r.render(mm, W, H)[0], plain["pixels"], f"{name}: plain render after visibility-only ones")
            assert_stats(r.stats(), plain, f"{name}: plain render after visibility-only ones")
    finally:
        r.close()


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["dense", "shipped"])
@pytest.mark.parametrize("colour", [True, False], ids=["colour", "visibility_only"])
def test_regrowth(which, colour, renderer_lib, oracle_port):
    """setup_capacity = 4: finish() asks for a repeat (the shipped scene needs fewer records than that: it is checked all
    the same), and the repeat's planes equal the oracle's."""
    import torch
    W, H = 320, 180
    sc, m = _scene(which, renderer_lib)
    want = expected(oracle_port.OracleScene(sc), sc.n_triangles, m, W, H)
    subset = (colour, True, True)
    r = renderer_lib.Renderer(0)
    try:
        r.load_scene(sc)
        r.set_option("setup_capacity", 4)
        bufs = [torch.full((H * W,), GUARD, dtype=torch.int32, device="cuda:0") if on else None for on in subset]
        ptrs = [b.data_ptr() if b is not None else 0 for b in bufs]
        r.render_device_visibility(m, W, H, *ptrs)
        assert r.finish() or which == "shipped", f"{which}: 4 setup records must overflow"
        for _ in range(4):
            r.render_device_visibility(m, W, H, *ptrs)
            if not r.finish():
                break
        assert r.stats()["overflow"] == 0
        got = [b if b is None else b.cpu().numpy().view(np.uint32).reshape(H, W) for b in bufs]
        check(got, want[:3], f"{which} repeat after regrowth", subset)
        assert_stats(r.stats(), want[3], f"{which} repeat after regrowth")
    finally:
        r.close()


@pytest.mark.gpu
@pytest.mark.parametrize("W,H", [(3840, 2160), (7681, 4321)], ids=["3840x2160", "7681x4321"])
@pytest.mark.parametrize("which", ["shipped", "dense"])
def test_large_frames(which, W, H, renderer_lib, oracle_port):
    """3840 x 2160 and a frame over 4K (odd sizes: partial tiles, shading blocks and key columns at both far edges),
    with and without colour."""
    import torch
    sc, m = _scene(which, renderer_lib)
    if which == "dense":
        m = flythrough(renderer_lib)[350]
    want = expected(oracle_port.OracleScene(sc), sc.n_triangles, m, W, H)[:3]
    r = renderer_lib.Renderer(0)
    try:
        r.load_scene(sc)
        for subset in ((True, True, True), (False, True, True)):
            got = [g if g is None else g[0] for g in device_planes(r, torch, m, W, H, subset=subset)]
            check(got, want, f"{which} {W}x{H} outputs {subset}", subset)
    finally:
        r.close()


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["shipped", "dense"])
def test_no_extra_launch(which, renderer_lib):
    """The planes are written inside the write-out kernels: a call launches exactly as many kernels as
    s3r_render_device for the same frame, with and without colour."""
    import torch
    W, H = 320, 180
    sc, m = _scene(which, renderer_lib)
    r = renderer_lib.Renderer(0)
    try:
        r.load_scene(sc)
        buf = torch.zeros((3, H * W), dtype=torch.int32, device="cuda:0")
        p = [buf[i].data_ptr() for i in range(3)]
        r.render_device(m, W, H, p[0])   # capacities settled before launches are counted
        assert r.finish() is False
        n0 = r.kernel_launches
        r.render_device(m, W, H, p[0])
        assert r.finish() is False
        plain = r.kernel_launches - n0
        for ptrs in ((p[0], p[1], p[2]), (0, p[1], p[2]), (0, p[1], 0), (p[0], 0, 0)):
            n1 = r.kernel_launches
            r.render_device_visibility(m, W, H, *ptrs)
            assert r.finish() is False
            assert r.kernel_launches - n1 == plain, f"{which} outputs {ptrs}"
    finally:
        r.close()


@pytest.mark.gpu
def test_rejected_arguments(renderer_lib):
    """All three outputs null, peer frames set and bad frame geometry return S3R_E_ARG with a message, and nothing is
    written to any output."""
    import torch
    r = renderer_lib.Renderer(0)
    try:
        r.load_scene(S.shipped_scene(1))
        m = flythrough(renderer_lib)[110]
        bufs = [torch.full((64 * 64 + PAD,), GUARD, dtype=torch.int32, device="cuda:0") for _ in range(3)]
        p = [b.data_ptr() for b in bufs]

        def rejected(call, what):
            with pytest.raises(renderer_lib.RendererError, match=f"s3r error {S3R_E_ARG}: .+"):
                call()
            assert r._lib.s3r_last_error().decode(), what

        rejected(lambda: r.render_device_visibility(m, 64, 64), "all three outputs null")
        for W, H, y0, y1 in ((0, 64, 0, 64), (64, 0, 0, 1), (65536, 1, 0, 1), (1, 65536, 0, 1),
                             (64, 64, 10, 10), (64, 64, 20, 10), (64, 64, 0, 65)):
            rejected(lambda: r.render_device_visibility(m, W, H, *p, y0=y0, y1=y1), f"geometry {W}x{H} {y0}..{y1}")
            rejected(lambda: r.render_device_visibility(m, W, H, 0, p[1], 0, y0=y0, y1=y1), f"geometry {W}x{H} {y0}..{y1}, triangle only")
        cams = np.ascontiguousarray(m, "<f4")
        rc = r._lib.s3r_render_device_visibility(r._h, cams.ctypes.data, 0, 64, 64, 0, 64, p[0], p[1], p[2], None)
        assert rc == S3R_E_ARG, "no views"
        peer = torch.zeros((64 * 64,), dtype=torch.int32, device="cuda:0")
        r.set_peer_frames([peer.data_ptr()])
        try:
            rejected(lambda: r.render_device_visibility(m, 64, 64, *p), "peer frames set")
            rejected(lambda: r.render_device_visibility(m, 64, 64, 0, p[1], p[2]), "peer frames set, planes only")
        finally:
            r.set_peer_frames([])
        torch.cuda.synchronize()
        for name, b in zip(("colour", "triangle", "depth"), bufs):
            assert (b.cpu().numpy().view(np.uint32) == GUARD).all(), f"a rejected call wrote to the {name} output"
        assert int(torch.count_nonzero(peer)) == 0
        r.render_device_visibility(m, 64, 64, *p)
        assert r.finish() is False
    finally:
        r.close()
