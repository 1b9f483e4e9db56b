"""Supersampled anti-aliasing (s3r_render_device_ssaa / s3r_render_host_ssaa) against the oracle, bit for bit.

An anti-aliased frame is defined as the reference's frame at k*W x k*H, box-resolved per channel with rounding half up
(include/s3r_b200.h).  Every expected pixel therefore comes from the oracle at the supersampled size and ``resolve``
below, and every comparison is exact.  The CPU test pins ``resolve`` itself on hand-made blocks.  The GPU tests cover the
small-scene path (tile_raster resolves in its write-out: tensor store, bulk row copies, plain stores, 24-bit host
transport, registered caller buffers), the general path (shade_tiles resolves its shading blocks) under every routing
with statistics, bands that start inside an output tile row, view batches, k = 1 as the plain call, capacity regrowth,
a 3840 x 2160 frame and the rejected arguments."""
import numpy as np
import pytest

from swift3drenderer_b200 import scene as S
from test_gpu_vis_edges import ROUTES, assert_same, assert_stats, restore_defaults, set_route

S3R_E_ARG = -4
GUARD = 0x55555555   # (pixels have a zero top byte: any word left at this value was never written)


def resolve(frame, k):
    """(..., k*H, k*W) 0x00RRGGBB frames -> (..., H, W): per channel (sum of the k x k block + k*k / 2) >> log2(k*k)."""
    f = np.asarray(frame, np.uint32)
    h, w = f.shape[-2] // k, f.shape[-1] // k
    blocks = f.reshape(f.shape[:-2] + (h, k, w, k))
    out = np.zeros(f.shape[:-2] + (h, w), np.uint32)
    for shift in (0, 8, 16):
        total = ((blocks >> np.uint32(shift)) & np.uint32(0xFF)).sum(axis=(-3, -1), dtype=np.uint32)
        out |= ((total + np.uint32(k * k // 2)) // np.uint32(k * k)) << np.uint32(shift)
    return out


def flythrough(lib):
    return lib.camera_path(S.input_script("flythrough", 600))


def oracle_ssaa(osc, m, W, H, k, **kw):
    """(expected output frame, the oracle's result at k*W x k*H)."""
    o = osc.render(m, k * W, k * H, **kw)
    return resolve(o["pixels"], k), o


def device_ssaa(r, torch, m, W, H, k, y0=0, y1=None):
    """render_device_ssaa into a guarded device buffer, repeated while finish() asks for it; (n, y1 - y0, W) frames."""
    y1 = H if y1 is None else y1
    n = np.asarray(m).reshape(-1, 12).shape[0]
    px = n * (y1 - y0) * W
    buf = torch.full((px + 64,), GUARD, dtype=torch.int32, device="cuda:0")
    for _ in range(4):
        r.render_device_ssaa(m, W, H, k, buf.data_ptr(), y0=y0, y1=y1)
        if not r.finish():
            break
    assert r.stats()["overflow"] == 0
    host = buf.cpu().numpy().view(np.uint32)
    assert (host[px:] == GUARD).all(), "the call wrote past its output"
    return host[:px].reshape(n, y1 - y0, W)


# ------------------------------------------------------------------------------------------------------------------
# CPU: the resolve rule
# ------------------------------------------------------------------------------------------------------------------
def test_resolve_rule_on_hand_made_blocks():
    # k = 2: a channel sum of 2 is half way between 0 and 1 and rounds up; 1 rounds down; 6 (1.5) rounds up to 2
    blk = np.array([[[0x000000, 0x000101], [0x010100, 0x000000]],      # blue 1, green 2, red 1
                    [[0x030102, 0x000001], [0x000200, 0x030203]]],     # blue 6, green 5, red 6
                   np.uint32)
    got = resolve(blk, 2)
    assert got.shape == (2, 1, 1)
    assert got[0, 0, 0] == 0x000100 and got[1, 0, 0] == 0x020102
    # channels do not carry into each other; saturated blocks stay saturated; the top byte stays zero
    assert resolve(np.array([[0xFF0000, 0x00FF00], [0x0000FF, 0x000000]], np.uint32), 2)[0, 0] == 0x404040
    assert resolve(np.full((4, 4), 0xFFFFFF, np.uint32), 4)[0, 0] == 0xFFFFFF
    assert resolve(np.full((4, 4), 0xFFFFFF, np.uint32), 2).tolist() == [[0xFFFFFF] * 2] * 2
    # k = 4: 8 of 16 is the half-way case and rounds up, 7 rounds down
    half = np.zeros((4, 4), np.uint32)
    half.flat[:8] = 0x010101
    assert resolve(half, 4)[0, 0] == 0x010101
    half.flat[7] = 0
    assert resolve(half, 4)[0, 0] == 0
    # k = 1 is the identity; blocks are the k x k squares at (k*y, k*x)
    rng = np.random.RandomState(5)
    f = rng.randint(0, 1 << 24, size=(3, 8, 12)).astype(np.uint32)
    assert np.array_equal(resolve(f, 1), f)
    for k in (2, 4):
        got = resolve(f, k)
        for v in range(3):
            for y in range(8 // k):
                for x in range(12 // k):
                    b = f[v, k * y:k * y + k, k * x:k * x + k]
                    want = 0
                    for shift in (0, 8, 16):
                        c = sum(int(p) >> shift & 255 for p in b.flat)
                        want |= int(np.floor(c / (k * k) + 0.5)) << shift
                    assert got[v, y, x] == want


# ------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------
SMALL_SIZES = [(160, 90), (101, 67), (320, 180)]


@pytest.mark.gpu
@pytest.mark.parametrize("W,H", SMALL_SIZES, ids=[f"{W}x{H}" for W, H in SMALL_SIZES])
def test_small_scene_path(W, H, renderer_lib, oracle_port):
    """Shipped scene (tile_raster resolves each 64 x 32 colour tile): device output through the tensor map (101 x 67:
    bulk row copies are not possible, plain stores), the bulk row copies and plain stores on request, and the host
    entry with 24-bit transport, 32-bit transport and a registered caller buffer."""
    import torch
    sc = S.shipped_scene(1)
    osc = oracle_port.OracleScene(sc)
    mats = flythrough(renderer_lib)
    r = renderer_lib.Renderer(0)
    try:
        r.load_scene(sc)
        for pose in (40, 110, 300):
            m = mats[pose]
            for k in (2, 4):
                want, o = oracle_ssaa(osc, m, W, H, k)
                what = f"shipped {W}x{H} pose {pose} k={k}"
                assert_same(device_ssaa(r, torch, m, W, H, k)[0], want, f"{what} device")
                assert_stats(r.stats(), o, f"{what} device")
                for opt, val in (("tensor_store", 0), ("tma_store", 0)):
                    r.set_option(opt, val)
                    assert_same(device_ssaa(r, torch, m, W, H, k)[0], want, f"{what} device {opt}=0")
                r.set_option("tensor_store", 1)
                r.set_option("tma_store", 1)
                for pack in (1, 0):
                    r.set_option("pack24", pack)
                    assert_same(r.render_ssaa(m, W, H, k)[0], want, f"{what} host pack24={pack}")
                    assert_stats(r.stats(), o, f"{what} host pack24={pack}")
                r.set_option("pack24", 1)
                r.set_option("pin_host", 1)
                buf = np.empty((1, H, W), np.uint32)
                assert_same(r.render_ssaa(m, W, H, k, out=buf)[0], want, f"{what} host pin_host=1")
                r.set_option("pin_host", 0)
    finally:
        r.close()


def general_cases(lib):
    mats = flythrough(lib)
    spin = lib.camera_path(S.input_script("spin", 12))
    return {"clip": (lambda: S.clip_stress_scene(3000), mats[350]),
            "dense": (lambda: S.icosahedron_field(20000, seed=9, extent=40, r_range=(0.3, 1.0)), mats[350]),
            "hazard": (lambda: S.hazard_scene(), spin[5])}


GENERAL_SIZES = [(320, 180), (1283, 721)]


@pytest.mark.gpu
@pytest.mark.parametrize("W,H", GENERAL_SIZES, ids=[f"{W}x{H}" for W, H in GENERAL_SIZES])
@pytest.mark.parametrize("name", ["clip", "dense", "hazard"])
def test_general_path_every_route(name, W, H, renderer_lib, oracle_port):
    """shade_tiles resolves its 32 x 16 shading blocks: host frames and statistics (those of the k*W x k*H frame) under
    every routing, and the device entry."""
    import torch
    build, m = general_cases(renderer_lib)[name]
    sc = build()
    osc = oracle_port.OracleScene(sc)
    r = renderer_lib.Renderer(0)
    try:
        r.load_scene(sc)
        r.set_option("fused_small", 0)   # (the hazard scene has 36 triangles: the general path only on request)
        for k in (2, 4):
            want, o = oracle_ssaa(osc, m, W, H, k)
            for route in ROUTES:
                set_route(r, route)
                what = f"{name} {W}x{H} k={k} route {route}"
                assert_same(r.render_ssaa(m, W, H, k)[0], want, what)
                assert_stats(r.stats(), o, what)
            restore_defaults(r)
            r.set_option("fused_small", 0)
            assert_same(device_ssaa(r, torch, m, W, H, k)[0], want, f"{name} {W}x{H} k={k} device")
            assert_stats(r.stats(), o, f"{name} {W}x{H} k={k} device")
    finally:
        r.close()


# bands in output rows: y0 % 4 in {1, 2, 3}, starts inside an output tile row (32 / k rows), a single row, the last row,
# and one that starts on a tile row for k = 2 and 4 (rendered row 32 / 64: the small-scene path's tensor store then
# writes from a nonzero output row)
BANDS = [(1, 50), (2, 91), (3, 180), (5, 6), (45, 46), (17, 33), (179, 180), (16, 100)]


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["shipped", "dense"])
def test_bands(which, renderer_lib, oracle_port):
    """Every band equals the same rows of the whole anti-aliased frame, on the device and on the host."""
    import torch
    W, H = 320, 180
    if which == "shipped":
        sc, m = S.shipped_scene(1), flythrough(renderer_lib)[110]
    else:
        build, m = general_cases(renderer_lib)["dense"]
        sc = build()
    osc = oracle_port.OracleScene(sc)
    r = renderer_lib.Renderer(0)
    try:
        r.load_scene(sc)
        for k in (2, 4):
            want, _ = oracle_ssaa(osc, m, W, H, k)
            for y0, y1 in BANDS:
                what = f"{which} k={k} band {y0}..{y1}"
                assert_same(device_ssaa(r, torch, m, W, H, k, y0, y1)[0], want[y0:y1], f"{what} device")
                assert_same(r.render_ssaa(m, W, H, k, y0=y0, y1=y1)[0], want[y0:y1], f"{what} host")
    finally:
        r.close()


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["shipped", "dense"])
def test_view_batches(which, renderer_lib):
    """Five views in chunks of two: every view equals its single-view render, on the device and on the host."""
    import torch
    W, H, k = 320, 180, 2
    mats = flythrough(renderer_lib)
    sc = S.shipped_scene(1) if which == "shipped" else general_cases(renderer_lib)["dense"][0]()
    views = mats[[40, 110, 200, 300, 350]]
    r = renderer_lib.Renderer(0)
    try:
        r.load_scene(sc)
        single = [device_ssaa(r, torch, v, W, H, k)[0] for v in views]
        r.set_option("views_per_chunk", 2)
        dev = device_ssaa(r, torch, views, W, H, k)
        host = r.render_ssaa(views, W, H, k)
        for i in range(len(views)):
            assert_same(dev[i], single[i], f"{which} view {i} of 5, device")
            assert_same(host[i], single[i], f"{which} view {i} of 5, host")
    finally:
        r.close()


@pytest.mark.gpu
def test_one_sample_is_the_plain_call(renderer_lib):
    """k = 1: the same frames as s3r_render_device / s3r_render_host, with the same number of kernel launches."""
    import torch
    W, H = 320, 180
    mats = flythrough(renderer_lib)
    for sc, m in ((S.shipped_scene(1), mats[110]), (general_cases(renderer_lib)["dense"][0](), mats[350])):
        r = renderer_lib.Renderer(0)
        try:
            r.load_scene(sc)
            r.render(m, W, H)   # capacities settled before launches are counted
            buf = torch.full((H, W), GUARD, dtype=torch.int32, device="cuda:0")
            n0 = r.kernel_launches
            r.render_device_ssaa(m, W, H, 1, buf.data_ptr())
            assert r.finish() is False
            n1 = r.kernel_launches
            a = buf.cpu().numpy().view(np.uint32).copy()
            buf.fill_(GUARD)
            r.render_device(m, W, H, buf.data_ptr())
            assert r.finish() is False
            n2 = r.kernel_launches
            assert_same(a, buf.cpu().numpy().view(np.uint32), "k=1 device")
            assert n1 - n0 == n2 - n1
            h1 = r.render_ssaa(m, W, H, 1)
            n3 = r.kernel_launches
            h2 = r.render(m, W, H)
            assert_same(h1[0], h2[0], "k=1 host")
            assert n3 - n2 == r.kernel_launches - n3
        finally:
            r.close()


@pytest.mark.gpu
def test_regrowth_and_clean_key_plane(renderer_lib, oracle_port):
    """With shrunk capacities the device call's finish() asks for a repeat that is the oracle's frame (the shipped scene
    needs fewer records than that: its frame is checked all the same), the host call regrows by itself, and a plain
    render after supersampled ones still equals the oracle (the key plane is clean)."""
    import torch
    W, H, k = 320, 180, 2
    build, m = general_cases(renderer_lib)["dense"]
    sc = build()
    osc = oracle_port.OracleScene(sc)
    want, _ = oracle_ssaa(osc, m, W, H, k)
    for which, scene in (("dense", sc), ("shipped", S.shipped_scene(1))):
        m_s = m if which == "dense" else flythrough(renderer_lib)[110]
        want_s = want if which == "dense" else oracle_ssaa(oracle_port.OracleScene(scene), m_s, W, H, k)[0]
        r = renderer_lib.Renderer(0)
        try:
            r.load_scene(scene)
            r.set_option("setup_capacity", 4)
            buf = torch.full((H, W), GUARD, dtype=torch.int32, device="cuda:0")
            r.render_device_ssaa(m_s, W, H, k, buf.data_ptr())
            overflowed = r.finish()
            assert overflowed or which == "shipped", f"{which}: 4 setup records must overflow"
            for _ in range(4):   # (a repeat may still overflow a capacity the short survivor list hid)
                r.render_device_ssaa(m_s, W, H, k, buf.data_ptr())
                if not r.finish():
                    break
            assert r.stats()["overflow"] == 0
            assert_same(buf.cpu().numpy().view(np.uint32), want_s, f"{which} device repeat after regrowth")
            r.set_option("setup_capacity", 4)
            assert_same(r.render_ssaa(m_s, W, H, k)[0], want_s, f"{which} host with regrowth")
        finally:
            r.close()
    r = renderer_lib.Renderer(0)
    try:
        r.load_scene(sc)
        for kk in (4, 2):
            r.render_ssaa(m, W, H, kk)
            device_ssaa(r, torch, m, W, H, kk, 7, 101)
        plain = osc.render(m, W, H)
        assert_same(r.render(m, W, H)[0], plain["pixels"], "plain render after supersampled ones")
        assert_stats(r.stats(), plain, "plain render after supersampled ones")
    finally:
        r.close()


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["shipped", "dense"])
def test_3840x2160(which, renderer_lib):
    """At 3840 x 2160 with k = 2 the output is the resolve of the plain 7680 x 4320 device frame (which the large-frame
    tests pin to the oracle)."""
    import torch
    W, H, k = 3840, 2160, 2
    mats = flythrough(renderer_lib)
    sc = S.shipped_scene(1) if which == "shipped" else general_cases(renderer_lib)["dense"][0]()
    m = mats[110] if which == "shipped" else mats[350]
    r = renderer_lib.Renderer(0)
    try:
        r.load_scene(sc)
        big = torch.full((k * H, k * W), GUARD, dtype=torch.int32, device="cuda:0")
        for _ in range(4):
            r.render_device(m, k * W, k * H, big.data_ptr())
            if not r.finish():
                break
        want = resolve(big.cpu().numpy().view(np.uint32), k)
        del big
        assert_same(device_ssaa(r, torch, m, W, H, k)[0], want, f"{which} 3840x2160 k=2 device")
        assert_same(r.render_ssaa(m, W, H, k)[0], want, f"{which} 3840x2160 k=2 host")
    finally:
        r.close()


@pytest.mark.gpu
def test_rejected_arguments(renderer_lib):
    """k not in {1, 2, 4}, k*W or k*H over 65535, and a supersampled call while peer frames are set return S3R_E_ARG
    with a message."""
    import torch
    r = renderer_lib.Renderer(0)
    try:
        r.load_scene(S.shipped_scene(1))
        m = flythrough(renderer_lib)[110]
        buf = torch.zeros((64 * 64,), dtype=torch.int32, device="cuda:0")

        def rejected(call, what):
            with pytest.raises(renderer_lib.RendererError, match=f"s3r error {S3R_E_ARG}: .+"):
                call()
            assert r._lib.s3r_last_error().decode(), what

        for k in (0, 3, 8):
            rejected(lambda: r.render_device_ssaa(m, 64, 64, k, buf.data_ptr()), f"k={k} device")
            rejected(lambda: r.render_ssaa(m, 64, 64, k), f"k={k} host")
        rejected(lambda: r.render_device_ssaa(m, 16384, 1, 4, buf.data_ptr()), "4 x 16384 = 65536 columns")
        rejected(lambda: r.render_device_ssaa(m, 1, 32768, 2, buf.data_ptr()), "2 x 32768 = 65536 rows")
        rejected(lambda: r.render_ssaa(m, 32768, 1, 2), "2 x 32768 = 65536 columns, host")
        # bands are checked before they are scaled: 2 x 2^31 would wrap to row 0
        for y0, y1 in ((2 ** 31, 10), (2 ** 30, 10), (10, 10), (20, 10), (0, 65)):
            rejected(lambda: r.render_device_ssaa(m, 64, 64, 2, buf.data_ptr(), y0=y0, y1=y1), f"band {y0}..{y1}, device")
            rejected(lambda: r.render_device_ssaa(m, 64, 64, 4, buf.data_ptr(), y0=y0, y1=y1), f"band {y0}..{y1}, device k=4")
            rejected(lambda: r.render_ssaa(m, 64, 64, 2, y0=y0, y1=y1), f"band {y0}..{y1}, host")
        assert int(torch.count_nonzero(buf)) == 0, "a rejected call wrote to its output"
        # the largest accepted frame is still fine: 4 x 16383 columns
        wide = torch.full((16383 + 64,), GUARD, dtype=torch.int32, device="cuda:0")
        r.render_device_ssaa(m, 16383, 1, 4, wide.data_ptr())
        r.finish()
        assert (wide.cpu().numpy().view(np.uint32)[16383:] == GUARD).all()
        peer = torch.zeros((64 * 64,), dtype=torch.int32, device="cuda:0")
        r.set_peer_frames([peer.data_ptr()])
        try:
            rejected(lambda: r.render_device_ssaa(m, 64, 64, 2, buf.data_ptr()), "peer frames set")
            rejected(lambda: r.render_ssaa(m, 64, 64, 2), "peer frames set, host")
        finally:
            r.set_peer_frames([])
        r.render_device_ssaa(m, 64, 64, 2, buf.data_ptr())
        assert r.finish() is False
    finally:
        r.close()
