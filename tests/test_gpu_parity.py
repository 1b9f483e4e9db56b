"""Parity tests proper: the CUDA path, called through the C ABI, against (a) the committed golden
frames of the unmodified reference, (b) the oracle on seeded inputs, (c) size-independent
properties at the benchmark's full 3840x2160.  Integer/byte outputs: bit-exact.  The north-star
tolerance (+-1 LSB on >= 99.9 % of pixels) is therefore met with zero differing pixels."""
import os
import subprocess
import sys

import numpy as np
import pytest

from swift3drenderer_b200 import scene as S
from cases import CASES

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def assert_same(a, b, what):
    if not np.array_equal(a, b):
        ys, xs = np.nonzero(a != b)
        raise AssertionError(f"{what}: {len(ys)} px differ, first (x={xs[0]}, y={ys[0]}) "
                             f"got {a[ys[0], xs[0]]:06x} want {b[ys[0], xs[0]]:06x}")


@pytest.mark.parametrize("name", sorted(CASES))
def test_cuda_matches_reference_golden_frames(name, gpu_renderer, renderer_lib, golden):
    (factory, script, n, keep, (W, H)), frames, pixels = golden(name)
    gpu_renderer.load_scene(factory())
    mats = renderer_lib.camera_path(S.input_script(script, n))
    for k, f in enumerate(frames):
        assert_same(gpu_renderer.render(mats[f], W, H)[0], pixels[k], f"{name} frame {f}")


@pytest.mark.parametrize("size", [(640, 360), (1280, 720), (333, 187), (64, 32), (65, 33), (1, 1), (7, 500)])
def test_cuda_matches_oracle_shipped_scene(size, gpu_renderer, renderer_lib, oracle_port):
    W, H = size
    sc = S.shipped_scene(1)
    gpu_renderer.load_scene(sc)
    osc = oracle_port.OracleScene(sc)
    mats = renderer_lib.camera_path(S.input_script("flythrough", 600))
    for f in range(0, 600, 40):
        assert_same(gpu_renderer.render(mats[f], W, H)[0], osc.render(mats[f], W, H)["pixels"], f"{W}x{H} frame {f}")


@pytest.mark.parametrize("kind", ["ico_tex", "ico_col", "clip", "regfloor", "dense_small"])
def test_cuda_matches_oracle_synthetic(kind, gpu_renderer, renderer_lib, oracle_port):
    sc = {
        "ico_tex": lambda: S.icosahedron_field(2000, seed=3, extent=60),
        "ico_col": lambda: S.icosahedron_field(2000, seed=4, extent=60, textured=False),
        "clip": lambda: S.clip_stress_scene(3000),
        "regfloor": lambda: S.shipped_scene(2, regular_floor=True),
        "dense_small": lambda: S.icosahedron_field(20000, seed=9, extent=40, r_range=(0.3, 1.0)),
    }[kind]()
    gpu_renderer.load_scene(sc)
    osc = oracle_port.OracleScene(sc)
    script = "flythrough" if kind == "regfloor" else "spin"
    mats = renderer_lib.camera_path(S.input_script(script, 120))
    for f in range(0, 120, 17):
        o = osc.render(mats[f], 640, 360)
        assert_same(gpu_renderer.render(mats[f], 640, 360)[0], o["pixels"], f"{kind} frame {f}")
        st = gpu_renderer.stats()
        assert st["near_rejected"] == o["stats"]["near_rejected"]
        assert st["clipped"] == o["stats"]["clipped"] and st["spawned"] == o["stats"]["spawned"]
        assert st["setups"] == o["stats"]["rasterized"]
        assert st["culled"] == o["stats"]["offscreen"] + o["stats"]["small_or_backfacing"]


def test_stage_dumps_are_bit_exact(gpu_renderer, renderer_lib, oracle_port):
    """Stage-level KATs: vertex stage (render.cpp:285-289) and clip/cull/setup (render.cpp:297-359)."""
    sc = S.clip_stress_scene(800)
    gpu_renderer.load_scene(sc)
    osc = oracle_port.OracleScene(sc)
    m = renderer_lib.camera_path(S.input_script("spin", 12))[11]
    W, H = 480, 270
    gpu_renderer.set_option("direct_small", 0)  # every survivor gets a setup record (the default walks small ones record-free)
    gpu_renderer.render(m, W, H)
    gpu_renderer.set_option("direct_small", 1)
    _, rv = osc.vertex_stage(m, W, H)
    assert np.array_equal(gpu_renderer.raster_vertices().view(np.uint32), rv.view(np.uint32))
    want = osc.render(m, W, H, want_setups=True)["setups"]
    got = gpu_renderer.setups()
    assert len(got) == len(want) > 50
    assert (np.diff(want["order"].astype(np.int64)) > 0).all()  # the reference's order is strictly increasing in our key
    for field in want.dtype.names:
        assert np.array_equal(got[field].view(np.uint32), want[field].view(np.uint32)), field
    assert (got["order"] >= sc.n_triangles).any()  # appended (clip-spawned) triangles present


def test_full_4k_frames_match_oracle(gpu_renderer, renderer_lib, oracle_port):
    """The benchmark configuration itself (C2: shipped scene, 3840x2160)."""
    sc = S.shipped_scene(1)
    gpu_renderer.load_scene(sc)
    osc = oracle_port.OracleScene(sc)
    mats = renderer_lib.camera_path(S.input_script("flythrough", 600))
    for f in (0, 100, 215, 330):
        assert_same(gpu_renderer.render(mats[f], 3840, 2160)[0], osc.render(mats[f], 3840, 2160)["pixels"], f"4K frame {f}")


def test_bands_reassemble_to_the_whole_frame(gpu_renderer, renderer_lib):
    """Screen-band partition (multi-GPU config) must not change a single pixel: every band walks
    the barycentrics from each triangle's own ymin exactly like the whole-frame render."""
    sc = S.shipped_scene(1)
    gpu_renderer.load_scene(sc)
    mats = renderer_lib.camera_path(S.input_script("flythrough", 600))
    W, H = 1920, 1080
    for f in (100, 330, 470):
        whole = gpu_renderer.render(mats[f], W, H)[0]
        for n in (2, 3, 8):
            edges = [H * k // n for k in range(n + 1)]
            parts = [gpu_renderer.render(mats[f], W, H, y0=edges[k], y1=edges[k + 1])[0] for k in range(n)]
            assert_same(np.concatenate(parts, 0), whole, f"{n} bands frame {f}")
        # bands that are not tile-aligned
        parts = [gpu_renderer.render(mats[f], W, H, y0=a, y1=b)[0] for a, b in ((0, 1), (1, 17), (17, 1000), (1000, 1080))]
        assert_same(np.concatenate(parts, 0), whole, f"ragged bands frame {f}")


def test_batched_views_equal_single_views(gpu_renderer, renderer_lib):
    sc = S.shipped_scene(1)
    gpu_renderer.load_scene(sc)
    mats = renderer_lib.camera_path(S.input_script("flythrough", 600))[::25]
    W, H = 512, 512
    batch = gpu_renderer.render(mats, W, H)
    assert batch.shape == (len(mats), H, W)
    for k in range(len(mats)):
        assert_same(batch[k], gpu_renderer.render(mats[k], W, H)[0], f"view {k}")
    gpu_renderer.set_option("views_per_chunk", 5)  # chunked submission gives the same frames
    assert np.array_equal(gpu_renderer.render(mats, W, H), batch)
    gpu_renderer.set_option("views_per_chunk", 256)


def test_tma_and_plain_write_out_agree(gpu_renderer, renderer_lib):
    """tile_raster's three write-outs — one TMA tensor store per tile, bulk row copies, plain stores — on the host path
    (24-bit packed transport, banded launches) and the device path (32-bit, whole frame and a band that cuts tile rows),
    with widths that are and are not multiples of the tile width."""
    import torch
    sc = S.shipped_scene(1)
    gpu_renderer.load_scene(sc)
    m = renderer_lib.camera_path(S.input_script("flythrough", 120))[110]
    variants = ((1, 1), (1, 0), (0, 0))   # (tma_store, tensor_store)
    for W, H in ((1280, 720), (1936, 1000), (1284, 722)):
        frames = []
        for tma, tmap in variants:
            gpu_renderer.set_option("tma_store", tma)
            gpu_renderer.set_option("tensor_store", tmap)
            host = gpu_renderer.render(m, W, H)[0]
            out = torch.zeros((H, W), dtype=torch.int32, device="cuda:0")
            gpu_renderer.render_device(m, W, H, out.data_ptr())
            assert gpu_renderer.finish() is False
            y0, y1 = H // 3 + 7, (2 * H) // 3 + 5
            band = torch.zeros((y1 - y0, W), dtype=torch.int32, device="cuda:0")
            gpu_renderer.render_device(m, W, H, band.data_ptr(), y0=y0, y1=y1)
            assert gpu_renderer.finish() is False
            frames.append((host, out.cpu().numpy().view(np.uint32), band.cpu().numpy().view(np.uint32), y0, y1))
        gpu_renderer.set_option("tma_store", 1)
        gpu_renderer.set_option("tensor_store", 1)
        ref = frames[-1][0]
        assert len(np.unique(ref)) > 100, len(np.unique(ref))
        for (tma, tmap), (host, dev, band, y0, y1) in zip(variants, frames):
            assert_same(host, ref, f"{W}x{H} host path, tma={tma} tensor={tmap}")
            assert_same(dev, ref, f"{W}x{H} device path, tma={tma} tensor={tmap}")
            assert_same(band, ref[y0:y1], f"{W}x{H} band, tma={tma} tensor={tmap}")


@pytest.mark.parametrize("direct_small", [1, 0])
def test_capacity_regrowth_is_transparent(direct_small, renderer_lib, oracle_port):
    sc = S.icosahedron_field(2000, seed=3, extent=60)
    r = renderer_lib.Renderer(0)
    r.load_scene(sc)
    r.set_option("direct_small", direct_small)
    r.set_option("setup_capacity", 8)  # far too small: forces the overflow -> regrow -> re-render path
    m = renderer_lib.camera_path(S.input_script("spin", 5))[4]
    got = r.render(m, 640, 360)[0]
    assert r.stats()["overflow"] == 0 and r.stats()["setups"] > 8
    assert_same(got, oracle_port.OracleScene(sc).render(m, 640, 360)["pixels"], "after regrow")
    r.close()


def test_empty_and_degenerate_scenes(renderer_lib, oracle_port):
    r = renderer_lib.Renderer(0)
    m = renderer_lib.camera_path(S.input_script("still", 1))[0]
    empty = S.Scene(np.ones((0, 4), "<f4"), np.zeros(0, "<u8"), np.zeros(0, S.ATTR_DTYPE), np.zeros(0, "<u8"),
                    S.procedural_textures(1))
    r.load_scene(empty)
    assert (r.render(m, 100, 50)[0] == 0x1E1E1E).all()
    # everything behind the camera / off screen
    sc = S.icosahedron_field(50, seed=2, extent=5, center=(0, 0, 500))
    r.load_scene(sc)
    got = r.render(m, 100, 50)[0]
    assert_same(got, oracle_port.OracleScene(sc).render(m, 100, 50)["pixels"], "behind camera")
    assert (got == 0x1E1E1E).all()
    r.close()


def test_invalid_scenes_are_rejected(renderer_lib):
    r = renderer_lib.Renderer(0)
    sc = S.shipped_scene(1)
    sc.vertices[0, 3] = 2.0
    with pytest.raises(renderer_lib.RendererError, match="w != 1"):
        r.load_scene(sc)
    sc = S.shipped_scene(1)
    sc.attributes["kind"][3] = 9
    with pytest.raises(renderer_lib.RendererError, match="kind"):
        r.load_scene(sc)
    with pytest.raises(renderer_lib.RendererError, match="no scene"):
        r.render(np.zeros(12, np.float32), 8, 8)
    r.close()


def test_drop_in_update_and_render(renderer_lib, oracle_port, tmp_path):
    """The reference's own calling pattern: private render.so beside data.bin, updateAndRender per frame
    into alternating halves of one pageable allocation (main.swift:117-118), live resize (main.swift:156-165)."""
    sc = S.shipped_scene(1)
    path = str(tmp_path / "data.bin")
    S.write_data_bin(path, sc)
    osc = oracle_port.OracleScene(sc)
    inp = S.input_script("flythrough", 600)[:140]
    mats = oracle_port.camera_path(inp)
    d = renderer_lib.DropIn(path)
    W, H = 320, 180
    double = np.zeros((2, H, W), np.uint32)
    for f in range(len(inp)):
        if f == 90:  # live resize
            W, H = 400, 220
            double = np.zeros((2, H, W), np.uint32)
        out = d.update_and_render(W, H, inp[f], out=double[f & 1])
        if f % 10 == 0 or f in (89, 90, 91):
            assert_same(out, osc.render(mats[f], W, H)["pixels"], f"drop-in frame {f}")
    d.close()


def test_drop_in_exits_666_without_data_bin(renderer_lib, tmp_path):
    """render-cpp/render.cpp:173 — exit(666) (status 666 & 0xFF = 154) when no data.bin is found."""
    code = (
        "import ctypes, shutil, sys\n"
        f"shutil.copy({renderer_lib.LIB_PATH!r}, {str(tmp_path / 'render.so')!r})\n"
        f"lib = ctypes.CDLL({str(tmp_path / 'render.so')!r})\n"
        "class PD(ctypes.Structure):\n"
        "    _fields_=[('b',ctypes.c_void_p),('w',ctypes.c_uint32),('h',ctypes.c_uint32),('p',ctypes.c_uint32),('s',ctypes.c_uint32)]\n"
        "buf=(ctypes.c_uint32*64)(); pd=PD(ctypes.addressof(buf),8,8,4,256); inp=(ctypes.c_float*6)()\n"
        "lib.updateAndRender(ctypes.byref(pd), ctypes.byref(inp))\n"
    )
    rc = subprocess.run([sys.executable, "-c", code]).returncode
    assert rc == (666 & 0xFF)


def test_device_resident_render_and_launch_count(gpu_renderer, renderer_lib):
    import torch
    sc = S.shipped_scene(1)
    gpu_renderer.load_scene(sc)
    m = renderer_lib.camera_path(S.input_script("flythrough", 120))[110]
    W, H = 1280, 720
    host = gpu_renderer.render(m, W, H)[0]
    out = torch.zeros((H, W), dtype=torch.int32, device="cuda:0")
    before = gpu_renderer.kernel_launches
    gpu_renderer.render_device(m, W, H, out.data_ptr())
    assert gpu_renderer.finish() is False
    assert gpu_renderer.kernel_launches - before >= 2
    assert np.array_equal(out.cpu().numpy().view(np.uint32), host)


def test_stale_host_registration_is_detected(gpu_renderer, renderer_lib):
    """Callers may free a frame buffer and get the same address back (large malloc = mmap); a cached
    cudaHostRegister would then DMA into the old pages.  The library must still fill what the CPU sees."""
    sc = S.shipped_scene(1)
    r = renderer_lib.Renderer(0)
    r.load_scene(sc)
    m = renderer_lib.camera_path(S.input_script("flythrough", 120))[110]
    W, H = 1280, 720
    want = r.render(m, W, H)[0].copy()
    r.set_option("pin_host", 1)  # opt-in fast path; the caller below then breaks its promise
    for _ in range(6):
        buf = np.zeros((1, H, W), np.uint32)  # fresh mmap each time, usually at a recycled address
        got = r.render(m, W, H, out=buf)
        assert np.array_equal(got[0], want)
        del buf, got
    r.set_option("pin_host", 0)  # drops every registration
    r.close()


def test_overflowing_bins_are_regrown(renderer_lib, oracle_port):
    """Inside a solid every triangle covers every tile: far more (triangle, tile) pairs than survivors."""
    sc = S.shipped_scene(1)
    r = renderer_lib.Renderer(0)
    r.load_scene(sc)
    r.set_option("setup_capacity", 64)  # also shrinks the bin-entry capacity to 64
    mats = renderer_lib.camera_path(S.input_script("flythrough", 600))
    osc = oracle_port.OracleScene(sc)
    for f in (110, 395, 520):
        assert_same(r.render(mats[f], 1920, 1080)[0], osc.render(mats[f], 1920, 1080)["pixels"], f"frame {f}")
    r.close()


def test_device_walk_jump_equals_sequential_adds(gpu_renderer, oracle_port):
    """The device build of walk_jump (division-free path) against true sequential binary32 adds, up to the longest jump
    a frame of 65535 pixels asks for (65534 steps, deltas down to about 1/65535)."""
    rs = np.random.RandomState(11)
    n = 20000
    s = rs.uniform(-2, 2, n).astype(np.float32)
    d = (rs.uniform(-3, 3, n) / rs.randint(1, 65536, n)).astype(np.float32)
    k = rs.randint(0, 65535, n).astype(np.uint32)
    # adversarial: ties, binade floors, zero crossings, stuck walks; the same kinds again at 65534 steps
    adv = [(2.0030441, -3.4061623e-06, 1845), (1.0, 2.0 ** -24, 3840), (1.0, -(2.0 ** -25), 3840), (1.0, 1.5 * 2.0 ** -23, 3840),
           (0.0, 1e-3, 3840), (-1.0, 1e-3, 3840), (16777216.0, 1.0, 100), (0.5, 0.0, 77),
           (1.0, 2.0 ** -24, 65534), (1.0, -(2.0 ** -25), 65534), (1.0, 1.5 * 2.0 ** -23, 65534),   # tie binades
           (1.0 + 65534 * 2.0 ** -23, -(2.0 ** -23), 65534),        # lands exactly on the binade floor at the last step
           (2.0 + 100 * 2.0 ** -22, -(2.0 ** -22), 65534),          # crosses a binade floor, then walks the finer binade
           (0.3, -1e-5, 65534), (-0.3, 1e-5, 65534), (0.0, -3.0 / 65535, 65534),   # zero crossings, a walk from zero
           (1.0, 1.0 / 65535, 65534), (-2.0, 3.0 / 65534, 65534)]
    for i, (a, b, c) in enumerate(adv):
        s[i], d[i], k[i] = a, b, c
    got = gpu_renderer.debug_walk(s, d, k)
    order = np.argsort(-k.astype(np.int64), kind="stable")   # longest walks first: walk i is live while step < k[i]
    want, dd, kk = s[order].copy(), d[order], k[order]
    live = np.searchsorted(-kk.astype(np.int64), -np.arange(int(k.max()), dtype=np.int64), side="left")
    for step in range(int(k.max())):  # vectorised sequential adds in binary32
        m = live[step]
        want[:m] = want[:m] + dd[:m]
    want = want[np.argsort(order)]
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), int((got.view(np.uint32) != want.view(np.uint32)).sum())


def test_fused_and_multi_kernel_geometry_agree(renderer_lib, oracle_port):
    """Small scenes take the single-CTA fused geometry kernel; it must produce the same frame and the same
    setup records as the general eight-launch path (and as the oracle)."""
    sc = S.shipped_scene(2, regular_floor=True)  # 1849 triangles: several 256-triangle chunks
    r = renderer_lib.Renderer(0)
    r.load_scene(sc)
    osc = oracle_port.OracleScene(sc)
    mats = renderer_lib.camera_path(S.input_script("flythrough", 600))
    for f in (40, 150, 275):
        r.set_option("fused_small", 1)
        a = r.render(mats[f], 1280, 720)[0]
        sa, la = r.setups(), r.stats()
        r.set_option("fused_small", 0)
        c = r.render(mats[f], 1280, 720)[0]   # general path, small triangles walked record-free (the default)
        lc = r.stats()
        r.set_option("direct_small", 0)
        b = r.render(mats[f], 1280, 720)[0]   # general path, every survivor recorded
        sb, lb = r.setups(), r.stats()
        r.set_option("direct_small", 1)
        assert_same(a, b, f"fused vs general frame {f}")
        assert_same(a, c, f"fused vs general (record-free small triangles) frame {f}")
        assert lc["setups"] == lb["setups"] and lc["culled"] == lb["culled"]
        assert sa.tobytes() == sb.tobytes()
        geo = ('triangles_in', 'near_rejected', 'clipped', 'spawned', 'culled', 'setups', 'overflow')
        assert {k: la[k] for k in geo} == {k: lb[k] for k in geo}  # the fused path keeps no bin statistics
        assert_same(a, osc.render(mats[f], 1280, 720)["pixels"], f"fused vs oracle frame {f}")
    r.close()


def test_host_transport_variants_agree(renderer_lib):
    """24-bit vs 32-bit PCIe transport, 1 vs 8 raster/copy bands, pinned vs staged: same bytes."""
    sc = S.shipped_scene(1)
    r = renderer_lib.Renderer(0)
    r.load_scene(sc)
    m = renderer_lib.camera_path(S.input_script("flythrough", 600))[330]
    for (W, H) in ((1920, 1080), (1000, 563), (48, 40)):
        ref = None
        for pack, bands, pin in ((1, 8, 0), (0, 8, 0), (1, 1, 0), (0, 3, 0), (1, 8, 1)):
            r.set_option("pack24", pack); r.set_option("host_bands", bands); r.set_option("pin_host", pin)
            out = np.full((1, H, W), 0x55555555, np.uint32)
            got = r.render(m, W, H, out=out)[0]
            ref = got.copy() if ref is None else ref
            assert_same(got, ref, f"{W}x{H} pack={pack} bands={bands} pin={pin}")
            assert (got >> 24 == 0).all()
        r.set_option("pin_host", 0)
    r.close()


def test_interleaved_tile_rows_reassemble_to_the_whole_frame(gpu_renderer, renderer_lib):
    """Multi-GPU load-balanced partition: tile rows dealt round-robin; the union must be the whole frame."""
    import torch
    th = renderer_lib.tile_height()
    for sc, script, fidx in ((S.shipped_scene(1), "flythrough", 330), (S.icosahedron_field(3000, seed=5, extent=50), "spin", 9)):
        gpu_renderer.load_scene(sc)
        m = renderer_lib.camera_path(S.input_script(script, 600 if script == "flythrough" else 10))[fidx]
        for (W, H) in ((1920, 1080), (640, 361)):
            whole = gpu_renderer.render(m, W, H)[0]
            for world in (2, 3, 8):
                frame = np.zeros((H, W), np.uint32)
                for phase in range(world):
                    rows, frame_rows, buf_rows = renderer_lib.rows_layout(H, world, phase, th)
                    if rows == 0:
                        continue
                    buf = torch.zeros((rows, W), dtype=torch.int32, device="cuda:0")
                    gpu_renderer.render_device_rows(m, W, H, world, phase, buf.data_ptr())
                    assert gpu_renderer.finish() is False
                    frame[frame_rows] = buf.cpu().numpy().view(np.uint32)[buf_rows]
                assert_same(frame, whole, f"{W}x{H} interleaved over {world}")


def _general_scenes():
    """Scenes that take the general (visibility-buffer) path: > 1920 triangles."""
    return (("clip", lambda: S.clip_stress_scene(3000), "spin", 9),          # straddlers, spawned, big and mid-size triangles
            ("dense", lambda: S.icosahedron_field(20000, seed=9, extent=40, r_range=(0.3, 1.0)), "spin", 5))  # tiny triangles


@pytest.mark.parametrize("which", [0, 1])
def test_general_path_variants_agree_with_the_oracle(which, gpu_renderer, renderer_lib, oracle_port):
    """Every routing of the general path must give the reference's frame: record-free direct walk on/off, and the
    flat-walk / tile-kernel split at different box sizes (16 = everything recorded goes to tiles ... 4096 = none)."""
    name, build, script, fidx = _general_scenes()[which]
    sc = build()
    gpu_renderer.load_scene(sc)
    m = renderer_lib.camera_path(S.input_script(script, 12))[fidx]
    W, H = 800, 450
    want = oracle_port.OracleScene(sc).render(m, W, H)["pixels"]
    try:
        for direct in (1, 0):
            for flat in (16, 128, 4096):
                gpu_renderer.set_option("direct_small", direct)
                gpu_renderer.set_option("flat_max", flat)
                assert_same(gpu_renderer.render(m, W, H)[0], want, f"{name} direct_small={direct} flat_max={flat}")
    finally:
        gpu_renderer.set_option("direct_small", 1)
        gpu_renderer.set_option("flat_max", 128)


@pytest.mark.parametrize("which", [0, 1])
def test_general_path_bands_rows_and_batches(which, gpu_renderer, renderer_lib):
    """Screen bands, interleaved tile rows and multi-view batches of the general path reassemble to the whole frame."""
    import torch
    name, build, script, fidx = _general_scenes()[which]
    gpu_renderer.load_scene(build())
    mats = renderer_lib.camera_path(S.input_script(script, 12))
    m = mats[fidx]
    W, H = 800, 450
    whole = gpu_renderer.render(m, W, H)[0]
    assert len(np.unique(whole)) > 50
    for n in (2, 5):
        edges = [H * k // n for k in range(n + 1)]
        parts = [gpu_renderer.render(m, W, H, y0=edges[k], y1=edges[k + 1])[0] for k in range(n)]
        assert_same(np.concatenate(parts, 0), whole, f"{name}: {n} bands")
    th = renderer_lib.tile_height()
    for world in (2, 8):
        frame = np.zeros((H, W), np.uint32)
        for phase in range(world):
            rows, frame_rows, buf_rows = renderer_lib.rows_layout(H, world, phase, th)
            if rows == 0:
                continue
            buf = torch.zeros((rows, W), dtype=torch.int32, device="cuda:0")
            gpu_renderer.render_device_rows(m, W, H, world, phase, buf.data_ptr())
            assert gpu_renderer.finish() is False
            frame[frame_rows] = buf.cpu().numpy().view(np.uint32)[buf_rows]
        assert_same(frame, whole, f"{name}: interleaved over {world}")
    batch = gpu_renderer.render(mats[3:9], W, H)
    for k in range(6):
        assert_same(batch[k], gpu_renderer.render(mats[3 + k], W, H)[0], f"{name}: view {k} of a batch")


def test_fused_assembly_writes_rows_to_every_destination(gpu_renderer, renderer_lib):
    """The shading kernel's fused frame assembly (s3r_set_peer_frames): the ranks' interleaved tile rows, stored
    straight into full-size destination frames, add up to the whole frame in every destination.  (One GPU here, two
    local destinations; across processes the destinations are CUDA-IPC mappings — tests/test_multigpu_peer.py.)"""
    sc = S.clip_stress_scene(3000)
    gpu_renderer.load_scene(sc)
    m = renderer_lib.camera_path(S.input_script("spin", 12))[9]
    W, H = 800, 450
    whole = gpu_renderer.render(m, W, H)[0]
    a, _ = gpu_renderer.peer_frame_alloc(W * H * 4)
    b, _ = gpu_renderer.peer_frame_alloc(W * H * 4)
    try:
        for world in (1, 3):
            for phase in range(world):
                gpu_renderer.set_peer_frames([a, b])
                gpu_renderer.render_device_rows(m, W, H, world, phase, 0)
                assert gpu_renderer.finish() is False
            gpu_renderer.set_peer_frames([])
            for ptr in (a, b):
                assert_same(gpu_renderer.read_device(ptr, (H, W)), whole, f"fused assembly over {world}")
        # small scenes (tile-kernel path) refuse destinations instead of silently ignoring them
        gpu_renderer.load_scene(S.shipped_scene(1))
        gpu_renderer.set_peer_frames([a])
        with pytest.raises(RuntimeError):
            gpu_renderer.render_device_rows(m, W, H, 1, 0, 0)
    finally:
        gpu_renderer.set_peer_frames([])
        gpu_renderer.peer_frame_release(a)
        gpu_renderer.peer_frame_release(b)


def test_span_tables_equal_in_tile_jumps_and_the_oracle(renderer_lib, oracle_port):
    """Small scenes, device path: the checkpoint tables of the largest survivors (span_walk, one row walk per frame)
    must give every tile exactly the weights its own exact jumps give — whole frames, bands, interleaved tile rows and
    view batches, with more than SPAN_MAX large survivors in some frames (the rest keep jumping)."""
    import torch
    th = renderer_lib.tile_height()
    r = renderer_lib.Renderer(0)
    cases = ((S.shipped_scene(1), (0, 110, 150, 230, 345, 350, 500, 550), (1920, 1080)),
             (S.shipped_scene(2, regular_floor=True), (40, 150), (1283, 721)),
             (S.icosahedron_field(60, seed=12, extent=12, r_range=(2.0, 5.0)), (3, 9), (1920, 1080)))
    for sc, frames, (W, H) in cases:
        r.load_scene(sc)
        osc = oracle_port.OracleScene(sc)
        mats = renderer_lib.camera_path(S.input_script("flythrough", 600))
        out = torch.zeros((len(frames), H, W), dtype=torch.int32, device="cuda:0")

        def dev(views, **kw):
            r.render_device(views, W, H, out.data_ptr(), **kw)
            assert r.finish() is False
            return out.cpu().numpy().view(np.uint32)

        want = np.stack([osc.render(mats[f], W, H)["pixels"] for f in frames])
        for spans in (1, 0):
            r.set_option("spans", spans)
            before = r.kernel_launches
            got = dev(mats[list(frames)])                       # one batch of views
            assert r.kernel_launches - before == (3 if spans else 2)
            for i, f in enumerate(frames):
                assert_same(got[i], want[i], f"spans={spans} batch frame {f} {W}x{H}")
        r.set_option("spans", 1)
        for f, w in zip(frames[:2], want[:2]):
            assert_same(dev(mats[f])[0], w, f"single view frame {f}")
            y0, y1 = H // 3 + 5, (2 * H) // 3 + 1               # a band that cuts tile rows
            band = dev(mats[f], y0=y0, y1=y1)
            assert_same(band.reshape(-1)[: (y1 - y0) * W].reshape(y1 - y0, W), w[y0:y1], f"band frame {f}")
            frame = np.zeros((H, W), np.uint32)
            for phase in range(3):
                rows, frame_rows, buf_rows = renderer_lib.rows_layout(H, 3, phase, th)
                buf = torch.zeros((rows, W), dtype=torch.int32, device="cuda:0")
                r.render_device_rows(mats[f], W, H, 3, phase, buf.data_ptr())
                assert r.finish() is False
                frame[frame_rows] = buf.cpu().numpy().view(np.uint32)[buf_rows]
            assert_same(frame, w, f"interleaved rows frame {f}")
    r.close()


def test_exact_math_equals_ieee_operators(gpu_renderer):
    """csrc/exact_math.cuh: the shading chain's hand-scheduled 1/sqrt and shared-reciprocal divisions must be the
    compiler's correctly rounded operators bit for bit — EVERY positive binary32 (and the negative/NaN fallbacks) for
    1/sqrt, 2^33 seeded operand sets incl. extreme mantissas and out-of-range operands for the division."""
    import ctypes
    lib, h = gpu_renderer._lib, gpu_renderer._h
    lib.s3r_debug_exact_math.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_uint32,
                                         ctypes.POINTER(ctypes.c_uint64)]
    res = (ctypes.c_uint64 * 5)()
    assert lib.s3r_debug_exact_math(h, 0, 0, 1 << 32, 0, res) == 0          # all 2^32 bit patterns
    assert res[0] == 0, f"1/sqrt: {res[0]} mismatches, first x={res[1]:08x} got={res[2]:08x} want={res[3]:08x}"
    for seed in (1, 2):
        assert lib.s3r_debug_exact_math(h, 1, 0, 1 << 32, seed, res) == 0
        assert res[0] == 0, f"div: {res[0]} mismatches, first a={res[1]:08x} b={res[2]:08x} got={res[3]:08x} want={res[4]:08x}"
    for seed in (3, 4):   # the vertex stage's two projections by one depth: operands of either sign, signed zeros
        assert lib.s3r_debug_exact_math(h, 2, 0, 1 << 32, seed, res) == 0
        assert res[0] == 0, f"signed div: {res[0]} mismatches, first a={res[1]:08x} b={res[2]:08x} got={res[3]:08x} want={res[4]:08x}"


def _i420_reference(px):
    """numpy restatement of the sink's BT.601 limited-range conversion (csrc/renderer.cu: bgr0_to_i420)."""
    H, W = px.shape
    r, g, b = ((px >> 16) & 255).astype(np.int64), ((px >> 8) & 255).astype(np.int64), (px & 255).astype(np.int64)
    y = ((66 * r + 129 * g + 25 * b + 128) >> 8) + 16
    ys, xs = np.minimum(np.arange(0, H + (H & 1)), H - 1), np.minimum(np.arange(0, W + (W & 1)), W - 1)
    mean = lambda c: (c[np.ix_(ys, xs)].reshape(len(ys) // 2, 2, len(xs) // 2, 2).sum(axis=(1, 3)) + 2) >> 2
    r2, g2, b2 = mean(r), mean(g), mean(b)
    u = ((-38 * r2 - 74 * g2 + 112 * b2 + 128) >> 8) + 128
    v = ((112 * r2 - 94 * g2 - 18 * b2 + 128) >> 8) + 128
    return np.concatenate([y.astype(np.uint8).ravel(), u.astype(np.uint8).ravel(), v.astype(np.uint8).ravel()])


def test_frame_sink_writes_device_frames(gpu_renderer, renderer_lib, tmp_path):
    """s3r_sink_*: device-resident frames go to a raw BGR0 file unchanged and to a YUV4MPEG2 file through the GPU colour
    conversion — more frames than the pinned ring holds, odd frame size, frames overwritten right after submission."""
    import torch
    sc = S.shipped_scene(1)
    gpu_renderer.load_scene(sc)
    mats = renderer_lib.camera_path(S.input_script("flythrough", 600))
    W, H, frames = 1283, 721, (0, 110, 150, 230, 330, 450, 599)
    want = [gpu_renderer.render(mats[f], W, H)[0] for f in frames]
    out = torch.zeros((H, W), dtype=torch.int32, device="cuda:0")
    raw_path, y4m_path = str(tmp_path / "frames.bgr0"), str(tmp_path / "frames.y4m")
    raw = renderer_lib.Sink(gpu_renderer, raw_path, W, H, fmt=0)
    y4m = renderer_lib.Sink(gpu_renderer, y4m_path, W, H, fps=(30, 1), fmt=1)
    for f in frames:                                   # one frame buffer, reused: the sinks are stream-ordered
        gpu_renderer.render_device(mats[f], W, H, out.data_ptr())
        raw.submit(out.data_ptr())
        y4m.submit(out.data_ptr())
    assert raw.close() == len(frames) and y4m.close() == len(frames)
    assert gpu_renderer.finish() is False
    got = np.fromfile(raw_path, np.uint32).reshape(len(frames), H, W)
    for i, f in enumerate(frames):
        assert_same(got[i], want[i], f"raw sink frame {f}")
    blob = open(y4m_path, "rb").read()
    head, _, body = blob.partition(b"\n")
    assert head.split()[:4] == [b"YUV4MPEG2", b"W%d" % W, b"H%d" % H, b"F30:1"] and b"C420jpeg" in head
    n = W * H + 2 * ((W + 1) // 2) * ((H + 1) // 2)
    assert len(body) == len(frames) * (6 + n)
    for i, f in enumerate(frames):
        rec = body[i * (6 + n):(i + 1) * (6 + n)]
        assert rec[:6] == b"FRAME\n"
        assert np.array_equal(np.frombuffer(rec[6:], np.uint8), _i420_reference(want[i])), f"y4m frame {f}"


def _cluster_scenes():
    return (("field", lambda: S.icosahedron_field(20000, seed=12, extent=(300.0, 170.0, 160.0), r_range=(0.5, 4.0), center=(0.0, 0.0, -420.0)), "spin"),
            ("inside", lambda: S.icosahedron_field(6000, seed=13, extent=60), "spin"),   # camera inside the field: clusters behind, beside, across the near plane
            ("clip", lambda: S.clip_stress_scene(3000), "strafe"),
            ("floor", lambda: S.shipped_scene(2, regular_floor=True), "flythrough"))


@pytest.mark.parametrize("which", [0, 1, 2, 3])
def test_cluster_front_equals_the_unclustered_front_and_the_oracle(which, renderer_lib, oracle_port):
    """The spatial pre-partition is invisible: frames AND the per-triangle statistics (near-rejected / clipped / culled /
    rasterised, render.cpp:306-317) are the same whether whole clusters are rejected by their bounds, every triangle of every
    cluster is tested, or the raw triangle stream is classified — whole frames, bands and interleaved tile rows."""
    import torch
    name, build, script = _cluster_scenes()[which]
    sc = build()
    r = renderer_lib.Renderer(0)
    try:
        r.set_option("fused_small", 0)   # ("floor" has 1 849 triangles: force it onto the general path)
        r.load_scene(sc)
        osc = oracle_port.OracleScene(sc)
        n = 600 if script == "flythrough" else 24
        mats = renderer_lib.camera_path(S.input_script(script, n))
        W, H = 800, 450
        th = renderer_lib.tile_height()
        for f in ((40, 100, 330) if script == "flythrough" else (0, 7, 23)):
            o = osc.render(mats[f], W, H)
            ref_stats = None
            for clusters, cull in ((1, 1), (1, 0), (0, 0)):
                r.set_option("clusters", clusters); r.set_option("cluster_cull", cull)
                got = r.render(mats[f], W, H)[0]
                assert_same(got, o["pixels"], f"{name} frame {f} clusters={clusters} cull={cull}")
                st = r.stats()
                assert st["near_rejected"] == o["stats"]["near_rejected"] and st["clipped"] == o["stats"]["clipped"]
                assert st["setups"] == o["stats"]["rasterized"] and st["culled"] == o["stats"]["offscreen"] + o["stats"]["small_or_backfacing"]
                ref_stats = ref_stats or st
                assert st == ref_stats
            r.set_option("clusters", 1); r.set_option("cluster_cull", 1)
            parts = [r.render(mats[f], W, H, y0=H * k // 3, y1=H * (k + 1) // 3)[0] for k in range(3)]
            assert_same(np.concatenate(parts, 0), o["pixels"], f"{name} frame {f}: 3 bands through the cluster front")
            frame = np.zeros((H, W), np.uint32)
            for phase in range(4):
                rows, frame_rows, buf_rows = renderer_lib.rows_layout(H, 4, phase, th)
                buf = torch.zeros((rows, W), dtype=torch.int32, device="cuda:0")
                for attempt in range(4):
                    r.render_device_rows(mats[f], W, H, 4, phase, buf.data_ptr())
                    if not r.finish():
                        break
                frame[frame_rows] = buf.cpu().numpy().view(np.uint32)[buf_rows]
            assert_same(frame, o["pixels"], f"{name} frame {f}: 4 interleaved phases through the cluster front")
    finally:
        r.close()


def test_cluster_rejection_is_conservative_for_any_matrix(renderer_lib, oracle_port):
    """s3r_render_device takes any 3x4 matrix, not only a camera's orthonormal rows: scaled, sheared and far-away views
    (most clusters too small, off screen or behind) still give the oracle's frame and statistics."""
    sc = S.icosahedron_field(8000, seed=21, extent=(200.0, 120.0, 100.0), r_range=(0.5, 6.0), center=(0.0, 0.0, -300.0))
    r = renderer_lib.Renderer(0)
    try:
        r.load_scene(sc)
        osc = oracle_port.OracleScene(sc)
        base = renderer_lib.camera_path(S.input_script("spin", 6))[5].reshape(3, 4)
        views = []
        for scale, shear, back in ((1.0, 0.0, 0.0), (1.7, 0.0, 0.0), (0.45, 0.0, 0.0), (1.0, 0.35, 0.0), (1.0, 0.0, 900.0), (1.0, 0.0, -250.0)):
            m = base.copy()
            m[:, :3] *= scale
            m[0, :3] += shear * m[1, :3]
            m[2, 3] -= back                      # camera-space z shifts: the field recedes (back > 0) or swallows the camera
            views.append(m.reshape(12).astype(np.float32))
        culled_clusters = 0
        for k, m in enumerate(views):
            o = osc.render(m, 640, 360)
            assert_same(r.render(m, 640, 360)[0], o["pixels"], f"matrix {k}")
            st = r.stats()
            assert st["near_rejected"] == o["stats"]["near_rejected"] and st["clipped"] == o["stats"]["clipped"]
            assert st["setups"] == o["stats"]["rasterized"] and st["culled"] == o["stats"]["offscreen"] + o["stats"]["small_or_backfacing"]
            culled_clusters += st["culled"]
        assert culled_clusters > 0
    finally:
        r.close()


@pytest.mark.parametrize("pin", ["1", "0"])
def test_multi_gpu_drop_in_matches_the_single_gpu_frames(pin, renderer_lib, tmp_path):
    """updateAndRender driving several GPUs from one process (S3R_DEVICES): interleaved tile rows, one host thread per
    GPU, every GPU copies its rows into the caller's buffer.  On a one-GPU box the same device is named three times —
    the threads, the row split and the copies are the same code.  Both scenes (tile-kernel path, general path), a live
    resize, registered caller memory (pin = 1) and the pinned-staging path (pin = 0)."""
    import torch
    n_gpu = torch.cuda.device_count()
    devices = ",".join(str(k % n_gpu) for k in range(max(3, min(n_gpu, 4))))
    field = S.icosahedron_field(4000, seed=17, extent=50)
    for name, sc, script in (("shipped", S.shipped_scene(1), "flythrough"), ("field", field, "spin")):
        path = str(tmp_path / f"{name}_{pin}.data.bin")
        S.write_data_bin(path, sc)
        inp = S.input_script(script, 40)
        d = renderer_lib.DropIn(path, devices=devices, env={"S3R_PIN_HOST": pin})
        r = renderer_lib.Renderer(0)
        try:
            r.load_scene(sc)
            cam = renderer_lib.Camera()
            buf = np.zeros((2, 1080, 1920), np.uint32)
            last_wh = None
            for f in range(40):
                W, H = (1920, 1080) if f < 25 or f >= 32 else (1283, 721)   # a live resize and back (main.swift:156-165)
                out = buf[f & 1].reshape(-1)[: W * H].reshape(H, W)
                d.update_and_render(W, H, inp[f], out=out)
                m = cam.update(inp[f])
                if f in (0, 1, 24, 25, 26, 31, 32, 39):
                    # the reference's stale-factor rule (render.cpp:275-280) is exercised by the resize: compare with a
                    # single-GPU drop-in semantics = s3r_factor of the CURRENT height whenever W*H changes, which it does here
                    assert_same(out, r.render(m, W, H)[0], f"{name} pin={pin} frame {f} at {W}x{H}")
                last_wh = (W, H)
            assert d.n_devices == len(devices.split(","))
        finally:
            d.close()
            r.close()
