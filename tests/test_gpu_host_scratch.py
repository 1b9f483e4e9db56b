"""Ownership of the renderer's device memory: every buffer a renderer allocates is freed when it is destroyed, and a
scene load drops the per-view scratch sized for the previous scene."""
import gc

import numpy as np
import pytest

from swift3drenderer_b200 import scene as S

pytestmark = pytest.mark.gpu

MIB = 1 << 20


def _free_bytes() -> int:
    import torch
    torch.cuda.synchronize(0)
    return torch.cuda.mem_get_info(0)[0]


def test_device_memory_returns_to_baseline(renderer_lib):
    """Create -> general-path scene -> whole frame, interleaved rows, host render, forced regrowth, debug_walk -> destroy,
    three times: free device memory comes back every time."""
    import torch
    field = S.icosahedron_field(4000)
    m = renderer_lib.camera_path(S.input_script("spin", 8))[7]
    W, H = 1280, 720
    rows, _, _ = renderer_lib.rows_layout(H, 3, 1)
    out = torch.zeros((H, W), dtype=torch.int32, device="cuda:0")
    band = torch.zeros((rows, W), dtype=torch.int32, device="cuda:0")
    walk = np.linspace(0, 1, 1000, dtype=np.float32), np.full(1000, 1e-3, np.float32), np.arange(1000, dtype=np.uint32)

    def cycle():
        r = renderer_lib.Renderer(0)
        try:
            r.load_scene(field)
            for _ in range(4):
                r.render_device(m, W, H, out.data_ptr())
                if not r.finish():
                    break
            for _ in range(4):
                r.render_device_rows(m, W, H, 3, 1, band.data_ptr())
                if not r.finish():
                    break
            host = r.render(m, W, H)[0]
            assert np.array_equal(host, out.cpu().numpy().view(np.uint32))
            r.set_option("setup_capacity", 8)
            assert np.array_equal(r.render(m, W, H)[0], host)
            r.debug_walk(*walk)
        finally:
            r.close()

    cycle()   # first launches load the kernels and size the context's own reservations: not the renderer's memory
    gc.collect()
    base = _free_bytes()
    for k in range(3):
        cycle()
        free = _free_bytes()
        assert base - free <= 16 * MIB, f"cycle {k}: {(base - free) / MIB:.1f} MiB of device memory not returned"


def test_scene_reload_frees_the_old_scratch(renderer_lib):
    """A 4K frame of a general-path scene sizes the key plane (8 bytes per pixel) and more; a small scene rendered at the
    same size needs none of it, so loading it must give that memory back."""
    W, H = 3840, 2160
    m = renderer_lib.camera_path(S.input_script("spin", 8))[7]
    r = renderer_lib.Renderer(0)
    try:
        r.load_scene(S.icosahedron_field(4000))
        r.render(m, W, H)
        before = _free_bytes()
        r.load_scene(S.shipped_scene(1))
        r.render(m, W, H)
        after = _free_bytes()
        assert after - before >= W * H * 8, f"only {(after - before) / MIB:.1f} MiB freed by the scene reload"
    finally:
        r.close()
