"""Host-side mirror of the renderer's C ABI (``include/render.h``, ``include/s3r_b200.h``) over ctypes.

The product is ``swift3drenderer_b200/lib/render.so`` (hand-written sm_100a CUDA behind an
``extern "C"`` layer).  This module only marshals pointers and sizes; it never renders anything
itself and there is no CPU fallback: if the shared library is missing or no CUDA device is
present, construction fails loudly.

``DropIn`` drives the library exactly the way the reference's main loop drives ``render.dylib``
(``main.swift:95-99,117-121``): a private copy of the shared object beside a ``data.bin``, the single
symbol ``updateAndRender(const PixelData*, const Input*)``, one call per frame.
"""
from __future__ import annotations

import ctypes
import os
import shutil
import subprocess
import tempfile
from typing import Optional

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("S3R_LIB") or os.path.join(HERE, "lib", "render.so")  # S3R_LIB: experiment builds
CSRC = os.path.join(HERE, "csrc")


class PixelData(ctypes.Structure):  # render-cpp/render.hpp:7-13
    _fields_ = [
        ("buffer", ctypes.POINTER(ctypes.c_uint32)),
        ("width", ctypes.c_uint32),
        ("height", ctypes.c_uint32),
        ("bytesPerPixel", ctypes.c_uint32),
        ("bufferSize", ctypes.c_uint32),
    ]


class Input(ctypes.Structure):  # render-cpp/render.hpp:15-21
    _fields_ = [
        ("up", ctypes.c_float), ("down", ctypes.c_float), ("left", ctypes.c_float), ("right", ctypes.c_float),
        ("mouse", ctypes.c_float * 2),
    ]


class CCamera(ctypes.Structure):
    _fields_ = [
        ("position", ctypes.c_float * 3), ("axis_x", ctypes.c_float * 3), ("axis_y", ctypes.c_float * 3),
        ("axis_z", ctypes.c_float * 3), ("matrix", ctypes.c_float * 12), ("mouse", ctypes.c_float * 2),
        ("started", ctypes.c_int32),
    ]


class CStats(ctypes.Structure):
    _fields_ = [(n, ctypes.c_uint32) for n in (
        "triangles_in", "near_rejected", "clipped", "spawned", "culled", "setups", "bin_entries",
        "big_triangles", "overflow")] + [("reserved", ctypes.c_uint32 * 7)]


SETUP_DTYPE = np.dtype([
    ("order", "<u4"), ("xmin", "<u4"), ("xmax", "<u4"), ("ymin", "<u4"), ("ymax", "<u4"), ("area", "<f4"),
    ("wstart", "<f4", (3,)), ("dx", "<f4", (3,)), ("dy", "<f4", (3,)), ("rvz", "<f4", (3,)),
    ("cv", "<f4", (3, 3)), ("n", "<f4", (3, 3)), ("kind", "<u4"), ("texture", "<u4"),
    ("payload", "<f4", (3, 3)), ("dz", "<f4", (2,)), ("tpp", "<f4", (2,)),
])

assert ctypes.sizeof(PixelData) == 24 and ctypes.sizeof(Input) == 24

EXPORTS = [
    "updateAndRender", "s3r_create", "s3r_destroy", "s3r_last_error", "s3r_load_scene_file",
    "s3r_load_scene_arrays", "s3r_scene_counts", "s3r_camera_reset", "s3r_camera_update", "s3r_factor",
    "s3r_render_device", "s3r_finish", "s3r_render_host", "s3r_get_stats", "s3r_dump_raster_vertices",
    "s3r_dump_setups", "s3r_kernel_launches", "s3r_set_option", "s3r_get_timing",
    "s3r_dropin_reset", "s3r_debug_walk", "s3r_debug_exact_math", "s3r_render_device_rows", "s3r_tile_height",
    "s3r_peer_frame_alloc", "s3r_peer_frame_open", "s3r_peer_frame_release", "s3r_set_peer_frames", "s3r_copy_from_device",
    "s3r_sink_open", "s3r_sink_submit", "s3r_sink_close", "s3r_debug_band_edges", "s3r_get_kernel_timing", "s3r_debug_clusters", "s3r_dropin_devices", "s3r_dropin_release_pins",
    "s3r_render_device_ssaa", "s3r_render_host_ssaa", "s3r_render_device_visibility",
    "s3r_update_vertices", "s3r_update_attributes", "s3r_update_texels", "s3r_dump_clusters",
]


class RendererError(RuntimeError):
    pass


def build_library(force: bool = False) -> str:
    """Compiles the CUDA sources for sm_100a (nvcc cross-compiles without a GPU)."""
    srcs = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [
        os.path.join(HERE, "..", "include", "render.h"), os.path.join(HERE, "..", "include", "s3r_b200.h")]
    stale = not os.path.exists(LIB_PATH) or any(
        os.path.getmtime(s) > os.path.getmtime(LIB_PATH) for s in srcs if os.path.exists(s))
    if force or stale:
        if shutil.which("nvcc") is None:
            if os.path.exists(LIB_PATH):
                return LIB_PATH
            raise RendererError("render.so is missing and nvcc is not available to build it")
        subprocess.check_call(["make", "-s", "-C", CSRC] + (["-B"] if force else []))
    return LIB_PATH


_lib = None


def load_library(path: Optional[str] = None) -> ctypes.CDLL:
    """Loads render.so and declares every entry point.  No fallback: a missing library is an error."""
    global _lib
    if path is None and _lib is not None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise RendererError(f"{p} not found: build it with swift3drenderer_b200.renderer.build_library() "
                            "(there is no CPU fallback)")
    lib = ctypes.CDLL(p)
    vp, u32, u64 = ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint64
    lib.updateAndRender.argtypes = [ctypes.POINTER(PixelData), ctypes.POINTER(Input)]
    lib.updateAndRender.restype = None
    lib.s3r_create.argtypes = [ctypes.POINTER(vp), ctypes.c_int]
    lib.s3r_destroy.argtypes = [vp]
    lib.s3r_destroy.restype = None
    lib.s3r_last_error.restype = ctypes.c_char_p
    lib.s3r_load_scene_file.argtypes = [vp, ctypes.c_char_p]
    lib.s3r_load_scene_arrays.argtypes = [vp, vp, u64, vp, vp, u64, vp, u64, vp, u64]
    lib.s3r_scene_counts.argtypes = [vp] + [ctypes.POINTER(u64)] * 4
    lib.s3r_camera_reset.argtypes = [ctypes.POINTER(CCamera)]
    lib.s3r_camera_reset.restype = None
    lib.s3r_camera_update.argtypes = [ctypes.POINTER(CCamera), ctypes.POINTER(Input)]
    lib.s3r_camera_update.restype = None
    lib.s3r_factor.argtypes = [u32]
    lib.s3r_factor.restype = ctypes.c_float
    lib.s3r_render_device.argtypes = [vp, vp, u32, u32, u32, u32, u32, vp, vp]
    lib.s3r_finish.argtypes = [vp]
    lib.s3r_render_host.argtypes = [vp, vp, u32, u32, u32, u32, u32, vp]
    lib.s3r_render_device_ssaa.argtypes = [vp, vp, u32, u32, u32, u32, u32, u32, vp, vp]
    lib.s3r_render_device_visibility.argtypes = [vp, vp, u32, u32, u32, u32, u32, vp, vp, vp, vp]
    lib.s3r_render_host_ssaa.argtypes = [vp, vp, u32, u32, u32, u32, u32, u32, vp]
    lib.s3r_get_stats.argtypes = [vp, u32, ctypes.POINTER(CStats)]
    lib.s3r_dump_raster_vertices.argtypes = [vp, u32, vp, u64]
    lib.s3r_dump_setups.argtypes = [vp, u32, vp, u64, ctypes.POINTER(u64)]
    lib.s3r_kernel_launches.argtypes = [vp]
    lib.s3r_kernel_launches.restype = u64
    lib.s3r_set_option.argtypes = [vp, ctypes.c_char_p, ctypes.c_int64]
    lib.s3r_get_timing.argtypes = [vp, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double),
                                   ctypes.POINTER(u64), ctypes.c_int]
    lib.s3r_debug_walk.argtypes = [vp, vp, vp, vp, vp, u32]
    lib.s3r_debug_exact_math.argtypes = [vp, u32, u64, u64, u32, ctypes.POINTER(u64)]
    lib.s3r_render_device_rows.argtypes = [vp, vp, u32, u32, u32, u32, u32, vp, vp]
    lib.s3r_tile_height.restype = u32
    lib.s3r_peer_frame_alloc.argtypes = [vp, u64, ctypes.POINTER(vp), ctypes.c_char_p]
    lib.s3r_peer_frame_open.argtypes = [vp, ctypes.c_char_p, ctypes.POINTER(vp)]
    lib.s3r_peer_frame_release.argtypes = [vp, vp]
    lib.s3r_set_peer_frames.argtypes = [vp, ctypes.POINTER(vp), u32]
    lib.s3r_copy_from_device.argtypes = [vp, vp, vp, u64]
    lib.s3r_sink_open.argtypes = [vp, ctypes.c_char_p, u32, u32, u32, u32, ctypes.c_int, ctypes.POINTER(vp)]
    lib.s3r_sink_submit.argtypes = [vp, vp, vp]
    lib.s3r_sink_close.argtypes = [vp, ctypes.POINTER(u64)]
    lib.s3r_debug_band_edges.argtypes = [u32, ctypes.c_int, ctypes.c_int, ctypes.POINTER(u32), ctypes.c_int]
    lib.s3r_debug_clusters.argtypes = [vp, u64, vp, u64, vp, u64, vp, u64, vp, ctypes.POINTER(u64)]
    lib.s3r_update_vertices.argtypes = [vp, u64, u64, vp, ctypes.c_int, vp]
    lib.s3r_update_attributes.argtypes = [vp, u64, u64, vp, vp]
    lib.s3r_update_texels.argtypes = [vp, u32, u32, vp, ctypes.c_int, vp]
    lib.s3r_dump_clusters.argtypes = [vp, vp, u64, vp, u64, ctypes.POINTER(u64)]
    lib.s3r_get_kernel_timing.argtypes = [vp, u32, ctypes.POINTER(ctypes.c_char_p), ctypes.POINTER(ctypes.c_double), ctypes.POINTER(u64)]
    if path is None:
        _lib = lib
    return lib


def make_input(rec) -> Input:
    i = Input()
    i.up, i.down, i.left, i.right = float(rec["up"]), float(rec["down"]), float(rec["left"]), float(rec["right"])
    i.mouse[0], i.mouse[1] = float(rec["mouse"][0]), float(rec["mouse"][1])
    return i


class Camera:
    """Host camera with the reference's ``update_camera`` semantics (render-cpp/render.cpp:134-156)."""

    def __init__(self):
        self._lib = load_library()
        self.c = CCamera()
        self._lib.s3r_camera_reset(ctypes.byref(self.c))

    def update(self, rec) -> np.ndarray:
        i = make_input(rec)
        self._lib.s3r_camera_update(ctypes.byref(self.c), ctypes.byref(i))
        return self.matrix

    @property
    def matrix(self) -> np.ndarray:
        return np.array(self.c.matrix[:], dtype=np.float32)


def camera_path(inputs) -> np.ndarray:
    """(n, 12) camera matrices: pose k is the state after k + 1 Input records."""
    cam = Camera()
    return np.stack([cam.update(r) for r in inputs]) if len(inputs) else np.zeros((0, 12), np.float32)


CLUSTER_HDR_DTYPE = np.dtype([("center", "<f4", (3,)), ("radius", "<f4"), ("max_edge", "<f4"), ("t0", "<u4"), ("v_off", "<u4"), ("tri_off", "<u4")])


def debug_clusters(scene) -> dict:
    """The load-time spatial pre-partition of ``scene``'s triangle stream (test hook, no GPU needed)."""
    lib = load_library()
    v = np.ascontiguousarray(scene.vertices, "<f4")
    vi = np.ascontiguousarray(scene.vertex_indices, "<u8")
    counts = (ctypes.c_uint64 * 3)()
    rc = lib.s3r_debug_clusters(v.ctypes.data, v.shape[0], vi.ctypes.data, vi.shape[0], None, 0, None, 0, None, counts)
    if rc < 0:
        raise RendererError(lib.s3r_last_error().decode())
    nc, nv, nt = int(counts[0]), int(counts[1]), int(counts[2])
    hdr = np.zeros(nc + 1, CLUSTER_HDR_DTYPE)
    pos = np.zeros((3, max(nv, 1)), np.float32)
    tri = np.zeros(max(nt, 1), np.uint32)
    rc = lib.s3r_debug_clusters(v.ctypes.data, v.shape[0], vi.ctypes.data, vi.shape[0], hdr.ctypes.data, nc + 1, pos.ctypes.data,
                                max(nv, 1), tri.ctypes.data, counts)
    if rc < 0:
        raise RendererError(lib.s3r_last_error().decode())
    return {"hdr": hdr, "pos": pos[:, :nv], "tri": tri[:nt]}


def tile_height() -> int:
    return int(load_library().s3r_tile_height())


def rows_layout(height: int, row_stride: int, row_phase: int, th: Optional[int] = None):
    """(compacted buffer rows, frame row -> buffer row map for the rows this phase owns) of
    ``s3r_render_device_rows``."""
    th = th or tile_height()
    tile_rows = (height + th - 1) // th
    owned = [a for a in range(tile_rows) if a % row_stride == row_phase]
    frame_rows, buf_rows = [], []
    for l, a in enumerate(owned):
        for i in range(th):
            if a * th + i < height:
                frame_rows.append(a * th + i)
                buf_rows.append(l * th + i)
    return len(owned) * th, np.asarray(frame_rows, np.int64), np.asarray(buf_rows, np.int64)


class Renderer:
    """One renderer bound to one GPU.  ``render`` is synchronous host-buffer rendering; ``render_device``
    enqueues on a stream and leaves the frame in HBM."""

    def __init__(self, device: int = 0):
        self._lib = load_library()
        self._h = ctypes.c_void_p()
        self._check(self._lib.s3r_create(ctypes.byref(self._h), device))
        self.device = device

    def _check(self, rc: int) -> int:
        if rc < 0:
            raise RendererError(f"s3r error {rc}: {self._lib.s3r_last_error().decode()}")
        return rc

    def close(self) -> None:
        if getattr(self, "_h", None) and self._h.value:
            self._lib.s3r_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- scene --------------------------------------------------------------------------------
    def load_scene_file(self, path: str) -> None:
        self._check(self._lib.s3r_load_scene_file(self._h, path.encode()))

    def load_scene(self, scene) -> None:
        v = np.ascontiguousarray(scene.vertices, "<f4")
        vi = np.ascontiguousarray(scene.vertex_indices, "<u8")
        ai = np.ascontiguousarray(scene.attribute_indices, "<u8")
        at = np.ascontiguousarray(scene.attributes)
        tx = np.ascontiguousarray(scene.textures, "<u4")
        assert at.dtype.itemsize == 48 and vi.shape == ai.shape
        self._check(self._lib.s3r_load_scene_arrays(
            self._h, v.ctypes.data, v.shape[0], vi.ctypes.data, ai.ctypes.data, vi.shape[0], at.ctypes.data,
            at.shape[0], tx.ctypes.data, tx.size))

    # ---- scene updates (include/s3r_b200.h): contents change in place, counts stay ---------------------------------------
    @staticmethod
    def _source(data, dtype, width):
        """(pointer, element count, on device, keep-alive) of a host array or a contiguous CUDA tensor."""
        if hasattr(data, "data_ptr") and getattr(data, "is_cuda", False):
            assert data.is_contiguous() and data.element_size() == np.dtype(dtype).itemsize
            return data.data_ptr(), data.numel() // width, 1, data
        a = np.ascontiguousarray(data, dtype)
        return a.ctypes.data, a.size // width, 0, a

    def update_vertices(self, xyz, first: int = 0, stream: int = 0) -> None:
        """New positions for vertices ``first ..``: a numpy (n, 3) float32 array (host) or a contiguous CUDA float32
        tensor of n x 3 values (device; it must stay unchanged until the enqueued update has run).  Ordered on ``stream``
        (0 = the renderer's own stream); the load-time clusters are refit on the GPU."""
        ptr, n, dev, _keep = self._source(xyz, "<f4", 3)
        self._check(self._lib.s3r_update_vertices(self._h, first, n, ctypes.c_void_p(ptr), dev, ctypes.c_void_p(stream)))

    def update_attributes(self, records, first: int = 0, stream: int = 0) -> None:
        """New attribute records (``scene.ATTR_DTYPE``, host) for attributes ``first ..``, checked by the load rules."""
        at = np.ascontiguousarray(records)
        assert at.dtype.itemsize == 48
        self._check(self._lib.s3r_update_attributes(self._h, first, at.shape[0], at.ctypes.data, ctypes.c_void_p(stream)))

    def update_textures(self, atlases, first: int = 0, stream: int = 0) -> None:
        """New 512 x 512 atlases (uint32 0x00RRGGBB rip-maps) from ``first`` on: an array or a contiguous CUDA tensor."""
        ptr, n, dev, _keep = self._source(atlases, "<u4", 1 << 18)
        self._check(self._lib.s3r_update_texels(self._h, first, n, ctypes.c_void_p(ptr), dev, ctypes.c_void_p(stream)))

    def cluster_dump(self) -> dict:
        """The device's cluster headers (``CLUSTER_HDR_DTYPE``, with the sentinel) and planar copies (3, cluster vertices)."""
        counts = (ctypes.c_uint64 * 3)()
        self._check(self._lib.s3r_dump_clusters(self._h, None, 0, None, 0, counts))
        nc, nv = int(counts[0]), int(counts[1])
        hdr = np.zeros(nc + 1, CLUSTER_HDR_DTYPE)
        pos = np.zeros((3, max(nv, 1)), np.float32)
        self._check(self._lib.s3r_dump_clusters(self._h, hdr.ctypes.data, nc + 1, pos.ctypes.data, max(nv, 1), counts))
        return {"hdr": hdr, "pos": pos[:, :nv]}

    def set_option(self, name: str, value: int) -> None:
        self._check(self._lib.s3r_set_option(self._h, name.encode(), int(value)))

    # ---- rendering ----------------------------------------------------------------------------
    def render(self, cameras, width: int, height: int, y0: int = 0, y1: Optional[int] = None,
               out: Optional[np.ndarray] = None) -> np.ndarray:
        cams = np.ascontiguousarray(cameras, "<f4").reshape(-1, 12)
        y1 = height if y1 is None else y1
        n = cams.shape[0]
        if out is None:
            out = np.empty((n, y1 - y0, width), np.uint32)
        assert out.dtype == np.uint32 and out.size == n * (y1 - y0) * width and out.flags.c_contiguous
        self._check(self._lib.s3r_render_host(self._h, cams.ctypes.data, n, width, height, y0, y1, out.ctypes.data))
        return out

    def render_device(self, cameras, width: int, height: int, dev_ptr: int, y0: int = 0, y1: Optional[int] = None,
                      stream: int = 0) -> None:
        cams = np.ascontiguousarray(cameras, "<f4").reshape(-1, 12)
        y1 = height if y1 is None else y1
        self._check(self._lib.s3r_render_device(self._h, cams.ctypes.data, cams.shape[0], width, height, y0, y1,
                                                 ctypes.c_void_p(dev_ptr), ctypes.c_void_p(stream)))

    def render_ssaa(self, cameras, width: int, height: int, samples: int, y0: int = 0, y1: Optional[int] = None,
                    out: Optional[np.ndarray] = None) -> np.ndarray:
        """``render`` with ``samples`` x ``samples`` samples per pixel (1, 2 or 4), box-resolved: the frame rendered at
        ``samples * width`` x ``samples * height``, each block averaged per channel with rounding half up.  Sizes and
        rows are output pixels."""
        cams = np.ascontiguousarray(cameras, "<f4").reshape(-1, 12)
        y1 = height if y1 is None else y1
        n = cams.shape[0]
        if out is None:
            out = np.empty((n, max(y1 - y0, 0), width), np.uint32)
        assert out.dtype == np.uint32 and out.size == n * max(y1 - y0, 0) * width and out.flags.c_contiguous
        self._check(self._lib.s3r_render_host_ssaa(self._h, cams.ctypes.data, n, width, height, y0, y1, samples,
                                                   out.ctypes.data))
        return out

    def render_device_ssaa(self, cameras, width: int, height: int, samples: int, dev_ptr: int, y0: int = 0,
                           y1: Optional[int] = None, stream: int = 0) -> None:
        """``render_device`` with ``samples`` x ``samples`` samples per pixel; see ``render_ssaa``."""
        cams = np.ascontiguousarray(cameras, "<f4").reshape(-1, 12)
        y1 = height if y1 is None else y1
        self._check(self._lib.s3r_render_device_ssaa(self._h, cams.ctypes.data, cams.shape[0], width, height, y0, y1,
                                                      samples, ctypes.c_void_p(dev_ptr), ctypes.c_void_p(stream)))

    def render_device_visibility(self, cameras, width: int, height: int, colour_ptr: int = 0, triangle_ptr: int = 0,
                                 depth_ptr: int = 0, y0: int = 0, y1: Optional[int] = None, stream: int = 0) -> None:
        """``render_device`` that also writes the visibility planes, each laid out like the colour output in device
        memory: per pixel the scene index of the winning triangle (uint32; a triangle the near-plane clip appended
        reports its parent; background 0xFFFFFFFF) and its interpolated 1/z (float32; background +0).  A pointer of 0
        leaves that output out; with ``colour_ptr`` = 0 nothing is shaded.  At least one pointer must be set."""
        cams = np.ascontiguousarray(cameras, "<f4").reshape(-1, 12)
        y1 = height if y1 is None else y1
        self._check(self._lib.s3r_render_device_visibility(self._h, cams.ctypes.data, cams.shape[0], width, height, y0, y1,
                                                            ctypes.c_void_p(colour_ptr), ctypes.c_void_p(triangle_ptr),
                                                            ctypes.c_void_p(depth_ptr), ctypes.c_void_p(stream)))

    def render_device_rows(self, cameras, width: int, height: int, row_stride: int, row_phase: int, dev_ptr: int,
                           stream: int = 0) -> None:
        """Interleaved tile rows (``a % row_stride == row_phase``), compacted output; see ``rows_layout``."""
        cams = np.ascontiguousarray(cameras, "<f4").reshape(-1, 12)
        self._check(self._lib.s3r_render_device_rows(self._h, cams.ctypes.data, cams.shape[0], width, height, row_stride,
                                                      row_phase, ctypes.c_void_p(dev_ptr), ctypes.c_void_p(stream)))

    # ---- fused frame assembly over peer memory (include/s3r_b200.h) ------------------------------
    def peer_frame_alloc(self, nbytes: int):
        """(device pointer, 64-byte IPC handle) of a new allocation on this renderer's GPU."""
        ptr, handle = ctypes.c_void_p(), ctypes.create_string_buffer(64)
        self._check(self._lib.s3r_peer_frame_alloc(self._h, nbytes, ctypes.byref(ptr), handle))
        return int(ptr.value), handle.raw

    def peer_frame_open(self, handle: bytes) -> int:
        ptr = ctypes.c_void_p()
        self._check(self._lib.s3r_peer_frame_open(self._h, handle, ctypes.byref(ptr)))
        return int(ptr.value)

    def peer_frame_release(self, ptr: int) -> None:
        self._check(self._lib.s3r_peer_frame_release(self._h, ctypes.c_void_p(ptr)))

    def set_peer_frames(self, ptrs) -> None:
        """Destinations of the following render_device(_rows) calls ([] = back to the call's own output)."""
        arr = (ctypes.c_void_p * max(len(ptrs), 1))(*[ctypes.c_void_p(p) for p in ptrs])
        self._check(self._lib.s3r_set_peer_frames(self._h, arr, len(ptrs)))

    def read_device(self, ptr: int, shape, dtype=np.uint32) -> np.ndarray:
        out = np.empty(shape, dtype)
        self._check(self._lib.s3r_copy_from_device(self._h, out.ctypes.data, ctypes.c_void_p(ptr), out.nbytes))
        return out

    def finish(self) -> bool:
        """Waits for enqueued work; True means a capacity overflowed and the last call must be repeated."""
        return self._check(self._lib.s3r_finish(self._h)) == 1

    # ---- introspection ------------------------------------------------------------------------
    def stats(self, view: int = 0) -> dict:
        st = CStats()
        self._check(self._lib.s3r_get_stats(self._h, view, ctypes.byref(st)))
        return {n: int(getattr(st, n)) for n, _ in CStats._fields_ if n != "reserved"}

    def raster_vertices(self, view: int = 0) -> np.ndarray:
        n = ctypes.c_uint64()
        self._check(self._lib.s3r_scene_counts(self._h, ctypes.byref(n), None, None, None))
        out = np.empty((n.value, 4), np.float32)
        self._check(self._lib.s3r_dump_raster_vertices(self._h, view, out.ctypes.data, n.value))
        return out[:, :3]

    def setups(self, view: int = 0) -> np.ndarray:
        n = ctypes.c_uint64()
        self._check(self._lib.s3r_dump_setups(self._h, view, None, 0, ctypes.byref(n)))
        out = np.zeros(n.value, SETUP_DTYPE)
        if n.value:
            self._check(self._lib.s3r_dump_setups(self._h, view, out.ctypes.data, n.value, ctypes.byref(n)))
        return out

    def debug_walk(self, start, delta, steps) -> np.ndarray:
        s = np.ascontiguousarray(start, "<f4"); d = np.ascontiguousarray(delta, "<f4"); n = np.ascontiguousarray(steps, "<u4")
        out = np.empty_like(s)
        self._check(self._lib.s3r_debug_walk(self._h, s.ctypes.data, d.ctypes.data, n.ctypes.data, out.ctypes.data, s.size))
        return out

    def timing(self, reset: bool = True) -> dict:
        g, q, n = ctypes.c_double(), ctypes.c_double(), ctypes.c_uint64()
        self._check(self._lib.s3r_get_timing(self._h, ctypes.byref(g), ctypes.byref(q), ctypes.byref(n), int(reset)))
        return {"geometry_ms": g.value, "raster_ms": q.value, "chunks": n.value}

    def kernel_timing(self) -> dict:
        """{kernel name: {"ms": summed CUDA-event time, "launches": n}} since the last ``timing(reset=True)``."""
        out, i = {}, 0
        while True:
            name, ms, n = ctypes.c_char_p(), ctypes.c_double(), ctypes.c_uint64()
            if self._check(self._lib.s3r_get_kernel_timing(self._h, i, ctypes.byref(name), ctypes.byref(ms), ctypes.byref(n))) != 0:
                return out
            out[name.value.decode()] = {"ms": ms.value, "launches": int(n.value)}
            i += 1

    @property
    def kernel_launches(self) -> int:
        return int(self._lib.s3r_kernel_launches(self._h))


class Sink:
    """Frame sink (``s3r_sink_*``): device-resident frames -> raw BGR0 (``fmt=0``) or YUV4MPEG2 4:2:0 (``fmt=1``) file."""

    def __init__(self, renderer: "Renderer", path: str, width: int, height: int, fps=(60, 1), fmt: int = 1):
        self._r, self._h = renderer, ctypes.c_void_p()
        renderer._check(renderer._lib.s3r_sink_open(renderer._h, path.encode(), width, height, fps[0], fps[1], fmt, ctypes.byref(self._h)))

    def submit(self, dev_ptr: int, stream: int = 0) -> None:
        self._r._check(self._r._lib.s3r_sink_submit(self._h, ctypes.c_void_p(dev_ptr), ctypes.c_void_p(stream)))

    def close(self) -> int:
        n = ctypes.c_uint64()
        h, self._h = self._h, ctypes.c_void_p()
        self._r._check(self._r._lib.s3r_sink_close(h, ctypes.byref(n)))
        return int(n.value)


class DropIn:
    """The reference's calling pattern: dlopen a private ``render.so`` that finds ``data.bin`` beside
    itself, then ``updateAndRender(&pixelData, &input)`` once per frame (main.swift:95-99,121).

    ``devices``: None = one GPU (``S3R_DEVICE`` or 0); "all" or "0,1,2,3" = the in-process multi-GPU drop-in
    (``S3R_DEVICES``; the library reads its environment at the first call)."""

    def __init__(self, data_bin_path: str, so_path: Optional[str] = None, devices: Optional[str] = None, env: Optional[dict] = None):
        so_path = so_path or LIB_PATH
        if not os.path.exists(so_path):
            raise RendererError(f"{so_path} not found (no CPU fallback)")
        self._dir = tempfile.mkdtemp(prefix="s3r_dropin_")
        self.so = os.path.join(self._dir, "render.so")
        shutil.copy(so_path, self.so)
        dst = os.path.join(self._dir, "data.bin")
        try:
            os.symlink(os.path.abspath(data_bin_path), dst)
        except OSError:
            shutil.copy(data_bin_path, dst)
        self._lib = ctypes.CDLL(self.so)
        self._fn = self._lib.updateAndRender
        self._fn.argtypes = [ctypes.POINTER(PixelData), ctypes.POINTER(Input)]
        self._fn.restype = None
        self._first_env = dict(env or {})
        if devices is not None:
            self._first_env["S3R_DEVICES"] = devices

    def update_and_render(self, width: int, height: int, rec, out: Optional[np.ndarray] = None) -> np.ndarray:
        if out is None:
            out = np.empty((height, width), np.uint32)
        pd = PixelData(out.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32)), width, height, 4, 4 * width * height)
        inp = make_input(rec)
        if self._first_env is not None:   # the library initialises itself inside its first call: give it its environment
            saved = {k: os.environ.get(k) for k in self._first_env}
            os.environ.update(self._first_env)
            try:
                self._fn(ctypes.byref(pd), ctypes.byref(inp))
            finally:
                for k, v in saved.items():
                    if v is None:
                        os.environ.pop(k, None)
                    else:
                        os.environ[k] = v
            self._first_env = None
            return out
        self._fn(ctypes.byref(pd), ctypes.byref(inp))
        return out

    @property
    def n_devices(self) -> int:
        return int(self._lib.s3r_dropin_devices())

    def reset_camera(self) -> None:
        self._lib.s3r_dropin_reset()

    def close(self) -> None:
        """Releases the library's registrations of caller memory (the library itself stays loaded, like the reference)."""
        try:
            self._lib.s3r_dropin_release_pins()
        except AttributeError:
            pass
        shutil.rmtree(self._dir, ignore_errors=True)
