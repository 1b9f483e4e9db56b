"""oracle/port.py — TEST INFRASTRUCTURE.  ctypes binding of oracle/_build/liboracle.so (the C
restatement in oracle/render_oracle.c).  Only tests/, __graft_entry__.smoke() and bench.py's CPU
baseline legs may import this module."""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "_build", "liboracle.so")


class CScene(ctypes.Structure):
    _fields_ = [
        ("vertex_count", ctypes.c_uint64), ("index_count", ctypes.c_uint64),
        ("attribute_count", ctypes.c_uint64), ("texel_count", ctypes.c_uint64),
        ("vertices", ctypes.c_void_p), ("vertex_indices", ctypes.c_void_p), ("attributes", ctypes.c_void_p),
        ("attribute_indices", ctypes.c_void_p), ("texels", ctypes.c_void_p), ("owned", ctypes.c_void_p),
    ]


class CInput(ctypes.Structure):
    _fields_ = [(n, ctypes.c_float) for n in ("up", "down", "left", "right", "mouse_x", "mouse_y")]


class CCamera(ctypes.Structure):
    _fields_ = [
        ("position", ctypes.c_float * 3), ("axis_x", ctypes.c_float * 3), ("axis_y", ctypes.c_float * 3),
        ("axis_z", ctypes.c_float * 3), ("matrix", ctypes.c_float * 12), ("mouse", ctypes.c_float * 2),
        ("started", ctypes.c_int),
    ]


SETUP_DTYPE = np.dtype([
    ("order", "<u4"), ("xmin", "<u4"), ("xmax", "<u4"), ("ymin", "<u4"), ("ymax", "<u4"), ("area", "<f4"),
    ("wstart", "<f4", (3,)), ("dx", "<f4", (3,)), ("dy", "<f4", (3,)), ("rvz", "<f4", (3,)),
    ("cv", "<f4", (3, 3)), ("n", "<f4", (3, 3)), ("kind", "<u4"), ("texture", "<u4"),
    ("payload", "<f4", (3, 3)), ("dz", "<f4", (2,)), ("tpp", "<f4", (2,)),
])

STATS_FIELDS = ("triangles_in", "near_rejected", "clipped", "spawned", "offscreen", "small_or_backfacing",
                "rasterized", "bbox_pixels", "covered_pixels", "shaded_pixels")


class CStats(ctypes.Structure):
    _fields_ = [(n, ctypes.c_uint64) for n in STATS_FIELDS] + [("scratch_overflow", ctypes.c_int)]


def build(force: bool = False) -> str:
    src = os.path.join(HERE, "render_oracle.c")
    if force or not os.path.exists(LIB) or os.path.getmtime(LIB) < os.path.getmtime(src):
        subprocess.check_call(["make", "-s", "-C", HERE, "port"])
    return LIB


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = ctypes.CDLL(build())
        _lib.oracle_scene_load.argtypes = [ctypes.POINTER(CScene), ctypes.c_char_p]
        _lib.oracle_scene_load.restype = ctypes.c_int
        _lib.oracle_scene_free.argtypes = [ctypes.POINTER(CScene)]
        _lib.oracle_camera_reset.argtypes = [ctypes.POINTER(CCamera)]
        _lib.oracle_camera_update.argtypes = [ctypes.POINTER(CCamera), ctypes.POINTER(CInput)]
        _lib.oracle_factor.argtypes = [ctypes.c_uint32]
        _lib.oracle_factor.restype = ctypes.c_float
        _lib.oracle_render.argtypes = [
            ctypes.POINTER(CScene), ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_void_p,
            ctypes.c_void_p, ctypes.POINTER(CStats), ctypes.c_void_p, ctypes.c_size_t,
            ctypes.POINTER(ctypes.c_size_t), ctypes.c_void_p]
        _lib.oracle_render.restype = ctypes.c_int
        _lib.oracle_vertex_stage.argtypes = [ctypes.POINTER(CScene), ctypes.c_void_p, ctypes.c_uint32,
                                             ctypes.c_uint32, ctypes.c_void_p, ctypes.c_void_p]
        _lib.oracle_walk.argtypes = [ctypes.c_float, ctypes.c_float, ctypes.c_uint32]
        _lib.oracle_walk.restype = ctypes.c_float
        assert ctypes.sizeof(CInput) == 24
    return _lib


class Camera:
    """Re-entrant camera with the reference's update semantics (render-cpp/render.cpp:134-156)."""

    def __init__(self):
        self.c = CCamera()
        lib().oracle_camera_reset(ctypes.byref(self.c))

    def update(self, rec) -> np.ndarray:
        i = CInput(float(rec["up"]), float(rec["down"]), float(rec["left"]), float(rec["right"]),
                   float(rec["mouse"][0]), float(rec["mouse"][1]))
        lib().oracle_camera_update(ctypes.byref(self.c), ctypes.byref(i))
        return self.matrix

    @property
    def matrix(self) -> np.ndarray:
        return np.array(self.c.matrix[:], dtype=np.float32)


def camera_path(inputs) -> np.ndarray:
    """Matrices (n, 12) after each Input record, starting from the reference's initial state."""
    cam = Camera()
    return np.stack([cam.update(r) for r in inputs])


class OracleScene:
    def __init__(self, scene=None, path: str | None = None):
        self.c = CScene()
        self._keep = None
        if path is not None:
            rc = lib().oracle_scene_load(ctypes.byref(self.c), path.encode())
            if rc:
                raise OSError(f"oracle_scene_load({path}) -> {rc}")
        else:
            v = np.ascontiguousarray(scene.vertices, "<f4")
            vi = np.ascontiguousarray(scene.vertex_indices, "<u8")
            at = np.ascontiguousarray(scene.attributes)
            ai = np.ascontiguousarray(scene.attribute_indices, "<u8")
            tx = np.ascontiguousarray(scene.textures, "<u4")
            self._keep = (v, vi, at, ai, tx)
            self.c.vertex_count, self.c.index_count = v.shape[0], vi.shape[0]
            self.c.attribute_count, self.c.texel_count = at.shape[0], tx.size
            self.c.vertices, self.c.vertex_indices = v.ctypes.data, vi.ctypes.data
            self.c.attributes, self.c.attribute_indices, self.c.texels = at.ctypes.data, ai.ctypes.data, tx.ctypes.data

    def render(self, matrix, width: int, height: int, want_depth=False, want_setups=False, setup_cap=None,
               want_winner=False):
        """want_winner: also return "winner", per pixel the order key of the triangle that wrote it last (its own index,
        or T + parent for a triangle appended by the clipper), 0xFFFFFFFF on background."""
        m = np.ascontiguousarray(matrix, "<f4")
        px = np.empty((height, width), np.uint32)
        depth = np.empty((height, width), np.float32) if want_depth else None
        winner = np.empty((height, width), np.uint32) if want_winner else None
        st = CStats()
        setups = None
        n = ctypes.c_size_t(0)
        if want_setups:
            cap = setup_cap or 2 * int(self.c.index_count // 3) + 8
            setups = np.zeros(cap, SETUP_DTYPE)
        lib().oracle_render(ctypes.byref(self.c), m.ctypes.data, width, height, px.ctypes.data,
                            depth.ctypes.data if want_depth else None, ctypes.byref(st),
                            setups.ctypes.data if want_setups else None, len(setups) if want_setups else 0,
                            ctypes.byref(n), winner.ctypes.data if want_winner else None)
        stats = {k: int(getattr(st, k)) for k in STATS_FIELDS}
        stats["scratch_overflow"] = int(st.scratch_overflow)
        out = {"pixels": px, "stats": stats}
        if want_depth:
            out["depth"] = depth
        if want_setups:
            out["setups"] = setups[: min(n.value, len(setups))]
        if want_winner:
            out["winner"] = winner
        return out

    def vertex_stage(self, matrix, width: int, height: int):
        m = np.ascontiguousarray(matrix, "<f4")
        V = int(self.c.vertex_count)
        cv = np.empty((V, 3), np.float32)
        rv = np.empty((V, 3), np.float32)
        lib().oracle_vertex_stage(ctypes.byref(self.c), m.ctypes.data, width, height, cv.ctypes.data, rv.ctypes.data)
        return cv, rv


def walk(start: float, delta: float, n: int) -> float:
    return float(lib().oracle_walk(start, delta, n))
