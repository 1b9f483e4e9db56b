"""Seeded random parity sweep: random triangle soups, views, frame sizes and option / entry-point combinations against
the oracle, bit for bit, case by case on fresh renderers and through long-lived ones.

Every other parity test renders a scene someone built for one purpose, under one axis of options.  Here every case is
a pure function of (seed, index): a shuffled soup mixing raster-space triangles of every box size, near-plane
straddlers (corners exactly on z = -0.1 and z = 0), exact duplicates and coplanar copies, fans, slivers, degenerate and
far-reaching triangles, crowds of tiny ones and randomly shared vertices, with per-corner attribute records; a pool of
views (the still camera, scripted paths, random rotations with roll, scaled and sheared matrices); a frame size biased
to the edges; and a plan of calls, each with the options it changes first.  Every call is compared with the oracle:
colour (or its box resolve for supersampling), triangle and depth planes, statistics of every view, setup records and
raster-space vertices, and the guard words behind every device output.  The long-lived sequences keep one renderer
through hundreds of random steps (calls, frame sizes, scene updates, reloads) without ever resetting its options.

The default run covers DEFAULT_CASES cases of DEFAULT_SEED and N_SEQUENCES sequences of SEQUENCE_STEPS steps.  A longer
or different run: S3R_SWEEP_SEED=<seed> S3R_SWEEP_CASES=<count> python -m pytest -m gpu tests/test_gpu_random_sweep.py.
One case alone: python -m pytest tests/test_gpu_random_sweep.py -k case_0137 (with the seed variable of its run).

The CPU tests keep the sweep honest: the generator is deterministic and stays inside the parity contract (DESIGN.md
§8), the default cases reach the paths and boundaries they exist for (from the oracle alone), every plan feature
occurs, and exact comparison has teeth on most cases (one ulp of one matrix entry changes a pixel or a winner)."""
import functools
import os

import numpy as np
import pytest

from swift3drenderer_b200 import scene as S
from test_gpu_shading_attributes import hash_atlases
from test_gpu_supersample import resolve
from test_gpu_vis_edges import KSCALE, NO_WINNER, assert_stats, block_winners, box_sizes
from test_gpu_visibility_planes import GUARD, PAD, device_planes, expected

DEFAULT_SEED = 20261022
DEFAULT_CASES = 48
SEED = int(os.environ.get("S3R_SWEEP_SEED", DEFAULT_SEED))
N_CASES = int(os.environ.get("S3R_SWEEP_CASES", DEFAULT_CASES))
N_SEQUENCES = 3
SEQUENCE_STEPS = 200
S3R_E_ARG = -4
SMALL_T = 1920                 # 2T <= 3840: the small-scene (fused) path
BIG_CASES = (11, 35)           # the only cases whose frames go up to 3840 x 2160
BOUNDARY_T = {1: 1920, 4: 1921}
MAX_PIXELS = 6 << 20           # views x (k W) x (k H) of one call
REPEATS = 6                    # finish() must stop asking for a repeat within this many submissions
EDGE_SIZES = (1, 2, 3, 15, 16, 17, 31, 32, 33, 63, 64, 65, 127, 128, 129)
DEFAULTS = {"clusters": 2, "cluster_cull": 1, "direct_small": 1, "flat_max": 128, "fused_small": 1, "spans": 1,
            "rowtab_capacity": -1, "tma_store": 1, "tensor_store": 1, "timing": 0, "pack24": 1, "host_bands": 12,
            "copy_threads": 0, "pin_host": 0, "views_per_chunk": 256}
ENTRIES = ("host", "device", "rows", "visibility", "ssaa_host", "ssaa_device", "peer", "refused")
REFUSALS = ("ssaa_peer", "visibility_peer", "ssaa_k3", "visibility_none")


def _option_value(rng, name):
    if name == "clusters":
        return int(rng.integers(0, 3))
    if name == "flat_max":
        return int(rng.choice([16, 128, 65536, int(rng.integers(17, 4097))]))
    if name == "rowtab_capacity":
        return int(rng.choice([-1, 0, int(rng.integers(1, 512))]))
    if name == "timing":
        return int(rng.choice([0, 1, 3]))
    if name == "host_bands":
        return int(rng.choice([1, 2, 3, 5, 12]))
    if name == "copy_threads":
        return int(rng.choice([0, 1, 3]))
    if name == "views_per_chunk":
        return int(rng.integers(1, 9))
    return int(rng.integers(0, 2))


# ------------------------------------------------------------------------------------------------------------------
# scenes
# ------------------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _procedural():
    return S.procedural_textures(2)


def _atlases(which):
    return hash_atlases() if which == "hash" else _procedural()


def _to_world(px, py, d, W, H):
    """Raster corners (px, py) at distance d of a W x H frame seen by the still camera -> world points."""
    factor = 0.1 * H / (2 * KSCALE)
    return np.stack([(px - W / 2) * d / factor, -(py - H / 2) * d / factor, -d], -1)


class _Soup:
    """Vertices (float64, rounded to float32 at the end) and triangles (vertex indices) of one scene, family by family;
    ``exact`` lists (original, copy) pairs with identical corners in identical order."""

    def __init__(self, rng, W, H):
        self.rng, self.W, self.H = rng, W, H
        self.v, self.t, self.nv = [], [], 0
        self.exact, self.flat = [], []        # flat: triangles at one constant depth (for coplanar copies)

    @property
    def n(self):
        return sum(len(t) for t in self.t)

    def add(self, verts, tris=None, flat=False):
        verts = np.asarray(verts, np.float64).reshape(-1, 3)
        tris = np.arange(len(verts)).reshape(-1, 3) if tris is None else np.asarray(tris).reshape(-1, 3)
        first = self.n
        self.v.append(verts)
        self.t.append(tris + self.nv)
        self.nv += len(verts)
        if flat:
            self.flat.extend(range(first, first + len(tris)))
        return first

    def raster(self, n, crowd=False):
        rng, W, H = self.rng, self.W, self.H
        if crowd:   # tiny triangles (twice the area just above the cull) packed into one 64 x 32 region
            x0, y0 = rng.uniform(0, max(W - 64, 1)), rng.uniform(0, max(H - 32, 1))
            c = np.stack([x0 + rng.uniform(0, 64, n), y0 + rng.uniform(0, 32, n)], -1)
            length, th = rng.uniform(4, 16, n), rng.uniform(0, np.pi, n)
            u = np.stack([np.cos(th), np.sin(th)], -1)
            wid = rng.uniform(10.5, 16, n) / length
            p = np.stack([c - u * length[:, None] / 2, c + u * length[:, None] / 2,
                          c + np.stack([-u[:, 1], u[:, 0]], -1) * wid[:, None]], 1)
            d = np.repeat(rng.uniform(0.1005, 0.11, n)[:, None], 3, 1) + rng.uniform(0, 0.001, (n, 3))   # in front of the rest
        else:       # box sizes log-uniform from sub-pixel to several frame widths
            c = np.stack([rng.uniform(-0.25, 1.25, n) * W, rng.uniform(-0.25, 1.25, n) * H], -1)
            size = np.exp(rng.uniform(np.log(0.3), np.log(4 * max(W, H) + 2), n))
            aspect = np.exp(rng.uniform(-1.5, 1.5, n))
            off = rng.uniform(-1, 1, (n, 3, 2)) * size[:, None, None]
            off[:, :, 0] *= aspect[:, None]
            p = c[:, None, :] + off
            d0 = np.exp(rng.uniform(np.log(0.2), np.log(300), n))
            slant = rng.random(n) < 0.5
            d = d0[:, None] * np.where(slant[:, None], np.exp(rng.uniform(-0.3, 0.3, (n, 3))), 1.0)
        # most triangles wound so that the reference's area is positive (the rest are back faces)
        area = (p[:, 2, 0] - p[:, 0, 0]) * (p[:, 0, 1] - p[:, 1, 1]) + (p[:, 2, 1] - p[:, 0, 1]) * (p[:, 1, 0] - p[:, 0, 0])
        flip = (area < 0) & (rng.random(n) < 0.85)
        p[flip] = p[flip][:, [0, 2, 1]]
        d[flip] = d[flip][:, [0, 2, 1]]
        first = self.add(_to_world(p[..., 0], p[..., 1], d, W, H))
        if not crowd:
            self.flat.extend(first + np.nonzero(~slant)[0])

    def near(self, n):
        """Triangles around the near plane of the still camera: 0 to 3 corners behind it, some corners exactly on
        z = -0.1 (on the plane is behind) or z = 0 (the eye plane)."""
        rng = self.rng
        behind = rng.integers(0, 4, n)
        z = np.where(np.arange(3)[None, :] < behind[:, None], rng.uniform(-0.1, 1.5, (n, 3)), -rng.uniform(0.1001, 4, (n, 3)))
        special = rng.random((n, 3))
        z = np.where((special < 0.12) & (z > -0.1), -0.1, z)
        z = np.where((special > 0.94) & (z > -0.1), 0.0, z)
        for k in range(n):
            rng.shuffle(z[k])
        xy = rng.uniform(-1, 1, (n, 3, 2)) * (np.abs(z)[..., None] + 0.3) * 0.35 + rng.uniform(-0.2, 0.2, (n, 1, 2))
        self.add(np.concatenate([xy, z[..., None]], -1))

    def far(self, n):
        rng = self.rng
        v = np.zeros((n, 3, 3))
        v[:, 0] = np.stack([rng.uniform(-5, 5, n), rng.uniform(-5, 5, n), -rng.uniform(2, 20, n)], -1)
        for k in (1, 2):
            v[:, k, :2] = rng.choice([-1, 1], (n, 2)) * rng.uniform(1000, 8000, (n, 2))
            v[:, k, 2] = -rng.uniform(1, 9000, n)
        self.add(v)

    def fan(self, n):
        rng, W, H = self.rng, self.W, self.H
        while n > 0:
            m = int(min(n, rng.integers(3, 9)))
            cx, cy = rng.uniform(0, W), rng.uniform(0, H)
            r = np.exp(rng.uniform(np.log(2), np.log(max(W, H) + 3)))
            ang = np.sort(rng.uniform(0, 2 * np.pi, m))
            px = np.concatenate([[cx], cx + r * np.cos(ang)])
            py = np.concatenate([[cy], cy + r * np.sin(ang)])
            d = rng.uniform(1, 50) * (1 + rng.uniform(0, 0.2, m + 1) * (rng.random() < 0.5))
            k = np.arange(m)
            self.add(_to_world(px, py, d, W, H), np.stack([np.zeros(m, int), 1 + (k + 1) % m, 1 + k], -1))
            n -= m

    def odd(self, n):
        """Slivers, triangles with two equal corners (by index or by value), back faces."""
        rng, W, H = self.rng, self.W, self.H
        for _ in range(n):
            a = np.array([rng.uniform(0, W), rng.uniform(0, H)])
            b = a + rng.uniform(-1, 1, 2) * rng.uniform(2, max(W, H) + 2)
            d = rng.uniform(0.5, 60)
            kind = rng.integers(0, 3)
            if kind == 0:    # sliver: the third corner a hair off the line a -> b
                c = a + (b - a) * rng.uniform(0.1, 0.9) + rng.uniform(-0.05, 0.05, 2)
                p = np.stack([a, b, c])
                self.add(_to_world(p[:, 0], p[:, 1], np.full(3, d), W, H))
            elif kind == 1:  # two corners the same vertex
                p = np.stack([a, b])
                self.add(_to_world(p[:, 0], p[:, 1], np.full(2, d), W, H), [[0, 0, 1]] if rng.random() < 0.5 else [[0, 1, 1]])
            else:            # two corners equal by value
                p = np.stack([a, b, b])
                self.add(_to_world(p[:, 0], p[:, 1], np.full(3, d), W, H))

    def copies(self, n):
        """Exact copies (same vertices, or new vertices with the same values, same corner order), copies with rotated
        corners, and coplanar triangles at the depth of a flat one."""
        rng, W, H = self.rng, self.W, self.H
        verts = np.concatenate(self.v)
        tris = np.concatenate(self.t)
        for _ in range(n):
            kind = rng.integers(0, 4)
            if kind == 3 and self.flat:
                src = self.flat[rng.integers(0, len(self.flat))]
                d = -verts[tris[src, 0], 2]
                c = np.array([rng.uniform(0, W), rng.uniform(0, H)])
                s = np.exp(rng.uniform(np.log(3), np.log(max(W, H) + 3)))
                p = c + rng.uniform(-1, 1, (3, 2)) * s
                area = (p[2, 0] - p[0, 0]) * (p[0, 1] - p[1, 1]) + (p[2, 1] - p[0, 1]) * (p[1, 0] - p[0, 0])
                if area < 0:
                    p = p[[0, 2, 1]]
                w = _to_world(p[:, 0], p[:, 1], np.full(3, d), W, H)
                w[:, 2] = verts[tris[src, 0], 2]
                self.add(w)
                continue
            src = int(rng.integers(0, len(tris)))
            if kind == 0:
                self.t.append(tris[src][None].copy())
                self.exact.append((src, self.n - 1))
            elif kind == 1:
                self.exact.append((src, self.add(verts[tris[src]])))
            else:
                self.add(verts[tris[src][list([(1, 2, 0), (2, 0, 1)][rng.integers(0, 2)])]])

    def scene_arrays(self, share):
        verts = np.concatenate(self.v).astype(np.float32)
        tris = np.concatenate(self.t).astype(np.int64)
        pinned = {b for _, b in self.exact} | {a for a, _ in self.exact}
        pick = np.nonzero(self.rng.random(len(tris)) < share)[0]
        for t in pick:   # index reuse across distant triangles: some clusters get huge bounds
            if t not in pinned:
                tris[t, self.rng.integers(0, 3)] = self.rng.integers(0, len(verts))
        return verts, tris


def _attributes(rng, T, n_tex, p_tex):
    """Per-corner records: corner 0 decides the kind; a textured corner 0 has texture records at every corner, a
    colour corner 0 may have texture records at the others (their words are lerped as colour, DESIGN.md §8)."""
    at = np.zeros((T, 3), S.ATTR_DTYPE)
    tex0 = rng.random(T) < p_tex
    kind = np.zeros((T, 3), bool)
    kind[:, 0] = tex0
    kind[:, 1:] = tex0[:, None] | (rng.random((T, 2)) < 0.15)
    direction = rng.normal(size=(T, 3, 3))
    direction /= np.linalg.norm(direction, axis=-1, keepdims=True)
    e = rng.uniform(-30, 30, (T, 1)) + np.where(rng.random((T, 1)) < 0.5, rng.uniform(-3, 3, (T, 3)), 0)
    at["normal"][..., :3] = (direction * np.exp2(np.clip(e, -30, 30))[..., None]).astype("<f4")
    rgb = rng.uniform(0, 255, (T, 3, 3)).astype("<f4")
    at["payload"][..., :3] = np.where(kind[..., None], 0, rgb.view("<u4"))
    mode = rng.integers(0, 3, T)
    uv = np.where(mode[:, None, None] == 0, rng.uniform(0, 1, (T, 1, 2)),
                  np.where(mode[:, None, None] == 1, rng.uniform(0, 1, (T, 3, 2)), rng.uniform(0, 255, (T, 3, 2))))
    tex_index = rng.integers(0, n_tex, (T, 3)).astype("<u4")
    at["payload"][..., 0] = np.where(kind, tex_index, at["payload"][..., 0])
    at["payload"][..., 1] = np.where(kind, 0, at["payload"][..., 1])
    at["payload"][..., 2:4] = np.where(kind[..., None], uv.astype("<f4").view("<u4"), at["payload"][..., 2:4])
    at["kind"] = kind
    return at.reshape(-1)


def make_scene(rng, T, W, H):
    """(scene, meta) of T triangles: meta["exact"] = (earlier, later) triangle pairs with identical corners,
    meta["textures"] = the atlas set's name."""
    soup = _Soup(rng, W, H)
    crowd = T >= 300 and W >= 64 and H >= 32 and rng.random() < 0.6
    p = np.array([0.50, 0.05, 0.12, 0.07, 0.07, 0.02, 0.15 if crowd else 0.0])
    n = rng.multinomial(T, p / p.sum())
    n_raster = max(int(n[0]), 1)
    soup.raster(n_raster)
    if n[6]:
        soup.raster(int(n[6]), crowd=True)
    if n[1]:
        soup.near(int(n[1]))
    if n[5]:
        soup.far(int(n[5]))
    if n[3]:
        soup.fan(int(n[3]))
    if n[4]:
        soup.odd(int(n[4]))
    soup.copies(max(T - soup.n, 0))
    verts, tris = soup.scene_arrays(share=0.03)
    tris = tris[:T]
    exact = [(a, b) for a, b in soup.exact if b < T]
    # shuffle: load-time clusters become ragged runs of unrelated triangles
    perm = rng.permutation(T)
    inv = np.empty(T, np.int64)
    inv[perm] = np.arange(T)
    tris = tris[perm]
    exact = sorted((min(inv[a], inv[b]), max(inv[a], inv[b])) for a, b in exact)
    textures = "hash" if rng.random() < 0.5 else "procedural"
    tx = _atlases(textures)
    at = _attributes(rng, T, tx.shape[0], rng.uniform(0.1, 0.9))
    v = np.ones((len(verts), 4), "<f4")
    v[:, :3] = verts
    sc = S.Scene(v, tris.reshape(-1).astype("<u8"), at, np.arange(3 * T, dtype="<u8"), tx)
    return sc, {"exact": [(int(a), int(b)) for a, b in exact], "textures": textures}


# ------------------------------------------------------------------------------------------------------------------
# views and frame sizes
# ------------------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _path(name, frames):
    from oracle import port
    return port.camera_path(S.input_script(name, frames))


def _rotation(rng):
    q = rng.normal(size=4)
    a, b, c, d = q / np.linalg.norm(q)
    return np.array([[a * a + b * b - c * c - d * d, 2 * (b * c - a * d), 2 * (b * d + a * c)],
                     [2 * (b * c + a * d), a * a - b * b + c * c - d * d, 2 * (c * d - a * b)],
                     [2 * (b * d - a * c), 2 * (c * d + a * b), a * a - b * b - c * c + d * d]])


def _matrix(R, c):
    return np.concatenate([R, -(R @ c)[:, None]], 1).astype(np.float32).reshape(12)


def make_views(rng, sc, n):
    """n views: the still camera, scripted-path poses, random rotations (roll included) from inside the soup's box or
    looking at it from outside, and scaled / sheared matrices."""
    xyz = sc.vertices[:, :3].astype(np.float64)
    lo, hi = np.percentile(xyz, 5, axis=0), np.percentile(xyz, 95, axis=0)
    centre, radius = (lo + hi) / 2, max(np.linalg.norm(hi - lo) / 2, 1.0)
    views, kinds = [], []
    for k in range(n):
        kind = "still" if k == 0 else str(rng.choice(["path", "inside", "outside", "nonrigid", "still"], p=[0.3, 0.2, 0.25, 0.2, 0.05]))
        if kind == "still":
            m = _path("still", 1)[0].copy()
        elif kind == "path":
            name = str(rng.choice(["spin", "flythrough", "strafe"]))
            frames = 600 if name == "flythrough" else 64
            m = _path(name, frames)[int(rng.integers(0, frames))].copy()
        elif kind == "inside":
            m = _matrix(_rotation(rng), rng.uniform(lo, hi))
        else:
            d = rng.normal(size=3)
            c = centre + d / np.linalg.norm(d) * radius * rng.uniform(1.2, 3)
            z = (c - centre) / np.linalg.norm(c - centre)
            x = np.cross(rng.normal(size=3), z)
            x /= np.linalg.norm(x)
            R = np.stack([x, np.cross(z, x), z])
            if kind == "nonrigid":
                shear = np.eye(3) + np.where(rng.random((3, 3)) < 0.5, rng.uniform(-0.5, 0.5, (3, 3)), 0) * (1 - np.eye(3))
                R = np.diag(rng.uniform(0.3, 3, 3)) @ shear @ R
            m = _matrix(R, c)
        views.append(m)
        kinds.append(kind)
    return np.stack(views), kinds


def make_size(rng, index=None):
    if index in BIG_CASES:
        return (3840, 2160) if index == BIG_CASES[0] else (int(rng.integers(1921, 3841)), int(rng.integers(1081, 2161)))
    u = rng.random()
    if u < 0.08:
        return (1, int(rng.integers(300, 701))) if rng.random() < 0.5 else (int(rng.integers(300, 701)), 1)

    def one():
        return int(rng.choice(EDGE_SIZES)) if rng.random() < 0.45 else int(2 * rng.integers(0, 700) + 1)
    return one(), one()


# ------------------------------------------------------------------------------------------------------------------
# plans
# ------------------------------------------------------------------------------------------------------------------
def _band(rng, H):
    kind = rng.integers(0, 3)
    if kind == 0:                       # one row
        y0 = int(rng.integers(0, H))
        return y0, y0 + 1
    if kind == 1:                       # starts inside a tile row and a 4-row key column
        y0 = int(rng.integers(0, H))
        y0 -= 0 if y0 % 16 else min(y0, 1)
        return y0, int(rng.integers(y0 + 1, H + 1))
    a, b = sorted(rng.choice(H + 1, 2, replace=False))
    return int(a), int(b)


def make_call(rng, state, T, W, H, n_views, first=False):
    """One call of the plan vocabulary.  ``state`` (the options as earlier calls left them) is updated with the
    options this call sets first."""
    opts = {}
    for name in DEFAULTS:
        if rng.random() < (0.5 if first else 0.2):
            opts[name] = _option_value(rng, name)
    if rng.random() < 0.08:
        opts["setup_capacity"] = int(rng.integers(1, 65))   # tiny: forces overflow and regrowth (not sticky)
    state.update({k: v for k, v in opts.items() if k in DEFAULTS})
    general = T > SMALL_T or state["fused_small"] == 0
    weights = {"host": 0.2, "device": 0.2, "rows": 0.1, "visibility": 0.16, "ssaa_host": 0.08, "ssaa_device": 0.1,
               "peer": 0.1 if general else 0.0, "refused": 0.08}
    names = list(weights)
    p = np.array([weights[k] for k in names])
    call = {"entry": str(rng.choice(names, p=p / p.sum())), "opts": opts}
    entry = call["entry"]
    k = 1
    if entry.startswith("ssaa"):
        k = int(rng.choice([2, 4]))
        if k * k * W * H > MAX_PIXELS or 4 * max(W, H) > 65535:
            k = 2
        if k * k * W * H > MAX_PIXELS:
            call["entry"] = entry = "device"
            k = 1
    call["k"] = k
    batch = entry in ("host", "device", "visibility", "ssaa_host", "ssaa_device") and rng.random() < 0.25
    nv = int(rng.integers(2, 8)) if batch else 1
    nv = max(1, min(nv, n_views, MAX_PIXELS // (k * k * W * H)))
    call["views"] = [int(v) for v in rng.choice(n_views, nv, replace=False)]
    call["band"] = _band(rng, H) if entry in ("host", "device", "visibility", "ssaa_host", "ssaa_device") and rng.random() < 0.35 else None
    call["stream"] = bool(entry in ("device", "rows", "visibility", "ssaa_device") and rng.random() < 0.25)
    if entry == "rows":
        stride = int(rng.integers(1, 6))
        call["stride"], call["phase"] = stride, int(rng.integers(0, stride))
    if entry == "peer":
        call["world"] = int(rng.integers(1, 4))
    if entry == "visibility":
        subset = [bool(b) for b in rng.integers(0, 2, 3)]
        if not any(subset):
            subset[int(rng.integers(0, 3))] = True
        call["subset"] = tuple(subset)
    if entry == "refused":
        call["refusal"] = str(rng.choice(REFUSALS))
    return call


def make_case(seed, index):
    """(scene, views, W, H, plan) of case ``index`` of ``seed``: plan = {"calls": [...], "exact": duplicate pairs,
    "textures", "view_kinds", "T_class"}."""
    return _make_case(int(seed), int(index))


@functools.lru_cache(maxsize=4)
def _make_case(seed, index):
    rng = np.random.default_rng([seed, index])
    W, H = make_size(rng, index)
    cls = ("small", "boundary", "general")[index % 3]
    if cls == "small":
        T = int(rng.integers(1, 65))
    elif cls == "boundary":
        T = BOUNDARY_T.get(index, int(rng.integers(1900, 1926)))
    else:
        T = int(np.exp(rng.uniform(np.log(2000), np.log(30000))))
    sc, meta = make_scene(rng, T, W, H)
    views, view_kinds = make_views(rng, sc, 8)
    state = dict(DEFAULTS)
    calls = [make_call(rng, state, T, W, H, len(views), first=(c == 0)) for c in range(int(rng.integers(3, 7)))]
    plan = {"calls": calls, "exact": meta["exact"], "textures": meta["textures"], "view_kinds": view_kinds, "T_class": cls}
    return sc, views, W, H, plan


def contract_problems(sc):
    """The generator's own rules (DESIGN.md §8) beyond S.validate."""
    out = list(S.validate(sc))
    at = sc.attributes
    if not np.isfinite(sc.vertices).all():
        out.append("non-finite vertex")
    n = at["normal"][:, :3].astype(np.float64)
    if not np.isfinite(n).all() or (np.linalg.norm(n, axis=1) == 0).any():
        out.append("zero or non-finite normal")
    kind = at["kind"][sc.attribute_indices.astype(np.int64)].reshape(-1, 3)
    if ((kind[:, 0] == 1) & (kind[:, 1:] != 1).any(1)).any():
        out.append("textured corner 0 with a colour record at another corner")
    tex = at["kind"] == 1
    if tex.any() and (at["payload"][tex, 0] >= sc.textures.shape[0]).any():
        out.append("texture index out of range")
    return out


# ------------------------------------------------------------------------------------------------------------------
# CPU: the generator is deterministic, valid, and reaches what the sweep exists for
# ------------------------------------------------------------------------------------------------------------------
def _scene_bytes(sc):
    return [np.ascontiguousarray(a).tobytes() for a in (sc.vertices, sc.vertex_indices, sc.attributes, sc.attribute_indices, sc.textures)]


def test_cases_are_deterministic_and_inside_the_contract():
    for i in range(N_CASES):
        a = _make_case.__wrapped__(SEED, i)
        b = _make_case.__wrapped__(SEED, i)
        assert _scene_bytes(a[0]) == _scene_bytes(b[0]), f"case {i}: scene differs between two calls"
        assert np.array_equal(a[1], b[1]) and a[2:4] == b[2:4] and repr(a[4]) == repr(b[4]), f"case {i}: views or plan differ"
        assert not contract_problems(a[0]), (i, contract_problems(a[0]))
        assert a[0].n_triangles == len(a[0].attribute_indices) // 3 and 1 <= a[2] <= 3840 and 1 <= a[3] <= 2160


def test_sequences_are_deterministic():
    for j in range(N_SEQUENCES):
        one = [repr(_step_key(s)) for s in sequence_steps(SEED, j, 40)]
        two = [repr(_step_key(s)) for s in sequence_steps(SEED, j, 40)]
        assert one == two


@functools.lru_cache(maxsize=1)
def _oracle_survey(seed, n_cases):
    """Per default case, the oracle's whole frame of the still camera (view 0, for which the raster-space families are
    placed): winner, depth, setups."""
    from oracle import port
    out = []
    for i in range(n_cases):
        if i in BIG_CASES:   # (seconds of oracle time each, and nothing the others lack)
            continue
        sc, views, W, H, plan = make_case(seed, i)
        o = port.OracleScene(sc).render(views[0], W, H, want_depth=True, want_setups=True, want_winner=True)
        out.append((i, sc.n_triangles, W, H, o, plan))
    return out


def test_coverage_premises(oracle_port):
    survey = _oracle_survey(SEED, N_CASES)
    stats = {k: sum(o["stats"][k] > 0 for *_, o, _ in survey) for k in ("near_rejected", "clipped", "spawned", "small_or_backfacing")}
    assert all(v >= 3 for v in stats.values()), stats
    flat_maxes = {16, 128} | {c["opts"]["flat_max"] for *_, p in survey for c in p["calls"] if "flat_max" in c["opts"]}
    big = np.concatenate([np.maximum(*box_sizes(o["setups"])) for *_, o, _ in survey])
    for limit in sorted(flat_maxes):
        if limit <= 1024:   # (the surveyed frames are at most 1399 px wide)
            assert (big < limit).sum() > 10 and (big >= limit).sum() > 3, (limit, (big >= limit).sum())
    wide = sum(((o["setups"]["xmin"] == 0) & (o["setups"]["xmax"] == W - 1) & (o["setups"]["ymin"] == 0) & (o["setups"]["ymax"] == H - 1)).any()
               for _, _, W, H, o, _ in survey if W > 1 and H > 1)
    assert wide >= 3
    ties = appended = textured = coloured = crowded = 0
    for i, T, W, H, o, plan in survey:
        w = o["winner"]
        won = w[w != NO_WINNER]
        appended += bool((won >= T).any())
        ties += bool(np.isin(won, [a for a, _ in plan["exact"]]).any())
        sc = make_case(SEED, i)[0]
        parent = np.where(won >= T, won - T, won).astype(np.int64)
        kind0 = sc.attributes["kind"][sc.attribute_indices[3 * parent].astype(np.int64)]
        textured += bool((kind0 == 1).any())
        coloured += bool((kind0 == 0).any())
        crowded += bool((block_winners(w) > 96).any())
    assert ties >= 3 and appended >= 3 and textured >= 5 and coloured >= 5 and crowded >= 1, (ties, appended, textured, coloured, crowded)
    Ts = [T for _, T, *_ in survey]
    assert min(Ts) <= 64 and max(Ts) > 2000 and 1920 in Ts and 1921 in Ts


def test_exact_copies_tie_by_order(oracle_port):
    """In some cases the earlier of two identical triangles wins pixels that the later one reaches at the same depth:
    with the earlier one collapsed to a point (order unchanged), the later one wins them at bit-identical depth."""
    from oracle import port
    found = 0
    for i, T, W, H, o, plan in _oracle_survey(SEED, N_CASES):
        firsts = [a for a, _ in plan["exact"] if (o["winner"] == a).any()]
        if not firsts:
            continue
        sc, views = make_case(SEED, i)[:2]
        vi = sc.vertex_indices.copy().reshape(-1, 3)
        pairs = {a: b for a, b in plan["exact"]}
        vi[firsts] = vi[firsts][:, :1]
        without = S.Scene(sc.vertices, vi.reshape(-1), sc.attributes, sc.attribute_indices, sc.textures)
        o2 = port.OracleScene(without).render(views[0], W, H, want_depth=True, want_winner=True)
        for a in firsts:
            px = o["winner"] == a
            same = (o2["winner"][px] == pairs[a]) & (o2["depth"][px].view(np.uint32) == o["depth"][px].view(np.uint32))
            found += int(same.sum())
    assert found > 20


def test_every_plan_feature_occurs():
    need = {f"entry={e}": 3 for e in ENTRIES}
    need.update({f"refusal={r}": 1 for r in REFUSALS})
    need.update({"batch": 5, "band": 5, "band_one_row": 1, "stream": 4, "k=2": 2, "k=4": 2, "opt:setup_capacity": 2,
                 "subset_planes_only": 1, "subset_all": 1, "rows_stride>1": 2})
    for name in DEFAULTS:
        need[f"opt:{name}"] = 3
    need.update({"clusters=0": 2, "clusters=1": 2, "flat_max=16": 1, "flat_max=65536": 1, "rowtab_capacity=0": 1, "timing=3": 1})
    seen = {}

    def see(f):
        seen[f] = seen.get(f, 0) + 1
    for i in range(N_CASES):
        for c in make_case(SEED, i)[4]["calls"]:
            see(f"entry={c['entry']}")
            if "refusal" in c:
                see(f"refusal={c['refusal']}")
            if len(c["views"]) > 1:
                see("batch")
            if c["band"]:
                see("band")
                if c["band"][1] - c["band"][0] == 1:
                    see("band_one_row")
            if c["stream"]:
                see("stream")
            if c["k"] > 1:
                see(f"k={c['k']}")
            if c.get("subset") == (False, True, True) or c.get("subset") == (False, True, False) or c.get("subset") == (False, False, True):
                see("subset_planes_only")
            if c.get("subset") == (True, True, True):
                see("subset_all")
            if c.get("stride", 1) > 1:
                see("rows_stride>1")
            for name, v in c["opts"].items():
                see(f"opt:{name}")
                see(f"{name}={v}")
    short = {f: (seen.get(f, 0), n) for f, n in need.items() if seen.get(f, 0) < n}
    assert not short, short


def test_exact_comparison_has_teeth(oracle_port):
    """For most cases a change no tolerance would notice changes an oracle pixel or winner: the order of one exact
    duplicate pair swapped (the earlier position keeps the tied pixels, now with the other copy's records), or one
    ulp of one diagonal entry of the still camera's matrix."""
    from oracle import port
    sensitive = 0
    survey = _oracle_survey(SEED, N_CASES)
    for i, T, W, H, o, plan in survey:
        sc, views = make_case(SEED, i)[:2]
        changed = []
        won = [(a, b) for a, b in plan["exact"] if (o["winner"] == a).any()]
        if won:
            a, b = won[0]
            vi, ai = sc.vertex_indices.reshape(-1, 3).copy(), sc.attribute_indices.reshape(-1, 3).copy()
            vi[[a, b]], ai[[a, b]] = vi[[b, a]], ai[[b, a]]
            changed.append(S.Scene(sc.vertices, vi.reshape(-1), sc.attributes, ai.reshape(-1), sc.textures))
        for scene, m in [(x, views[0]) for x in changed] + [(sc, None)]:
            osc = port.OracleScene(scene)
            for e in ((None,) if m is not None else (0, 5, 10)):
                m2 = views[0].copy()
                if e is not None:
                    m2[e] = np.nextafter(m2[e], np.float32(np.inf))
                o2 = osc.render(m2, W, H, want_winner=True)
                if not (np.array_equal(o2["pixels"], o["pixels"]) and np.array_equal(o2["winner"], o["winner"])):
                    sensitive += 1
                    break
            else:
                continue
            break
    assert sensitive >= 0.6 * len(survey), (sensitive, len(survey))


# ------------------------------------------------------------------------------------------------------------------
# GPU: running a call against the oracle
# ------------------------------------------------------------------------------------------------------------------
class Ctx:
    """One renderer, the scene it holds (and its oracle), the frame size and the options as the calls left them."""

    def __init__(self, lib, port, torch, r):
        self.lib, self.port, self.torch, self.r = lib, port, torch, r
        self.th = lib.tile_height()
        self.state = dict(DEFAULTS)
        self.pinned = []
        self.side = None

    def load(self, sc):
        self.sc = sc
        self.osc = self.port.OracleScene(sc)
        self.cache = {}
        self.r.load_scene(sc)

    def oracle(self, m, W, H, setups=False):
        key = (m.tobytes(), W, H, setups)
        if key not in self.cache:
            if len(self.cache) > 24:
                self.cache.clear()
            self.cache[key] = self.osc.render(m, W, H, want_depth=True, want_winner=True, want_setups=setups)
        return self.cache[key]

    def stream(self, on):
        if not on:
            return 0
        if self.side is None:
            self.side = self.torch.cuda.Stream()
        return self.side.cuda_stream

    def set_options(self, opts):
        for name, value in opts.items():
            self.r.set_option(name, value)
            if name in DEFAULTS:
                self.state[name] = value
            if name == "pin_host" and not value:
                self.pinned.clear()


def _first_diff(got, want, winner, what, k=1):
    if np.array_equal(got, want):
        return
    ys, xs = np.nonzero(got != want)
    y, x = int(ys[0]), int(xs[0])
    win = winner[k * y:k * y + k, k * x:k * x + k].ravel().tolist() if winner is not None else "?"
    raise AssertionError(f"{what}: {len(ys)} px differ, first (x={x}, y={y}) got {int(got[y, x]):06x} want {int(want[y, x]):06x}, "
                         f"oracle winner {win}")


def _guarded(torch, n):
    return torch.full((n + PAD,), GUARD, dtype=torch.int32, device="cuda:0")


def _read(torch, buf, n, what):
    torch.cuda.synchronize()
    host = buf.cpu().numpy().view(np.uint32)
    assert (host[n:] == GUARD).all(), f"{what}: the call wrote past its output"
    return host[:n]


def _submit(ctx, launch, stream=0):
    """Submits, repeating while finish() asks for it (a regrown capacity may still be short once).  A call on a caller
    stream first waits for the outputs' initialisation on torch's stream."""
    if stream:
        ctx.torch.cuda.synchronize()
    for _ in range(REPEATS):
        launch()
        if not ctx.r.finish():
            return
    raise AssertionError(f"finish() still asks for a repeat after {REPEATS} submissions")


def _stages(ctx, m, W, H, o, what, k=1):
    """Setup records (with every survivor recorded) and raster-space vertices of the last whole-frame submission."""
    r = ctx.r
    if ctx.state["direct_small"] == 0:
        got, want = r.setups(), o["setups"]
        assert len(got) == len(want), f"{what}: {len(got)} setups != oracle {len(want)}"
        for field in want.dtype.names:
            same = got[field].view(np.uint32) == want[field].view(np.uint32)
            if got[field].dtype.kind == "f":   # (a NaN's payload is not part of the contract)
                same |= np.isnan(got[field]) & np.isnan(want[field])
            if not same.all():
                bad = np.nonzero(~same.reshape(len(want), -1).all(1))[0]
                raise AssertionError(f"{what}: setup field {field} differs in {len(bad)} records, first order {want['order'][bad[0]]}")
    if k == 1:
        rv = ctx.osc.vertex_stage(m, W, H)[1]
        got = r.raster_vertices()
        same = (got.view(np.uint32) == rv.view(np.uint32)) | (np.isnan(got) & np.isnan(rv))
        assert same.all(), f"{what}: raster vertices differ at {np.nonzero(~same.all(1))[0][:5].tolist()}"


def run_call(ctx, call, views, W, H, what):
    """Executes one plan call on ctx's renderer and checks every output against the oracle."""
    torch, r, lib = ctx.torch, ctx.r, ctx.lib
    ctx.set_options(call["opts"])
    entry, k = call["entry"], call["k"]
    ms = views[call["views"]]
    n = len(ms)
    y0, y1 = call["band"] or (0, H)
    whole = call["band"] is None
    sp = ctx.stream(call["stream"])
    if sp:
        torch.cuda.synchronize()
    want = [ctx.oracle(m, k * W, k * H, setups=(whole and n == 1 and entry != "peer")) for m in ms]
    colour = [resolve(o["pixels"], k) if k > 1 else o["pixels"] for o in want]
    T = ctx.sc.n_triangles

    def check_stats():
        if whole:
            for v, o in enumerate(want):
                assert_stats(r.stats(v), o, f"{what}: view {v}")

    if entry == "host" or entry == "ssaa_host":
        out = None
        if ctx.state["pin_host"]:
            out = np.empty((n, y1 - y0, W), np.uint32)
            ctx.pinned.append(out)
        got = r.render(ms, W, H, y0=y0, y1=y1, out=out) if entry == "host" else r.render_ssaa(ms, W, H, k, y0=y0, y1=y1, out=out)
        for v in range(n):
            _first_diff(got[v], colour[v][y0:y1], want[v]["winner"][k * y0:], f"{what}: view {v}", k)
        check_stats()
    elif entry in ("device", "ssaa_device"):
        px = n * (y1 - y0) * W
        buf = _guarded(torch, px)
        if entry == "device":
            _submit(ctx, lambda: r.render_device(ms, W, H, buf.data_ptr(), y0=y0, y1=y1, stream=sp), sp)
        else:
            _submit(ctx, lambda: r.render_device_ssaa(ms, W, H, k, buf.data_ptr(), y0=y0, y1=y1, stream=sp), sp)
        got = _read(torch, buf, px, what).reshape(n, y1 - y0, W)
        for v in range(n):
            _first_diff(got[v], colour[v][y0:y1], want[v]["winner"][k * y0:], f"{what}: view {v}", k)
        check_stats()
    elif entry == "visibility":
        subset = call["subset"]
        if sp:
            px = n * (y1 - y0) * W
            bufs = [_guarded(torch, px) if on else None for on in subset]
            ptrs = [b.data_ptr() if b is not None else 0 for b in bufs]
            _submit(ctx, lambda: r.render_device_visibility(ms, W, H, *ptrs, y0=y0, y1=y1, stream=sp), sp)
            got = [_read(torch, b, px, f"{what}: {name}").reshape(n, y1 - y0, W) if b is not None else None
                   for name, b in zip(("colour", "triangle", "depth"), bufs)]
        else:
            got = device_planes(r, torch, ms, W, H, y0, y1, subset)
        for v in range(n):
            c, tri, dep, o = expected(ctx.osc, T, ms[v], W, H)
            for name, g, w in zip(("colour", "triangle", "depth"), got, (c, tri, dep)):
                if g is not None:
                    _first_diff(g[v], w[y0:y1], o["winner"][y0:], f"{what}: view {v} {name}")
        check_stats()
    elif entry == "rows":
        m = ms[0]
        rows, frame_rows, buf_rows = lib.rows_layout(H, call["stride"], call["phase"], ctx.th)
        px = rows * W
        buf = _guarded(torch, px)
        _submit(ctx, lambda: r.render_device_rows(m, W, H, call["stride"], call["phase"], buf.data_ptr(), stream=sp), sp)
        got = _read(torch, buf, px, what).reshape(rows, W)
        _first_diff(got[buf_rows], colour[0][frame_rows], want[0]["winner"][frame_rows], what)
    elif entry == "peer":
        m, world = ms[0], call["world"]
        a, _ = r.peer_frame_alloc(W * H * 4)
        b, _ = r.peer_frame_alloc(W * H * 4)
        try:
            for phase in range(world):
                r.set_peer_frames([a, b])
                _submit(ctx, lambda: r.render_device_rows(m, W, H, world, phase, 0))
                r.set_peer_frames([])
            for ptr in (a, b):
                _first_diff(r.read_device(ptr, (H, W)), colour[0], want[0]["winner"], f"{what}: peer frame over {world}")
        finally:
            r.set_peer_frames([])
            r.peer_frame_release(a)
            r.peer_frame_release(b)
    elif entry == "refused":
        px = n * (y1 - y0) * W
        bufs = [_guarded(torch, px) for _ in range(4)]
        p = [bb.data_ptr() for bb in bufs]
        kind = call["refusal"]
        torch.cuda.synchronize()
        if kind.endswith("_peer"):
            r.set_peer_frames([p[3]])
        try:
            calls = {"ssaa_peer": [lambda: r.render_device_ssaa(ms, W, H, 2, p[0], y0=y0, y1=y1),
                                   lambda: r.render_ssaa(ms, W, H, 2, y0=y0, y1=y1)],
                     "visibility_peer": [lambda: r.render_device_visibility(ms, W, H, p[0], p[1], p[2], y0=y0, y1=y1),
                                         lambda: r.render_device_visibility(ms, W, H, 0, p[1], 0, y0=y0, y1=y1)],
                     "ssaa_k3": [lambda: r.render_device_ssaa(ms, W, H, 3, p[0], y0=y0, y1=y1),
                                 lambda: r.render_ssaa(ms, W, H, 3, y0=y0, y1=y1)],
                     "visibility_none": [lambda: r.render_device_visibility(ms, W, H, 0, 0, 0, y0=y0, y1=y1)]}[kind]
            for c in calls:
                with pytest.raises(lib.RendererError, match=f"s3r error {S3R_E_ARG}: .+"):
                    c()
        finally:
            r.set_peer_frames([])
        for bb in bufs:
            _read(torch, bb, 0, f"{what}: a refused call")   # every word of every buffer is still the guard
        assert r.finish() is False
    else:
        raise AssertionError(entry)
    if entry in ("host", "device", "ssaa_host", "ssaa_device", "visibility") and whole and n == 1:
        _stages(ctx, ms[0], k * W, k * H, want[0], what, k)
    if ctx.state["timing"]:
        r.timing()


def describe(call):
    return {k: v for k, v in call.items() if v not in (None, False) and not (k == "opts" and not v)}


# ------------------------------------------------------------------------------------------------------------------
# GPU: independent cases
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("index", range(N_CASES), ids=[f"case_{i:04d}" for i in range(N_CASES)])
def test_case(index, renderer_lib, oracle_port, tmp_path):
    import torch
    sc, views, W, H, plan = make_case(SEED, index)
    r = renderer_lib.Renderer(0)
    ctx = Ctx(renderer_lib, oracle_port, torch, r)
    try:
        ctx.load(sc)
        for c, call in enumerate(plan["calls"]):
            what = f"case {index} of seed {SEED}: T={sc.n_triangles} {W}x{H}, call {c} {describe(call)}"
            try:
                run_call(ctx, call, views, W, H, what)
            except AssertionError as e:
                path = tmp_path / f"case_{index:04d}.bin"
                S.write_data_bin(str(path), sc)
                raise AssertionError(f"{e}\n  plan: {[describe(x) for x in plan['calls']]}\n  views: {plan['view_kinds']}\n"
                                     f"  scene written to {path}\n  replay: S3R_SWEEP_SEED={SEED} python -m pytest "
                                     f"tests/test_gpu_random_sweep.py -k case_{index:04d}") from None
    finally:
        r.close()


# ------------------------------------------------------------------------------------------------------------------
# GPU: long-lived sequences on one renderer
# ------------------------------------------------------------------------------------------------------------------
def _moved(rng, xyz):
    """New positions for the same vertices: a rigid motion, a push along the view axis (across the near plane, out of
    the frame), a scale about a point, or noise on a subset."""
    kind = rng.integers(0, 4)
    out = xyz.astype(np.float64)
    if kind == 0:
        out = (out - out.mean(0)) @ _rotation(rng).T + out.mean(0) + rng.normal(size=3)
    elif kind == 1:
        out[:, 2] += rng.uniform(-4, 4)
        out[:, :2] += rng.uniform(-3, 3, 2)
    elif kind == 2:
        c = out[rng.integers(0, len(out))]
        out = (out - c) * rng.uniform(0.2, 3) + c
    else:
        pick = rng.random(len(out)) < 0.3
        out[pick] += rng.normal(size=(int(pick.sum()), 3)) * rng.uniform(0.01, 2)
    return out.astype(np.float32)


def sequence_steps(seed, j, n_steps):
    """The steps of sequence j: dicts with "step" in {load, call, resize, vertices, attributes, textures}."""
    rng = np.random.default_rng([seed, 1 << 20, j])
    W, H = make_size(rng)
    T = int(rng.choice([int(rng.integers(1, 65)), int(rng.integers(1900, 1926)), int(rng.integers(2000, 8000))]))
    sc, _ = make_scene(rng, T, W, H)
    views, _ = make_views(rng, sc, 8)
    yield {"step": "load", "scene": sc, "views": views, "W": W, "H": H}
    state = dict(DEFAULTS)
    for s in range(1, n_steps):
        u = rng.random()
        if u < 0.62:
            yield {"step": "call", "call": make_call(rng, state, sc.n_triangles, W, H, len(views))}
        elif u < 0.72:
            W, H = make_size(rng)
            W, H = min(W, 1400), min(H, 1400)
            yield {"step": "resize", "W": W, "H": H}
        elif u < 0.84:
            xyz = _moved(rng, sc.vertices[:, :3])
            v = sc.vertices.copy()
            v[:, :3] = xyz
            sc = S.Scene(v, sc.vertex_indices, sc.attributes, sc.attribute_indices, sc.textures)
            yield {"step": "vertices", "xyz": xyz, "device": bool(rng.random() < 0.5), "stream": bool(rng.random() < 0.4), "scene": sc}
        elif u < 0.91:
            at = _attributes(rng, sc.n_triangles, sc.textures.shape[0], rng.uniform(0.1, 0.9))
            sc = S.Scene(sc.vertices, sc.vertex_indices, at, sc.attribute_indices, sc.textures)
            yield {"step": "attributes", "scene": sc}
        elif u < 0.95:
            tx = sc.textures[::-1].copy() if rng.random() < 0.5 else (sc.textures ^ np.uint32(rng.integers(1, 1 << 24))) & np.uint32(0xFFFFFF)
            sc = S.Scene(sc.vertices, sc.vertex_indices, sc.attributes, sc.attribute_indices, tx)
            yield {"step": "textures", "device": bool(rng.random() < 0.5), "scene": sc}
        else:
            T = int(rng.choice([int(rng.integers(1, 65)), int(rng.integers(1900, 1926)), int(rng.integers(2000, 12000))]))
            sc, _ = make_scene(rng, T, W, H)
            views, _ = make_views(rng, sc, 8)
            yield {"step": "load", "scene": sc, "views": views, "W": W, "H": H}


def _step_key(step):
    return {k: (v if k in ("step", "call", "W", "H", "device", "stream") else "...") for k, v in step.items()}


@pytest.mark.gpu
@pytest.mark.parametrize("j", range(N_SEQUENCES), ids=[f"sequence_{j}" for j in range(N_SEQUENCES)])
def test_sequence(j, renderer_lib, oracle_port):
    """One renderer through SEQUENCE_STEPS random steps, never reset: every call equals the oracle of the scene arrays
    as they stand.  A failing call is run once more on a fresh renderer with the same scene, options and frame size, and
    the message says whether the failure depends on the renderer's history."""
    import torch
    r = renderer_lib.Renderer(0)
    ctx = Ctx(renderer_lib, oracle_port, torch, r)
    calls = 0
    try:
        for s, step in enumerate(sequence_steps(SEED, j, SEQUENCE_STEPS)):
            kind = step["step"]
            if kind == "load":
                ctx.load(step["scene"])
                views, W, H = step["views"], step["W"], step["H"]
            elif kind == "resize":
                W, H = step["W"], step["H"]
            elif kind == "vertices":
                src = torch.from_numpy(np.ascontiguousarray(step["xyz"])).cuda() if step["device"] else step["xyz"]
                sp = ctx.stream(step["stream"])
                torch.cuda.synchronize()
                r.update_vertices(src, stream=sp)
                if sp:
                    ctx.side.synchronize()
                ctx.sc, ctx.osc, ctx.cache = step["scene"], oracle_port.OracleScene(step["scene"]), {}
            elif kind == "attributes":
                r.update_attributes(step["scene"].attributes)
                ctx.sc, ctx.osc, ctx.cache = step["scene"], oracle_port.OracleScene(step["scene"]), {}
            elif kind == "textures":
                tx = step["scene"].textures
                r.update_textures(torch.from_numpy(tx.view(np.int32)).cuda() if step["device"] else tx)
                torch.cuda.synchronize()
                ctx.sc, ctx.osc, ctx.cache = step["scene"], oracle_port.OracleScene(step["scene"]), {}
            else:
                call = step["call"]
                calls += 1
                what = f"sequence {j} of seed {SEED}, step {s}: T={ctx.sc.n_triangles} {W}x{H} {describe(call)}"
                try:
                    run_call(ctx, call, views, W, H, what)
                except AssertionError as e:
                    fresh = renderer_lib.Renderer(0)
                    try:
                        fctx = Ctx(renderer_lib, oracle_port, torch, fresh)
                        fctx.load(ctx.sc)
                        fctx.set_options({k: v for k, v in ctx.state.items() if v != DEFAULTS[k]})
                        run_call(fctx, call, views, W, H, what + " (fresh renderer)")
                        verdict = "passes on a fresh renderer: a state-carrying bug"
                    except AssertionError as e2:
                        verdict = f"fails on a fresh renderer too: {e2}"
                    finally:
                        fresh.close()
                    raise AssertionError(f"{e}\n  {verdict}\n  options: {ctx.state}\n  replay: steps 0..{s} of "
                                         f"sequence_steps({SEED}, {j}, {s + 1}) on one renderer "
                                         f"(S3R_SWEEP_SEED={SEED} python -m pytest tests/test_gpu_random_sweep.py -k sequence_{j})") from None
        assert calls > SEQUENCE_STEPS // 2
    finally:
        r.close()
