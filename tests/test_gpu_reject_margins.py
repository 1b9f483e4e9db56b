"""The two conservative rejection tests against the oracle, at their boundaries: frames and statistics.

Everywhere else the renderer is bit-exact by construction.  Two tests only have to be safe, and they use approximate
arithmetic with a hand-derived margin:
  * tile_outside_triangle drops a (triangle, tile) pair when one barycentric weight is provably negative over the tile
    (tile-list collection of the small-scene path, count_tiles and bin_big_body of the general path).  Its margin covers
    the drift of the reference's incremental walk (render.cpp:374-379), which can turn a weight that is negative at a
    pixel centre into one that is not.
  * cluster_verdict rejects whole clusters from a bounding sphere and a longest edge (cluster_cull): behind the near
    plane, off the frame or the band, outside the interleaved tile rows a submission owns, or too small for the area cull.
A rejection that is wrong in the unsafe direction loses a triangle the reference draws.  The scenes here put probes on
purpose at the boundaries: slivers whose edge passes a few hundredths of a pixel outside a tile corner's pixel centre,
kept only where the oracle draws the pixel although the kernel's own evaluation says the weight is negative (the margin
alone keeps the pair), and ladders of single-triangle clusters across every boundary of cluster_verdict.  The CPU
tests at the top prove from the oracle (and a float64 restatement of cluster_verdict with exact division and square
root) that every scene reaches the boundary it exists for; the GPU tests compare frames and statistics.  A cluster
wrongly culled shows as fewer setups than the oracle's rasterized triangles, a wrong near-plane verdict as a near /
clipped mismatch, even where the lost triangle is hidden."""
import functools

import numpy as np
import pytest

from swift3drenderer_b200 import scene as S
from test_gpu_vis_edges import ROUTES, _Mesh, assert_same, assert_stats, set_route, still, textures

TILE_W, TILE_H = 64, 32          # csrc/pipeline.cuh
BIG_TILES = 16                   # csrc/pipeline.cuh: triangles over more tiles are binned by bin_big_body
K_NEAR = np.float32(0.1)         # csrc/pipeline.cuh kNear
f32 = np.float32


# ------------------------------------------------------------------------------------------------------------------
# A. tile_outside_triangle
# ------------------------------------------------------------------------------------------------------------------
def tile_best(st, k, tx0, ylo_t, yhi_t):
    """tile_outside_triangle (csrc/kernels.cu) for setup record k and the tile at column tx0 whose rows [ylo_t, yhi_t)
    are in the submission, in binary32 and the kernel's operation order: [(best, margin)] per weight.  The pair is
    dropped when some best < -margin."""
    xmin, xmax, ymin, ymax = (int(st[n][k]) for n in ("xmin", "xmax", "ymin", "ymax"))
    x0, x1 = max(tx0, xmin), min(tx0 + TILE_W - 1, xmax)
    y0, y1 = max(ylo_t, ymin), min(yhi_t - 1, ymax)
    bw, bh = f32(xmax - xmin), f32(ymax - ymin)
    fx0, fx1, fy0, fy1 = f32(x0 - xmin), f32(x1 - xmin), f32(y0 - ymin), f32(y1 - ymin)
    out = []
    for c in range(3):
        ws, dx, dy = st["wstart"][k][c], st["dx"][k][c], st["dy"][k][c]
        wmax = (abs(ws) + abs(dx) * bw) + abs(dy) * bh
        margin = ((bw + bh) + f32(16)) * f32(2.4e-7) * (wmax + f32(1))
        best = (ws + (fx1 if dx > 0 else fx0) * dx) + (fy1 if dy > 0 else fy0) * dy
        out.append((best, margin))
    return out


MARGIN_W, MARGIN_H = 2560, 1440
MARGIN_BANDS = [0, 16 * TILE_H + 11, 32 * TILE_H + 21, MARGIN_H]   # y0 and y1 cut tile rows
N_WHOLE_SLOTS = 120


def _probe_slots():
    """Probe slots: (kind, tile column, pixel row of the target corner, box size range).  'tl': the tile's top-left pixel
    (the sliver lies up-left of it), 'br': its bottom-right pixel (the sliver lies down-right).  The band kinds target
    the first / last row of a tile row that a band edge cuts."""
    slots = []
    rng = np.random.RandomState(11)
    tiles_x, tiles_y = MARGIN_W // TILE_W, MARGIN_H // TILE_H
    used = set()

    def tile():
        while True:
            t = (rng.randint(2, tiles_x - 2), rng.randint(2, tiles_y - 2))
            if t not in used:
                used.add(t)
                return t
    for corner in ("tl", "br"):
        for k in range(N_WHOLE_SLOTS // 2):
            tx, ty = tile()
            y = ty * TILE_H if corner == "tl" else ty * TILE_H + TILE_H - 1
            slots.append((corner, tx, y, (20, 250) if k < 20 else (250, 3000)))
    for e in MARGIN_BANDS[1:-1]:
        for k in range(12):
            tx = 3 + 3 * k + (e % 7)
            slots.append(("tl", tx, e, (300, 3000)))        # first row of the band below the edge
            slots.append(("br", tx + 1, e - 1, (300, 3000)))  # last row of the band above it
    return slots


def _probe(rng, corner, tx, y, sizes):
    """A sliver with one edge along a line that passes ~0..0.002 px outside the centre of pixel (x, y), the triangle on
    the far side of the tile: long along the line (its box, and the reference's walk to the pixel, is `size` px), a few
    pixels thick."""
    th = rng.uniform(0.2, 1.37)
    if corner == "tl":
        p, nrm = np.array([tx * TILE_W + 0.5, y + 0.5]), -np.array([np.cos(th), np.sin(th)])
    else:
        p, nrm = np.array([tx * TILE_W + TILE_W - 0.5, y + 0.5]), np.array([np.cos(th), np.sin(th)])
    t = np.array([np.sin(th), -np.cos(th)])
    size = np.exp(rng.uniform(np.log(sizes[0]), np.log(sizes[1])))
    a = size * rng.uniform(0.3, 0.7)
    q = p + (rng.uniform(-0.0005, 0.002) if size > 250 else rng.uniform(-0.0002, 0.0002)) * nrm
    return [q + a * t, q - (size - a) * t, q + rng.uniform(2.5, 5) * nrm + rng.uniform(-1, 1) * t]


def _filler(mesh, n, rng, W, H):
    for _ in range(n):
        x, y = rng.uniform(-20, W), rng.uniform(-20, H)
        sx, sy = rng.uniform(8, 120), rng.uniform(8, 120)
        mesh.tri([(x, y), (x + sx, y + rng.uniform(0, 8)), (x + rng.uniform(0, 8), y + sy)], rng.uniform(20, 30),
                 tuple(rng.uniform(40, 255, 3)))


def margin_pairs(o, probes, band=None):
    """The (probe, tile) pairs only the margin keeps: the oracle's winner shows the probe on a pixel of the tile (of the
    band's part of it), the kernel's own best is negative for some weight, and no weight is below -margin (that would
    be an unsound rejection).  Returns (pairs, unsound)."""
    st, win = o["setups"], o["winner"]
    row = {int(t): i for i, t in enumerate(st["order"])}
    pairs, unsound = [], []
    for k, (corner, tx, y) in enumerate(probes):
        if k not in row:
            continue
        ty0 = (y // TILE_H) * TILE_H
        ylo_t, yhi_t = ty0, ty0 + TILE_H
        if band is not None:
            if not band[0] <= y < band[1]:
                continue
            ylo_t, yhi_t = max(ty0, band[0]), min(ty0 + TILE_H, band[1])
        if not (win[ylo_t:yhi_t, tx * TILE_W:(tx + 1) * TILE_W] == k).any():
            continue
        bm = tile_best(st, row[k], tx * TILE_W, ylo_t, yhi_t)
        if any(b < -m for b, m in bm):
            unsound.append((k, corner, tx, y))
        elif any(b < 0 for b, _ in bm):
            pairs.append((k, corner, tx, y))
    return pairs, unsound


@functools.lru_cache(maxsize=None)
def _margin_probes(oracle_port):
    """Settles the probes against the oracle (as tie_field settles its tie sites): a slot whose probe is not a
    margin-only pair is drawn again, up to 40 times.  Returns [(corner, tile column, target row, corners)] of the slots
    that settled."""
    rng = np.random.RandomState(7)
    slots = _probe_slots()
    drawn = [_probe(rng, *s) for s in slots]
    good = np.zeros(len(slots), bool)
    m = oracle_port.camera_path(still())[0]
    W, H = MARGIN_W, MARGIN_H
    for _ in range(40):
        mesh = _Mesh(W, H)
        for k, pts in enumerate(drawn):
            mesh.tri(pts, 2.0 + 0.002 * k, (255.0 * (k % 2), 40.0 + (k * 37) % 200, 255.0 - (k * 53) % 200))
        o = oracle_port.OracleScene(mesh.scene()).render(m, W, H, want_winner=True, want_setups=True)
        probes = [s[:3] for s in slots]
        # whole-frame slots need a margin-only pair in the whole frame, band slots one in their band
        whole = {p[0] for p in margin_pairs(o, probes)[0]}
        banded = {p[0] for band in zip(MARGIN_BANDS[:-1], MARGIN_BANDS[1:]) for p in margin_pairs(o, probes, band)[0]}
        good = np.array([k in (whole if k < N_WHOLE_SLOTS else banded) for k in range(len(slots))])
        bad = np.nonzero(~good)[0]
        if len(bad) == 0:
            break
        for k in bad:
            drawn[k] = _probe(rng, *slots[k])
    return [(s[0], s[1], s[2], drawn[k]) for k, s in enumerate(slots) if good[k]]


def margin_scene(oracle_port, n_filler):
    """The settled probes at depths 2.0.., then ``n_filler`` triangles behind them all."""
    mesh = _Mesh(MARGIN_W, MARGIN_H)
    probes = _margin_probes(oracle_port)
    for k, (_, _, _, pts) in enumerate(probes):
        mesh.tri(pts, 2.0 + 0.002 * k, (255.0 * (k % 2), 40.0 + (k * 37) % 200, 255.0 - (k * 53) % 200))
    _filler(mesh, n_filler, np.random.RandomState(5), MARGIN_W, MARGIN_H)
    return mesh.scene(), [p[:3] for p in probes]


# ------------------------------------------------------------------------------------------------------------------
# B. cluster_verdict: a float64 restatement with exact division and square root
# ------------------------------------------------------------------------------------------------------------------
def verdict64(m, hdr, W, H, band=(0, None), world=1, phase=0, sigma=None, tangent=True):
    """cluster_verdict (csrc/kernels.cu) for one cluster header in float64, MUFU replaced by exact operations (and the
    kernel's 1.00001 / 0.99999 factors kept).  Returns (verdict, quantities): verdict 0 keep, 1 near-rejected, 2 culled;
    sigma / tangent override the Gram bound and the tangent factor (to show that each is needed)."""
    a = np.asarray(m, np.float64).reshape(3, 4)
    c = np.asarray(hdr["center"], np.float64)
    radius, max_edge = float(hdr["radius"]), float(hdr["max_edge"])
    y0, y1 = band[0], H if band[1] is None else band[1]
    factor = _factor(H)
    fw, fh, half_w, half_h = float(W), float(H), W / 2.0, H / 2.0
    cc = a[:, :3] @ c + a[:, 3]
    ax = np.abs(c) + radius
    norm = np.sqrt((a[:, :3] ** 2).sum(1))
    gram = a[:, :3] @ a[:, :3].T
    sig = np.sqrt(np.abs(gram).sum(1).max()) if sigma is None else sigma
    e = 2.0 ** -21 * (np.abs(a[:, :3]) @ ax + np.abs(a[:, 3]))
    rho = (norm * radius + 2 * e) * 1.000001 + 1e-30
    err = e.max()
    d = -cc[2]
    q = {"d_max": d + rho[2], "d_min": d - rho[2]}
    d_min, d_max = q["d_min"], q["d_max"]
    if d_max < 0 or (d_min > 0 and d_max <= float(K_NEAR)):
        return 1, q
    if not d_min > float(K_NEAR) * 1.000001:
        return 0, q
    x_lo, x_hi, yy_lo, yy_hi = cc[0] - rho[0], cc[0] + rho[0], -cc[1] - rho[1], -cc[1] + rho[1]
    inv_min, inv_max = factor / d_min * 1.00001, factor / d_max * 0.99999
    qx_hi = x_hi * (inv_min if x_hi >= 0 else inv_max)
    qx_lo = x_lo * (inv_max if x_lo >= 0 else inv_min)
    qy_hi = yy_hi * (inv_min if yy_hi >= 0 else inv_max)
    qy_lo = yy_lo * (inv_max if yy_lo >= 0 else inv_min)
    sx = 2.0 ** -18 * (max(abs(qx_lo), abs(qx_hi)) + fw) + 0.01
    sy = 2.0 ** -18 * (max(abs(qy_lo), abs(qy_hi)) + fh) + 0.01
    q.update(sx_hi=qx_hi + half_w + sx, sx_lo=qx_lo + half_w - sx, sy_hi=qy_hi + half_h + sy, sy_lo=qy_lo + half_h - sy)
    if q["sx_hi"] < 0 or q["sy_hi"] < y0 or q["sx_lo"] >= fw or q["sy_lo"] >= y1:
        return 2, q
    if world != 1:
        ylo, yhi = int(max(0.0, np.floor(q["sy_lo"]))), int(min(fh - 1, q["sy_hi"]))
        if ylo > yhi or not any(a_ % world == phase for a_ in range(ylo // TILE_H, yhi // TILE_H + 1)):
            return 2, q
    length = sig * max_edge + 4 * err
    rcp_min = 1.0 / d_min * 1.00001
    tu, tv = max(abs(x_lo), abs(x_hi)) * rcp_min, max(abs(yy_lo), abs(yy_hi)) * rcp_min
    tan = np.sqrt(1 + tu * tu + tv * tv) * 1.00001 if tangent else 1.0
    q["pixels"] = inv_min * length * tan * 1.00001 + 2 * (sx + sy)
    if q["pixels"] <= 3.09:
        return 2, q
    return 0, q


def _tri_world(p, m):
    """World positions of camera-space points p (3 x 3) under the 3 x 4 matrix m."""
    a = np.asarray(m, np.float64).reshape(3, 4)
    return (np.linalg.solve(a[:, :3], (np.asarray(p, np.float64) - a[:, 3]).T)).T


def world_scene(tris, colours):
    n = len(tris)
    v = np.ones((3 * n, 4), "<f4")
    v[:, :3] = np.asarray(tris, np.float64).reshape(-1, 3)
    at = np.zeros(n, S.ATTR_DTYPE)
    at["normal"][:, 2] = 1.0
    at["payload"][:, :3] = np.asarray(colours, "<f4").view("<u4")
    return S.Scene(v, np.arange(3 * n, dtype="<u8"), at, np.repeat(np.arange(n, dtype="<u8"), 3), textures())


def _camera_point(xr, yr, d, factor, W, H):
    """Camera-space point at depth d that projects to raster (xr, yr)."""
    return np.array([(xr - W / 2) * d / factor, -(yr - H / 2) * d / factor, -d])


def _factor(H):
    return float(np.float32(np.float32(0.1) * np.float32(H) / (np.float32(2) * np.float32(float.fromhex("0x1.0a2c9ap-5")))))


def _needle(tip, direction, length, width, d, factor, W, H):
    """Raster-space needle at depth d: its tip at ``tip``, pointing along ``direction``; camera-space corners."""
    u = np.asarray(direction, np.float64) / np.linalg.norm(direction)
    n = np.array([-u[1], u[0]])
    tip = np.asarray(tip, np.float64)
    base = tip - length * u
    return [_camera_point(*pt, d, factor, W, H) for pt in (tip, base + n * width / 2, base - n * width / 2)]


IDENTITY = np.array([1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0], np.float32)


def ladder(name):
    """One ladder: (W, H, matrix, scene, rungs, role).  rungs[k] describes triangle k (a cluster of its own).  role is
    what the ladder exists for (see the premise test)."""
    rng = np.random.RandomState(abs(hash(name)) % 1000)
    tris, rungs = [], []

    def add(p, rung):
        tris.append(p)
        rungs.append(rung)
    if name == "near":
        # slivers along the view ray, 0.01 long, whose far vertex lies at depth kNear + k ulps, at kNear (1 +- r), and
        # around the eye plane (depth 0: the reference's 0 / 0)
        W, H, m = 800, 450, IDENTITY
        ulp = float(np.spacing(K_NEAR))
        fars = [float(K_NEAR) + k * ulp for k in (-8, -2, -1, 0, 1, 2, 8)]
        fars += [float(K_NEAR) * (1 + r) for r in (-3e-3, -1e-3, -2e-4, 5e-5, 2e-4, 1e-3, 3e-3)]
        fars += [-1e-3, -1e-6, 0.0, 1e-6, 1e-3, 0.05]
        for k, far in enumerate(fars):
            x, y = -0.1 + 0.05 * (k % 5), -0.075 + 0.05 * (k // 5)
            p = np.array([[x, y, -far], [x, y, -(far - 0.01)], [x + 1e-5, y + 2e-5, -(far - 0.01)]])
            add(p.astype(np.float32), {"far": far})
        role = "near"
    elif name in ("edges_narrow", "edges_wide"):
        # needles pointing at the left / right frame edge, tips from -2 to +2 px around x = 0 and x = W
        W, H = (24, 4096) if name == "edges_narrow" else (800, 450)
        m, F = IDENTITY, _factor(H)
        tips = [-2, -1, -0.5, -0.25, -0.12, -0.06, -0.03, -0.01, 0.0, 0.01, 0.05, 0.2, 0.45, 1, 2]
        if name == "edges_wide":   # the sphere's depth extent loosens the bound far from the optical axis: ~6 px here
            tips = [-16, -12, -9, -7, -5, -3] + tips
        step = 100 if H > 1000 else 20
        for k, t in enumerate(tips):
            y = H / 2 + (k - len(tips) / 2) * step
            add(_needle((t, y + 0.37), (1, 0), 20, 1.1, 5.0, F, W, H), {"side": "left", "tip": t})
            add(_needle((W - t, y + 3.71), (-1, 0), 20, 1.1, 5.0, F, W, H), {"side": "right", "tip": t})
        role = "screen"
    elif name == "rows":
        # vertical needles near the centre column ending just above / below the 32-row boundaries around the centre row,
        # and at the band edges of ROWS_BANDS (y0 % 32 != 0), pointing up and down
        W, H = 800, 450
        m, F = IDENTITY, _factor(H)
        k = 0
        for yb in (192, 224, 256) + tuple(ROWS_BANDS[1:-1]):
            for t in (-1.5, -0.6, -0.2, -0.05, -0.02, 0.02, 0.05, 0.2, 0.6, 1.5):
                x = 300 + 4 * k
                add(_needle((x + 0.3, yb + t), (0, 1), 12, 1.8, 5.0, F, W, H), {"boundary": yb, "tip": t, "dir": "down"})
                add(_needle((x + 2.6, yb + t), (0, -1), 12, 1.8, 5.0, F, W, H), {"boundary": yb, "tip": t, "dir": "up"})
                k += 1
        role = "rows"
    elif name == "small":
        # equilateral triangles at the frame centre, reference area 9.9 .. 10.9, and smaller ones with room
        W, H = 800, 450
        m, F = IDENTITY, _factor(H)
        for k, area in enumerate((5.0, 6.0, 6.5, 7.0, 7.5, 7.9, 8.5, 9.5, 9.9, 9.95, 10.0, 10.02, 10.05, 10.1, 10.3, 10.6, 10.9)):
            L = np.sqrt(2 * area / np.sqrt(3))
            cx, cy = W / 2 + 20 * (k % 6 - 3) + 0.31, H / 2 + 20 * (k // 6 - 1) + 0.17
            th = rng.uniform(0, 2 * np.pi)
            pts = [(cx + L / np.sqrt(3) * np.cos(th + j * 2 * np.pi / 3), cy + L / np.sqrt(3) * np.sin(th + j * 2 * np.pi / 3)) for j in range(3)]
            add([_camera_point(x, y, 5.0, F, W, H) for x, y in pts], {"area": area})
        role = "small"
    elif name == "oblique":
        # near both ends of a wide frame: triangles in the plane perpendicular to the view ray (their longest edge
        # projects sqrt(1 + tu^2) ~ 10 times longer than factor * L / d)
        W, H = 8192, 256
        m, F = IDENTITY, _factor(H)
        k = 0
        for xr in (30.0, W - 30.0):
            for j, (lpx, hpx) in enumerate(((9.0, 1.2), (12.0, 1.0), (16.0, 0.8), (24.0, 0.6), (40.0, 0.35), (60.0, 0.25))):
                yr = 40.0 + 34 * j
                c = _camera_point(xr, yr, 5.0, F, W, H)
                ray = c / np.linalg.norm(c)
                u = np.cross(ray, [0.0, 1.0, 0.0]); u /= np.linalg.norm(u)
                s = lpx * 5.0 / F / np.sqrt(1 + (c[0] / c[2]) ** 2)   # world length whose projection is ~lpx px
                add([c + u * s / 2, c - u * s / 2, c + np.array([0.0, hpx * 5.0 / F, 0.0])], {"px": lpx, "end": xr})
                k += 1
        role = "tangent"
    elif name == "scaled":
        # a matrix with its x row scaled by 8 and its y row sheared: world edges along x project 8 times longer
        W, H = 800, 450
        m = np.array([8, 0, 0, 0, 0.7, 1, 0, 0, 0, 0, 1, 0], np.float32)
        F = _factor(H)
        for k, (lpx, hpx) in enumerate(((9.0, 1.2), (12.0, 1.0), (16.0, 0.8), (20.0, 0.6), (24.0, 0.5))):
            cx, cy = 300 + 50 * k + 0.3, 200 + 12 * k + 0.6
            p = [_camera_point(cx - lpx / 2, cy, 5.0, F, W, H), _camera_point(cx + lpx / 2, cy, 5.0, F, W, H),
                 _camera_point(cx, cy + hpx, 5.0, F, W, H)]
            add(_tri_world(p, m), {"px": lpx})
        role = "sigma"
    elif name == "far_offset":
        # probes near |c| = 1e5 seen through a matrix whose translation cancels the offset: the transform's rounding
        # (the e term) dominates the bounds; needles across the left frame edge
        W, H = 800, 450
        m = np.array([1, 0, 0, -1e5, 0, 1, 0, 0, 0, 0, 1, 0], np.float32)
        F = _factor(H)
        for k, t in enumerate((-40, -20, -10, -6, -4, -3, -2, -1, -0.5, 0.0, 0.3, 1, 3)):
            y = 40 + 30 * k + 0.4
            p = _needle((t, y), (1, 0), 20, 1.5, 50.0, F, W, H)
            add(_tri_world(p, m), {"tip": t})
        role = "screen"
    else:
        raise KeyError(name)
    # consecutive triangles of the list go to different clusters only when they are far apart (cluster.cpp): the rungs,
    # placed in spatial order, are dealt from the two halves of the ladder in turn
    if name != "near":
        half = (len(tris) + 1) // 2
        order = [j for i in range(half) for j in (i, half + i) if j < len(tris)]
        tris, rungs = [tris[j] for j in order], [rungs[j] for j in order]
    colours = [tuple(rng.uniform(60, 255, 3)) for _ in tris]
    return W, H, m, world_scene(tris, colours), rungs, role


ROWS_BANDS = [0, 219, 235, 450]
LADDERS = ["near", "edges_narrow", "edges_wide", "rows", "small", "oblique", "scaled", "far_offset"]


def ladder_clusters(sc):
    """Cluster header of each triangle; asserts that every triangle is a cluster of its own."""
    from swift3drenderer_b200 import renderer as R
    hdr = R.debug_clusters(sc)["hdr"]
    n_tris = np.diff(hdr["tri_off"].astype(np.int64))
    assert (n_tris == 1).all(), f"{(n_tris > 1).sum()} clusters hold more than one probe"
    by_t0 = {int(h["t0"]): h for h in hdr[:-1]}
    return [by_t0[t] for t in range(sc.n_triangles)]


# ------------------------------------------------------------------------------------------------------------------
# premise checks (CPU)
# ------------------------------------------------------------------------------------------------------------------
def test_margin_scene_premises(oracle_port):
    """At least 20 (probe, tile) pairs at top-left corners and 20 at bottom-right corners of the whole frame are kept
    by the margin alone, at few-tile (count_tiles) and many-tile (bin_big_body) box sizes; at least 5 more at the
    cut tile rows of each band edge; no pair is rejected unsoundly; the general-path variant keeps every probe's pixels."""
    m = oracle_port.camera_path(still())[0]
    W, H = MARGIN_W, MARGIN_H
    small, probes = margin_scene(oracle_port, 300)
    assert small.n_triangles <= 1920
    o = oracle_port.OracleScene(small).render(m, W, H, want_winner=True, want_setups=True)
    pairs, unsound = margin_pairs(o, probes)
    assert not unsound, unsound[:5]
    tl, br = [p for p in pairs if p[1] == "tl"], [p for p in pairs if p[1] == "br"]
    assert len(tl) >= 20 and len(br) >= 20, (len(tl), len(br))
    st = o["setups"]
    row = {int(t): i for i, t in enumerate(st["order"])}
    ntiles = []
    for k, *_ in pairs:
        i = row[k]
        ntiles.append((int(st["xmax"][i]) // TILE_W - int(st["xmin"][i]) // TILE_W + 1)
                      * (int(st["ymax"][i]) // TILE_H - int(st["ymin"][i]) // TILE_H + 1))
        assert max(int(st["xmax"][i]) - int(st["xmin"][i]), int(st["ymax"][i]) - int(st["ymin"][i])) >= 16
    ntiles = np.asarray(ntiles)
    assert ((ntiles > 1) & (ntiles <= BIG_TILES)).sum() >= 3 and (ntiles > BIG_TILES).sum() >= 20, sorted(ntiles)
    # walks of over 2000 steps reach some of the pixels
    assert max(int(st["xmax"][row[k]]) - int(st["xmin"][row[k]]) + int(st["ymax"][row[k]]) - int(st["ymin"][row[k]])
               for k, *_ in pairs) > 2000
    for e in MARGIN_BANDS[1:-1]:
        j = MARGIN_BANDS.index(e)
        cut = [p for band in ((MARGIN_BANDS[j - 1], e), (e, MARGIN_BANDS[j + 1]))
               for p in margin_pairs(o, probes, band)[0] if p[3] in (e, e - 1)]
        assert len(cut) >= 5, (e, len(cut))
    big, probes2 = margin_scene(oracle_port, 2100)
    assert big.n_triangles > 1920 and probes2 == probes
    o2 = oracle_port.OracleScene(big).render(m, W, H, want_winner=True)
    won = o["winner"] < len(probes)
    assert np.array_equal(o2["winner"][won], o["winner"][won])


@pytest.mark.parametrize("name", LADDERS)
def test_ladder_premises(name, oracle_port):
    """Every rung is a cluster of its own; the float64 restatement of cluster_verdict rejects some rungs with a relative
    room of at least 1e-4 (approximate reciprocals and square roots cannot flip them) and keeps some that the oracle
    rasterizes close to the boundary; no rung the oracle rasterizes (or does not near-reject) is rejected; and for the
    oblique and scaled ladders the tangent factor resp. the Gram bound is necessary."""
    W, H, m, sc, rungs, role = ladder(name)
    hdr = ladder_clusters(sc)
    o = oracle_port.OracleScene(sc).render(m, W, H, want_setups=True)
    kept_by_oracle = set(o["setups"]["order"].tolist())
    cv, rv = oracle_port.OracleScene(sc).vertex_stage(m, W, H)
    near_by_oracle = {t for t in range(sc.n_triangles) if np.nanmax(rv[3 * t:3 * t + 3, 2]) <= K_NEAR}
    v = [verdict64(m, h, W, H) for h in hdr]
    for t, (vd, q) in enumerate(v):
        assert not (vd == 2 and t in kept_by_oracle), (t, rungs[t], q)
        assert not (vd == 1 and t not in near_by_oracle), (t, rungs[t], q)
    if role == "near":
        room = [t for t, (vd, q) in enumerate(v) if vd == 1 and q["d_max"] <= float(K_NEAR) * (1 - 1e-4)]
        close = [t for t, (vd, q) in enumerate(v) if vd == 0 and t not in near_by_oracle
                 and q["d_max"] <= float(K_NEAR) * (1 + 1e-3)]
        assert len(room) >= 3 and len(close) >= 2, (room, close)
        assert any(r["far"] == 0.0 for r in rungs) and sum(t in near_by_oracle for t in range(len(rungs))) >= 8
    elif role == "screen":
        def gap(q):   # how far the nearest frame-edge test is from rejecting (negative: rejected), in pixels
            return min(q["sx_hi"], W - q["sx_lo"])
        room = [t for t, (vd, q) in enumerate(v) if vd == 2 and gap(q) < -1e-4 * max(1.0, abs(q["sx_hi"]))]
        close = [t for t, (vd, q) in enumerate(v) if vd == 0 and t in kept_by_oracle and gap(q) <= 0.25]
        assert len(room) >= 3, room
        if name == "edges_narrow":   # near the optical axis the sphere is within a few hundredths of the tip
            assert len(close) >= 2, close
        elif name == "edges_wide":   # 400 px off the axis the sphere's depth extent loosens the bound by ~6 px
            assert any(vd == 0 and t not in kept_by_oracle for t, (vd, _) in enumerate(v))
        else:   # far_offset: the transform's rounding dominates: kept rungs sit a few pixels from the edge, the oracle still culls some
            assert any(vd == 0 and t not in kept_by_oracle for t, (vd, _) in enumerate(v))
            assert any(vd == 0 and t in kept_by_oracle for t, (vd, _) in enumerate(v))
    elif role == "rows":
        for world in (2, 3, 4):
            for phase in range(world):
                owned = lambda t: any(a % world == phase for a in range(int(o["setups"]["ymin"][t]) // TILE_H,
                                                                    int(o["setups"]["ymax"][t]) // TILE_H + 1))
                row = {int(tt): i for i, tt in enumerate(o["setups"]["order"])}
                vs = [verdict64(m, h, W, H, world=world, phase=phase) for h in hdr]
                for t, (vd, q) in enumerate(vs):
                    assert not (vd == 2 and t in row and owned(row[t])), (world, phase, t, rungs[t])
                rej = [t for t, (vd, _) in enumerate(vs) if vd == 2 and t in row]
                assert len(rej) >= 2, (world, phase)
        for y0, y1 in zip(ROWS_BANDS[:-1], ROWS_BANDS[1:]):
            vs = [verdict64(m, h, W, H, band=(y0, y1)) for h in hdr]
            kept_band = [t for t in range(len(rungs)) if t in kept_by_oracle
                         and np.max(rv[3 * t:3 * t + 3, 1]) >= y0 and np.min(rv[3 * t:3 * t + 3, 1]) < y1]
            assert all(vs[t][0] == 0 for t in kept_band)
            room = [t for t, (vd, q) in enumerate(vs) if vd == 2 and (q["sy_hi"] < y0 - 1e-4 * y0 or q["sy_lo"] >= y1 * (1 + 1e-4))]
            close = [t for t in kept_band if min(vs[t][1]["sy_hi"] - y0, y1 - vs[t][1]["sy_lo"]) <= 0.25]
            assert len(room) >= 3 and len(close) >= 1, (y0, y1, room, close)
    else:
        # too small: pixel bounds against 3.09
        room = [t for t, (vd, q) in enumerate(v) if vd == 2 and q["pixels"] <= 3.09 * (1 - 1e-4)]
        close = [t for t, (vd, q) in enumerate(v) if vd == 0 and t in kept_by_oracle and q["pixels"] <= 3.09 + 0.5]
        if role == "small":
            # the equilateral shape has the largest area for its longest edge: area >= 10 needs L >= 3.40 px, so the
            # closest a kept rung can come is L plus the slack terms (~3.46)
            assert len(room) >= 3 and len(close) >= 3, (room, close, [round(q.get("pixels", 0), 3) for _, q in v])
            assert all(v[t][1]["pixels"] <= 3.6 for t in close)
        else:
            kept = [t for t in range(len(rungs)) if t in kept_by_oracle]
            assert len(kept) >= 4, kept
            what = {"tangent": {"tangent": False}, "sigma": {"sigma": 1.0}}[role]
            needed = [t for t in kept if verdict64(m, hdr[t], W, H, **what)[0] == 2]
            assert len(needed) >= 3, (role, needed, kept)


# ------------------------------------------------------------------------------------------------------------------
# GPU: frames and statistics against the oracle
# ------------------------------------------------------------------------------------------------------------------
def _device_frame(r, m, W, H, y0=0, y1=None):
    import torch
    y1 = H if y1 is None else y1
    out = torch.full((y1 - y0, W), 0x55555555, dtype=torch.int32, device="cuda:0")
    for _ in range(4):   # a fresh renderer's first general-path frame may overflow a capacity: finish() asks for a repeat
        r.render_device(m, W, H, out.data_ptr(), y0=y0, y1=y1)
        if not r.finish():
            break
    assert r.stats()["overflow"] == 0
    return out.cpu().numpy().view(np.uint32)


def expected_part_stats(o, rv, T, band=None, world=1, phase=0):
    """(near, clipped, spawned, setups, culled, overflow) of a band or of one interleaved phase, for scenes without
    near-plane triangles: the oracle's rasterized triangles whose float rows meet the band (render.cpp:311-314 against
    [y0, y1)) resp. whose box rows meet a tile row the phase owns; everything else not near-rejected is culled."""
    st = o["setups"]
    keep = 0
    for i, t in enumerate(st["order"].tolist()):
        ys = rv[3 * t:3 * t + 3, 1]
        if band is not None and not (ys.max() >= band[0] and ys.min() < band[1]):
            continue
        if world != 1 and not any(a % world == phase for a in range(int(st["ymin"][i]) // TILE_H, int(st["ymax"][i]) // TILE_H + 1)):
            continue
        keep += 1
    near = o["stats"]["near_rejected"]
    return (near, 0, 0, keep, T - near - keep, 0)


def _got(st):
    return (st["near_rejected"], st["clipped"], st["spawned"], st["setups"], st["culled"], st["overflow"])


def _check_parts(r, renderer_lib, m, W, H, o, rv, T, what, bands, worlds, part_stats=True):
    """Bands (pixels and, when part_stats, statistics) and interleaved rows (pixels, per-phase statistics)."""
    import torch
    for y0, y1 in zip(bands[:-1], bands[1:]):
        assert_same(_device_frame(r, m, W, H, y0, y1), o["pixels"][y0:y1], f"{what}: band {y0}..{y1}")
        if part_stats:
            want = expected_part_stats(o, rv, T, band=(y0, y1))
            assert _got(r.stats()) == want, f"{what}: band {y0}..{y1} statistics {_got(r.stats())} != {want}"
    th = renderer_lib.tile_height()
    for world in worlds:
        frame = np.zeros((H, W), np.uint32)
        for phase in range(world):
            rows, frame_rows, buf_rows = renderer_lib.rows_layout(H, world, phase, th)
            if rows == 0:
                continue
            buf = torch.zeros((rows, W), dtype=torch.int32, device="cuda:0")
            for _ in range(4):
                r.render_device_rows(m, W, H, world, phase, buf.data_ptr())
                if not r.finish():
                    break
            assert r.stats()["overflow"] == 0
            if part_stats:
                want = expected_part_stats(o, rv, T, world=world, phase=phase)
                assert _got(r.stats()) == want, f"{what}: phase {phase}/{world} statistics {_got(r.stats())} != {want}"
            frame[frame_rows] = buf.cpu().numpy().view(np.uint32)[buf_rows]
        assert_same(frame, o["pixels"], f"{what}: {world} interleaved phases")


@pytest.mark.gpu
def test_tile_margin_small_scene_path(renderer_lib, oracle_port):
    """A: probes kept by the margin alone, on the fused small-scene path (tile-list collection in tile_raster), with
    span tables and without, whole frame, bands that cut tile rows, interleaved rows over 2 and 3 phases."""
    sc, _ = margin_scene(oracle_port, 300)
    W, H = MARGIN_W, MARGIN_H
    m = renderer_lib.camera_path(still())[0]
    o = oracle_port.OracleScene(sc).render(m, W, H, want_setups=True)
    rv = oracle_port.OracleScene(sc).vertex_stage(m, W, H)[1]
    r = renderer_lib.Renderer(0)
    try:
        r.load_scene(sc)
        for spans in (1, 0):
            r.set_option("spans", spans)
            what = f"margin probes, small-scene path, spans={spans}"
            assert_same(_device_frame(r, m, W, H), o["pixels"], what)
            assert_stats(r.stats(), o, what)
            assert_same(r.render(m, W, H)[0], o["pixels"], f"{what} host")
            _check_parts(r, renderer_lib, m, W, H, o, rv, sc.n_triangles, what, MARGIN_BANDS, (2, 3))
    finally:
        r.close()


@pytest.mark.gpu
def test_tile_margin_general_path(renderer_lib, oracle_port):
    """A: the same probes padded over 1920 triangles on the general path; at flat_max = 16 the few-tile probes are
    binned by count_tiles and the many-tile ones by bin_big_body.  Every routing, bands, interleaved rows."""
    sc, _ = margin_scene(oracle_port, 2100)
    W, H = MARGIN_W, MARGIN_H
    m = renderer_lib.camera_path(still())[0]
    o = oracle_port.OracleScene(sc).render(m, W, H, want_setups=True)
    rv = oracle_port.OracleScene(sc).vertex_stage(m, W, H)[1]
    r = renderer_lib.Renderer(0)
    try:
        r.load_scene(sc)
        for route in [rt for rt in ROUTES if rt[3] == 16]:
            set_route(r, route)
            what = f"margin probes, general path, route {route}"
            assert_same(_device_frame(r, m, W, H), o["pixels"], what)
            assert_stats(r.stats(), o, what)
            # (the cluster front on bands and rows: the filler's clusters are not single triangles, so only pixels and
            # the per-part statistics, which do not depend on how triangles were grouped)
            _check_parts(r, renderer_lib, m, W, H, o, rv, sc.n_triangles, what, MARGIN_BANDS, (2, 3))
    finally:
        r.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", LADDERS)
def test_cluster_ladders(name, renderer_lib, oracle_port):
    """B: each ladder on the general path with the cluster front and cluster rejection, the cluster front without
    rejection, and no cluster front: whole frame (pixels and statistics), bands and interleaved rows over 2, 3 and 4
    phases (pixels, and statistics where the ladder has no near-plane triangle)."""
    W, H, m, sc, _, _ = ladder(name)
    osc = oracle_port.OracleScene(sc)
    o = osc.render(m, W, H, want_setups=True)
    rv = osc.vertex_stage(m, W, H)[1]
    bands = ROWS_BANDS if name == "rows" else [0, H // 3 + 5, (2 * H) // 3 + 1, H]
    r = renderer_lib.Renderer(0)
    try:
        r.set_option("fused_small", 0)
        r.load_scene(sc)
        for c, cc in ((1, 1), (1, 0), (0, 0)):
            r.set_option("clusters", c)
            r.set_option("cluster_cull", cc)
            what = f"ladder {name} {W}x{H} clusters={c} cluster_cull={cc}"
            assert_same(_device_frame(r, m, W, H), o["pixels"], what)
            assert_stats(r.stats(), o, what)
            _check_parts(r, renderer_lib, m, W, H, o, rv, sc.n_triangles, what, bands, (2, 3, 4),
                         part_stats=name != "near")
    finally:
        r.close()
