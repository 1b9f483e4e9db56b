"""Per-corner attributes against the oracle, bit for bit: smooth normals and per-corner texture indices through the
near-plane clip, on every shading path.  Frames, statistics and setup records.

A triangle whose three corners carry the same normal is shaded with N * (sum of b_k / z_k), and unit() removes the
scale: a wrong corner, a wrong 1/z or a swapped blend then moves a colour by its last bit at most.  A triangle whose
corners name the same atlas cannot show which corner the clipper took the index from.  The scenes here give every
corner its own normal and every textured corner its own atlas:
  * hash atlases: every texel of the four atlases is a distinct colour with all channels >= 64, so a wrong atlas, level
    or texel always changes the colour (a box-filtered atlas has equal neighbours);
  * smooth-normal probes: colour triangles with one colour and three normals — tilted up to ~60 degrees apart, of
    lengths 1, 0.05 and 20 (the reference blends raw normals and normalises afterwards), an opposite pair whose blend
    passes through zero inside the triangle, and lengths 2^-55 and 2^55 (inv_sqrt_rn's fallback outside
    [2^-100, 2^100], csrc/exact_math.cuh) — at depths that differ per corner, with boxes under 16 px (record-free),
    16..127 px (flat walk) and 128 px and more (tile kernel);
  * clip probes: triangles through the near plane z = -0.1 in all six arrangements (one corner in front at position
    0, 1 or 2; two in front with the behind corner at 0, 1 or 2, which appends a triangle), each as (a) a textured
    triangle with three distinct atlases and normals, (b) a colour triangle with distinct colours and normals and (c) a
    colour corner 0 with texture records at the other corners, whose words the clipper lerps as colour (hazard H5);
  * filler for the general path: 2 000 small triangles of both kinds with per-corner normals, colours and atlases.
A vertex the clipper makes on edge a -> b takes a's texture index (render.cpp:233), and the setup takes the index of
whatever lies at position 0 afterwards, so a clipped triangle can sample another atlas than its corner 0 named; the
CPU tests restate that bookkeeping (render.cpp:212-262) in Python, check it against the oracle's setup records and
show from the oracle alone that every probe reaches what it exists for.

Not built here, and outside the parity contract: a textured corner 0 with colour records at corners the clipper
interpolates from.  The made vertex would then carry a colour word as its texture index; the reference reads outside
its atlases with it, while the kernels take the index modulo the atlas count (make_setup)."""
import functools

import numpy as np
import pytest

from swift3drenderer_b200 import scene as S
from test_gpu_vis_edges import KSCALE, ROUTES, assert_same, assert_stats, render_rows, restore_defaults, set_route, still

W, H = 960, 540
N_TEX = 4
GUARD_LO, GUARD_HI = 2.0 ** -100, 2.0 ** 100      # inv_sqrt_rn's fast range, csrc/exact_math.cuh
SHAPES = ("tilt", "lengths", "opposite", "tiny", "huge")
SIZES = {"small": 10, "mid": 3, "large": 1}        # smooth probes per shape and size class
ARRANGEMENTS = [("one", 0), ("one", 1), ("one", 2), ("two", 0), ("two", 1), ("two", 2)]   # (corners in front, position)
FORMS = ("tex", "col", "mixed")
N_FILLER = 2000


@functools.lru_cache(maxsize=None)
def hash_atlases(n=N_TEX):
    """n 512 x 512 atlases in which every texel is a distinct colour 0x00RRGGBB with every channel in 64..255:
    texel i gets colour number (i * 2654435761 + 12345) mod 192^3 (the multiplier is prime to 2 and 3: a bijection)."""
    i = np.arange(n << 18, dtype=np.int64)
    k = (i * 2654435761 + 12345) % 192 ** 3
    r, g, b = 64 + k // (192 * 192), 64 + (k // 192) % 192, 64 + k % 192
    return ((r << 16) | (g << 8) | b).astype(np.uint32).reshape(n, S.ATLAS, S.ATLAS)


def front_flags(arrangement):
    many, pos = arrangement
    return tuple((k == pos) if many == "one" else (k != pos) for k in range(3))


def clip_bookkeeping(front):
    """render.cpp:212-262 for corners in front of the near plane (``front``): the corners of the in-place triangle and
    of the appended one (None when one corner is in front), as (source corner, made) per position.  A vertex made on
    edge i -> i + 1 carries corner i's texture index (render.cpp:233)."""
    made, cur, nxt, pre, two = {}, 0, 0, 0, False
    for i in range(3):
        j = (i + 1) % 3
        if front[i] == front[j]:
            cur, nxt, pre, two = i, j, (i + 2) % 3, front[i]
        else:
            made[i] = (i, True)
    d = [(0, False), (1, False), (2, False)]
    if not two:
        d[cur], d[nxt] = made[pre], made[nxt]
        return d, None
    d[pre] = made[nxt]
    return d, [(cur, False), made[nxt], made[pre]]


class _Builder:
    """Triangles given by raster corners of the W x H frame seen by the still camera, a depth per corner and a
    48-byte attribute record per corner.  Corner order is kept as given (the clip arrangements depend on it)."""

    def __init__(self):
        self.factor = 0.1 * H / (2 * KSCALE)   # render.cpp:279
        self.v, self.at, self.info = [], [], []

    def tri(self, pts, depth, attrs, info):
        for (x, y), z in zip(np.asarray(pts, np.float64), np.asarray(depth, np.float64)):
            self.v.append(((x - W / 2) * z / self.factor, -(y - H / 2) * z / self.factor, -z))
        self.at.extend(attrs)
        self.info.append(info)
        return len(self.info) - 1

    def scene(self):
        n = len(self.info)
        v = np.ones((3 * n, 4), "<f4")
        v[:, :3] = np.asarray(self.v, np.float64).reshape(-1, 3)
        at = np.array(self.at, S.ATTR_DTYPE)
        idx = np.arange(3 * n, dtype="<u8")
        return S.Scene(v, idx, at, idx.copy(), hash_atlases())


def _oriented(pts):
    """Raster corners wound so that the reference's area is positive: corners 1 and 2 trade places (only their
    positions: depths and records stay with the corner index)."""
    p = np.asarray(pts, np.float64)
    area = (p[2, 0] - p[0, 0]) * (p[0, 1] - p[1, 1]) + (p[2, 1] - p[0, 1]) * (p[1, 0] - p[0, 0])
    return p[[0, 2, 1]] if area < 0 else p


def _tilted(rng, n=3, lo=15.0, hi=32.0):
    """n unit normals facing the camera (+z), tilted lo..hi degrees off the axis at azimuths about 120 degrees apart."""
    phi0 = rng.uniform(0, 2 * np.pi)
    out = []
    for k in range(n):
        th, ph = np.radians(rng.uniform(lo, hi)), phi0 + 2 * np.pi * k / n + rng.uniform(-0.3, 0.3)
        out.append(np.array([np.sin(th) * np.cos(ph), np.sin(th) * np.sin(ph), np.cos(th)]))
    return out


def _normals(shape, rng, k):
    if shape == "tilt":
        return _tilted(rng)
    if shape == "lengths":
        lengths = np.roll([1.0, 0.05, 20.0], k)
        return [n * s for n, s in zip(_tilted(rng), lengths)]
    if shape == "opposite":   # n1 = -n0, n2 parallel to n0: the blend is a multiple of n0 that changes sign inside
        v = _tilted(rng, 1)[0]
        return [v, -v, rng.uniform(0.3, 2.0) * v]
    return [n * 2.0 ** (-55 if shape == "tiny" else 55) for n in _tilted(rng)]


def _cell_tri(rng, x0, y0, sx, sy):
    """A triangle spanning about sx by sy pixels from (x0, y0), corners jittered."""
    return [(x0 + rng.uniform(0, 2), y0 + rng.uniform(0, 2)), (x0 + sx - rng.uniform(0, 2), y0 + rng.uniform(0, 0.3 * sy)),
            (x0 + rng.uniform(0, 0.3 * sx), y0 + sy - rng.uniform(0, 2))]


def _rgb(rng):
    return tuple(rng.uniform(60, 255, 3))


def _smooth_probes(b, rng):
    """Large probes in the top row (5 cells of 192 x 180 px), mid probes below (15 cells of 64 x 64 px), small probes in
    a row of 50 cells of 19 x 19 px; per corner depths 2, 3 and 4.5 in some order."""
    cells = {"large": [(4 + 192 * i, 4, 184, 174) for i in range(5)],
             "mid": [(4 + 64 * i, 190, rng.uniform(22, 58), rng.uniform(22, 58)) for i in range(15)],
             "small": [(4 + 19 * i, 258, rng.uniform(9, 13.5), rng.uniform(9, 13.5)) for i in range(50)]}
    for size, per in SIZES.items():
        for j, (x0, y0, sx, sy) in enumerate(cells[size]):
            shape = SHAPES[j // per]
            pts = _oriented(_cell_tri(rng, x0, y0, sx, sy))
            depth = rng.permutation([2.0, 3.0, 4.5]) * rng.uniform(0.9, 1.1)
            col = _rgb(rng)
            attrs = [S.color_attr(n, col) for n in _normals(shape, rng, j)]
            b.tri(pts, depth, attrs, {"what": "smooth", "shape": shape, "size": size})


def _behind_corners_out(pts, depth, front):
    """Moves each behind corner's raster position away from the corners in front so that the near plane cuts its
    edges near where the corner was: the point at depth 0.1 on the edge from a corner in front (raster p, depth
    df) to a behind one (raster q, depth db) projects to p + w (q - p), w = db (0.1 - df) / (0.1 (db - df)).  Exact
    with one corner in front; with two, about (w averaged over both edges, from the middle of the front edge)."""
    p = np.array(pts, np.float64)
    fronts = [k for k in range(3) if front[k]]
    centre = p[fronts].mean(0)
    for k in range(3):
        if not front[k]:
            w = np.mean([depth[k] * (0.1 - depth[f]) / (0.1 * (depth[k] - depth[f])) for f in fronts])
            p[k] = centre + (p[k] - centre) / w
    return p


def _clip_probes(b, rng):
    """6 arrangements x 3 forms x 2 sizes in 12 x 3 cells of 80 x 78 px below the smooth probes.  Corners in front lie
    at depth 1.2..3 (in the smaller probes the first of them at 0.13..0.19), behind ones at 0.03..0.07, their raster
    positions moved out so that the clipped pieces fill about the triangle drawn in the cell."""
    cells = [(2 + 80 * (i % 12), 300 + 80 * (i // 12)) for i in range(36)]
    k = 0
    for arrangement in ARRANGEMENTS:
        front = front_flags(arrangement)
        for form in FORMS:
            for scale in (1.0, 0.6):
                x0, y0 = cells[k]
                pts = _oriented(_cell_tri(rng, x0, y0, 76 * scale, 74 * scale))
                depth = [rng.uniform(1.2, 3.0) if f else rng.uniform(0.03, 0.07) for f in front]
                if scale < 1:   # the first corner in front lies just beyond the plane: a step forward changes the arrangement
                    depth[front.index(True)] = rng.uniform(0.13, 0.19)
                pts = _behind_corners_out(pts, depth, front)
                normals = [n * s for n, s in zip(_tilted(rng), rng.uniform(0.5, 2.0, 3))]
                tex = rng.permutation(N_TEX)[:3] if form != "col" else None
                uv = rng.uniform(0.0, 3.0, (3, 2))
                if form == "tex":
                    attrs = [S.texture_attr(n, int(t), c) for n, t, c in zip(normals, tex, uv)]
                elif form == "col":
                    attrs = [S.color_attr(n, _rgb(rng)) for n in normals]
                else:
                    attrs = [S.color_attr(normals[0], _rgb(rng))] + [S.texture_attr(n, int(t), c) for n, t, c in zip(normals[1:], tex[1:], uv[1:])]
                b.tri(pts, depth, attrs, {"what": "clip", "arrangement": arrangement, "form": form,
                                          "tex": None if tex is None else [int(t) for t in tex]})
                k += 1


def _filler(b, rng, n):
    """Small camera-facing triangles behind every probe, both kinds, per-corner normals, colours and atlases."""
    for k in range(n):
        x, y = rng.uniform(-6, W), rng.uniform(-6, H)
        pts = _oriented(_cell_tri(rng, x, y, rng.uniform(5, 14), rng.uniform(5, 14)))
        depth = rng.uniform(8, 20) + rng.uniform(0, 0.5, 3)
        normals = _tilted(rng)
        if k % 2:
            tex = rng.permutation(N_TEX)[:3]
            attrs = [S.texture_attr(nn, int(t), c) for nn, t, c in zip(normals, tex, rng.uniform(0, 4, (3, 2)))]
        else:
            attrs = [S.color_attr(nn, _rgb(rng)) for nn in normals]
        b.tri(pts, depth, attrs, {"what": "filler"})


@functools.lru_cache(maxsize=None)
def probe_scene(filler=False):
    """(scene, info): info[k] says what triangle k is for.  The probes come first, so their indices do not depend on
    whether the filler follows."""
    b = _Builder()
    _smooth_probes(b, np.random.RandomState(3))
    _clip_probes(b, np.random.RandomState(4))
    if filler:
        _filler(b, np.random.RandomState(5), N_FILLER)
    return b.scene(), tuple(b.info)


def views(oracle_port):
    """Still, a small turn, a step back (every corner comes in front: nothing is clipped) and a step forward with a
    turn (the smaller clip probes' first corner in front goes behind: their arrangements change)."""
    out = [oracle_port.camera_path(still())[0]]
    for rec in ({"mouse": (4.0, -3.0)}, {"down": 1.0}, {"up": 1.0, "mouse": (-5.0, 2.0)}):
        inp = np.zeros(1, S.INPUT_DTYPE)
        for key, value in rec.items():
            inp[0][key] = value
        out.append(oracle_port.camera_path(inp)[0])
    return np.stack(out)


def skewed():
    """A non-orthonormal view: the x row scaled, the y row sheared (normals come out neither unit nor orthogonal)."""
    m = np.array([1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0], np.float64).reshape(3, 4)
    m[0, :3] *= 1.25
    m[1, :3] += 0.3 * m[0, :3]
    return m.reshape(12).astype(np.float32)


def indices(info, **want):
    return [k for k, i in enumerate(info) if all(i.get(a) == v for a, v in want.items())]


# ------------------------------------------------------------------------------------------------------------------
# float64 restatement of the shading of one colour triangle (exact barycentrics at pixel centres)
# ------------------------------------------------------------------------------------------------------------------
def _unit(a):
    return a / np.sqrt((a * a).sum(-1, keepdims=True))


def shade64(cv, rv, n, col, xs, ys):
    """Colour of the pixels (xs, ys) of a colour triangle with camera-space corners cv, raster corners rv, camera-space
    normals n and one colour col, in float64: (colour as (k, 3) levels, blended normals)."""
    (x0, y0, _), (x1, y1, _), (x2, y2, _) = rv
    px, py = xs + 0.5, ys + 0.5
    area = (x2 - x0) * (y0 - y1) + (y2 - y0) * (x1 - x0)
    w = np.stack([((px - x1) * (y1 - y2) + (py - y1) * (x2 - x1)) / area,
                  ((px - x2) * (y2 - y0) + (py - y2) * (x0 - x2)) / area,
                  ((px - x0) * (y0 - y1) + (py - y0) * (x1 - x0)) / area], -1)
    rvz = 1.0 / rv[:, 2]
    b = w / (w @ rvz)[:, None]
    point = -_unit(b @ (cv * rvz[:, None]))
    nb = b @ (n * rvz[:, None])
    normal = _unit(nb)
    shade = (_unit(point + normal) * normal).sum(-1)
    return np.floor(shade[:, None] * np.asarray(col)[None, :]), nb


# ------------------------------------------------------------------------------------------------------------------
# premise checks (CPU)
# ------------------------------------------------------------------------------------------------------------------
def test_hash_atlases_and_texture_indices(oracle_port):
    """Every texel is distinct, every channel >= 64; every setup the oracle makes names an atlas that exists."""
    tx = hash_atlases()
    assert tx.shape == (N_TEX, S.ATLAS, S.ATLAS) and len(np.unique(tx)) == tx.size
    assert min(int((tx >> s & 255).min()) for s in (0, 8, 16)) >= 64
    sc, _ = probe_scene(True)
    assert not S.validate(sc) and 2 * sc.n_triangles > 3840 and 2 * probe_scene()[0].n_triangles <= 3840
    for m in list(views(oracle_port)) + [skewed()]:
        st = oracle_port.OracleScene(sc).render(m, W, H, want_setups=True)["setups"]
        assert (st["texture"][st["kind"] == 1] < N_TEX).all()


def _clip_render(oracle_port, sc):
    m = oracle_port.camera_path(still())[0]
    return oracle_port.OracleScene(sc).render(m, W, H, want_setups=True, want_winner=True)


def test_clip_probes_show_both_pieces(oracle_port):
    """Every arrangement x form has visible pixels of the in-place triangle and, with two corners in front, of the
    appended one (order T + parent); the oracle clips and appends exactly the probes that straddle the plane."""
    sc, info = probe_scene()
    T = sc.n_triangles
    o = _clip_render(oracle_port, sc)
    win, st = o["winner"], o["setups"]
    clip = indices(info, what="clip")
    assert o["stats"]["clipped"] == len(clip) and o["stats"]["spawned"] == len(clip) // 2
    for arrangement in ARRANGEMENTS:
        for form in FORMS:
            for t in indices(info, what="clip", arrangement=arrangement, form=form):
                assert (win == t).sum() >= 50, (arrangement, form, t)
                if arrangement[0] == "two":
                    assert (win == T + t).sum() >= 50, (arrangement, form, t)
                    assert T + t in st["order"]
                else:
                    assert T + t not in st["order"]


def test_clip_texture_indices_follow_the_restated_bookkeeping(oracle_port):
    """A Python restatement of render.cpp:212-262 predicts the texture index of every clipped and appended textured
    probe, and the oracle's setup records agree.  Where a made vertex lands at position 0 and carries another corner's
    index — one corner in front at position 2, two in front with the behind corner at 0 (both pieces) or at 1 (the
    appended piece) — the probe's visible pixels use another atlas than its corner 0 named."""
    sc, info = probe_scene()
    T = sc.n_triangles
    o = _clip_render(oracle_port, sc)
    st, win = o["setups"], o["winner"]
    row = {int(t): i for i, t in enumerate(st["order"])}
    moved = set()
    for t in indices(info, what="clip", form="tex"):
        arrangement, tex = info[t]["arrangement"], info[t]["tex"]
        in_place, appended = clip_bookkeeping(front_flags(arrangement))
        for order, corners in ((t, in_place), (T + t, appended)):
            if corners is None:
                continue
            src, made = corners[0]
            assert int(st["texture"][row[order]]) == tex[src], (arrangement, order)
            if tex[src] != tex[0]:
                assert (win == order).sum() >= 50
                moved.add((arrangement, order >= T, made))
    # (the appended piece of ("two", 1) starts at original corner 2; the others at a made vertex)
    assert moved == {(("one", 2), False, True), (("two", 0), False, True), (("two", 0), True, False),
                     (("two", 1), True, False)}, moved


def _with_attrs(sc, edit):
    at = sc.attributes.copy()
    edit(at.reshape(-1, 3))
    return S.Scene(sc.vertices, sc.vertex_indices, at, sc.attribute_indices, sc.textures)


def test_ablations_change_the_probes(oracle_port):
    """The scene makes each rule visible: corner 0's normal on every corner changes most smooth-probe pixels, and in
    every textured clip arrangement both a single atlas the probe did not name and corner 0's atlas on every corner
    change pixels — the latter exactly where the bookkeeping moves another corner's index to position 0."""
    sc, info = probe_scene()
    T = sc.n_triangles
    osc = oracle_port.OracleScene(sc)
    m = oracle_port.camera_path(still())[0]
    o = osc.render(m, W, H, want_winner=True)
    win = o["winner"]

    def flat_normals(at):
        at["normal"][:] = at["normal"][:, :1]
    smooth = np.isin(win, indices(info, what="smooth"))
    changed = oracle_port.OracleScene(_with_attrs(sc, flat_normals)).render(m, W, H)["pixels"] != o["pixels"]
    assert changed[smooth].mean() >= 0.3, changed[smooth].mean()
    for shape in SHAPES:
        mine = np.isin(win, indices(info, what="smooth", shape=shape))
        assert changed[mine].mean() >= 0.15, (shape, changed[mine].mean())

    tex_probes = indices(info, what="clip", form="tex")

    def retexture(pick):
        def edit(at):
            for t in tex_probes:
                at["payload"][t, :, 0] = pick(info[t]["tex"])
        return oracle_port.OracleScene(_with_attrs(sc, edit)).render(m, W, H)["pixels"] != o["pixels"]
    unused = retexture(lambda tex: (set(range(N_TEX)) - set(tex)).pop())
    first = retexture(lambda tex: tex[0])
    for t in tex_probes:
        arrangement = info[t]["arrangement"]
        in_place, appended = clip_bookkeeping(front_flags(arrangement))
        for order, corners in ((t, in_place), (T + t, appended)):
            if corners is None:
                continue
            assert unused[win == order].any(), (arrangement, order)
            assert first[win == order].any() == (corners[0][0] != 0), (arrangement, order)


def test_normal_blend_in_float64(oracle_port):
    """The colour of the smooth probes follows the blend of the raw corner normals: a float64 evaluation (exact
    barycentrics from the oracle's raster vertices) is within one level of the oracle at every pixel away from the
    opposite probes' zero line, and equal at most; the 2^-55 and 2^55 probes put dot(n, n) at least 2^4 outside
    inv_sqrt_rn's guard at every shaded pixel; the opposite probes' blend changes sign inside the visible triangle."""
    sc, info = probe_scene()
    m = oracle_port.camera_path(still())[0]
    osc = oracle_port.OracleScene(sc)
    o = osc.render(m, W, H, want_winner=True)
    cv, rv = osc.vertex_stage(m, W, H)
    a = np.asarray(m, np.float64).reshape(3, 4)
    total = exact = 0
    for t in indices(info, what="smooth"):
        ys, xs = np.nonzero(o["winner"] == t)
        assert len(ys) >= 10, (info[t], len(ys))
        n = sc.attributes["normal"][3 * t:3 * t + 3, :3].astype(np.float64) @ a[:, :3].T
        col = sc.attributes["payload"][3 * t, :3].view("<f4").astype(np.float64)
        want, nb = shade64(cv[3 * t:3 * t + 3].astype(np.float64), rv[3 * t:3 * t + 3].astype(np.float64), n, col, xs, ys)
        got = np.stack([(o["pixels"][ys, xs] >> s) & 255 for s in (16, 8, 0)], -1).astype(np.float64)
        shape = info[t]["shape"]
        dot = (nb * nb).sum(-1)
        if shape == "tiny":
            assert dot.max() <= GUARD_LO / 16, (t, dot.max())
        if shape == "huge":
            assert dot.min() >= GUARD_HI * 16, (t, dot.min())
        keep = np.ones(len(ys), bool)
        if shape == "opposite":
            s = nb @ n[0]
            assert (s > 0).any() and (s < 0).any(), t
            keep = np.abs(s) > 1e-3 * np.abs(s).max()
        diff = np.abs(got[keep] - want[keep])
        assert diff.max() <= 1, (info[t], diff.max())
        total += diff.size
        exact += (diff == 0).sum()
    assert exact >= 0.9 * total, (exact, total)


def test_smooth_probe_routes(oracle_port):
    """Every shape has boxes under 16 px, 16..127 px and 128 px or more."""
    sc, info = probe_scene()
    st = _clip_render(oracle_port, sc)["setups"]
    big = np.maximum(st["xmax"].astype(np.int64) - st["xmin"], st["ymax"].astype(np.int64) - st["ymin"])
    box = dict(zip(st["order"].tolist(), big.tolist()))
    for shape in SHAPES:
        sizes = [box[t] for t in indices(info, what="smooth", shape=shape)]
        assert min(sizes) < 16 and any(16 <= s < 128 for s in sizes) and max(sizes) >= 128, (shape, sorted(sizes))


def test_views_change_the_arrangements(oracle_port):
    """The batch's step back leaves nothing to clip; its step forward near-rejects the smaller one-in-front probes
    and turns the smaller two-in-front probes into one-in-front ones (fewer appended triangles)."""
    sc, info = probe_scene()
    osc = oracle_port.OracleScene(sc)
    st = [osc.render(m, W, H)["stats"] for m in views(oracle_port)]
    n = len(indices(info, what="clip"))
    assert (st[0]["clipped"], st[0]["spawned"], st[0]["near_rejected"]) == (n, n // 2, 0)
    assert st[1]["clipped"] == n and st[2]["clipped"] == 0
    assert st[3]["near_rejected"] == n // 4 and st[3]["spawned"] == n // 4 and st[3]["clipped"] == 3 * n // 4


# ------------------------------------------------------------------------------------------------------------------
# GPU: setup records, frames and statistics against the oracle
# ------------------------------------------------------------------------------------------------------------------
def assert_same_setups(got, want, what):
    assert len(got) == len(want), f"{what}: {len(got)} setups != oracle {len(want)}"
    for field in want.dtype.names:
        g, w = got[field].view(np.uint32), want[field].view(np.uint32)
        if not np.array_equal(g, w):
            bad = np.nonzero((g != w).reshape(len(want), -1).any(1))[0]
            raise AssertionError(f"{what}: field {field} differs in {len(bad)} setups, first order {want['order'][bad[0]]}: "
                                 f"{got[field][bad[0]]} != oracle {want[field][bad[0]]}")


@pytest.mark.gpu
def test_setup_records_equal_the_oracle(renderer_lib, oracle_port):
    """Every field of every setup record, as bits — corner normals / z, texture index, payload, dz, tpp — on the
    small-scene path (probes alone) and on the general path with every survivor recorded (probes and filler), for
    the still view and a scaled and sheared one (normals are transformed with w = 0 and not renormalised)."""
    for filler in (False, True):
        sc, _ = probe_scene(filler)
        osc = oracle_port.OracleScene(sc)
        r = renderer_lib.Renderer(0)
        try:
            r.load_scene(sc)
            r.set_option("direct_small", 0)
            for name, m in (("still", oracle_port.camera_path(still())[0]), ("skewed", skewed())):
                what = f"{'general' if filler else 'small-scene'} path, {name} view"
                o = osc.render(m, W, H, want_setups=True)
                assert_same(r.render(m, W, H)[0], o["pixels"], what)
                assert_stats(r.stats(), o, what)
                assert_same_setups(r.setups(), o["setups"], what)
        finally:
            r.close()


@pytest.mark.gpu
def test_small_scene_path(renderer_lib, oracle_port):
    """The probes alone (fused geometry, tile_raster): whole frame, a band that cuts tile rows, 3 interleaved phases and
    a batch of 4 views, span tables on and off."""
    sc, _ = probe_scene()
    osc = oracle_port.OracleScene(sc)
    vs = views(oracle_port)
    want = [osc.render(m, W, H) for m in vs]
    y0, y1 = 45, 301
    r = renderer_lib.Renderer(0)
    try:
        r.load_scene(sc)
        for spans in (1, 0):
            r.set_option("spans", spans)
            what = f"small-scene path, spans={spans}"
            assert_same(r.render(vs[0], W, H)[0], want[0]["pixels"], what)
            assert_stats(r.stats(), want[0], what)
            assert_same(r.render(vs[0], W, H, y0=y0, y1=y1)[0], want[0]["pixels"][y0:y1], f"{what}: band {y0}..{y1}")
            assert_same(render_rows(r, renderer_lib, vs[0], W, H, 3), want[0]["pixels"], f"{what}: 3 interleaved phases")
            got = r.render(vs, W, H)
            for k, o in enumerate(want):
                assert_same(got[k], o["pixels"], f"{what}: batch view {k}")
                assert_stats(r.stats(k), o, f"{what}: batch view {k}")
    finally:
        r.close()


@pytest.mark.gpu
def test_general_path_every_route(renderer_lib, oracle_port):
    """Probes and filler on the general path (record-free direct walks, the flat walk, the tile kernel, shade_tiles
    staging from records and from the raw scene) under every routing: whole frame, 2 bands, 3 interleaved phases, a
    batch of 4 views and a 1283 x 721 frame."""
    sc, _ = probe_scene(True)
    osc = oracle_port.OracleScene(sc)
    vs = views(oracle_port)
    want = [osc.render(m, W, H) for m in vs]
    W2, H2 = 1283, 721
    big = osc.render(vs[0], W2, H2)
    bands = [0, 203, H]
    r = renderer_lib.Renderer(0)
    try:
        r.load_scene(sc)
        for route in ROUTES:
            set_route(r, route)
            what = f"general path clusters={route[0]} cull={route[1]} direct_small={route[2]} flat_max={route[3]}"
            assert_same(r.render(vs[0], W, H)[0], want[0]["pixels"], what)
            assert_stats(r.stats(), want[0], what)
            parts = [r.render(vs[0], W, H, y0=a, y1=b)[0] for a, b in zip(bands[:-1], bands[1:])]
            assert_same(np.concatenate(parts, 0), want[0]["pixels"], f"{what}: bands {bands}")
            assert_same(render_rows(r, renderer_lib, vs[0], W, H, 3), want[0]["pixels"], f"{what}: 3 interleaved phases")
            got = r.render(vs, W, H)
            for k, o in enumerate(want):
                assert_same(got[k], o["pixels"], f"{what}: batch view {k}")
                assert_stats(r.stats(k), o, f"{what}: batch view {k}")
            assert_same(r.render(vs[0], W2, H2)[0], big["pixels"], f"{what}: {W2}x{H2}")
            assert_stats(r.stats(), big, f"{what}: {W2}x{H2}")
    finally:
        restore_defaults(r)
        r.close()
