"""Edge cases of the general (visibility-buffer) path against the oracle, bit for bit, frames and statistics.

The general path resolves visibility in several kernels that must agree with each other and with the reference's
strict '>' depth test (render.cpp:364): record-free direct walks (raw-stream classify or the cluster front's queue),
the flat walk of post_setup and the tile kernel all publish 64-bit keys depth << 32 | ~order, and shade_tiles stages
the winners of each 32 x 16 block in passes of 96 setups.  The scenes here are built so that each of those paths is
reached on purpose — exact depth ties between copies far apart in list order, blocks with more than 96 and 192
distinct winners, boxes on the routing thresholds and the frame border, capacity overflows — and the CPU tests at
the top prove from the oracle alone that every scene reaches what it exists for.  Every GPU test runs under the
routings that can disagree: cluster front on/off (with and without cluster rejection), record-free small triangles
on/off and three flat-walk limits."""
import numpy as np
import pytest

from swift3drenderer_b200 import scene as S

BG = 0x1E1E1E
NO_WINNER = 0xFFFFFFFF
KSCALE = float.fromhex("0x1.0a2c9ap-5")   # near * tan(fov / 2), render.cpp:81-97
ROUTES = [(c, cc, ds, fm) for c, cc in ((0, 0), (1, 0), (1, 1)) for ds in (1, 0) for fm in (16, 128, 4096)]
SHADE_TRIS = 96            # setups shade_tiles stages per pass (32 x 16 blocks)
BLOCK_W, BLOCK_H = 32, 16

_textures = []


def textures():
    if not _textures:
        _textures.append(S.procedural_textures(2))
    return _textures[0]


def still():
    """The initial camera: camera space is world space, so scene coordinates (z = -0.1 included) stay exact."""
    return S.input_script("still", 1)


# ------------------------------------------------------------------------------------------------------------------
# scene builders: triangles placed in raster space of a W x H frame seen by the still camera
# ------------------------------------------------------------------------------------------------------------------
class _Mesh:
    def __init__(self, W, H):
        self.W, self.H = W, H
        self.factor = 0.1 * H / (2 * KSCALE)   # render.cpp:279
        self.v, self.col = [], []

    def tri(self, pts, depth, rgb):
        """Adds one colour triangle with raster corners ``pts`` (3 x 2) at distances ``depth`` (scalar or 3); returns
        its index.  The corners are wound so that the reference's area is positive."""
        p = np.asarray(pts, np.float64)
        d = np.broadcast_to(np.asarray(depth, np.float64), (3,))
        area = (p[2, 0] - p[0, 0]) * (p[0, 1] - p[1, 1]) + (p[2, 1] - p[0, 1]) * (p[1, 0] - p[0, 0])
        if area < 0:
            p, d = p[[0, 2, 1]], d[[0, 2, 1]]
        for (x, y), z in zip(p, d):
            self.v.append(((x - self.W / 2) * z / self.factor, -(y - self.H / 2) * z / self.factor, -z))
        self.col.append(rgb)
        return len(self.col) - 1

    def scene(self):
        n = len(self.col)
        v = np.ones((3 * n, 4), "<f4")
        v[:, :3] = np.asarray(self.v, np.float64).reshape(-1, 3)
        at = np.zeros(n, S.ATTR_DTYPE)
        at["normal"][:, 2] = 1.0
        at["payload"][:, :3] = np.asarray(self.col, "<f4").view("<u4")
        return S.Scene(v, np.arange(3 * n, dtype="<u8"), at, np.repeat(np.arange(n, dtype="<u8"), 3), textures())


def _right_tri(x0, y0, sx, sy, rng, skew=3.0):
    """A triangle with its box corner at (x0, y0), about sx by sy pixels, edges slightly skewed."""
    return [(x0, y0), (x0 + sx, y0 + rng.uniform(0, skew)), (x0 + rng.uniform(0, skew), y0 + sy)]


TIE_NEED = {"small": 1, "mid": 1, "large": 1, "coplanar": 3, "small_first": 3, "large_first": 3}   # exact ties per site


def tie_pixels(sc, sites, osc_of, m, W, H):
    """Per tie site, the pixels its later copy reaches at exactly the depth of its earlier copy, which wins them by
    list order alone: the winner of the scene is the earlier copy, and with every earlier copy collapsed to a point
    (culled, list order unchanged) the winner is the later copy at bit-identical depth."""
    first = np.array([a for _, a, _ in sites])
    later = np.array([b for _, _, b in sites])
    without = S.Scene(sc.vertices, sc.vertex_indices.copy(), sc.attributes, sc.attribute_indices, sc.textures)
    vi = without.vertex_indices.reshape(-1, 3)
    vi[first] = vi[first][:, :1]
    o1 = osc_of(sc).render(m, W, H, want_winner=True, want_depth=True)
    o2 = osc_of(without).render(m, W, H, want_winner=True, want_depth=True)
    site_of = np.full(sc.n_triangles + 1, -1)
    site_of[first] = np.arange(len(sites))
    w1, w2 = o1["winner"], o2["winner"]
    s = site_of[np.minimum(w1, sc.n_triangles)]
    tied = (s >= 0) & (w2 == later[np.maximum(s, 0)]) & (o1["depth"].view(np.uint32) == o2["depth"].view(np.uint32))
    return np.bincount(s[tied], minlength=len(sites)), tied, o1, o2


def tie_field(oracle_port, W=800, H=450):
    """Tie sites: the same triangle twice, the copies in the first and the second half of the list (different
    clusters, walk rounds, CTAs and kernels), the second copy a different colour and either identical or with its
    corners rotated (v1, v2, v0 or v2, v0, v1: the depths may round differently).  Boxes under 16 px (record-free),
    16..127 px (flat walk) and 128 px and more (tile kernel), flat and slanted; small-and-large coplanar pairs in both
    orders, whose two triangles take different kernels; partly overlapping coplanar triangles at constant z.
    hazard_scene() follows, so its near-plane vertices, slivers, corner-0 kinds and constant uv run through the
    cluster front too.  The sites avoid the part of the frame that the hazard scene's near triangles cover (x 50..409).

    Whether two different triangles reach a pixel at the same binary32 depth depends on roundings no simple rule
    predicts, so the sites are settled against the oracle: a site whose copies tie at fewer than TIE_NEED[kind]
    pixels of the still view is drawn again (new shape, rotation and order) until every site has them.
    Returns (scene, sites): sites = [(kind, earlier index, later index)]."""
    rng = np.random.RandomState(5)
    gens = []   # one generator per site: () -> (kind, first (pts, depth, rgb), second (pts, depth, rgb))

    def colours():
        return ((rng.uniform(150, 255), rng.uniform(0, 60), rng.uniform(0, 60)),
                (rng.uniform(0, 60), rng.uniform(150, 255), rng.uniform(0, 60)))

    def copy_pair(kind, shape, depth, rotated):
        def gen():
            a, b = colours()
            pts = np.asarray(shape(), np.float64)
            d = np.broadcast_to(np.asarray(depth() if callable(depth) else depth, np.float64), (3,)).copy()
            if not rotated:
                return kind, (pts, d, a), (pts, d, b)
            rot = [(1, 2, 0), (2, 0, 1)][rng.randint(2)]
            one, other = (pts, d), (pts[list(rot)], d[list(rot)])
            if rng.randint(2):
                one, other = other, one
            return kind, one + (a,), other + (b,)
        gens.append(gen)

    def small_shape(cx, cy):
        def shape():
            a, b, th = rng.uniform(4.5, 6), rng.uniform(4.5, 6), rng.uniform(0, 2 * np.pi)
            rot = np.array([[np.cos(th), -np.sin(th)], [np.sin(th), np.cos(th)]])
            p = np.array([[0, 0], [a, 0], [0, b]]) @ rot.T
            return p - p.mean(0) + (cx + 4.5, cy + 4.5)
        return shape

    # small: one per 9 x 9 cell, right triangles with 4.5..6 px legs at any angle
    k = 0
    for cy in range(0, H - 8, 9):
        for cx in list(range(0, 50, 9)) + list(range(410, W - 8, 9)):
            if rng.uniform() < 0.08:
                continue
            copy_pair("small", small_shape(cx, cy), 2.0 if k % 4 < 2 else (lambda: 2.0 + rng.uniform(0, 0.4, 3)), k % 2 == 1)
            k += 1
    # mid (16..127 px boxes) and coplanar overlaps: 78 x 75 cells of the right part
    for j, cy in enumerate(range(0, H - 74, 75)):
        for i, cx in enumerate(range(410, W - 77, 78)):
            if (i + j) % 4 == 3:
                def gen(cx=cx, cy=cy):
                    s = rng.uniform(30, 60)
                    a, b = colours()
                    t1 = _right_tri(cx + 2, cy + 2, s, s, rng)
                    t2 = _right_tri(cx + 2 + s / 3, cy + 2 + s / 4, 0.9 * s, 0.9 * s, rng)
                    return "coplanar", (np.asarray(t1), np.full(3, 3.5), a), (np.asarray(t2), np.full(3, 3.5), b)
                gens.append(gen)
            else:
                copy_pair("mid", lambda cx=cx, cy=cy: _right_tri(cx + 2, cy + 2, *rng.uniform(17, 72, 2), rng),
                          3.0 if (i + j) % 2 else (lambda: 3.0 + rng.uniform(0, 0.6, 3)), (i + 2 * j) % 2 == 1)
    # large (128 px and more) in the upper-left halves of 195 x 150 cells; small-and-large coplanar pairs in the
    # lower-right halves (constant z: the depths of the two differ by the weights' rounding only)
    for j, cy in enumerate(range(0, H - 149, 150)):
        for i, cx in enumerate(range(410, W - 194, 195)):
            copy_pair("large", lambda cx=cx, cy=cy: [(cx + 2, cy + 2), (cx + 2 + rng.uniform(135, 185), cy + 3),
                                                     (cx + 3, cy + 2 + rng.uniform(100, 140))],
                      4.5 if (i + j) % 2 else (lambda: 4.5 + rng.uniform(0, 0.8, 3)), (i + j) % 2 == 1)

            def gen(cx=cx, cy=cy, small_first=(i + j) % 2 == 1):
                x1, y1 = cx + 192.5, cy + 147.5
                big = np.array([(x1, cy + 6.5), (x1, y1), (x1 - 185.0, y1)]) + rng.uniform(-0.5, 0.5, (3, 2))
                small = np.array([(x1 - 24.0, y1 - 14.0), (x1 - 12.5, y1 - 3.0), (x1 - 26.0, y1 - 2.5)]) + rng.uniform(-0.9, 0.9, (3, 2))
                a, b = colours()
                if small_first:
                    return "small_first", (small, np.full(3, 4.0), a), (big, np.full(3, 4.0), b)
                return "large_first", (big, np.full(3, 4.0), a), (small, np.full(3, 4.0), b)
            gens.append(gen)
    # two huge sites behind everything (boxes over 128 px in both directions)
    for k in range(2):
        copy_pair("large", lambda k=k: _right_tri(412 + 10 * k, 4 + 20 * k, 370 - 30 * k, 430 - 40 * k, rng), 5.5 - 0.3 * k, k == 1)

    pairs = [g() for g in gens]
    hazard = S.hazard_scene(textures=textures())
    m = oracle_port.camera_path(still())[0]
    for _ in range(60):
        mesh = _Mesh(W, H)
        first = [mesh.tri(*p[1]) for p in pairs]
        second = [mesh.tri(*p[2]) for p in pairs]
        sites = [(p[0], a, b) for p, a, b in zip(pairs, first, second)]
        sc = S.concat_scenes(mesh.scene(), hazard)
        count = tie_pixels(sc, sites, oracle_port.OracleScene, m, W, H)[0]
        short = [k for k, (kind, _, _) in enumerate(sites) if count[k] < TIE_NEED[kind]]
        if not short:
            return sc, sites
        for k in short:
            pairs[k] = gens[k]()
    raise AssertionError(f"tie sites without exact ties: {[sites[k] for k in short][:5]}")


def needle_field(W=800, H=450, n=6000, seed=31):
    """Long thin triangles (area just above the cull) at random depths and angles, packed into a 128 x 64 pixel
    region: many 32 x 16 shading blocks have more than 96 distinct winners, some more than 192."""
    rng = np.random.RandomState(seed)
    m = _Mesh(W, H)
    x0, y0 = 400, 208
    for _ in range(n):
        c = np.array([x0 + rng.uniform(0, 128), y0 + rng.uniform(0, 64)])
        length, th = rng.uniform(6, 40), rng.uniform(0, np.pi)
        u = np.array([np.cos(th), np.sin(th)])
        wid = rng.uniform(10.5, 12.5) / length   # the reference's area (twice the triangle's) just above 10
        p = [c - u * length / 2, c + u * length / 2, c + np.array([-u[1], u[0]]) * wid]
        m.tri(p, rng.uniform(3, 30) + rng.uniform(0, 0.05, 3), tuple(rng.uniform(30, 255, 3)))
    return m.scene()


LIMIT_W, LIMIT_H = 803, 451


def limit_scene(W=LIMIT_W, H=LIMIT_H):
    """Boxes on the routing thresholds (15/16/17 and 127/128/129 px wide or high), large triangles with one corner
    inside each border, corner triangles whose boxes are small only because they are clamped to the frame, and
    boxes that start on the last column or row.  Returns (scene, names): names[k] says what triangle k is for."""
    rng = np.random.RandomState(9)
    m = _Mesh(W, H)
    names = []

    def add(name, pts, depth=5.0):
        m.tri(pts, depth, tuple(rng.uniform(40, 255, 3)))
        names.append(name)

    # clamped box edges: min at x + 0.5, max at x + d + 0.5 -> xmax - xmin == d whatever the projection's rounding
    for k, d in enumerate((15, 16, 17)):
        add(f"w{d}", [(20.5 + 40 * k, 20.5), (20.5 + 40 * k + d, 20.5), (20.5 + 40 * k, 30.5)])
        add(f"h{d}", [(160.5 + 20 * k, 20.5), (170.5 + 20 * k, 20.5), (160.5 + 20 * k, 20.5 + d)])
        add(f"s{d}", [(240.5 + 30 * k, 20.5), (240.5 + 30 * k + d, 20.5), (240.5 + 30 * k, 20.5 + d)])
    for k, d in enumerate((127, 128, 129)):
        add(f"w{d}", [(20.5, 60.5 + 20 * k), (20.5 + d, 60.5 + 20 * k), (20.5, 72.5 + 20 * k)])
        add(f"h{d}", [(360.5 + 20 * k, 20.5), (372.5 + 20 * k, 20.5), (360.5 + 20 * k, 20.5 + d)])
        add(f"s{d}", [(440.5 + 15 * k, 30.5 + 10 * k), (440.5 + 15 * k + d, 30.5 + 10 * k), (440.5 + 15 * k, 30.5 + 10 * k + d)], 6.0 + k)
    # one corner inside each border, the other two far outside: boxes clamped to the frame
    cx, cy = W / 2, H / 2
    add("border_left", [(3.5, cy + 0.5), (-2000.0, cy - 1500.0), (-2000.0, cy + 1500.0)], 9.0)
    add("border_right", [(W - 3.5, cy - 40.5), (W + 2000.0, cy - 1500.0), (W + 2000.0, cy + 1500.0)], 9.0)
    add("border_top", [(cx + 60.5, 2.5), (cx - 1500.0, -2000.0), (cx + 1500.0, -2000.0)], 9.0)
    add("border_bottom", [(cx - 60.5, H - 2.5), (cx - 1500.0, H + 2000.0), (cx + 1500.0, H + 2000.0)], 9.0)
    # corners: one vertex inside, the wedge opens away from the frame -> clamped boxes of 5 x 5 pixels
    for name, (x, y), (sx, sy) in (("corner_tl", (4.5, 4.5), (-1, -1)), ("corner_tr", (W - 4.5, 4.5), (1, -1)),
                                   ("corner_bl", (4.5, H - 4.5), (-1, 1)), ("corner_br", (W - 4.5, H - 4.5), (1, 1))):
        add(name, [(x, y), (x + sx * 3000.0, y + sy * 200.0), (x + sx * 200.0, y + sy * 3000.0)], 4.0)
    # boxes that start on the last column / row (and both)
    add("last_col", [(W - 0.75, 100.5), (W + 30.0, 100.5), (W - 0.75, 130.5)])
    add("last_col_small", [(W - 0.75, 300.5), (W + 8.0, 300.5), (W - 0.75, 310.5)])
    add("last_row", [(300.5, H - 0.75), (340.5, H - 0.75), (300.5, H + 30.0)])
    add("last_row_small", [(500.5, H - 0.75), (510.5, H - 0.75), (500.5, H + 8.0)])
    add("last_pixel", [(W - 0.75, H - 0.75), (W + 20.0, H - 0.75), (W - 0.75, H + 20.0)], 3.0)
    # busy background: mid-size triangles at random depths behind the probes
    for _ in range(300):
        x, y = rng.uniform(-20, W), rng.uniform(-20, H)
        add("filler", _right_tri(x, y, rng.uniform(4, 60), rng.uniform(4, 60), rng, skew=8.0), rng.uniform(7, 12))
    return m.scene(), names


# ------------------------------------------------------------------------------------------------------------------
# helpers
# ------------------------------------------------------------------------------------------------------------------
def assert_same(a, b, what):
    if not np.array_equal(a, b):
        ys, xs = np.nonzero(a != b)
        raise AssertionError(f"{what}: {len(ys)} px differ, first (x={xs[0]}, y={ys[0]}) "
                             f"got {a[ys[0], xs[0]]:06x} want {b[ys[0], xs[0]]:06x}")


def assert_stats(st, o, what):
    want = o["stats"]
    got = (st["near_rejected"], st["clipped"], st["spawned"], st["setups"], st["culled"], st["overflow"])
    ref = (want["near_rejected"], want["clipped"], want["spawned"], want["rasterized"],
           want["offscreen"] + want["small_or_backfacing"], 0)
    assert got == ref, f"{what}: statistics (near, clipped, spawned, setups, culled, overflow) {got} != oracle {ref}"


def set_route(r, route):
    c, cc, ds, fm = route
    r.set_option("clusters", c)
    r.set_option("cluster_cull", cc)
    r.set_option("direct_small", ds)
    r.set_option("flat_max", fm)


def restore_defaults(r):
    for name, value in (("clusters", 2), ("cluster_cull", 1), ("direct_small", 1), ("flat_max", 128), ("fused_small", 1),
                        ("spans", 1), ("rowtab_capacity", -1)):
        r.set_option(name, value)


def render_rows(r, renderer_lib, m, W, H, world):
    """Interleaved tile rows over ``world`` phases, reassembled to a whole frame (a phase is submitted again when
    finish() asks for it: a capacity regrown for an earlier submission may still be short)."""
    import torch
    th = renderer_lib.tile_height()
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
        frame[frame_rows] = buf.cpu().numpy().view(np.uint32)[buf_rows]
    return frame


def check_routes(r, renderer_lib, m, W, H, o, name, routes=ROUTES, bands=None, world=None):
    """Whole frame (pixels and statistics) under every routing; optionally bands (edges) and interleaved rows."""
    for route in routes:
        set_route(r, route)
        what = f"{name} clusters={route[0]} cull={route[1]} direct_small={route[2]} flat_max={route[3]}"
        assert_same(r.render(m, W, H)[0], o["pixels"], what)
        assert_stats(r.stats(), o, what)
        if bands:
            parts = [r.render(m, W, H, y0=a, y1=b)[0] for a, b in zip(bands[:-1], bands[1:])]
            assert_same(np.concatenate(parts, 0), o["pixels"], f"{what}: bands {bands}")
        if world:
            assert_same(render_rows(r, renderer_lib, m, W, H, world), o["pixels"], f"{what}: {world} interleaved phases")


def box_sizes(setups):
    return (setups["xmax"].astype(np.int64) - setups["xmin"], setups["ymax"].astype(np.int64) - setups["ymin"])


def block_winners(winner):
    """Distinct winning triangles of every 32 x 16 block of the frame."""
    H, W = winner.shape
    out = []
    for y in range(0, H, BLOCK_H):
        for x in range(0, W, BLOCK_W):
            w = winner[y:y + BLOCK_H, x:x + BLOCK_W]
            out.append(len(np.unique(w[w != NO_WINNER])))
    return np.asarray(out)


def _spin_poses(renderer_lib, frames):
    return renderer_lib.camera_path(S.input_script("spin", max(frames) + 1))[list(frames)]


# ------------------------------------------------------------------------------------------------------------------
# premise checks (CPU): every scene reaches the paths it exists for
# ------------------------------------------------------------------------------------------------------------------
def test_oracle_winner_plane_is_consistent(oracle_port):
    sc = S.clip_stress_scene(600)
    osc = oracle_port.OracleScene(sc)
    m = oracle_port.camera_path(S.input_script("spin", 10))[9]
    o = osc.render(m, 320, 180, want_winner=True, want_setups=True)
    w = o["winner"]
    assert (o["pixels"][w == NO_WINNER] == BG).all()
    won = np.unique(w[w != NO_WINNER])
    assert len(won) > 20 and np.isin(won, o["setups"]["order"]).all()
    assert (won >= sc.n_triangles).any()   # clip-spawned winners carry T + parent
    # the extra output changes nothing else
    plain = osc.render(m, 320, 180)
    assert np.array_equal(plain["pixels"], o["pixels"]) and plain["stats"] == o["stats"]


def test_tie_field_premises(oracle_port):
    """Every tie site has pixels where its two copies reach the same binary32 depth and the earlier one wins by list
    order alone (so a tie rule broken the other way changes the frame), and every routing class is present."""
    sc, sites = tie_field(oracle_port)
    assert 4000 <= sc.n_triangles <= 8000
    m = oracle_port.camera_path(still())[0]
    count, tied, o1, o2 = tie_pixels(sc, sites, oracle_port.OracleScene, m, 800, 450)
    missing = [(sites[k], int(count[k])) for k in range(len(sites)) if count[k] < TIE_NEED[sites[k][0]]]
    assert not missing, f"{len(missing)} tie sites without enough exact ties, e.g. {missing[:5]}"
    assert (o1["pixels"][tied] != o2["pixels"][tied]).all()   # the copies' colours tell the winner
    o = oracle_port.OracleScene(sc).render(m, 800, 450, want_setups=True)
    w1 = o1["winner"]
    # routing classes of the sites' triangles (boxes from the oracle's setups)
    st = o["setups"]
    bw, bh = box_sizes(st)
    big = np.maximum(bw, bh)
    cls = dict(zip(st["order"].tolist(), big.tolist()))
    kinds = {}
    for kind, a, b in sites:
        kinds.setdefault(kind, []).append((cls.get(a, -1), cls.get(b, -1)))
    for kind in ("small", "mid", "large", "small_first", "large_first", "coplanar"):
        assert kind in kinds, kind
    assert all(0 <= a < 16 and 0 <= b < 16 for a, b in kinds["small"])
    assert all(16 <= a < 128 and 16 <= b < 128 for a, b in kinds["mid"])
    assert all(a >= 128 and b >= 128 for a, b in kinds["large"])
    assert all(0 <= a < 16 and b >= 128 for a, b in kinds["small_first"])
    assert all(a >= 128 and 0 <= b < 16 for a, b in kinds["large_first"])
    assert sum(1 for k, *_ in sites if k == "small") > 1500
    # the hazard scene follows the sites and is not all hidden
    assert (w1[w1 != NO_WINNER] >= 2 * len(sites)).sum() > 1000


def test_needle_field_premises(oracle_port):
    sc = needle_field()
    m = oracle_port.camera_path(still())[0]
    o = oracle_port.OracleScene(sc).render(m, 800, 450, want_winner=True, want_setups=True)
    n = block_winners(o["winner"])
    assert (n > SHADE_TRIS).sum() >= 4 and (n > 2 * SHADE_TRIS).any(), sorted(n)[-8:]
    bw, bh = box_sizes(o["setups"])
    assert (np.maximum(bw, bh) < 16).sum() > 500 and (np.maximum(bw, bh) >= 16).sum() > 500


def test_limit_scene_premises(oracle_port):
    sc, names = limit_scene()
    W, H = LIMIT_W, LIMIT_H
    assert W % 4 and H % 4
    m = oracle_port.camera_path(still())[0]
    o = oracle_port.OracleScene(sc).render(m, W, H, want_setups=True, want_winner=True)
    st = o["setups"]
    box = {int(t): (int(st["xmin"][k]), int(st["xmax"][k]), int(st["ymin"][k]), int(st["ymax"][k])) for k, t in enumerate(st["order"])}
    idx = {name: k for k, name in enumerate(names) if name != "filler"}
    for d in (15, 16, 17, 127, 128, 129):
        x0, x1, y0, y1 = box[idx[f"w{d}"]]
        assert x1 - x0 == d and y1 - y0 < 16, (d, box[idx[f"w{d}"]])
        x0, x1, y0, y1 = box[idx[f"h{d}"]]
        assert y1 - y0 == d and x1 - x0 < 16, (d, box[idx[f"h{d}"]])
        x0, x1, y0, y1 = box[idx[f"s{d}"]]
        assert x1 - x0 == d and y1 - y0 == d
    for side in ("left", "right", "top", "bottom"):
        x0, x1, y0, y1 = box[idx[f"border_{side}"]]
        assert max(x1 - x0, y1 - y0) >= 128 and (x0 == 0 or y0 == 0 or x1 == W - 1 or y1 == H - 1)
    for corner in ("tl", "tr", "bl", "br"):
        x0, x1, y0, y1 = box[idx[f"corner_{corner}"]]
        assert x1 - x0 < 16 and y1 - y0 < 16 and (x0 == 0 or x1 == W - 1) and (y0 == 0 or y1 == H - 1)
    assert box[idx["last_col"]][0] == W - 1 and box[idx["last_col_small"]][0] == W - 1
    assert box[idx["last_row"]][2] == H - 1 and box[idx["last_row_small"]][2] == H - 1
    assert box[idx["last_pixel"]][0] == W - 1 and box[idx["last_pixel"]][2] == H - 1
    for name in ("corner_tl", "corner_tr", "corner_bl", "corner_br", "last_col", "last_row", "last_pixel", "w16", "h128"):
        assert (o["winner"] == idx[name]).any(), f"{name} wins no pixel"


def test_row_table_scene_premise(oracle_port):
    """The clip scene at flat_max = 16 has many tile-path triangles of different heights (see the row-table test)."""
    need = _tile_path_rows(oracle_port)
    assert len(need) > 50 and need.max() < need.sum() // 2


def _tile_path_rows(oracle_port):
    sc = S.clip_stress_scene(3000)
    m = oracle_port.camera_path(S.input_script("spin", 12))[9]
    st = oracle_port.OracleScene(sc).render(m, 800, 450, want_setups=True)["setups"]
    bw, bh = box_sizes(st)
    tile = (bw >= 16) | (bh >= 16)
    return 3 * (bh[tile] + 1)


# ------------------------------------------------------------------------------------------------------------------
# GPU: frames and statistics against the oracle
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_exact_ties_across_kernels(renderer_lib, oracle_port):
    """A: the earlier copy keeps every tied pixel whichever kernels the two copies went through."""
    sc, _ = tie_field(oracle_port)
    r = renderer_lib.Renderer(0)
    try:
        r.load_scene(sc)
        osc = oracle_port.OracleScene(sc)
        W, H = 800, 450
        cams = [(f"still", renderer_lib.camera_path(still())[0])]
        cams += [(f"spin {k}", m) for k, m in zip((1, 4), _spin_poses(renderer_lib, (1, 4)))]
        for name, m in cams:
            o = osc.render(m, W, H)
            if name == "still":
                check_routes(r, renderer_lib, m, W, H, o, f"ties {name}", bands=[0, 150, 300, 450], world=4)
            else:
                check_routes(r, renderer_lib, m, W, H, o, f"ties {name}")
    finally:
        restore_defaults(r)
        r.close()


@pytest.mark.gpu
def test_crowded_shading_blocks(renderer_lib, oracle_port):
    """B: blocks with more than 96 and 192 distinct winners take a second and a third staging pass in shade_tiles."""
    sc = needle_field()
    r = renderer_lib.Renderer(0)
    try:
        r.set_option("fused_small", 0)
        r.load_scene(sc)
        m = renderer_lib.camera_path(still())[0]
        W, H = 800, 450
        o = oracle_port.OracleScene(sc).render(m, W, H)
        check_routes(r, renderer_lib, m, W, H, o, "needles", bands=[0, 213, 229, 450], world=3)
    finally:
        restore_defaults(r)
        r.close()


@pytest.mark.gpu
def test_routing_limits_and_odd_frames(renderer_lib, oracle_port):
    """C: boxes on the 16 px and flat_max thresholds, boxes clamped by the frame border, boxes on the last column or
    row, frame sizes that are no multiple of 4, 32 or 64, and bands that start at y0 % 4 = 1, 2, 3."""
    sc, _ = limit_scene()
    r = renderer_lib.Renderer(0)
    try:
        r.set_option("fused_small", 0)
        r.load_scene(sc)
        osc = oracle_port.OracleScene(sc)
        m = renderer_lib.camera_path(still())[0]
        W, H = LIMIT_W, LIMIT_H
        o = osc.render(m, W, H)
        check_routes(r, renderer_lib, m, W, H, o, f"limits {W}x{H}", bands=[0, 5, 150, 303, H], world=3)
        for W2, H2 in ((33, 17), (1, 1), (800, 450)):
            check_routes(r, renderer_lib, m, W2, H2, osc.render(m, W2, H2), f"limits {W2}x{H2}")
    finally:
        restore_defaults(r)
        r.close()


def _dense():
    return S.icosahedron_field(20000, seed=9, extent=40, r_range=(0.3, 1.0))


def _away(m):
    """The same view with the whole scene behind the camera: no candidate at all."""
    a = np.asarray(m, np.float32).reshape(3, 4).copy()
    a[2, 3] += 1.0e4
    return a.reshape(12)


@pytest.mark.gpu
def test_walk_queue_overflow_is_reported_and_regrown(renderer_lib, oracle_port):
    """D: the cluster front's candidate queue overflows (bit 8), finish() asks for the repeat, and the repeat is the
    oracle's frame — whole frame, band, interleaved rows, a batch in which only some views overflow, host path."""
    import torch
    sc = _dense()
    osc = oracle_port.OracleScene(sc)
    mats = renderer_lib.camera_path(S.input_script("spin", 12))
    W, H = 800, 450
    th = renderer_lib.tile_height()
    r = renderer_lib.Renderer(0)
    try:
        r.load_scene(sc)
        r.set_option("clusters", 1)
        views = [mats[3], _away(mats[4]), mats[5], _away(mats[6]), mats[7], _away(mats[8])]
        want = [osc.render(v, W, H) for v in views]
        setups = max(o["stats"]["rasterized"] for o in want) + 1024

        def shrink():
            r.set_option("setup_capacity", setups)   # survivor buffers large enough; the walk queue holds 8 records

        for cull in (1, 0):
            r.set_option("cluster_cull", cull)
            # whole frame
            shrink()
            out = torch.zeros((H, W), dtype=torch.int32, device="cuda:0")
            r.render_device(views[0], W, H, out.data_ptr())
            assert r.finish() is True
            assert r.stats()["overflow"] & 8, r.stats()
            r.render_device(views[0], W, H, out.data_ptr())
            assert r.finish() is False
            assert_same(out.cpu().numpy().view(np.uint32), want[0]["pixels"], f"cull={cull} whole frame after regrowth")
            assert_stats(r.stats(), want[0], f"cull={cull} whole frame after regrowth")
            # band
            y0, y1 = 97, 333
            shrink()
            band = torch.zeros((y1 - y0, W), dtype=torch.int32, device="cuda:0")
            r.render_device(views[0], W, H, band.data_ptr(), y0=y0, y1=y1)
            assert r.finish() is True and r.stats()["overflow"] & 8
            r.render_device(views[0], W, H, band.data_ptr(), y0=y0, y1=y1)
            assert r.finish() is False and r.stats()["overflow"] == 0
            assert_same(band.cpu().numpy().view(np.uint32), want[0]["pixels"][y0:y1], f"cull={cull} band after regrowth")
            # interleaved rows: every phase overflows first
            frame = np.zeros((H, W), np.uint32)
            for phase in range(3):
                rows, frame_rows, buf_rows = renderer_lib.rows_layout(H, 3, phase, th)
                buf = torch.zeros((rows, W), dtype=torch.int32, device="cuda:0")
                shrink()
                r.render_device_rows(views[2], W, H, 3, phase, buf.data_ptr())
                assert r.finish() is True and r.stats()["overflow"] & 8, f"phase {phase}"
                r.render_device_rows(views[2], W, H, 3, phase, buf.data_ptr())
                assert r.finish() is False and r.stats()["overflow"] == 0
                frame[frame_rows] = buf.cpu().numpy().view(np.uint32)[buf_rows]
            assert_same(frame, want[2]["pixels"], f"cull={cull} interleaved rows after regrowth")
            # a batch: the views that see the field overflow, the ones that look away do not
            shrink()
            batch = torch.zeros((len(views), H, W), dtype=torch.int32, device="cuda:0")
            r.render_device(np.stack(views), W, H, batch.data_ptr())
            assert r.finish() is True
            flags = [r.stats(k)["overflow"] & 8 for k in range(len(views))]
            assert all(flags[0::2]) and not any(flags[1::2]), flags
            r.render_device(np.stack(views), W, H, batch.data_ptr())
            assert r.finish() is False
            got = batch.cpu().numpy().view(np.uint32)
            for k, o in enumerate(want):
                assert_same(got[k], o["pixels"], f"cull={cull} batch view {k} after regrowth")
                assert_stats(r.stats(k), o, f"cull={cull} batch view {k} after regrowth")
            # host path: regrows by itself
            shrink()
            assert_same(r.render(views[4], W, H)[0], want[4]["pixels"], f"cull={cull} host path")
            assert_stats(r.stats(), want[4], f"cull={cull} host path")
    finally:
        restore_defaults(r)
        r.close()


@pytest.mark.gpu
def test_row_start_table_full_or_absent(renderer_lib, oracle_port):
    """D: tile-path triangles that do not fit the row-start table keep their exact jumps — a table that holds only
    some of them, an empty table, and no table at all (spans = 0)."""
    need = _tile_path_rows(oracle_port)
    sc = S.clip_stress_scene(3000)
    m = renderer_lib.camera_path(S.input_script("spin", 12))[9]
    W, H = 800, 450
    o = oracle_port.OracleScene(sc).render(m, W, H)
    routes = [(c, cc, ds, 16) for c, cc in ((0, 0), (1, 0), (1, 1)) for ds in (1, 0)]
    r = renderer_lib.Renderer(0)
    try:
        r.load_scene(sc)
        for cap, spans in ((0, 1), (int(need.sum() // 2), 1), (-1, 0)):   # (an empty table first: a fresh renderer)
            r.set_option("rowtab_capacity", cap)
            r.set_option("spans", spans)
            check_routes(r, renderer_lib, m, W, H, o, f"rowtab_capacity={cap} spans={spans}", routes=routes,
                         bands=[0, 131, 450], world=3)
    finally:
        restore_defaults(r)
        r.close()


@pytest.mark.gpu
def test_overflowed_peer_frame_rows_are_overwritten(renderer_lib, oracle_port):
    """D: an overflowed pass of the fused frame assembly writes background rows into every destination; its repeat
    must overwrite them (one GPU, two local destinations), under every routing."""
    sc = S.clip_stress_scene(3000)
    m = renderer_lib.camera_path(S.input_script("spin", 12))[9]
    W, H = 800, 450
    want = oracle_port.OracleScene(sc).render(m, W, H)["pixels"]
    th = renderer_lib.tile_height()
    r = renderer_lib.Renderer(0)
    r.load_scene(sc)
    a, _ = r.peer_frame_alloc(W * H * 4)
    b, _ = r.peer_frame_alloc(W * H * 4)
    try:
        for route in ROUTES:
            set_route(r, route)
            for world in (1, 3):
                for phase in range(world):
                    _, frame_rows, _ = renderer_lib.rows_layout(H, world, phase, th)
                    r.set_option("setup_capacity", 8)
                    r.set_peer_frames([a, b])
                    r.render_device_rows(m, W, H, world, phase, 0)
                    assert r.finish() is True
                    for ptr in (a, b):
                        assert (r.read_device(ptr, (H, W))[frame_rows] == BG).all(), f"{route} world {world} phase {phase}: overflowed rows"
                    for _ in range(4):   # (the first pass measured only what fit: a later capacity may need a second regrowth)
                        r.render_device_rows(m, W, H, world, phase, 0)
                        if not r.finish():
                            break
                    assert r.stats()["overflow"] == 0
                r.set_peer_frames([])
                for ptr in (a, b):
                    assert_same(r.read_device(ptr, (H, W)), want, f"{route}: fused assembly over {world} after an overflowed pass")
    finally:
        r.set_peer_frames([])
        r.peer_frame_release(a)
        r.peer_frame_release(b)
        restore_defaults(r)
        r.close()


@pytest.mark.gpu
def test_key_plane_is_clean_between_submissions(renderer_lib, oracle_port):
    """E: keys are zero between submissions, whatever the previous one was — a band, interleaved rows, an overflowed
    frame (repeated, or abandoned for the next camera), a batch, another frame size, a peer-frame submission — under
    every routing.  Consecutive submissions never share a camera, so a key left behind cannot equal what the next
    frame writes."""
    import torch
    sc = S.clip_stress_scene(3000)
    osc = oracle_port.OracleScene(sc)
    poses = renderer_lib.camera_path(S.input_script("spin", 32))[1::2]
    r = renderer_lib.Renderer(0)
    r.load_scene(sc)
    peer, _ = r.peer_frame_alloc(800 * 450 * 4)
    oracle = {}

    def want(m, W, H):
        key = (m.tobytes(), W, H)
        if key not in oracle:
            oracle[key] = osc.render(m, W, H)["pixels"]
        return oracle[key]

    def device_frame(m, W, H):
        """Renders, repeating the submission as long as finish() asks for it; returns (frame, submissions)."""
        out = torch.zeros((np.asarray(m).reshape(-1, 12).shape[0], H, W), dtype=torch.int32, device="cuda:0")
        for n in range(1, 5):
            r.render_device(m, W, H, out.data_ptr())
            if not r.finish():
                break
        assert r.stats()["overflow"] == 0
        return out.cpu().numpy().view(np.uint32), n

    try:
        for route in ROUTES:
            set_route(r, route)
            cams = iter(poses)
            W, H = 800, 450
            m = next(cams)
            assert_same(r.render(m, W, H)[0], want(m, W, H), f"{route} whole frame")
            m = next(cams)
            assert_same(r.render(m, W, H, y0=17, y1=301)[0], want(m, W, H)[17:301], f"{route} ragged band")
            m = next(cams)
            assert_same(render_rows(r, renderer_lib, m, W, H, 3), want(m, W, H), f"{route} interleaved rows")
            m = next(cams)
            r.set_option("setup_capacity", 64)
            got, n = device_frame(m, W, H)
            assert n > 1
            assert_same(got[0], want(m, W, H), f"{route} repeat of an overflowed frame")
            m = next(cams)
            r.set_option("setup_capacity", 64)
            out = torch.zeros((H, W), dtype=torch.int32, device="cuda:0")
            r.render_device(m, W, H, out.data_ptr())
            assert r.finish() is True   # abandoned: the caller goes on with the next camera
            m = next(cams)
            assert_same(device_frame(m, W, H)[0][0], want(m, W, H), f"{route} frame after an abandoned overflowed frame")
            views = np.stack([next(cams) for _ in range(3)])
            got = device_frame(views, W, H)[0]
            for k in range(3):
                assert_same(got[k], want(views[k], W, H), f"{route} batch view {k}")
            for W, H in ((800, 450), (803, 451), (640, 360)):
                m = next(cams)
                assert_same(r.render(m, W, H)[0], want(m, W, H), f"{route} size {W}x{H}")
            W, H = 800, 450
            m = next(cams)
            r.set_peer_frames([peer])
            for _ in range(4):
                r.render_device_rows(m, W, H, 1, 0, 0)
                if not r.finish():
                    break
            r.set_peer_frames([])
            assert_same(r.read_device(peer, (H, W)), want(m, W, H), f"{route} peer-frame submission")
            m = next(cams)
            assert_same(r.render(m, W, H)[0], want(m, W, H), f"{route} last whole frame")
    finally:
        r.set_peer_frames([])
        r.peer_frame_release(peer)
        restore_defaults(r)
        r.close()


@pytest.mark.gpu
def test_walk_queue_may_need_more_records_than_triangles(renderer_lib, oracle_port):
    """The cluster front reserves the direct walk's queue in chunks of 64 records per warp and pads them with holes, so
    a scene whose triangles nearly all take the direct walk needs more records than it has triangles.  The first frame
    (queue sized to the triangle count) overflows, and the regrowth must not stop at the triangle count: the repeat, and
    the host path, give the oracle's frame."""
    import torch
    rng = np.random.RandomState(41)
    W, H = 800, 450
    mesh = _Mesh(W, H)
    for _ in range(2000):
        x, y = rng.uniform(0, W - 12), rng.uniform(0, H - 12)
        mesh.tri(_right_tri(x, y, rng.uniform(5, 12), rng.uniform(5, 12), rng), rng.uniform(2, 20), tuple(rng.uniform(40, 255, 3)))
    sc = mesh.scene()
    m = renderer_lib.camera_path(still())[0]
    o = oracle_port.OracleScene(sc).render(m, W, H)
    assert o["stats"]["rasterized"] == sc.n_triangles   # every triangle is a record-free candidate
    for cull in (1, 0):
        r = renderer_lib.Renderer(0)
        try:
            r.set_option("fused_small", 0)
            r.set_option("clusters", 1)
            r.set_option("cluster_cull", cull)
            r.load_scene(sc)
            out = torch.zeros((H, W), dtype=torch.int32, device="cuda:0")
            r.render_device(m, W, H, out.data_ptr())
            assert r.finish() is True and r.stats()["overflow"] & 8, r.stats()
            r.render_device(m, W, H, out.data_ptr())
            assert r.finish() is False
            assert_same(out.cpu().numpy().view(np.uint32), o["pixels"], f"cull={cull} repeat")
            assert_stats(r.stats(), o, f"cull={cull} repeat")
            assert_same(r.render(m, W, H)[0], o["pixels"], f"cull={cull} host path")
        finally:
            r.close()
