"""Scene updates (s3r_update_vertices / _attributes / _texels): a loaded scene animated in place, against the oracle.

Every expected frame is the oracle's frame of the UPDATED scene arrays (a new ``Scene`` with the new vertices, records or
atlases), and every comparison is exact: pixels, statistics, visibility planes.  After a vertex update the general path's
cluster front must see the new positions in the clusters' private copies and bounds that still bound them, so the
refit headers are also compared, bit for bit, with a float64 numpy restatement of the bounds rule (cluster.hpp) applied to
the load-time partition.  The CPU tests pin that restatement to the load-time build and prove from the oracle alone that
each animation changes what it exists to change: triangles entering and leaving the frame, near-plane straddles, boxes
crossing the routing thresholds."""
import numpy as np
import pytest

from swift3drenderer_b200 import scene as S
from test_gpu_supersample import BANDS, resolve
from test_gpu_vis_edges import (NO_WINNER, ROUTES, assert_same, assert_stats, box_sizes, render_rows, restore_defaults,
                                set_route, still)
from test_gpu_visibility_planes import device_colour, device_planes, expected

S3R_E_SCENE, S3R_E_ARG, S3R_E_NOSCENE = -3, -4, -5
W, H = 320, 180
VERTEX_UPDATE_KERNELS = 2   # scene_scatter + cluster_refit (include/s3r_b200.h)


# ------------------------------------------------------------------------------------------------------------------
# the bounds rule, restated in float64 numpy (std::min / std::max argument order kept: it decides the sign of a zero)
# ------------------------------------------------------------------------------------------------------------------
def _mn(a, b):
    return np.where(b < a, b, a)


def _mx(a, b):
    return np.where(a < b, b, a)


def bounds_rule(hdr, pos, tri):
    """Headers {center, radius, max_edge} of the partition ``hdr`` / ``tri`` over the cluster copies ``pos`` (3, NV);
    t0, v_off, tri_off and the sentinel are taken from ``hdr``."""
    n = len(hdr) - 1
    out = hdr.copy()
    if n == 0:
        return out
    v_off = hdr["v_off"].astype(np.int64)
    t_off = hdr["tri_off"].astype(np.int64)
    nv, nt = np.diff(v_off), np.diff(t_off)
    P = np.asarray(pos, np.float32).astype(np.float64)
    lo, hi, me2 = np.zeros((n, 3)), np.zeros((n, 3)), np.zeros(n)
    with np.errstate(invalid="ignore", over="ignore"):
        for j in range(int(nt.max())):
            act = nt > j
            w = tri[np.where(act, t_off[:-1] + j, 0)].astype(np.int64)
            c = [P[:, v_off[:-1] + ((w >> (8 * k)) & 255)].T for k in range(3)]
            l, h = _mn(c[0], _mn(c[1], c[2])), _mx(c[0], _mx(c[1], c[2]))
            a = act[:, None]
            lo = np.where(a, l if j == 0 else _mn(lo, l), lo)
            hi = np.where(a, h if j == 0 else _mx(hi, h), hi)
            e2 = np.zeros(n)
            for e in range(3):
                d = c[e] - c[(e + 1) % 3]
                e2 = _mx(e2, (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2])
            me2 = np.where(act, _mx(me2, e2), me2)
        centre = (0.5 * (lo + hi)).astype(np.float32)
        c64 = centre.astype(np.float64)
        r2 = np.zeros(n)
        finite = np.ones(n, bool)
        for k in range(int(nv.max())):
            act = nv > k
            p = P[:, np.where(act, v_off[:-1] + k, 0)].T
            d = p - c64
            r2 = np.where(act, _mx(r2, (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]), r2)
            finite &= ~act | np.isfinite(p).all(1)

        def round_up(v):
            f = v.astype(np.float32)
            f = np.where(~(f.astype(np.float64) >= v), np.nextafter(f, np.float32(np.inf)), f)
            return np.nextafter(f, np.float32(np.inf))

        radius = round_up(np.sqrt(r2) * (1.0 + 1e-9))
        max_edge = round_up(np.sqrt(me2) * (1.0 + 1e-9))
    bad = ~finite | ~np.isfinite(radius) | ~np.isfinite(max_edge)
    centre[bad] = 0
    radius[bad] = np.inf
    max_edge[bad] = np.inf
    out["center"][:n], out["radius"][:n], out["max_edge"][:n] = centre, radius, max_edge
    return out


def cluster_sources(sc, clusters):
    """Per cluster vertex: the original vertex it copies (from the triangle words and the index stream)."""
    hdr, tri = clusters["hdr"], clusters["tri"]
    n = len(hdr) - 1
    nt = np.diff(hdr["tri_off"].astype(np.int64))
    owner = np.repeat(np.arange(n), nt)
    orig = hdr["t0"][owner].astype(np.int64) + np.arange(len(tri)) - np.repeat(hdr["tri_off"][:n].astype(np.int64), nt)
    vi = np.asarray(sc.vertex_indices, np.int64).reshape(-1, 3)
    src = np.zeros(clusters["pos"].shape[1], np.int64)
    for k in range(3):
        src[hdr["v_off"][owner].astype(np.int64) + ((tri >> (8 * k)) & 255)] = vi[orig, k]
    return src


def expected_clusters(clusters, src, xyz):
    """(headers, copies) the device must hold after its positions became ``xyz`` (V, 3)."""
    pos = np.ascontiguousarray(np.asarray(xyz, np.float32)[src].T)
    return bounds_rule(clusters["hdr"], pos, clusters["tri"]), pos


def same_bits(a, b):
    return np.array_equal(np.ascontiguousarray(a).view(np.uint8), np.ascontiguousarray(b).view(np.uint8))


# ------------------------------------------------------------------------------------------------------------------
# animations: (scene at load, camera, updated positions)
# ------------------------------------------------------------------------------------------------------------------
def _dense():
    """3000 icosahedrons in and around the still camera's view: some behind the camera, some beside the frame."""
    return S.icosahedron_field(3000, seed=21, extent=(10.0, 6.0, 8.0), r_range=(0.2, 0.6), center=(0.0, 0.0, -8.0))


def _small_field():
    """1000 small icosahedrons well inside the view: most of their triangles fail the area cull at load."""
    return S.icosahedron_field(1000, seed=23, extent=(6.0, 3.5, 3.0), r_range=(0.08, 0.25), center=(0.0, 0.0, -12.0))


def _rigid(sc, seed, scale=1.0, shift=(6.0, 4.0, 7.0)):
    """A seeded rigid motion (rotation about its centre, centre moved by up to ``shift``) per icosahedron (12 consecutive
    vertices), optionally scaled about its centre."""
    rng = np.random.RandomState(seed)
    p = np.asarray(sc.vertices[:, :3], np.float64).reshape(-1, 12, 3)
    n = p.shape[0]
    c = p.mean(1, keepdims=True)
    q, _ = np.linalg.qr(rng.normal(size=(n, 3, 3)))
    new_c = c + rng.uniform(-1, 1, (n, 1, 3)) * np.asarray(shift)
    out = np.einsum("nij,nkj->nki", q, (p - c) * scale) + new_c
    return out.reshape(-1, 3).astype(np.float32)


def _with_positions(sc, xyz):
    v = sc.vertices.copy()
    v[:, :3] = xyz
    return S.Scene(v, sc.vertex_indices, sc.attributes, sc.attribute_indices, sc.textures)


def animation(name, lib):
    """(scene at load, camera matrix, new positions (V, 3) float32)."""
    m = lib.camera_path(still())[0]
    if name == "dense":
        sc = _dense()
        return sc, m, _rigid(sc, 3)
    if name == "dense_x3":
        sc = _small_field()
        return sc, m, _rigid(sc, 4, scale=3.0, shift=(1.0, 1.0, 1.0))
    if name == "clip":
        sc = S.clip_stress_scene(4000)
        xyz = np.asarray(sc.vertices[:, :3], np.float32).copy()
        xyz[:, 2] += np.float32(0.9)   # the slab slides through the near plane
        return sc, m, xyz
    if name == "hazards":
        sc = S.hazard_scene()
        xyz = np.asarray(sc.vertices[:, :3], np.float64)
        xyz = xyz * np.array([0.8, 1.1, 1.0]) + np.array([1.5, -0.4, 0.35])   # slides sideways and towards the camera
        return sc, m, xyz.astype(np.float32)
    if name == "shipped":
        sc = S.shipped_scene(1)
        m = lib.camera_path(S.input_script("flythrough", 600))[110]
        xyz = np.asarray(sc.vertices[:, :3], np.float64)
        rng = np.random.RandomState(2)
        xyz = xyz + rng.uniform(-1.5, 1.5, (1, 3)) + rng.uniform(-0.6, 0.6, xyz.shape)
        return sc, m, xyz.astype(np.float32)
    raise KeyError(name)


ANIMATIONS = ["dense", "dense_x3", "clip", "hazards", "shipped"]
# (triangles that were no survivor at load and win pixels after the update, winners at load that win none after it):
# the camera sits inside the clip scene's slab, where a few clipped giants win at load; the two small scenes exist for
# the small-scene path and only need a changed frame
PREMISE_WINNERS = {"dense": (300, 300), "dense_x3": (300, 300), "clip": (20, 2), "hazards": (0, 3), "shipped": (0, 0)}


# ------------------------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("which", ["dense", "clip", "hazards", "shipped"])
def test_bounds_restatement_matches_the_load_build(which, renderer_lib, oracle_port):
    """The numpy restatement, applied to the load-time positions, gives the load-time headers bit for bit."""
    sc = {"dense": _dense, "clip": lambda: S.clip_stress_scene(4000), "hazards": S.hazard_scene,
          "shipped": lambda: S.shipped_scene(1)}[which]()
    c = renderer_lib.debug_clusters(sc)
    src = cluster_sources(sc, c)
    hdr, pos = expected_clusters(c, src, sc.vertices[:, :3])
    assert same_bits(pos, c["pos"])
    assert same_bits(hdr, c["hdr"])
    # ... and with a NaN vertex, exactly its clusters get the never-culling bounds
    xyz = np.asarray(sc.vertices[:, :3], np.float32).copy()
    xyz[int(src[len(src) // 2]), 1] = np.nan
    hdr2, _ = expected_clusters(c, src, xyz)
    v_off = c["hdr"]["v_off"].astype(np.int64)
    has_nan = np.add.reduceat(np.isnan(xyz[src]).any(1), v_off[:-1])
    assert np.array_equal(np.isinf(hdr2["radius"][:-1]), has_nan > 0)


@pytest.mark.parametrize("name", ANIMATIONS)
def test_animation_premises(name, renderer_lib, oracle_port):
    """From the oracle alone: triangles rejected (near plane, off screen or culled) at load win pixels after the update,
    winners at load are gone after it, the clip scene's straddles change, and boxes cross the 16 / 128 px routing limits."""
    sc, m, xyz = animation(name, renderer_lib)
    new = _with_positions(sc, xyz)
    T = sc.n_triangles
    before = oracle_port.OracleScene(sc).render(m, W, H, want_setups=True, want_winner=True)
    after = oracle_port.OracleScene(new).render(m, W, H, want_setups=True, want_winner=True)

    def winners(o):
        w = o["winner"][o["winner"] != NO_WINNER].astype(np.int64)
        return set(np.unique(np.where(w >= T, w - T, w)).tolist())

    def recorded(o):
        s = o["setups"]["order"].astype(np.int64)
        return set(np.where(s >= T, s - T, s).tolist())

    wb, wa = winners(before), winners(after)
    entering = wa - recorded(before)   # not even a survivor at load
    enter_min, leave_min = PREMISE_WINNERS[name]
    assert len(entering) >= enter_min, f"{name}: {len(entering)} triangles enter"
    assert len(wb - wa) >= leave_min, f"{name}: {len(wb - wa)} winners leave"
    assert (before["pixels"] != after["pixels"]).mean() > 0.01, f"{name}: the update hardly changes the frame"
    if name == "dense_x3":
        # more survivors than the initial survivor capacity, max(4096, T / 4), which the load-time frame stays under
        cap = max(4096, T // 4)
        assert before["stats"]["rasterized"] < cap < after["stats"]["rasterized"]
    if name == "clip":
        assert before["stats"]["clipped"] != after["stats"]["clipped"] and after["stats"]["clipped"] > 100

    def size_class(o):
        sx, sy = box_sizes(o["setups"])
        big = np.maximum(sx, sy)
        order = o["setups"]["order"].astype(np.int64)
        return dict(zip(order.tolist(), np.digitize(big, [16, 128]).tolist()))

    cb, ca = size_class(before), size_class(after)
    moved = [t for t in cb if t in ca and cb[t] != ca[t]]
    if T > 1920:   # general path: flat_max and the record-free limit route by box size
        assert len(moved) >= 20, f"{name}: {len(moved)} boxes cross a routing limit"


# ------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------
def _clusters_now(r):
    d = r.cluster_dump()
    return d["hdr"], d["pos"]


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["dense", "clip", "hazards"])
def test_refit_headers_and_copies(which, renderer_lib, oracle_port):
    """After a full update, a partial range (first > 0, count not a multiple of 4), two updates in a row, the load-time
    positions and a NaN vertex made finite again, the device's headers and copies equal the restatement bit for bit."""
    import torch
    sc, m, xyz = animation(which, renderer_lib)
    base = np.asarray(sc.vertices[:, :3], np.float32)
    c = renderer_lib.debug_clusters(sc)
    src = cluster_sources(sc, c)
    r = renderer_lib.Renderer(0)
    try:
        r.load_scene(sc)
        hdr0, pos0 = _clusters_now(r)
        assert same_bits(hdr0, c["hdr"]) and same_bits(pos0, c["pos"])
        state = base.copy()

        def check(what):
            want_hdr, want_pos = expected_clusters(c, src, state)
            got_hdr, got_pos = _clusters_now(r)
            assert same_bits(got_pos, want_pos), f"{which} {what}: copies differ"
            assert same_bits(got_hdr, want_hdr), f"{which} {what}: headers differ " \
                f"({int((got_hdr != want_hdr).sum())} records)"
            return got_hdr

        r.update_vertices(xyz)                           # full, host source
        state = xyz.copy()
        check("full update")
        V = len(base)
        a, b = 5, max(6, V - 7)                          # partial, device source
        part = np.ascontiguousarray(base[a:b] * np.float32(1.01))
        r.update_vertices(torch.from_numpy(part).cuda(), first=a)
        torch.cuda.synchronize()
        state[a:b] = part
        check(f"partial {a}..{b}")
        r.update_vertices(xyz[:3] + np.float32(0.5))    # two in a row, without a synchronisation between them
        r.update_vertices(xyz[V - 1:] - np.float32(0.25), first=V - 1)
        state[:3] = xyz[:3] + np.float32(0.5)
        state[V - 1:] = xyz[V - 1:] - np.float32(0.25)
        check("two in a row")
        r.update_vertices(base)
        state = base.copy()
        assert same_bits(check("load-time positions"), c["hdr"])
        k = int(src[len(src) // 2])
        nan = base[k:k + 1].copy()
        nan[0, 2] = np.nan
        r.update_vertices(nan, first=k)
        state[k] = nan[0]
        got = check("NaN vertex")
        v_off = c["hdr"]["v_off"].astype(np.int64)
        owners = np.searchsorted(v_off, np.nonzero(src == k)[0], side="right") - 1
        inf = np.nonzero(np.isinf(got["radius"][:-1]))[0]
        assert set(inf.tolist()) == set(owners.tolist()) | set(np.nonzero(np.isinf(c["hdr"]["radius"][:-1]))[0].tolist())
        r.update_vertices(base[k:k + 1], first=k)
        state[k] = base[k]
        assert same_bits(check("finite again"), c["hdr"])
    finally:
        r.close()


def _check_frames(r, renderer_lib, oracle_port, sc, m, what, routes=ROUTES, extras=True):
    """Every frame of ``r`` (whose scene must now equal ``sc``) equals the oracle's: all routes (whole frame and bands),
    and with ``extras`` device bands, interleaved rows over 2 and 3 phases, a view batch, 2 x 2 supersampling and the
    visibility planes."""
    import torch
    osc = oracle_port.OracleScene(sc)
    colour, tri, depth, o = expected(osc, sc.n_triangles, m, W, H)
    for route in routes:
        set_route(r, route)
        rw = f"{what} route={route}"
        assert_same(r.render(m, W, H)[0], colour, rw)
        assert_stats(r.stats(), o, rw)
        parts = [r.render(m, W, H, y0=a, y1=b)[0] for a, b in ((0, 61), (61, 62), (62, 180))]
        assert_same(np.concatenate(parts, 0), colour, f"{rw}: bands")
    restore_defaults(r)
    if not extras:
        return colour
    for y0, y1 in BANDS[:4]:
        assert_same(device_colour(r, torch, m, W, H, y0, y1), colour[y0:y1], f"{what}: device band {y0}..{y1}")
    for world in (2, 3):
        assert_same(render_rows(r, renderer_lib, m, W, H, world), colour, f"{what}: {world} interleaved phases")
    spin = renderer_lib.camera_path(S.input_script("spin", 6))
    views = np.stack([m, spin[2], spin[5]])
    r.set_option("views_per_chunk", 2)
    batch = r.render(views, W, H)
    r.set_option("views_per_chunk", 256)
    for i, v in enumerate(views):
        assert_same(batch[i], osc.render(v, W, H)["pixels"], f"{what}: view {i} of a batch of 3")
    assert_same(r.render_ssaa(m, W, H, 2)[0], resolve(osc.render(m, 2 * W, 2 * H)["pixels"], 2), f"{what}: ssaa k=2")
    got = device_planes(r, torch, m, W, H)
    for name, g, w in zip(("colour", "triangle", "depth"), got, (colour, tri, depth)):
        assert_same(g[0], w, f"{what}: visibility {name}")
    return colour


@pytest.mark.gpu
@pytest.mark.parametrize("name", ANIMATIONS)
def test_frames_after_update(name, renderer_lib, oracle_port):
    """Frames before and after the update equal the oracle's frames of the load-time and the updated arrays, under every
    routing and partition; a renderer freshly loaded with the updated arrays (another partition) renders the same."""
    import torch
    sc, m, xyz = animation(name, renderer_lib)
    new = _with_positions(sc, xyz)
    r = renderer_lib.Renderer(0)
    fresh = renderer_lib.Renderer(0)
    try:
        r.load_scene(sc)
        _check_frames(r, renderer_lib, oracle_port, sc, m, f"{name} at load", routes=ROUTES[:1] + ROUTES[-1:], extras=False)
        r.update_vertices(torch.from_numpy(np.ascontiguousarray(xyz)).cuda())
        if name == "dense_x3":
            # the scaled field needs more survivor / bin room than the load-time frames did: the first frame asks for
            # a repeat, and the repeat is the oracle's
            buf = torch.zeros((H, W), dtype=torch.int32, device="cuda:0")
            set_route(r, (1, 1, 0, 128))
            r.render_device(m, W, H, buf.data_ptr())
            assert r.finish() is True, "the scaled field should have overflowed a capacity"
            restore_defaults(r)
        colour = _check_frames(r, renderer_lib, oracle_port, new, m, f"{name} updated")
        fresh.load_scene(new)
        assert_same(fresh.render(m, W, H)[0], colour, f"{name}: fresh load")
        parts = [fresh.render(m, W, H, y0=a, y1=b)[0] for a, b in ((0, 61), (61, 180))]
        assert_same(np.concatenate(parts, 0), colour, f"{name}: fresh load, bands")
    finally:
        restore_defaults(r)
        r.close()
        fresh.close()


@pytest.mark.gpu
@pytest.mark.parametrize("source", ["device", "host"])
def test_updates_are_ordered_on_the_stream(source, renderer_lib, oracle_port):
    """render -> update -> render -> update -> render, enqueued on one stream without a host synchronisation: every frame
    is the oracle's frame of its own scene state (bands, so the cluster front reads copies and bounds)."""
    import torch
    sc, m, xyz = animation("dense", renderer_lib)
    states = [np.asarray(sc.vertices[:, :3], np.float32), xyz, _rigid(sc, 9)]
    want = [oracle_port.OracleScene(_with_positions(sc, s)).render(m, W, H)["pixels"] for s in states]
    r = renderer_lib.Renderer(0)
    try:
        r.load_scene(sc)
        for _ in range(2):   # settle capacities for all three states first
            for s in states:
                r.update_vertices(s)
                for a, b in ((0, 90), (90, 180)):
                    r.render(m, W, H, y0=a, y1=b)
        r.update_vertices(states[0])
        r.render(m, W, H)
        if source == "device":
            stream = torch.cuda.Stream()
            sp = stream.cuda_stream
            srcs = [torch.from_numpy(np.ascontiguousarray(s)).cuda() for s in states]
            torch.cuda.synchronize()
        else:
            sp = 0
            srcs = states
        bufs = [torch.zeros((H, W), dtype=torch.int32, device="cuda:0") for _ in states]
        torch.cuda.synchronize()
        for k in range(3):
            if k:
                r.update_vertices(srcs[k], stream=sp)
            for a, b in ((0, 90), (90, 180)):
                r.render_device(m, W, H, bufs[k].data_ptr() + 4 * a * W, y0=a, y1=b, stream=sp)
        assert r.finish() is False
        torch.cuda.synchronize()
        for k in range(3):
            assert_same(bufs[k].cpu().numpy().view(np.uint32), want[k], f"{source} source: frame {k}")
    finally:
        r.close()


def _recoloured(sc):
    at = sc.attributes.copy()
    n = len(at)
    rng = np.random.RandomState(4)
    # recolour the colour records, switch a third of the records colour <-> texture, change corner normals
    col = at["kind"] == S.KIND_COLOR
    at["payload"][col, :3] = rng.uniform(0, 255, (int(col.sum()), 3)).astype("<f4").view("<u4")
    sw = np.arange(n) % 3 == 1
    to_tex = sw & col
    to_col = sw & ~col
    at["kind"][to_tex] = S.KIND_TEXTURE
    at["payload"][to_tex, 0] = 1
    at["payload"][to_tex, 2:4] = rng.uniform(0, 1, (int(to_tex.sum()), 2)).astype("<f4").view("<u4")
    at["kind"][to_col] = S.KIND_COLOR
    at["payload"][to_col, :3] = rng.uniform(0, 255, (int(to_col.sum()), 3)).astype("<f4").view("<u4")
    nrm = at["normal"][:, :3].astype(np.float64) + rng.uniform(-0.5, 0.5, (n, 3))
    at["normal"][:, :3] = (nrm / np.linalg.norm(nrm, axis=1, keepdims=True)).astype("<f4")
    return at


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["shipped", "dense"])
def test_attributes_and_atlases(which, renderer_lib, oracle_port):
    """Recoloured records, colour <-> texture switches, new corner normals and a replaced atlas (a different procedural
    image) on the small-scene and the general path; an invalid record is refused and changes nothing."""
    import torch
    sc, m, _ = animation(which, renderer_lib)
    r = renderer_lib.Renderer(0)
    try:
        r.load_scene(sc)
        at = _recoloured(sc)
        first = 7
        r.update_attributes(at[first:], first=first)
        r.update_attributes(at[:first])
        cur = S.Scene(sc.vertices, sc.vertex_indices, at, sc.attribute_indices, sc.textures)
        for route in (ROUTES[0], ROUTES[-1]):
            set_route(r, route)
            assert_same(r.render(m, W, H)[0], oracle_port.OracleScene(cur).render(m, W, H)["pixels"], f"{which} records {route}")
            assert_same(np.concatenate([r.render(m, W, H, y0=a, y1=b)[0] for a, b in ((0, 77), (77, 180))]),
                        oracle_port.OracleScene(cur).render(m, W, H)["pixels"], f"{which} records, bands {route}")
        restore_defaults(r)
        tex = sc.textures.copy()
        tex[1] = S.build_ripmap_atlas(S.procedural_image(5))
        r.update_textures(torch.from_numpy(tex[1:2].view(np.int32)).cuda(), first=1)
        cur = S.Scene(sc.vertices, sc.vertex_indices, at, sc.attribute_indices, tex)
        want = oracle_port.OracleScene(cur).render(m, W, H)["pixels"]
        assert not np.array_equal(want, oracle_port.OracleScene(
            S.Scene(sc.vertices, sc.vertex_indices, at, sc.attribute_indices, sc.textures)).render(m, W, H)["pixels"])
        assert_same(r.render(m, W, H)[0], want, f"{which} atlas 1 replaced (device source)")
        r.update_textures(sc.textures[1:2], first=1)
        r.update_textures(tex[1:2], first=1)
        assert_same(r.render(m, W, H)[0], want, f"{which} atlas 1 replaced (host source)")
        for field, value in (("kind", 2), ("texture", sc.textures.shape[0]), ("normal_w", 1.0)):
            bad = at[:4].copy()
            if field == "kind":
                bad["kind"][2] = value
            elif field == "texture":
                bad["kind"][2] = S.KIND_TEXTURE
                bad["payload"][2, 0] = value
            else:
                bad["normal"][2, 3] = value
            with pytest.raises(renderer_lib.RendererError, match=f"error {S3R_E_SCENE}"):
                r.update_attributes(bad, first=3)
            assert_same(r.render(m, W, H)[0], want, f"{which}: frame after the refused record ({field})")
    finally:
        restore_defaults(r)
        r.close()


@pytest.mark.gpu
def test_rejected_arguments_and_launch_counts(renderer_lib, oracle_port):
    """Each rejected argument returns its code and changes nothing; count = 0 launches nothing; a vertex update launches
    its documented kernels; a render launches as many kernels after an update as before it."""
    import ctypes
    import torch
    sc, m, xyz = animation("dense", renderer_lib)
    lib = renderer_lib.load_library()
    r = renderer_lib.Renderer(0)
    try:
        h = r._h
        assert lib.s3r_update_vertices(h, 0, 1, xyz.ctypes.data, 0, None) == S3R_E_NOSCENE
        assert lib.s3r_update_attributes(h, 0, 1, sc.attributes.ctypes.data, None) == S3R_E_NOSCENE
        assert lib.s3r_update_texels(h, 0, 1, sc.textures.ctypes.data, 0, None) == S3R_E_NOSCENE
        r.load_scene(sc)
        V, A, NT = len(xyz), len(sc.attributes), sc.textures.shape[0]
        want = oracle_port.OracleScene(sc).render(m, W, H)["pixels"]
        for mode in ("whole", "band"):
            y1 = H if mode == "whole" else 90
            r.render(m, W, H, y0=0, y1=y1)
        hdr0, pos0 = _clusters_now(r)
        dev = torch.from_numpy(np.ascontiguousarray(xyz)).cuda()
        atl = torch.from_numpy(sc.textures[:1].view(np.int32)).cuda()
        n0 = r.kernel_launches
        rejected = [
            ("vertices past the end", lib.s3r_update_vertices(h, V - 2, 3, xyz.ctypes.data, 0, None)),
            ("vertices first > V", lib.s3r_update_vertices(h, V + 1, 0, xyz.ctypes.data, 0, None)),
            ("vertices huge count", lib.s3r_update_vertices(h, 1, 2 ** 64 - 1, xyz.ctypes.data, 0, None)),
            ("vertices null", lib.s3r_update_vertices(h, 0, 1, None, 0, None)),
            ("vertices flag 2", lib.s3r_update_vertices(h, 0, 1, xyz.ctypes.data, 2, None)),
            ("vertices host flagged device", lib.s3r_update_vertices(h, 0, 1, xyz.ctypes.data, 1, None)),
            ("vertices device flagged host", lib.s3r_update_vertices(h, 0, 1, ctypes.c_void_p(dev.data_ptr()), 0, None)),
            ("attributes past the end", lib.s3r_update_attributes(h, A - 1, 2, sc.attributes.ctypes.data, None)),
            ("attributes null", lib.s3r_update_attributes(h, 0, 1, None, None)),
            ("attributes from device", lib.s3r_update_attributes(h, 0, 1, ctypes.c_void_p(dev.data_ptr()), None)),
            ("texels past the end", lib.s3r_update_texels(h, NT - 1, 2, sc.textures.ctypes.data, 0, None)),
            ("texels null", lib.s3r_update_texels(h, 0, 1, None, 0, None)),
            ("texels flag -1", lib.s3r_update_texels(h, 0, 1, sc.textures.ctypes.data, -1, None)),
            ("texels device flagged host", lib.s3r_update_texels(h, 0, 1, ctypes.c_void_p(atl.data_ptr()), 0, None)),
        ]
        for what, rc in rejected:
            assert rc == S3R_E_ARG, f"{what}: {rc}"
        for what, rc in (("vertices", lib.s3r_update_vertices(h, 3, 0, None, 0, None)),
                         ("attributes", lib.s3r_update_attributes(h, A, 0, None, None)),
                         ("texels", lib.s3r_update_texels(h, NT, 0, None, 1, None))):
            assert rc == 0, f"count 0 ({what}): {rc}"
        assert r.kernel_launches == n0, "a rejected or empty update launched a kernel"
        hdr1, pos1 = _clusters_now(r)
        assert same_bits(hdr1, hdr0) and same_bits(pos1, pos0)
        assert_same(r.render(m, W, H)[0], want, "frame after the rejected calls")
        assert_same(np.concatenate([r.render(m, W, H, y0=0, y1=90)[0], r.render(m, W, H, y0=90, y1=H)[0]]), want,
                    "bands after the rejected calls")
        # launches of a render before and after an update (same positions: capacities are settled)
        counts = []
        for _ in range(2):
            for y0, y1 in ((0, H), (0, 90)):
                n1 = r.kernel_launches
                r.render(m, W, H, y0=y0, y1=y1)
                counts.append(r.kernel_launches - n1)
            n1 = r.kernel_launches
            r.update_vertices(dev)
            torch.cuda.synchronize()
            assert r.kernel_launches - n1 == VERTEX_UPDATE_KERNELS
            n1 = r.kernel_launches
            r.update_attributes(sc.attributes)
            r.update_textures(sc.textures)
            assert r.kernel_launches == n1, "attribute and atlas updates are copies"
            r.update_vertices(np.asarray(sc.vertices[:, :3], np.float32))
        assert counts[:2] == counts[2:], f"launches per render before / after an update: {counts}"
    finally:
        r.close()


@pytest.mark.gpu
def test_device_memory_is_stable_over_update_cycles(renderer_lib, oracle_port):
    """Device memory after 50 update + render cycles equals that after the first cycle."""
    import torch
    sc, m, xyz = animation("dense", renderer_lib)
    base = np.asarray(sc.vertices[:, :3], np.float32)
    srcs = [torch.from_numpy(np.ascontiguousarray(s)).cuda() for s in (xyz, base)]
    r = renderer_lib.Renderer(0)
    try:
        r.load_scene(sc)
        for k in range(4):   # capacities for both states
            r.update_vertices(srcs[k % 2])
            r.render(m, W, H, y0=0, y1=90)
            r.render(m, W, H)
        torch.cuda.synchronize()
        free0 = torch.cuda.mem_get_info()[0]
        for k in range(50):
            r.update_vertices(srcs[k % 2] if k % 3 else (xyz if k % 2 == 0 else base))
            r.render(m, W, H, y0=0, y1=90)
            r.render(m, W, H)
        torch.cuda.synchronize()
        assert torch.cuda.mem_get_info()[0] == free0
        want = oracle_port.OracleScene(_with_positions(sc, base)).render(m, W, H)["pixels"]
        assert_same(r.render(m, W, H)[0], want, "after 50 cycles")
    finally:
        r.close()
