// cluster.cpp — load-time clustering of the triangle stream (see cluster.hpp).  Host only; no arithmetic of the parity
// chain lives here: clusters only decide which triangles the front kernel may skip, and every skip is justified on the
// device by a conservative test against the bounds computed below (rounded outwards).
#include "cluster.hpp"

#include <math.h>
#include <string.h>

#include <algorithm>
#include <numeric>

namespace s3r {

namespace {

struct Building {
    uint32_t verts[CL_MAX_VERTS];
    uint32_t n_verts = 0, n_tris = 0, t0 = 0;
    double lo[3], hi[3];
    double max_edge2 = 0;
};

struct Raw {            // one finished cluster before sorting
    uint32_t t0, n_tris;
    float cx, cy, cz, radius, max_edge;
    uint32_t morton;
};

inline uint32_t spread3(uint32_t v) {   // 10 bits -> every third bit
    v &= 1023u;
    v = (v | (v << 16)) & 0x030000FFu;
    v = (v | (v << 8)) & 0x0300F00Fu;
    v = (v | (v << 4)) & 0x030C30C3u;
    v = (v | (v << 2)) & 0x09249249u;
    return v;
}

}  // namespace

void build_clusters(const float *px, const float *py, const float *pz, const uint32_t *vi0, const uint32_t *vi1,
                    const uint32_t *vi2, uint64_t T, ClusterSet &out) {
    const float *pos[3] = {px, py, pz};
    std::vector<Raw> raw;
    raw.reserve((size_t)(T / 8 + 16));
    Building cur;

    auto flush = [&]() {
        if (cur.n_tris == 0) { return; }
        Raw r;
        r.t0 = cur.t0; r.n_tris = cur.n_tris;
        const ClusterBounds b = cluster_bounds(
            cur.n_tris, cur.n_verts,
            [&](uint32_t j, int c, int a) { return pos[a][(c == 0 ? vi0 : c == 1 ? vi1 : vi2)[cur.t0 + j]]; },
            [&](uint32_t k, int a) { return pos[a][cur.verts[k]]; });
        r.cx = b.cx; r.cy = b.cy; r.cz = b.cz; r.radius = b.radius; r.max_edge = b.max_edge;
        r.morton = 0;
        raw.push_back(r);
        cur.n_verts = 0; cur.n_tris = 0; cur.max_edge2 = 0;
    };

    for (uint64_t t = 0; t < T; t++) {
        const uint32_t id[3] = {vi0[t], vi1[t], vi2[t]};
        double lo[3], hi[3], e2 = 0;
        for (int a = 0; a < 3; a++) {
            const double v0 = pos[a][id[0]], v1 = pos[a][id[1]], v2 = pos[a][id[2]];
            lo[a] = std::min(v0, std::min(v1, v2)); hi[a] = std::max(v0, std::max(v1, v2));
        }
        for (int e = 0; e < 3; e++) {
            double d2 = 0;
            for (int a = 0; a < 3; a++) { const double d = (double)pos[a][id[e]] - (double)pos[a][id[(e + 1) % 3]]; d2 += d * d; }
            e2 = std::max(e2, d2);
        }
        bool accept = false;
        uint32_t fresh = 0;
        if (cur.n_tris > 0 && cur.n_tris < CL_MAX_TRIS) {
            for (int k = 0; k < 3; k++) {
                bool seen = false;
                for (int j = 0; j < k; j++) { seen = seen || id[j] == id[k]; }
                for (uint32_t j = 0; j < cur.n_verts && !seen; j++) { seen = cur.verts[j] == id[k]; }
                fresh += seen ? 0u : 1u;
            }
            if (cur.n_verts + fresh <= CL_MAX_VERTS) {
                double diag2 = 0;
                for (int a = 0; a < 3; a++) { const double d = std::max(cur.hi[a], hi[a]) - std::min(cur.lo[a], lo[a]); diag2 += d * d; }
                accept = diag2 <= (double)CL_SPREAD * CL_SPREAD * std::max(cur.max_edge2, e2);   // false for NaN
            }
        }
        if (!accept) {
            flush();
            cur.t0 = (uint32_t)t;
            for (int a = 0; a < 3; a++) { cur.lo[a] = lo[a]; cur.hi[a] = hi[a]; }
        } else {
            for (int a = 0; a < 3; a++) { cur.lo[a] = std::min(cur.lo[a], lo[a]); cur.hi[a] = std::max(cur.hi[a], hi[a]); }
        }
        for (int k = 0; k < 3; k++) {
            bool seen = false;
            for (uint32_t j = 0; j < cur.n_verts && !seen; j++) { seen = cur.verts[j] == id[k]; }
            if (!seen) { cur.verts[cur.n_verts++] = id[k]; }
        }
        cur.max_edge2 = std::max(cur.max_edge2, e2);
        cur.n_tris++;
    }
    flush();

    // Morton order of the cluster centres over the scene's bounding box (10 bits per axis)
    float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (const Raw &r : raw) {
        if (!std::isfinite(r.radius)) { continue; }
        const float c[3] = {r.cx, r.cy, r.cz};
        for (int a = 0; a < 3; a++) { lo[a] = std::min(lo[a], c[a]); hi[a] = std::max(hi[a], c[a]); }
    }
    for (Raw &r : raw) {
        if (!std::isfinite(r.radius)) { continue; }
        const float c[3] = {r.cx, r.cy, r.cz};
        uint32_t q[3];
        for (int a = 0; a < 3; a++) {
            const double span = (double)hi[a] - (double)lo[a];
            q[a] = span > 0 ? (uint32_t)std::min(1023.0, ((double)c[a] - lo[a]) / span * 1024.0) : 0u;
        }
        r.morton = spread3(q[0]) | (spread3(q[1]) << 1) | (spread3(q[2]) << 2);
    }
    std::vector<uint32_t> order(raw.size());
    std::iota(order.begin(), order.end(), 0u);
    std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return raw[a].morton < raw[b].morton; });

    out.n_clusters = (uint32_t)raw.size();
    out.hdr.resize(raw.size() + 1);
    out.tri.resize((size_t)T);
    out.px.clear(); out.py.clear(); out.pz.clear(); out.src.clear();
    out.px.reserve((size_t)T); out.py.reserve((size_t)T); out.pz.reserve((size_t)T); out.src.reserve((size_t)T);
    uint32_t tri_off = 0;
    for (size_t k = 0; k < order.size(); k++) {
        const Raw &r = raw[order[k]];
        ClusterHeader &h = out.hdr[k];
        h.cx = r.cx; h.cy = r.cy; h.cz = r.cz; h.radius = r.radius; h.max_edge = r.max_edge;
        h.t0 = r.t0; h.v_off = (uint32_t)out.px.size(); h.tri_off = tri_off;
        uint32_t verts[CL_MAX_VERTS], n_verts = 0;
        for (uint32_t j = 0; j < r.n_tris; j++) {
            const uint64_t t = (uint64_t)r.t0 + j;
            const uint32_t id[3] = {vi0[t], vi1[t], vi2[t]};
            uint32_t local[3];
            for (int c = 0; c < 3; c++) {
                uint32_t at = n_verts;
                for (uint32_t q = 0; q < n_verts; q++) { if (verts[q] == id[c]) { at = q; break; } }
                if (at == n_verts) {
                    verts[n_verts++] = id[c];
                    out.px.push_back(px[id[c]]); out.py.push_back(py[id[c]]); out.pz.push_back(pz[id[c]]);
                    out.src.push_back(id[c]);
                }
                local[c] = at;
            }
            out.tri[tri_off++] = local[0] | (local[1] << 8) | (local[2] << 16);
        }
    }
    ClusterHeader &end = out.hdr[raw.size()];
    memset(&end, 0, sizeof(end));
    end.v_off = (uint32_t)out.px.size(); end.tri_off = tri_off; end.t0 = (uint32_t)T;
}

}  // namespace s3r
