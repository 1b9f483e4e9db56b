// cluster.hpp — spatial pre-partition of the triangle stream, built once at scene load (host); a scene update keeps the
// partition and refits the bounds on the device (cluster_refit, kernels.cu).
//
// The reference walks its triangle list front to back every frame (render-cpp/render.cpp:297-317) and rejects most of a
// large scene triangle by triangle.  Here the list is cut into CLUSTERS — runs of consecutive triangles that sit close
// together (at most CL_MAX_VERTS distinct vertices, CL_MAX_TRIS triangles, bounding box no larger than a few of their
// edges) — each with a bounding sphere and its longest edge, so that a whole cluster can be rejected by one
// conservative test (behind the near plane, off screen, outside the rows a GPU owns, or too small to pass the
// `area < 10` cull) before any of its vertices is transformed.  Clusters are stored in Morton order of their centres (what a
// warp of the front kernel touches is close together in space and in memory); every cluster owns private copies of its
// vertices (streamed, coalesced) and its triangles become one 32-bit word each (three cluster-local vertex numbers).
// The reference's processing order survives as the order key: triangle j of a cluster is original triangle t0 + j.
#pragma once
#include <math.h>
#include <stdint.h>
#include <string.h>

#include <vector>

#ifdef __CUDACC__
#define CL_HD __host__ __device__
#else
#define CL_HD
#endif

namespace s3r {

constexpr uint32_t CL_MAX_VERTS = 16;    // distinct vertices per cluster (an icosahedron has 12)
constexpr uint32_t CL_MAX_TRIS = 32;     // triangles per cluster (an icosahedron has 20)
constexpr float CL_SPREAD = 4.0f;        // a cluster's bounding-box diagonal stays within CL_SPREAD of its longest edge

struct ClusterHeader {                   // 32 bytes, two 16-byte loads
    float cx, cy, cz, radius;            // bounding sphere of the cluster's vertices (radius rounded up)
    float max_edge;                      // longest triangle edge in object space (rounded up)
    uint32_t t0;                         // original index of the cluster's first triangle (the rest follow consecutively)
    uint32_t v_off;                      // first entry in the cluster-vertex arrays
    uint32_t tri_off;                    // first entry in the triangle-word array
};
static_assert(sizeof(ClusterHeader) == 32, "ClusterHeader must be 32 bytes");

struct ClusterSet {
    std::vector<ClusterHeader> hdr;      // n_clusters + 1: the last one is a sentinel that carries the end offsets
    std::vector<float> px, py, pz;       // cluster-private vertex copies, in cluster order
    std::vector<uint32_t> src;           // per cluster vertex: the original vertex it copies (scene updates re-gather from it)
    std::vector<uint32_t> tri;           // v0 | v1 << 8 | v2 << 16 (cluster-local vertex numbers), in cluster order
    uint32_t n_clusters = 0;
};

// ---- the bounds rule -----------------------------------------------------------------------------------------------
// One definition for the load-time build (host) and the refit after a scene update (device, cluster_refit in kernels.cu):
// both compile it without contraction (-ffp-contract=off on the host, -fmad=false on the device), so the same partition
// and positions give bit-identical headers.  min / max keep std::min / std::max's argument order (which one wins a tie
// of +0 and -0 is part of the centre's bits).
struct ClusterBounds { float cx, cy, cz, radius, max_edge; };

CL_HD inline double bound_min(double a, double b) { return (b < a) ? b : a; }
CL_HD inline double bound_max(double a, double b) { return (a < b) ? b : a; }
CL_HD inline bool bound_finite(float v) { uint32_t u; memcpy(&u, &v, 4); return (u & 0x7F800000u) != 0x7F800000u; }
CL_HD inline float round_up(double v) {   // smallest-ish binary32 >= v, with one extra ulp of slack
    float f = (float)v;
    if (!(f >= v)) { f = nextafterf(f, INFINITY); }
    return nextafterf(f, INFINITY);
}

// Bounds of a cluster of n_tris triangles over n_verts distinct vertices.  corner(j, c, a): coordinate a of corner c of the
// cluster's triangle j; vert(k, a): coordinate a of its vertex k.  Centre: the double-precision box centre rounded to
// binary32; radius and max_edge: sqrt of the double r^2 / edge^2 times (1 + 1e-9), rounded up.  A non-finite vertex (or
// bound) gives centre 0 and radius = max_edge = inf: bounds that never justify a skip.
#ifdef __CUDACC__
#pragma nv_exec_check_disable
#endif
template <typename Corner, typename Vert>
CL_HD inline ClusterBounds cluster_bounds(uint32_t n_tris, uint32_t n_verts, const Corner &corner, const Vert &vert) {
    double lo[3] = {0, 0, 0}, hi[3] = {0, 0, 0}, max_edge2 = 0;
    for (uint32_t j = 0; j < n_tris; j++) {
        for (int a = 0; a < 3; a++) {
            const double v0 = corner(j, 0, a), v1 = corner(j, 1, a), v2 = corner(j, 2, a);
            const double l = bound_min(v0, bound_min(v1, v2)), h = bound_max(v0, bound_max(v1, v2));
            lo[a] = j == 0 ? l : bound_min(lo[a], l);
            hi[a] = j == 0 ? h : bound_max(hi[a], h);
        }
        double e2 = 0;
        for (int e = 0; e < 3; e++) {
            double d2 = 0;
            for (int a = 0; a < 3; a++) { const double d = (double)corner(j, e, a) - (double)corner(j, (e + 1) % 3, a); d2 += d * d; }
            e2 = bound_max(e2, d2);
        }
        max_edge2 = bound_max(max_edge2, e2);
    }
    ClusterBounds b;
    b.cx = (float)(0.5 * (lo[0] + hi[0])); b.cy = (float)(0.5 * (lo[1] + hi[1])); b.cz = (float)(0.5 * (lo[2] + hi[2]));
    const float c[3] = {b.cx, b.cy, b.cz};
    double r2 = 0;
    bool finite = true;
    for (uint32_t k = 0; k < n_verts; k++) {
        double d2 = 0;
        for (int a = 0; a < 3; a++) { const double d = (double)vert(k, a) - (double)c[a]; d2 += d * d; finite = finite && bound_finite(vert(k, a)); }
        r2 = bound_max(r2, d2);   // (a NaN never wins here; non-finite clusters are handled below)
    }
    b.radius = round_up(sqrt(r2) * (1.0 + 1e-9));
    b.max_edge = round_up(sqrt(max_edge2) * (1.0 + 1e-9));
    if (!finite || !bound_finite(b.radius) || !bound_finite(b.max_edge)) {
        b.cx = b.cy = b.cz = 0.f; b.radius = INFINITY; b.max_edge = INFINITY;
    }
    return b;
}

// positions: planar float[V]; vi0..2: planar uint32[T] (corner k of triangle t).
void build_clusters(const float *px, const float *py, const float *pz, const uint32_t *vi0, const uint32_t *vi1,
                    const uint32_t *vi2, uint64_t T, ClusterSet &out);

}  // namespace s3r
