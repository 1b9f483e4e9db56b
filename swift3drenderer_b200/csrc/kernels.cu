// kernels.cu — hand-written sm_100a kernels of the frame pipeline (DESIGN.md section 5).
//
// Small scenes (2T <= 3840), three launches per batch of views:
//   geometry_small     one CTA per view: vertex stage, classify, clip, setup; picks the largest survivors for span_walk
//                                                                                        (render.cpp:285-359, 212-262)
//   span_walk          once per frame: the reference's own row walk of the (<= 8) largest survivors, dropping the
//                      weights at every tile column (whole-frame launches only)          (render.cpp:374-379)
//   tile_raster        per 64x32 tile, 4 CTAs/SM: exact barycentric walk + depth in registers, deferred perspective-
//                      correct shading + rip-map fetch, colour tile in shared memory, cp.async.bulk (TMA) write-out
//                                                                                        (render.cpp:360-382, 124-132)
// General path (visibility buffer of 64-bit depth|order keys), six launches per frame:
//   vertex_stage       K1   model/view/projection over planar float4 position streams   (render.cpp:285-289)
//   triangle_classify  K2a  near reject / straddle / cull with warp-ballot compaction; unclipped triangles under 16x16
//                           pixels are walked right here, record-free                    (render.cpp:297-317, 360-382)
//   triangle_setup     K2b  gather, near-plane clip (0/1/2 out), setup records, block-scan compaction, inline binning
//                                                                                        (render.cpp:297-359, 212-262)
//   post_setup         K3   cooperative binning of the largest triangles, their row-start blocks, flat row walk of
//                           recorded triangles under 128x128, tile work queue + overflow record
//   tile_raster_queue  K4   tile kernel over (tile, chunk) items for triangles over 128 pixels
//   shade_tiles        K5   visibility buffer -> colour: per 32x32 block, distinct triangles set up once, one covered
//                           pixel per lane; clears the keys; optional fused frame assembly into peer frames
//                                                                                        (render.cpp:363-372, 339-359, 124-132)
//
// PARITY RULES (see DESIGN.md): this translation unit is compiled with -fmad=false -prec-div=true
// -prec-sqrt=true -ftz=false; every expression is written in the reference's evaluation order so
// that each binary32 intermediate equals the CPU's.  Do not "simplify" arithmetic here.  The only
// hand-scheduled operators are in exact_math.cuh (device-checked against the compiler's, bit for bit).
#include <cstddef>
#include <type_traits>
#include "pipeline.cuh"
#include "cluster.hpp"
#include "walk.cuh"
#include "exact_math.cuh"

namespace s3r {

// ------------------------------------------------------------------------------------------------
// small helpers
// ------------------------------------------------------------------------------------------------
struct Cam { float m[12]; };

// The view's 3 x 4 camera matrix: from the parameter block when the submission has a single view (no upload, no global
// load), otherwise from the uploaded array.
__device__ __forceinline__ Cam load_cam(const Frame &f, uint32_t view) {
    Cam c;
    if (f.cam_inline) {
#pragma unroll
        for (int i = 0; i < 12; i++) { c.m[i] = f.cam0[i]; }
    } else {
        const float *p = f.cams + 12 * view;
#pragma unroll
        for (int i = 0; i < 12; i++) { c.m[i] = __ldg(p + i); }
    }
    return c;
}

// simd_mul(float4x3, float4) = ((c0*x + c1*y) + c2*z) + c3*w
__device__ __forceinline__ float3 xform(const Cam &c, float x, float y, float z, float w) {
    return make_float3(((c.m[0] * x + c.m[1] * y) + c.m[2] * z) + c.m[3] * w,
                       ((c.m[4] * x + c.m[5] * y) + c.m[6] * z) + c.m[7] * w,
                       ((c.m[8] * x + c.m[9] * y) + c.m[10] * z) + c.m[11] * w);
}

// render.cpp:288 — (v.x, -v.y, 0) * factor / -v.z + (W/2, H/2, -v.z)
__device__ __forceinline__ float3 project(float3 cv, float factor, float half_w, float half_h) {
    const float nz = -cv.z;
    // the two quotients share one reciprocal refinement (exact_math.cuh: bit-identical to the `/` operator, checked on
    // the device); the third component, 0 * factor / nz + nz, IS nz unless nz is zero (0 / 0): +-0 / nz is a zero for
    // every other nz, infinities included, and x + (+-0) == x
    float qx, qy;
    div2_rn_signed(cv.x * factor, -cv.y * factor, nz, qx, qy);
    return make_float3(qx + half_w, qy + half_h, nz != 0.f ? nz : 0.f * factor / nz + nz);
}

__device__ __forceinline__ float3 add3(float3 a, float3 b) { return make_float3(a.x + b.x, a.y + b.y, a.z + b.z); }
__device__ __forceinline__ float3 scale3(float3 a, float s) { return make_float3(a.x * s, a.y * s, a.z * s); }
__device__ __forceinline__ float dot3(float3 a, float3 b) { return (a.x * b.x + a.y * b.y) + a.z * b.z; }
// simd_fast_normalize as pinned by the oracle shim: v * (1 / sqrt(dot(v, v)))
// (1.0f / x is the correctly rounded reciprocal, and so is __frcp_rn(x): same bits, fewer instructions)
__device__ __forceinline__ float3 unit3(float3 a) { return scale3(a, inv_sqrt_rn(dot3(a, a))); }   // == __frcp_rn(__fsqrt_rn(.)), exact_math.cuh
// EDGE_FUNCTION(a, b, c), render.cpp:9
__device__ __forceinline__ float edge_fn(float ax, float ay, float bx, float by, float cx, float cy) {
    return (cx - ax) * (ay - by) + (cy - ay) * (bx - ax);
}

__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31u; }

// Programmatic dependent launch: the general path's kernels are launched with programmatic stream serialization, so a
// kernel's CTAs are placed while its predecessor drains and wait here — before they touch anything the predecessor wrote —
// until it has completed and flushed.  Without the launch attribute this is a no-op.
__device__ __forceinline__ void wait_for_predecessor() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// fire-and-forget 64-bit max on a visibility key: always the reduction form (REDG.E.MAX.64).  atomicMax() with an unused
// result is sometimes compiled to the returning ATOMG form instead, and a walk loop then waits for each atomic to
// come back before it may reuse the address registers (45 % of post_setup's warp time on the clipping-stress scene).
__device__ __forceinline__ void red_max_u64(unsigned long long *p, unsigned long long v) {
    asm volatile("red.global.max.u64 [%0], %1;" :: "l"(p), "l"(v) : "memory");
}

// n sequential additions of d onto s (render.cpp:374-379): true steps when the target is near, the exact
// jump (walk.cuh) otherwise.  Both give the same bits; the loop is cheaper for short distances.
__device__ __forceinline__ float walk_near(float s, float d, uint32_t n) {
    if (n > 24u) { return walk_jump(s, d, n); }
    for (uint32_t i = 0; i < n; i++) { s = add_rn(s, d); }
    return s;
}

// The weight at box offset (nx, ny) from the one at the box's first pixel: down ny rows (render.cpp:378), then nx pixels
// along the row (render.cpp:374), each by walk_near.
__device__ __forceinline__ float weight_at(float ws, float dy, uint32_t ny, float dx, uint32_t nx) {
    return walk_near(walk_near(ws, dy, ny), dx, nx);
}

// mark on a tile-list entry: this small triangle passed a depth pre-check in pass 1 (top bit of the entry type)
constexpr uint32_t SMALL_MAX = 16;      // triangles whose whole bbox is narrower and lower than this take the per-triangle path

// ------------------------------------------------------------------------------------------------
// K0 — reset
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void reset_body(const Frame &f, uint32_t view, uint32_t i, uint32_t stride) {
    if (!f.counters) { return; }   // (vertex stage re-run for a raster-vertex dump: the frame's counters stay)
    if (i < C_COUNT) { f.counters[view * C_COUNT + i] = 0; }
    for (uint32_t t = i; t < f.n_tiles; t += stride) { f.tile_count[view * f.tile_stride + t] = 0; }
}

// ------------------------------------------------------------------------------------------------
// K1 — vertex stage: 4 vertices per thread, float4 loads of the planar streams, float4 stores.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void vertex_body(const Frame &f, const Cam &cam, uint32_t view, uint32_t i4) {
    const float4 x = __ldg(reinterpret_cast<const float4 *>(f.pos_x + i4));
    const float4 y = __ldg(reinterpret_cast<const float4 *>(f.pos_y + i4));
    const float4 z = __ldg(reinterpret_cast<const float4 *>(f.pos_z + i4));
    float4 *out = f.rv + (size_t)view * f.Vpad + i4;
    const float xs[4] = {x.x, x.y, x.z, x.w}, ys[4] = {y.x, y.y, y.z, y.w}, zs[4] = {z.x, z.y, z.z, z.w};
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const float3 cv = xform(cam, xs[k], ys[k], zs[k], 1.0f);
        const float3 rv = project(cv, f.factor, f.half_w, f.half_h);
        out[k] = make_float4(rv.x, rv.y, rv.z, 0.f);
    }
}

__global__ void __launch_bounds__(256) vertex_stage(const __grid_constant__ Frame f) {
    // first kernel of a frame: also zeroes the per-view counters and tile histograms (no separate reset launch)
    reset_body(f, blockIdx.y, blockIdx.x * blockDim.x + threadIdx.x, gridDim.x * blockDim.x);
    const uint32_t i4 = (blockIdx.x * blockDim.x + threadIdx.x) * 4u;
    if (i4 >= f.Vpad) { return; }
    vertex_body(f, load_cam(f, blockIdx.y), blockIdx.y, i4);
}

// ------------------------------------------------------------------------------------------------
// K2 — triangle setup
// ------------------------------------------------------------------------------------------------
struct Corner {
    float3 cv, rv, n;
    uint4 pay;      // raw payload words: colour = floats 0..2; texture = {index, -, u, v}
    uint32_t kind;
};

__device__ __forceinline__ float3 lerp3(float3 a, float3 b, float u, float t) {  // x*(1-a) + y*a
    return add3(scale3(a, u), scale3(b, t));
}

// render.cpp:222-236 — the vertex where edge (a -> b) meets z = near
__device__ __forceinline__ Corner clip_vertex(const Corner &a, const Corner &b, uint32_t kind0, const Frame &f) {
    const float t = (kNear - a.rv.z) / (b.rv.z - a.rv.z);
    const float u = 1 - t;
    Corner c;
    c.cv = lerp3(a.cv, b.cv, u, t);
    c.rv = make_float3(c.cv.x * f.factor / kNear + f.half_w, -c.cv.y * f.factor / kNear + f.half_h,
                       0.f * f.factor / kNear + kNear);
    c.kind = kind0;
    c.pay = make_uint4(0, 0, 0, 0);
    if (kind0 == 0) {
        const float3 ca = make_float3(__uint_as_float(a.pay.x), __uint_as_float(a.pay.y), __uint_as_float(a.pay.z));
        const float3 cb = make_float3(__uint_as_float(b.pay.x), __uint_as_float(b.pay.y), __uint_as_float(b.pay.z));
        const float3 col = lerp3(ca, cb, u, t);
        c.pay.x = __float_as_uint(col.x); c.pay.y = __float_as_uint(col.y); c.pay.z = __float_as_uint(col.z);
    } else if (kind0 == 1) {
        c.pay.x = a.pay.x;  // texture index of the edge's first endpoint, render.cpp:233
        c.pay.z = __float_as_uint(__uint_as_float(a.pay.z) * u + __uint_as_float(b.pay.z) * t);
        c.pay.w = __float_as_uint(__uint_as_float(a.pay.w) * u + __uint_as_float(b.pay.w) * t);
    }
    c.n = lerp3(a.n, b.n, u, t);
    return c;
}

// A triangle's screen bounds from its raster-space vertices (render.cpp:311-321): the float extremes the culls compare, and
// the pixel box clamped to the frame.  One definition for every kernel that routes, sets up or re-derives a triangle, so
// that all of them find the same box.
struct Bounds { float min_x, max_x, min_y, max_y; uint32_t xmin, xmax, ymin, ymax; };

__device__ __forceinline__ Bounds bounds_of(const Frame &f, float x0, float y0, float x1, float y1, float x2, float y2) {
    const float max_x = fmaxf(fmaxf(x0, x1), x2), max_y = fmaxf(fmaxf(y0, y1), y2);
    const float min_x = fminf(fminf(x0, x1), x2), min_y = fminf(fminf(y0, y1), y2);
    return {min_x, max_x, min_y, max_y, (uint32_t)fmaxf(0, min_x), (uint32_t)fminf(f.fw - 1, max_x),
            (uint32_t)fmaxf(0, min_y), (uint32_t)fminf(f.fh - 1, max_y)};
}

// The coverage half of the setup (render.cpp:318-334): barycentric weights at the first pixel centre, their
// per-pixel / per-row increments, 1/z per corner.  One function for every place that needs these values (setup
// records, the classify kernel's direct walk, deferred shading) so that all of them produce the same bits.
struct VisCore { float ws[3], dx[3], dy[3], rz[3]; };

__device__ __forceinline__ void vis_core(float3 a, float3 b, float3 c, float area, uint32_t xmin, uint32_t ymin, VisCore &o) {
    const float inv_area = __frcp_rn(area);  // 1 / area
    const float px = (float)xmin + 0.5f, py = (float)ymin + 0.5f;
    o.ws[0] = edge_fn(b.x, b.y, c.x, c.y, px, py) * inv_area;
    o.ws[1] = edge_fn(c.x, c.y, a.x, a.y, px, py) * inv_area;
    o.ws[2] = edge_fn(a.x, a.y, b.x, b.y, px, py) * inv_area;
    o.dx[0] = (b.y - c.y) * inv_area; o.dx[1] = (c.y - a.y) * inv_area; o.dx[2] = (a.y - b.y) * inv_area;
    o.dy[0] = (c.x - b.x) * inv_area; o.dy[1] = (a.x - c.x) * inv_area; o.dy[2] = (b.x - a.x) * inv_area;
    o.rz[0] = __frcp_rn(a.z); o.rz[1] = __frcp_rn(b.z); o.rz[2] = __frcp_rn(c.z);  // 1 / z
}

// A survivor's head {xmin | xmax << 16, ymin | ymax << 16, order, kind} (Frame::head): the first 16 bytes of its SetupVis
// record, also stored alone for the kernels that only bin or size a triangle.
struct Head { uint32_t xmin, xmax, ymin, ymax, order, kind; };
static_assert(offsetof(SetupVis, xmin) == 0 && offsetof(SetupVis, xmax) == 2 && offsetof(SetupVis, ymin) == 4 &&
              offsetof(SetupVis, ymax) == 6 && offsetof(SetupVis, order) == 8 && offsetof(SetupVis, kind) == 12,
              "a head is the first 16 bytes of a SetupVis record");

__device__ __forceinline__ Head unpack_head(uint4 h) { return {h.x & 0xFFFFu, h.x >> 16, h.y & 0xFFFFu, h.y >> 16, h.z, h.w}; }

// A SetupVis record read as four 16-byte words (in any memory space), its fields by name.
struct VisRecord { Head head; VisCore c; };
static_assert(offsetof(SetupVis, wstart) == 16 && offsetof(SetupVis, dx) == 28 && offsetof(SetupVis, dy) == 40 &&
              offsetof(SetupVis, rvz) == 52, "load_vis reads the coverage fields of SetupVis at these offsets");

__device__ __forceinline__ VisRecord load_vis(const SetupVis *p) {
    const uint4 *q = reinterpret_cast<const uint4 *>(p);
    const uint4 q0 = q[0], q1 = q[1], q2 = q[2], q3 = q[3];
    VisRecord r;
    r.head = unpack_head(q0);
    r.c.ws[0] = __uint_as_float(q1.x); r.c.ws[1] = __uint_as_float(q1.y); r.c.ws[2] = __uint_as_float(q1.z);
    r.c.dx[0] = __uint_as_float(q1.w); r.c.dx[1] = __uint_as_float(q2.x); r.c.dx[2] = __uint_as_float(q2.y);
    r.c.dy[0] = __uint_as_float(q2.z); r.c.dy[1] = __uint_as_float(q2.w); r.c.dy[2] = __uint_as_float(q3.x);
    r.c.rz[0] = __uint_as_float(q3.y); r.c.rz[1] = __uint_as_float(q3.z); r.c.rz[2] = __uint_as_float(q3.w);
    return r;
}

// render.cpp:311-359.  Returns false when the triangle is culled.
__device__ __forceinline__ bool make_setup(const Corner &d0, const Corner &d1, const Corner &d2, uint32_t order,
                                           const Frame &f, SetupVis &v, SetupShade &s) {
    const float area = edge_fn(d0.rv.x, d0.rv.y, d1.rv.x, d1.rv.y, d2.rv.x, d2.rv.y);
    const Bounds b = bounds_of(f, d0.rv.x, d0.rv.y, d1.rv.x, d1.rv.y, d2.rv.x, d2.rv.y);
    if (b.max_x < 0 || b.max_y < 0) { return false; }
    if (b.min_x >= f.fw || b.min_y >= f.fh) { return false; }
    if (area < 10) { return false; }
    v.xmin = (uint16_t)b.xmin; v.xmax = (uint16_t)b.xmax; v.ymin = (uint16_t)b.ymin; v.ymax = (uint16_t)b.ymax;
    v.order = order;
    v.kind = d0.kind;
    VisCore vc;
    vis_core(d0.rv, d1.rv, d2.rv, area, b.xmin, b.ymin, vc);
#pragma unroll
    for (int k = 0; k < 3; k++) { v.wstart[k] = vc.ws[k]; v.dx[k] = vc.dx[k]; v.dy[k] = vc.dy[k]; v.rvz[k] = vc.rz[k]; }
    const Corner *d[3] = {&d0, &d1, &d2};
#pragma unroll
    for (int k = 0; k < 3; k++) {
        const float3 c = scale3(d[k]->cv, v.rvz[k]), n = scale3(d[k]->n, v.rvz[k]);
        s.cv[3 * k] = c.x; s.cv[3 * k + 1] = c.y; s.cv[3 * k + 2] = c.z;
        s.n[3 * k] = n.x; s.n[3 * k + 1] = n.y; s.n[3 * k + 2] = n.z;
    }
    s.kind = d0.kind;
    s.texture = 0;
    s.area = area;
    s.tpp[0] = 0.f; s.tpp[1] = 0.f;
    if (d0.kind == 0) {
#pragma unroll
        for (int k = 0; k < 3; k++) {
            s.pay[3 * k] = __uint_as_float(d[k]->pay.x) * v.rvz[k];
            s.pay[3 * k + 1] = __uint_as_float(d[k]->pay.y) * v.rvz[k];
            s.pay[3 * k + 2] = __uint_as_float(d[k]->pay.z) * v.rvz[k];
        }
    } else {
        s.texture = d0.pay.x % f.n_tex;   // valid scenes: unchanged (checked at load); a mixed-kind triangle's reinterpreted payload stays inside the atlases
#pragma unroll
        for (int k = 0; k < 3; k++) {
            s.pay[2 * k] = __uint_as_float(d[k]->pay.z) * v.rvz[k];
            s.pay[2 * k + 1] = __uint_as_float(d[k]->pay.w) * v.rvz[k];
        }
        s.pay[6] = (v.rvz[0] * v.dx[0] + v.rvz[1] * v.dx[1]) + v.rvz[2] * v.dx[2];  // dz.x = dot(rvz, dx)
        s.pay[7] = (v.rvz[0] * v.dy[0] + v.rvz[1] * v.dy[1]) + v.rvz[2] * v.dy[2];  // dz.y = dot(rvz, dy)
        s.pay[8] = 0.f;
        s.tpp[0] = (s.pay[0] * v.dx[0] + s.pay[2] * v.dx[1]) + s.pay[4] * v.dx[2];
        s.tpp[1] = (s.pay[1] * v.dy[0] + s.pay[3] * v.dy[1]) + s.pay[5] * v.dy[2];
    }
    return true;
}

// Conservative trivial reject of a (triangle, tile) pair: true only if one barycentric weight is
// provably negative at every pixel of the tile (clipped to the bbox), i.e. no pixel there can pass the
// inside test (render.cpp:362), so skipping the pair cannot change the frame.
// The walked weight differs from the real-valued linear function L(x, y) = wstart + (x - xmin) dx +
// (y - ymin) dy only by accumulated rounding: each of the at most (bw + bh) additions is off by at most
// half an ulp, i.e. 2^-24 of the largest magnitude on the way (<= max |L| over the bbox corners).  The
// margin used is more than twice that bound plus the error of evaluating L in binary32 here.
__device__ __forceinline__ bool tile_outside_triangle(const SetupVis &v, uint32_t tx0, uint32_t ylo_t, uint32_t yhi_t) {
    const uint32_t x0 = max(tx0, (uint32_t)v.xmin), x1 = min(tx0 + TILE_W - 1u, (uint32_t)v.xmax);
    const uint32_t y0 = max(ylo_t, (uint32_t)v.ymin), y1 = min(yhi_t - 1u, (uint32_t)v.ymax);
    const float bw = (float)(v.xmax - v.xmin), bh = (float)(v.ymax - v.ymin);
    const float fx0 = (float)(x0 - v.xmin), fx1 = (float)(x1 - v.xmin), fy0 = (float)(y0 - v.ymin), fy1 = (float)(y1 - v.ymin);
#pragma unroll
    for (int c = 0; c < 3; c++) {
        const float ws = v.wstart[c], dx = v.dx[c], dy = v.dy[c];
        const float wmax = fabsf(ws) + fabsf(dx) * bw + fabsf(dy) * bh;          // >= max |L| over the bbox
        const float margin = (bw + bh + 16.f) * 2.4e-7f * (wmax + 1.f);
        const float best = ws + (dx > 0.f ? fx1 : fx0) * dx + (dy > 0.f ? fy1 : fy0) * dy;   // max of L over the rectangle
        if (best < -margin) { return true; }
    }
    return false;
}

// Tile-row ownership.  Absolute tile row `a` (counted from the top of the full frame) belongs to this
// submission iff it meets the band [y0, y1) and a % row_stride == row_phase.  row_stride == 1 is the
// contiguous band; row_stride == n GPUs interleaves the tile rows for load balance.  The local row index
// (grid row, tile arrays, compacted output) is a - tile_row0 resp. a / row_stride.
// a / row_stride and a % row_stride without a hardware division (exact for a * row_stride < 2^32; row_stride > 1)
__device__ __forceinline__ uint32_t div_stride(const Frame &f, uint32_t a) { return __umulhi(a, f.rs_magic); }
__device__ __forceinline__ uint32_t mod_stride(const Frame &f, uint32_t a) { return a - div_stride(f, a) * f.row_stride; }
__device__ __forceinline__ bool owns_row(const Frame &f, uint32_t a) { return f.row_stride == 1u || mod_stride(f, a) == f.row_phase; }
__device__ __forceinline__ uint32_t local_row(const Frame &f, uint32_t a) { return f.row_stride == 1u ? a - f.tile_row0 : div_stride(f, a); }
__device__ __forceinline__ uint32_t abs_row(const Frame &f, uint32_t l) { return f.row_stride == 1u ? l + f.tile_row0 : l * f.row_stride + f.row_phase; }
// output row of pixel row yy (inside absolute tile row a)
__device__ __forceinline__ size_t out_row(const Frame &f, uint32_t yy, uint32_t a) {
    return f.row_stride == 1u ? (size_t)(yy - f.y0) : (size_t)(div_stride(f, a) * TILE_H + (yy - a * TILE_H));
}
// pixel row of output row r (inverse of out_row)
__device__ __forceinline__ uint32_t pixel_y(const Frame &f, uint32_t r) {
    return f.row_stride == 1u ? r + f.y0 : ((r / TILE_H) * f.row_stride + f.row_phase) * TILE_H + r % TILE_H;
}
// position of the key of output row r, column x inside a view's key plane (see Frame::keys): columns of 4 rows per sector;
// one step along x is 4 keys
constexpr uint32_t KEY_STEP = 4;
__device__ __forceinline__ size_t key_at(const Frame &f, size_t r, uint32_t x) { return ((r >> 2) * f.W + x) * KEY_STEP + (r & 3u); }
// The reference's walk along one pixel row (render.cpp:362-364, 374) from pixel x0, where the weights are w, to pixel x1:
// every covered pixel x publishes its key depth << 32 | key_lo to krow[KEY_STEP * x] — depth starts at 0, strict '>'
// (render.cpp:364) — with a fire-and-forget red.max that nothing waits for.
__device__ __forceinline__ void publish_row(unsigned long long *krow, uint32_t x0, uint32_t x1, float3 w, float3 d, float3 rz,
                                            unsigned long long key_lo) {
    for (uint32_t x = x0; x <= x1; x++) {
        const bool inside = w.x >= 0 && w.y >= 0 && w.z >= 0;                  // render.cpp:362
        const float ooz = (rz.x * w.x + rz.y * w.y) + rz.z * w.z;              // render.cpp:363
        if (inside && ooz > 0.f) { red_max_u64(krow + KEY_STEP * x, ((unsigned long long)__float_as_uint(ooz) << 32) | key_lo); }
        w.x = add_rn(w.x, d.x); w.y = add_rn(w.y, d.y); w.z = add_rn(w.z, d.z);   // render.cpp:374
    }
}
__device__ __forceinline__ uint32_t owned_rows_in(const Frame &f, uint32_t a0, uint32_t a1) {   // #owned rows in [a0, a1]
    if (f.row_stride == 1u) { return a1 - a0 + 1u; }
    const uint32_t first = a0 + mod_stride(f, f.row_phase + f.row_stride - mod_stride(f, a0));
    return first > a1 ? 0u : div_stride(f, a1 - first) + 1u;
}

// Pixel rows of [ylo, yhi] this submission owns, as a count and an index -> row map (flat walk work items).
// Interleaved ownership: the first owned tile row may be cut by ylo, the last by yhi, the ones between are whole.
struct OwnedRows { uint32_t count, first_y, first_n, next_a; };

__device__ __forceinline__ OwnedRows owned_pixel_rows(const Frame &f, uint32_t ylo, uint32_t yhi) {
    OwnedRows o;
    if (f.row_stride == 1u) { o.count = yhi - ylo + 1u; o.first_y = ylo; o.first_n = o.count; o.next_a = 0; return o; }
    const uint32_t a0 = ylo / TILE_H, a1 = yhi / TILE_H;
    const uint32_t af = a0 + mod_stride(f, f.row_phase + f.row_stride - mod_stride(f, a0));   // first owned tile row >= a0
    if (af > a1) { o.count = 0; o.first_y = 0; o.first_n = 0; o.next_a = 0; return o; }
    o.first_y = max(ylo, af * TILE_H);
    o.first_n = min(yhi, af * TILE_H + TILE_H - 1u) - o.first_y + 1u;
    o.next_a = af + f.row_stride;
    o.count = o.first_n;
    if (o.next_a <= a1) {
        const uint32_t more = div_stride(f, a1 - o.next_a) + 1u, last = o.next_a + (more - 1u) * f.row_stride;   // owned tile rows after the first
        o.count += (more - 1u) * TILE_H + (min(yhi, last * TILE_H + TILE_H - 1u) - last * TILE_H + 1u);
    }
    return o;
}
__device__ __forceinline__ uint32_t owned_row_at(const Frame &f, const OwnedRows &o, uint32_t i) {
    if (i < o.first_n) { return o.first_y + i; }
    const uint32_t j = i - o.first_n;
    return (o.next_a + (j / TILE_H) * f.row_stride) * TILE_H + j % TILE_H;
}

struct TileRange { uint32_t tx0, tx1, a0, a1; bool empty; };   // tile columns and ABSOLUTE tile rows, clamped to the band

__device__ __forceinline__ TileRange tile_range(const Frame &f, uint32_t xmin, uint32_t xmax, uint32_t ymin, uint32_t ymax) {
    TileRange r;
    const uint32_t ylo = max(ymin, f.y0), yhi = min(ymax, f.y1 - 1u);
    r.empty = ylo > yhi;
    r.tx0 = xmin / TILE_W; r.tx1 = xmax / TILE_W;
    r.a0 = ylo / TILE_H; r.a1 = yhi / TILE_H;
    return r;
}

// Single-pass binning: every tile owns a fixed-capacity list (tile_cap slots); one atomic reserves the
// position.  Lists are unordered (the depth keys carry the order).  Overflowing tiles are detected by
// post_setup's closing step; the host regrows tile_cap and renders the frame again.
__device__ __forceinline__ void bin_one(const Frame &f, uint32_t view, uint32_t tile, uint32_t slot) {
    const uint32_t pos = atomicAdd(f.tile_count + view * f.tile_stride + tile, 1u);
    if (pos < f.tile_cap) { f.entries[((size_t)view * f.tile_stride + tile) * f.tile_cap + pos] = slot; }
}

struct SetupShared {
    uint32_t list[256];
    uint32_t count;
    uint32_t stats[4];   // near, clipped, spawned, culled
    uint32_t warp_sum[8];
    uint32_t base;
};

// Block-wide ordered slot allocation for `keep` flags: warp ballot -> per-warp counts -> one
// global atomicAdd per block -> slot.  All 256 threads must call.
__device__ __forceinline__ uint32_t allocate_slots(bool keep, uint32_t *global_counter, SetupShared &sh) {
    const uint32_t mask = __ballot_sync(0xFFFFFFFFu, keep);
    const uint32_t warp = threadIdx.x >> 5, lane = lane_id();
    if (lane == 0) { sh.warp_sum[warp] = __popc(mask); }
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t total = 0;
#pragma unroll
        for (int w = 0; w < 8; w++) { const uint32_t c = sh.warp_sum[w]; sh.warp_sum[w] = total; total += c; }
        sh.base = total ? atomicAdd(global_counter, total) : 0u;
    }
    __syncthreads();
    const uint32_t slot = sh.base + sh.warp_sum[warp] + __popc(mask & ((1u << lane) - 1u));
    __syncthreads();  // warp_sum/base reusable by the next call
    return slot;
}

__device__ __forceinline__ void store_setup(const Frame &f, uint32_t view, uint32_t slot, const SetupVis &v,
                                            const SetupShade &s) {
    uint4 *dv = reinterpret_cast<uint4 *>(f.vis + (size_t)view * f.setup_cap + slot);
    const uint4 *sv = reinterpret_cast<const uint4 *>(&v);
#pragma unroll
    for (int i = 0; i < 4; i++) { dv[i] = sv[i]; }
    uint4 *ds = reinterpret_cast<uint4 *>(f.shade + (size_t)view * f.setup_cap + slot);
    const uint4 *ss = reinterpret_cast<const uint4 *>(&s);
#pragma unroll
    for (int i = 0; i < 8; i++) { ds[i] = ss[i]; }
    f.head[(size_t)view * f.setup_cap + slot] = sv[0];   // bbox + order key + kind: all binning needs
    if (!f.direct_bin) { f.slot_of[(size_t)view * 2u * f.T + v.order] = slot; }   // lets a depth key find its triangle again
}

__device__ __forceinline__ bool is_small_bbox(uint32_t xmin, uint32_t xmax, uint32_t ymin, uint32_t ymax) {
    return xmax - xmin < SMALL_MAX && ymax - ymin < SMALL_MAX;
}
// The record-free route: with direct_small, a triangle that does not straddle the near plane (z: its corners' raster z) and
// whose pixel box is under SMALL_MAX x SMALL_MAX is walked straight from its raster-space vertices and shaded from the raw
// scene; it never gets a setup record.  The front kernels route by this rule and shade_tiles finds records by it.
__device__ __forceinline__ bool is_record_free(const Frame &f, float z0, float z1, float z2, const Bounds &b) {
    return f.direct_small && !(fminf(fminf(z0, z1), z2) < kNear) && is_small_bbox(b.xmin, b.xmax, b.ymin, b.ymax);
}
// Recorded triangles whose box stays under flat_max pixels in both directions are walked row by row straight into the
// visibility buffer (post_setup); only larger ones pay for tile binning and the tile kernel.
__device__ __forceinline__ bool is_flat_bbox(const Frame &f, uint32_t xmin, uint32_t xmax, uint32_t ymin, uint32_t ymax) {
    return xmax - xmin < f.flat_max && ymax - ymin < f.flat_max;
}

// K3 for one survivor, fused into setup: triangles over few tiles are binned right here (with the
// conservative outside test), everything larger goes to the cooperative big list.
__device__ __forceinline__ void count_tiles(const Frame &f, uint32_t view, uint32_t slot, const SetupVis &v) {
    const TileRange r = tile_range(f, v.xmin, v.xmax, v.ymin, v.ymax);
    if (r.empty) { return; }
    const uint32_t ntiles = (r.tx1 - r.tx0 + 1u) * owned_rows_in(f, r.a0, r.a1);
    if (ntiles == 0u) { return; }
    if (ntiles > BIG_TILES) {
        const uint32_t pos = atomicAdd(f.counters + view * C_COUNT + C_BIG, 1u);
        if (pos < f.big_cap) { f.big_list[(size_t)view * f.big_cap + pos] = slot; }
        else { atomicOr(f.counters + view * C_COUNT + C_OVERFLOW, 4u); }
        return;
    }
    for (uint32_t a = r.a0; a <= r.a1; a++) {
        if (!owns_row(f, a)) { continue; }
        const uint32_t ya = a * TILE_H, ylo_t = max(ya, f.y0), yhi_t = min(ya + TILE_H, f.y1);
        for (uint32_t tx = r.tx0; tx <= r.tx1; tx++) {
            if (ntiles > 1u && tile_outside_triangle(v, tx * TILE_W, ylo_t, yhi_t)) { continue; }
            bin_one(f, view, local_row(f, a) * f.tiles_x + tx, slot);
        }
    }
}

__device__ __forceinline__ void emit_block(bool valid, const Corner &d0, const Corner &d1, const Corner &d2,
                                           uint32_t order, const Frame &f, uint32_t view, SetupShared &sh,
                                           bool count_culled) {
    SetupVis v;
    SetupShade s;
    const bool keep = valid && make_setup(d0, d1, d2, order, f, v, s);
    if (count_culled) {
        const uint32_t culled = __ballot_sync(0xFFFFFFFFu, valid && !keep);
        if (lane_id() == 0 && culled) { atomicAdd(&sh.stats[3], __popc(culled)); }
    }
    const uint32_t slot = allocate_slots(keep, f.counters + view * C_COUNT + C_SETUPS, sh);
    if (keep) {
        if (slot < f.setup_cap) {
            store_setup(f, view, slot, v, s);
            // general path: only triangles too large for the flat per-triangle walk are binned into tiles
            if (!f.direct_bin && !is_flat_bbox(f, v.xmin, v.xmax, v.ymin, v.ymax)) { count_tiles(f, view, slot, v); }
        } else {
            atomicOr(f.counters + view * C_COUNT + C_OVERFLOW, 1u);
        }
    }
}

// HAS_RV: the vertex stage left raster-space vertices in HBM (raw-stream front, small scenes); otherwise (cluster front,
// which keeps them on chip) the vertex stage's own expression is evaluated again — the same bits.
template <bool HAS_RV>
__device__ __forceinline__ Corner gather_corner(const Frame &f, const Cam &cam, uint32_t view, uint32_t vi, uint32_t ai) {
    Corner c;
    c.cv = xform(cam, __ldg(f.pos_x + vi), __ldg(f.pos_y + vi), __ldg(f.pos_z + vi), 1.0f);
    if (HAS_RV) {
        const float4 r = f.rv[(size_t)view * f.Vpad + vi];
        c.rv = make_float3(r.x, r.y, r.z);
    } else {   // cluster front: raster-space vertices never reach HBM; the vertex stage's own expression gives the same bits
        c.rv = project(c.cv, f.factor, f.half_w, f.half_h);
    }
    const uint4 a = __ldg(f.attr + 2 * (size_t)ai);
    c.n = xform(cam, __uint_as_float(a.x), __uint_as_float(a.y), __uint_as_float(a.z), 0.0f);
    c.kind = a.w;
    c.pay = __ldg(f.attr + 2 * (size_t)ai + 1);
    return c;
}

constexpr uint32_t ITEM_STRADDLE = 0x80000000u;

// clip(), render.cpp:212-262.  On return d0..d2 hold the in-place triangle; when two corners were in
// front, (s0, s1, s2) is the appended triangle (current, I_np, I_pc) and the function returns true.
__device__ __forceinline__ bool clip_near(Corner &d0, Corner &d1, Corner &d2, Corner &s0, Corner &s1, Corner &s2,
                                          const Frame &f) {
    const bool f0 = d0.rv.z > kNear, f1 = d1.rv.z > kNear, f2 = d2.rv.z > kNear;
    const uint32_t kind0 = d0.kind;  // render.cpp:225: the kind always comes from corner 0
    // The edge whose endpoints lie on the same side fixes (current, next, preceding); the loop in
    // the reference keeps the last such edge.
    int cur = 0;
    if (f0 == f1) { cur = 0; }
    if (f1 == f2) { cur = 1; }
    if (f2 == f0) { cur = 2; }
    const Corner c = cur == 0 ? d0 : (cur == 1 ? d1 : d2);  // current
    const Corner n = cur == 0 ? d1 : (cur == 1 ? d2 : d0);  // next
    const Corner p = cur == 0 ? d2 : (cur == 1 ? d0 : d1);  // preceding
    const bool two_in_front = c.rv.z > kNear;
    const Corner i_np = clip_vertex(n, p, kind0, f);  // data_new[next]:      edge next -> preceding
    const Corner i_pc = clip_vertex(p, c, kind0, f);  // data_new[preceding]: edge preceding -> current
    Corner e0, e1, e2;                                // new (current, next, preceding)
    if (two_in_front) {
        e0 = c; e1 = n; e2 = i_np;                    // data[preceding] = data_new[next]       (:240)
        s0 = c; s1 = i_np; s2 = i_pc;                 // appended (current, I_np, I_pc)         (:241-254)
    } else {
        e0 = i_pc; e1 = i_np; e2 = p;                 // data[current], data[next] replaced     (:259-260)
    }
    if (cur == 0) { d0 = e0; d1 = e1; d2 = e2; }
    else if (cur == 1) { d1 = e0; d2 = e1; d0 = e2; }
    else { d2 = e0; d0 = e1; d1 = e2; }
    return two_in_front;
}

struct FrontCounts { uint32_t n_near, n_clip, n_cull, n_direct; };

// The front tests of one triangle from its raster-space vertices (render.cpp:306-317): 0 rejected, 1 candidate,
// 2 candidate that straddles the near plane.
__device__ __forceinline__ uint32_t front_test(const Frame &f, const float4 &r0, const float4 &r1, const float4 &r2, FrontCounts &n) {
    if (fmaxf(fmaxf(r0.z, r1.z), r2.z) <= kNear) {  // render.cpp:306
        n.n_near++;
        return 0u;
    }
    if (fminf(fminf(r0.z, r1.z), r2.z) < kNear) {  // render.cpp:308
        n.n_clip++;
        return 2u;
    }
    // the order of the three culls does not matter for the result (all are 'continue's before any side
    // effect, render.cpp:311-317); the area test removes ~80 % of a dense field
    const Bounds b = bounds_of(f, r0.x, r0.y, r1.x, r1.y, r2.x, r2.y);
    // screen partition: a triangle whose rows cannot meet this submission's rows contributes nothing
    // (ymax = (uint)min(H - 1, max_y) < y0 follows from max_y < y0; ymin >= y1 from min_y >= y1; and 0 <= y0, y1 <= H)
    const bool off = (b.max_x < 0 || b.max_y < f.band_lo) || (b.min_x >= f.fw || b.min_y >= f.band_hi);
    if (edge_fn(r0.x, r0.y, r1.x, r1.y, r2.x, r2.y) < 10 || off) { n.n_cull++; return 0u; }
    return 1u;
}

// Phase 1 of K2 for one 256-triangle chunk (one 256-thread CTA, all threads call): classify from the
// raster-space vertices only and compact the work items into sh.list[0 .. sh.count).
__device__ __forceinline__ void classify_body(const Frame &f, uint32_t view, uint32_t chunk, SetupShared &sh) {
    const uint32_t tid = threadIdx.x, lane = lane_id();
    if (tid == 0) { sh.count = 0; }
    if (tid < 4) { sh.stats[tid] = 0; }
    __syncthreads();

    // ---- phase 1: classify one triangle per thread from raster-space vertices only ----------
    const uint32_t t = chunk * 256u + tid;
    uint32_t cls = 0;  // 0 rejected, 1 rasterisable as is, 2 straddles the near plane
    FrontCounts n = {0u, 0u, 0u, 0u};
    if (t < f.T) {
        const float4 *rv = f.rv + (size_t)view * f.Vpad;
        const float4 r0 = rv[__ldg(f.vi0 + t)], r1 = rv[__ldg(f.vi1 + t)], r2 = rv[__ldg(f.vi2 + t)];
        cls = front_test(f, r0, r1, r2, n);
        if (cls == 1u && f.row_stride != 1u) {   // interleaved tile rows: does it touch a row we own?
            const Bounds b = bounds_of(f, r0.x, r0.y, r1.x, r1.y, r2.x, r2.y);
            if (b.ymin > b.ymax || owned_rows_in(f, b.ymin / TILE_H, b.ymax / TILE_H) == 0u) { cls = 0; n.n_cull++; }
        }
    }
    {   // warp-ballot compaction of the work items into shared memory
        const uint32_t m_near = __ballot_sync(0xFFFFFFFFu, n.n_near != 0u), m_cull = __ballot_sync(0xFFFFFFFFu, n.n_cull != 0u);
        const uint32_t m_clip = __ballot_sync(0xFFFFFFFFu, cls == 2), m_work = __ballot_sync(0xFFFFFFFFu, cls != 0);
        uint32_t base = 0;
        if (lane == 0) {
            if (m_near) { atomicAdd(&sh.stats[0], __popc(m_near)); }
            if (m_clip) { atomicAdd(&sh.stats[1], __popc(m_clip)); }
            if (m_cull) { atomicAdd(&sh.stats[3], __popc(m_cull)); }
            if (m_work) { base = atomicAdd(&sh.count, __popc(m_work)); }
        }
        base = __shfl_sync(0xFFFFFFFFu, base, 0);
        if (cls != 0) { sh.list[base + __popc(m_work & ((1u << lane) - 1u))] = t | (cls == 2 ? ITEM_STRADDLE : 0u); }
    }
    __syncthreads();
}

// Phase 2 of K2: dense full setup of up to 256 work items held in sh.list (all 256 threads call).
template <bool HAS_RV>
__device__ __forceinline__ void process_items(const Frame &f, const Cam &cam, uint32_t view, SetupShared &sh) {
    const uint32_t tid = threadIdx.x, lane = lane_id();
    const uint32_t count = sh.count;
    const bool valid = tid < count;
    Corner d0, d1, d2, s0, s1, s2;
    bool spawn = false;
    uint32_t tri = 0;
    if (valid) {
        const uint32_t item = sh.list[tid];
        tri = item & ~ITEM_STRADDLE;
        d0 = gather_corner<HAS_RV>(f, cam, view, __ldg(f.vi0 + tri), __ldg(f.ai0 + tri));
        d1 = gather_corner<HAS_RV>(f, cam, view, __ldg(f.vi1 + tri), __ldg(f.ai1 + tri));
        d2 = gather_corner<HAS_RV>(f, cam, view, __ldg(f.vi2 + tri), __ldg(f.ai2 + tri));
        if (item & ITEM_STRADDLE) { spawn = clip_near(d0, d1, d2, s0, s1, s2, f); }
    }
    if (count) { emit_block(valid, d0, d1, d2, tri, f, view, sh, /*count_culled=*/true); }
    if (__syncthreads_or(spawn)) {
        const uint32_t m_sp = __ballot_sync(0xFFFFFFFFu, spawn);
        if (lane == 0 && m_sp) { atomicAdd(&sh.stats[2], __popc(m_sp)); }
        // appended triangles run after all originals, in parent order: key = T + parent index
        emit_block(spawn, s0, s1, s2, f.T + tri, f, view, sh, /*count_culled=*/true);
    }
    __syncthreads();
    if (tid < 4 && sh.stats[tid]) { atomicAdd(f.counters + view * C_COUNT + C_NEAR + tid, sh.stats[tid]); }
    __syncthreads();
}

// K2a: classify every input triangle and, for the common case, finish its visibility right here.
//
// A triangle that does not straddle the near plane and whose screen bounding box is under 16 x 16 pixels needs
// nothing but its three raster-space vertices to be rasterised: the thread that classified it computes the
// coverage setup (vis_core) into shared memory and cuts the box into (triangle, row) work items; the whole CTA then
// walks those items — replaying the reference's own additions from the box's first pixel (render.cpp:374-379) — and
// publishes depth << 32 | ~order keys with fire-and-forget 64-bit atomicMax.  No setup record, no attribute
// gather, no bin entry is ever written for such a triangle; the pixels it wins are shaded from the raw scene
// (shade_tiles).  Everything else (straddling or larger triangles) is appended to the work list of K2b.
constexpr uint32_t CLS_PER_CTA = 1024;   // triangles per classify CTA (four per thread)

struct WalkShared {
    float par[12][256];                // per parked box: ws[3], dx[3], dy[3], rz[3]  (SoA: conflict-free)
    float ck[9][256];                  // row-start weights at box rows 4, 8, 12 (checkpoints: a row item replays at most 3 row steps)
    uint32_t xy[256];                  // xmin | ymin << 16
    uint32_t bwrows[256];              // xmax - xmin | owned-row mask << 16
    uint32_t tri[256];                 // order key of the box's triangle
    uint16_t items[256 * SMALL_MAX];   // parked slot | owned row << 8, grouped by box width
    uint32_t n_cand;
    uint32_t cls_count[SMALL_MAX];     // row items per box width (1 .. 16 pixels): a warp's items are equally wide
    uint32_t stats[4];                 // near-rejected, clipped, walked here, culled
    uint32_t work_base;
};

// Where a candidate (front tests passed, not straddling) goes: its exact pixel box (render.cpp:318-321), and for a box
// under 16 x 16 pixels the box rows this submission owns (bit r: row ymin + r; under 16 rows meet at most two tile rows).
// route 3: walked record-free (direct walk); 1: work item for K2b (larger box); 0: owns no row of it — culled here.
struct BoxRoute { uint32_t xmin, xmax, ymin, ymax, rows, route; };

__device__ __forceinline__ BoxRoute route_candidate(const Frame &f, const float4 &r0, const float4 &r1, const float4 &r2) {
    BoxRoute b;
    const Bounds bb = bounds_of(f, r0.x, r0.y, r1.x, r1.y, r2.x, r2.y);
    b.xmin = bb.xmin; b.xmax = bb.xmax; b.ymin = bb.ymin; b.ymax = bb.ymax;
    const uint32_t ylo = max(b.ymin, f.y0), yhi = min(b.ymax, f.y1 - 1u);
    b.rows = 0;
    if (is_record_free(f, r0.z, r1.z, r2.z, bb)) {
        const uint32_t lo = ylo - b.ymin, hi = yhi - b.ymin;
        uint32_t rows = (2u << hi) - (1u << lo);
        if (f.row_stride != 1u) {
            const uint32_t a0 = ylo / TILE_H, a1 = yhi / TILE_H;
            const uint32_t split = (a0 + 1u) * TILE_H - b.ymin;   // first box row inside tile row a0 + 1
            const uint32_t low = split < SMALL_MAX ? (1u << split) - 1u : 0xFFFFu;
            rows &= (owns_row(f, a0) ? low : 0u) | (a1 != a0 && owns_row(f, a1) ? ~low : 0u);
        }
        b.rows = rows;
        b.route = rows ? 3u : 0u;
    } else {
        b.route = owned_rows_in(f, ylo / TILE_H, yhi / TILE_H) != 0u ? 1u : 0u;
    }
    return b;
}

// One round of up to 256 candidates, one per thread (valid: this thread has one; item: its order key, | ITEM_STRADDLE
// for a straddler whose vertices are not looked at): routing, coverage setup (vis_core) into shared memory, and the
// direct walk of the boxes under 16 x 16 pixels — one (triangle, owned row) work item per lane, grouped by box width,
// row starts from checkpoints every 4 rows, true additions along the row (render.cpp:374-379), keys published with
// fire-and-forget 64-bit red.max.  Everything else becomes a work item of K2b.  All 256 threads call.
// (Work items of two rows each were measured and lose in both kernels once the keys are in columns: profiles/r02_experiments.md.)
__device__ __forceinline__ void walk_round(const Frame &f, uint32_t view, WalkShared &wsh, FrontCounts &n, bool valid, uint32_t item,
                                           const float4 &r0, const float4 &r1, const float4 &r2) {
    const uint32_t tid = threadIdx.x, lane = lane_id();
    unsigned long long *keys = f.keys + (size_t)view * f.key_view_stride;
    if (tid < SMALL_MAX) { wsh.cls_count[tid] = 0; }
    __syncthreads();
    uint32_t route = 0;   // 1 work item for K2b, 3 walked here
    uint32_t my_cls = 0, my_rows = 0, my_off = 0;
    if (valid) {
        if (item & ITEM_STRADDLE) {
            route = 1;
        } else {
            const BoxRoute b = route_candidate(f, r0, r1, r2);
            route = b.route;
            if (route == 0u) { n.n_cull++; }
            if (route == 3u) {
                n.n_direct++;
                VisCore vc;
                vis_core(make_float3(r0.x, r0.y, r0.z), make_float3(r1.x, r1.y, r1.z), make_float3(r2.x, r2.y, r2.z),
                         edge_fn(r0.x, r0.y, r1.x, r1.y, r2.x, r2.y), b.xmin, b.ymin, vc);
#pragma unroll
                for (int k = 0; k < 3; k++) {
                    wsh.par[k][tid] = vc.ws[k]; wsh.par[3 + k][tid] = vc.dx[k]; wsh.par[6 + k][tid] = vc.dy[k]; wsh.par[9 + k][tid] = vc.rz[k];
                }
                wsh.xy[tid] = b.xmin | (b.ymin << 16);
                wsh.bwrows[tid] = (b.xmax - b.xmin) | (b.rows << 16);
                wsh.tri[tid] = item;
                float w0 = vc.ws[0], w1 = vc.ws[1], w2 = vc.ws[2];
                const uint32_t top = 31u - (uint32_t)__clz((int)b.rows);   // last owned box row
                for (uint32_t r = 1; r <= (top & ~3u); r++) {            // render.cpp:378, row by row; keep rows 4, 8, 12
                    w0 = add_rn(w0, vc.dy[0]); w1 = add_rn(w1, vc.dy[1]); w2 = add_rn(w2, vc.dy[2]);
                    if ((r & 3u) == 0u) { const uint32_t g = (r >> 2) - 1u; wsh.ck[3 * g][tid] = w0; wsh.ck[3 * g + 1][tid] = w1; wsh.ck[3 * g + 2][tid] = w2; }
                }
                my_rows = (uint32_t)__popc(b.rows);   // work items: the owned rows
                my_cls = b.xmax - b.xmin;
                my_off = atomicAdd(&wsh.cls_count[my_cls], my_rows);
            }
        }
    }
    {   // work items for K2b: one global atomic per warp
        const uint32_t m = __ballot_sync(0xFFFFFFFFu, route == 1);
        uint32_t base = 0;
        if (lane == 0 && m) { base = atomicAdd(f.counters + view * C_COUNT + C_WORK, __popc(m)); }
        base = __shfl_sync(0xFFFFFFFFu, base, 0);
        if (route == 1) { f.worklist[(size_t)view * f.T + base + __popc(m & ((1u << lane) - 1u))] = item; }
    }
    __syncthreads();
    uint32_t n_items = 0, cls_base = 0;   // items of narrower boxes come first
#pragma unroll
    for (uint32_t c = 0; c < SMALL_MAX; c++) { const uint32_t k = wsh.cls_count[c]; if (c < my_cls) { cls_base += k; } n_items += k; }
    if (route == 3) {
        uint32_t pos = my_off + cls_base;
        for (uint32_t i = 0; i < my_rows; i++) { wsh.items[pos++] = (uint16_t)(tid | (i << 8)); }
    }
    __syncthreads();
    // The direct walk: one work item per thread and pass.  The owned rows of a box are always one contiguous range (a box
    // under 16 rows meets at most two tile rows), so item k is row k of that range.
    for (uint32_t i = tid; i < n_items; i += 256u) {
        const uint32_t it = wsh.items[i], ow = it & 255u;
        const uint32_t br = wsh.bwrows[ow], bw = br & 0xFFFFu, mask = br >> 16;
        const uint32_t r = (uint32_t)__ffs((int)mask) - 1u + (it >> 8);
        const float dy0 = wsh.par[6][ow], dy1 = wsh.par[7][ow], dy2 = wsh.par[8][ow];
        const float dx0 = wsh.par[3][ow], dx1 = wsh.par[4][ow], dx2 = wsh.par[5][ow];
        const float rz0 = wsh.par[9][ow], rz1 = wsh.par[10][ow], rz2 = wsh.par[11][ow];
        const uint32_t xy = wsh.xy[ow];
        const unsigned long long key_lo = (unsigned long long)(~wsh.tri[ow]);
        const uint32_t g = r >> 2;
        float w0, w1, w2;
        if (g == 0u) { w0 = wsh.par[0][ow]; w1 = wsh.par[1][ow]; w2 = wsh.par[2][ow]; }
        else { w0 = wsh.ck[3 * g - 3][ow]; w1 = wsh.ck[3 * g - 2][ow]; w2 = wsh.ck[3 * g - 1][ow]; }
        for (uint32_t q = 0; q < (r & 3u); q++) { w0 = add_rn(w0, dy0); w1 = add_rn(w1, dy1); w2 = add_rn(w2, dy2); }   // render.cpp:378
        const uint32_t y = (xy >> 16) + r, a = y / TILE_H;
        unsigned long long *krow = keys + key_at(f, out_row(f, y, a), xy & 0xFFFFu);   // neighbouring lanes: neighbouring rows, same x
        // (leaving the row once it has left its run of inside pixels — the weights are monotone along a row — was
        // measured and does not pay: the warp's longest row decides, and the test costs every lane)
        publish_row(krow, 0u, bw, make_float3(w0, w1, w2), make_float3(dx0, dx1, dx2), make_float3(rz0, rz1, rz2), key_lo);
    }
    __syncthreads();   // parked boxes and items are rewritten by the next round
}

// statistics: one shared-memory atomic per warp, one global atomic per CTA and counter (all 256 threads call)
__device__ __forceinline__ void publish_front_counts(const Frame &f, uint32_t view, WalkShared &wsh, FrontCounts n) {
    const uint32_t tid = threadIdx.x, lane = lane_id();
    n.n_near = __reduce_add_sync(0xFFFFFFFFu, n.n_near); n.n_clip = __reduce_add_sync(0xFFFFFFFFu, n.n_clip);
    n.n_direct = __reduce_add_sync(0xFFFFFFFFu, n.n_direct); n.n_cull = __reduce_add_sync(0xFFFFFFFFu, n.n_cull);
    if (lane == 0) {
        if (n.n_near) { atomicAdd(&wsh.stats[0], n.n_near); }
        if (n.n_clip) { atomicAdd(&wsh.stats[1], n.n_clip); }
        if (n.n_direct) { atomicAdd(&wsh.stats[2], n.n_direct); }
        if (n.n_cull) { atomicAdd(&wsh.stats[3], n.n_cull); }
    }
    __syncthreads();
    if (tid < 4 && wsh.stats[tid]) {
        atomicAdd(f.counters + view * C_COUNT + (tid == 2u ? (uint32_t)C_DIRECT : (uint32_t)C_NEAR + tid), wsh.stats[tid]);   // C_NEAR, C_CLIPPED, C_DIRECT, C_CULLED
    }
}

struct ClassifyShared {
    WalkShared w;
    uint32_t cand[CLS_PER_CTA];        // triangles that passed the front tests (| ITEM_STRADDLE)
};

__global__ void __launch_bounds__(256) triangle_classify(const __grid_constant__ Frame f) {
    wait_for_predecessor();
    __shared__ ClassifyShared csh;
    WalkShared &wsh = csh.w;
    const uint32_t view = blockIdx.y, tid = threadIdx.x, lane = lane_id();
    if (tid == 0) { wsh.n_cand = 0; }
    if (tid < 4) { wsh.stats[tid] = 0; }
    __syncthreads();
    const float4 *rv = f.rv + (size_t)view * f.Vpad;
    FrontCounts n = {0u, 0u, 0u, 0u};   // per-thread statistics, reduced once at the end

    // ---- front: near reject, straddle, area cull, screen/band reject (render.cpp:306-317), 4 triangles per thread ----
#pragma unroll 2
    for (uint32_t pass = 0; pass < CLS_PER_CTA / 256u; pass++) {
        const uint32_t t = blockIdx.x * CLS_PER_CTA + pass * 256u + tid;
        uint32_t cand = 0;   // 1 candidate, 2 candidate that straddles the near plane
        if (t < f.T) {
            const float4 r0 = rv[__ldg(f.vi0 + t)], r1 = rv[__ldg(f.vi1 + t)], r2 = rv[__ldg(f.vi2 + t)];
            cand = front_test(f, r0, r1, r2, n);
        }
        const uint32_t m = __ballot_sync(0xFFFFFFFFu, cand != 0);
        uint32_t base = 0;
        if (lane == 0 && m) { base = atomicAdd(&wsh.n_cand, __popc(m)); }
        base = __shfl_sync(0xFFFFFFFFu, base, 0);
        if (cand) { csh.cand[base + __popc(m & ((1u << lane) - 1u))] = t | (cand == 2 ? ITEM_STRADDLE : 0u); }
    }
    __syncthreads();
    const uint32_t n_cand = wsh.n_cand;
    for (uint32_t cbase = 0; cbase < n_cand; cbase += 256u) {   // candidates, densely packed, 256 per round
        const bool valid = cbase + tid < n_cand;
        uint32_t item = 0;
        float4 r0 = make_float4(0.f, 0.f, 0.f, 0.f), r1 = r0, r2 = r0;
        if (valid) {
            item = csh.cand[cbase + tid];
            if (!(item & ITEM_STRADDLE)) { r0 = rv[__ldg(f.vi0 + item)]; r1 = rv[__ldg(f.vi1 + item)]; r2 = rv[__ldg(f.vi2 + item)]; }
        }
        walk_round(f, view, wsh, n, valid, item, r0, r1, r2);
    }
    publish_front_counts(f, view, wsh, n);
}

// ------------------------------------------------------------------------------------------------
// K1 + K2a over the spatial pre-partition (cluster.hpp), three kernels:
//   cluster_cull    one thread per cluster: a conservative verdict from the bounding sphere — every vertex at or behind the
//                   near plane (all its triangles are near-rejected, render.cpp:306), or every triangle certainly culled: off
//                   screen, outside the rows this submission owns, or too small to reach `area >= 10` (render.cpp:311-317).
//                   Such a cluster costs 48 bytes of header; its vertices are never transformed.  On an n-GPU screen
//                   partition a rank skips what misses its rows, so the geometry work shrinks with n.
//   cluster_front   one warp per group of four surviving clusters: the vertex stage (render.cpp:285-289) streamed from the
//                   cluster-private position arrays into SHARED memory — raster-space vertices never travel to HBM —, the
//                   front tests with corners gathered from shared memory, routing, and a 40-byte record per candidate of
//                   the direct walk into a queue in HBM;
//   direct_walk     coverage setup and direct walk of the queue, 256 records per round (walk_round).
// Every skipped triangle is proven rejected by the reference's own per-triangle tests, so the frame cannot change.
// ------------------------------------------------------------------------------------------------
constexpr uint32_t FRONT_GROUP = 4;                                  // clusters a warp of the front kernel takes at a time
constexpr uint32_t FRONT_VERTS = FRONT_GROUP * CL_MAX_VERTS;         // <= 64 vertices ...
constexpr uint32_t FRONT_TRIS = FRONT_GROUP * CL_MAX_TRIS;           // ... and <= 128 triangles per group

struct FrontWarp {                       // a warp's private staging: nothing in the front kernel crosses warps
    float4 rv[FRONT_VERTS];              // raster-space vertices of the group's clusters
    uint16_t cand[FRONT_TRIS];           // triangles that passed the front tests: position in the group | 0x8000 for a straddler
};

// One candidate of the direct walk as the front kernel hands it to the walk kernel through HBM: the three raster-space
// vertices and the order key (40 bytes; a warp's candidates are contiguous).
struct __align__(8) WalkRecord { float v[9]; uint32_t order; };
static_assert(sizeof(WalkRecord) == 40, "WalkRecord must be 40 bytes");

// A record is written and read as five 8-byte words.
__device__ __forceinline__ void store_walk_record(WalkRecord *p, const float4 &r0, const float4 &r1, const float4 &r2, uint32_t order) {
    uint2 *q = reinterpret_cast<uint2 *>(p);
    q[0] = make_uint2(__float_as_uint(r0.x), __float_as_uint(r0.y)); q[1] = make_uint2(__float_as_uint(r0.z), __float_as_uint(r1.x));
    q[2] = make_uint2(__float_as_uint(r1.y), __float_as_uint(r1.z)); q[3] = make_uint2(__float_as_uint(r2.x), __float_as_uint(r2.y));
    q[4] = make_uint2(__float_as_uint(r2.z), order);
}

__device__ __forceinline__ uint32_t load_walk_record(const WalkRecord *p, float4 &r0, float4 &r1, float4 &r2) {   // returns the order key
    const uint2 *q = reinterpret_cast<const uint2 *>(p);
    const uint2 a = q[0], b = q[1], c = q[2], d = q[3], e = q[4];
    r0 = make_float4(__uint_as_float(a.x), __uint_as_float(a.y), __uint_as_float(b.x), 0.f);
    r1 = make_float4(__uint_as_float(b.y), __uint_as_float(c.x), __uint_as_float(c.y), 0.f);
    r2 = make_float4(__uint_as_float(d.x), __uint_as_float(d.y), __uint_as_float(e.x), 0.f);
    return e.y;
}

// The rejection tests only have to err on the safe side, so they use the approximate units (MUFU, a few ulps) with a margin
// instead of the correctly rounded operators this translation unit is compiled with (-prec-div / -prec-sqrt: ten times the
// instructions).  fast_sqrt_up(x) >= sqrt(x), fast_div_up(a, b) >= a / b for a >= 0, b > 0.
__device__ __forceinline__ float fast_sqrt_up(float x) { return x > 0.f ? x * mufu_rsq(x) * 1.00001f : 0.f; }
__device__ __forceinline__ float fast_div_up(float a, float b) { return a * mufu_rcp(b) * 1.00001f; }

// What the rejection tests need from the view's matrix: the norms of its rows and a bound of its largest singular value
// (Gershgorin on the Gram matrix; 1 for a camera's orthonormal rows).
struct ViewBounds { float norm[3], sigma; };

__device__ __forceinline__ ViewBounds view_bounds(const Cam &cam) {
    ViewBounds vb;
    float gram = 0.f;
#pragma unroll
    for (int i = 0; i < 3; i++) {
        const float m0 = cam.m[4 * i], m1 = cam.m[4 * i + 1], m2 = cam.m[4 * i + 2];
        vb.norm[i] = fast_sqrt_up(m0 * m0 + m1 * m1 + m2 * m2);
        float row = 0.f;
#pragma unroll
        for (int j = 0; j < 3; j++) { row += fabsf(m0 * cam.m[4 * j] + m1 * cam.m[4 * j + 1] + m2 * cam.m[4 * j + 2]); }
        gram = fmaxf(gram, row);
    }
    vb.sigma = fast_sqrt_up(gram);
    return vb;
}

// Conservative verdict on a bounding sphere (centre, radius) whose triangles have no edge longer than max_edge:
// 0: process per triangle; 1: every triangle near-rejected; 2: every triangle culled (off screen / not ours / too small).
// Every comparison is written so that NaN / infinite bounds end in 0.
__device__ __forceinline__ uint32_t cluster_verdict(const Frame &f, const Cam &cam, const ViewBounds &vb, float cx, float cy, float cz,
                                                    float radius, float max_edge) {
    const float3 cc = xform(cam, cx, cy, cz, 1.0f);
    const float ax = fabsf(cx) + radius, ay = fabsf(cy) + radius, az = fabsf(cz) + radius;
    float rho[3], err = 0.f;
#pragma unroll
    for (int i = 0; i < 3; i++) {
        // |binary32 transform - exact transform| of any point of the sphere: four products and three sums, each within
        // 2^-24 of the running magnitude; 2^-21 of the summed magnitudes is more than twice that
        const float e = 0x1p-21f * (fabsf(cam.m[4 * i]) * ax + fabsf(cam.m[4 * i + 1]) * ay + fabsf(cam.m[4 * i + 2]) * az + fabsf(cam.m[4 * i + 3]));
        // every vertex's computed camera-space coordinate i lies within rho[i] of the computed centre's
        rho[i] = (vb.norm[i] * radius + 2.f * e) * 1.000001f + 1e-30f;
        err = fmaxf(err, e);
    }
    const float d = -cc.z, d_min = d - rho[2], d_max = d + rho[2];
    // near reject (render.cpp:306): every vertex has rv.z = -cv.z <= near.  -cv.z == 0 makes rv.z NaN in the reference's
    // expression (0 / 0), so only spheres strictly behind the eye plane or strictly between it and the near plane count.
    if (d_max < 0.f || (d_min > 0.f && d_max <= kNear)) { return 1u; }
    if (!(d_min > kNear * 1.000001f)) { return 0u; }   // may touch the near plane (or bounds are not finite): per triangle
    // every vertex strictly in front: raster coordinates by interval arithmetic over the box [cc - rho, cc + rho]
    const float x_lo = cc.x - rho[0], x_hi = cc.x + rho[0], y_lo = -cc.y - rho[1], y_hi = -cc.y + rho[1];   // raster y grows downwards (-cv.y)
    // factor / d_min rounded up, factor / d_max rounded down (d_min < d_max, both positive): an upper bound takes the
    // larger scale for a positive coordinate and the smaller one for a negative coordinate, a lower bound the other way round
    const float inv_min = fast_div_up(f.factor, d_min), inv_max = f.factor * mufu_rcp(d_max) * 0.99999f;
    const float qx_hi = x_hi * (x_hi >= 0.f ? inv_min : inv_max), qx_lo = x_lo * (x_lo >= 0.f ? inv_max : inv_min);
    const float qy_hi = y_hi * (y_hi >= 0.f ? inv_min : inv_max), qy_lo = y_lo * (y_lo >= 0.f ? inv_max : inv_min);
    // slack: rounding of the vertices' own projections and of this evaluation (a few 2^-24 of the magnitudes)
    const float sx = 0x1p-18f * (fmaxf(fabsf(qx_lo), fabsf(qx_hi)) + f.fw) + 0.01f, sy = 0x1p-18f * (fmaxf(fabsf(qy_lo), fabsf(qy_hi)) + f.fh) + 0.01f;
    const float sx_hi = qx_hi + f.half_w + sx, sx_lo = qx_lo + f.half_w - sx, sy_hi = qy_hi + f.half_h + sy, sy_lo = qy_lo + f.half_h - sy;
    // off screen / outside the band (render.cpp:311-314 and the partition's row range)
    if (sx_hi < 0.f || sy_hi < f.band_lo || sx_lo >= f.fw || sy_lo >= f.band_hi) { return 2u; }
    if (f.row_stride != 1u) {   // interleaved tile rows: does the sphere reach a row this submission owns?
        const uint32_t ylo = (uint32_t)fmaxf(0.f, floorf(sy_lo)), yhi = (uint32_t)fminf(f.fh - 1.f, sy_hi);
        if (ylo > yhi || owned_rows_in(f, ylo / TILE_H, yhi / TILE_H) == 0u) { return 2u; }
    }
    // too small (render.cpp:316-317): |area| <= product of two projected edges.  A camera-space segment of length L at
    // depth >= d_min whose endpoints project at tangents (tu, tv) is at most factor / d_min * L * sqrt(1 + tu^2 + tv^2)
    // pixels long.  L: the longest object-space edge through the matrix plus the endpoints' rounding.
    const float len = vb.sigma * max_edge + 4.f * err;
    const float rcp_min = mufu_rcp(d_min) * 1.00001f;
    const float tu = fmaxf(fabsf(x_lo), fabsf(x_hi)) * rcp_min, tv = fmaxf(fabsf(y_lo), fabsf(y_hi)) * rcp_min;
    const float pixels = inv_min * len * fast_sqrt_up(1.f + tu * tu + tv * tv) * 1.00001f + 2.f * (sx + sy);
    if (pixels <= 3.09f) { return 2u; }   // (3.09 + rounding)^2 < 10
    return 0u;
}

constexpr int FRONT_CTAS = 4;                 // cluster_front CTAs per SM
constexpr uint32_t WALK_HOLE = 0xFFFFFFFFu;   // order key of a queue slot that holds no candidate
constexpr uint32_t WALK_CHUNK = 64;           // queue slots a warp of the front kernel reserves at a time

// Rejection of whole clusters by their bounds, one thread per cluster: the sphere around the cluster's vertices and its
// longest edge against the view (cluster_verdict).  Surviving clusters are appended to a compact list as {first vertex,
// first triangle word, original index of the first triangle, vertices | triangles << 16} — everything the front kernel
// needs, so it never reads a header; the triangles of what is rejected are accounted for here (near-rejected or culled,
// exactly what the reference's per-triangle tests would have said).  The front kernel's work is then proportional to what
// may actually be visible to this submission: on an n-GPU screen partition, 1/n of it.  (A coarser test on spheres around
// batches of 64 clusters in front of this one was measured: the 32-byte headers it saves cost less than its extra step.)
// (Each CTA judges CULL_ROUNDS x 256 consecutive clusters with no barrier and no atomic between the rounds, so the header loads
// of one round overlap the arithmetic of another; then one block scan and ONE global atomic reserve the CTA's list slots, and
// the survivors' entries are rebuilt from their headers, which are still in L1/L2.  One list atomic per 256 clusters kept a
// dependent round trip in every round — 23 us for the benchmark field —, a global atomic per warp for the statistics put tens
// of thousands of operations on two addresses — 36 us.)
constexpr uint32_t CULL_ROUNDS = 8;
constexpr int CULL_UNROLL = 2;

__global__ void __launch_bounds__(256) cluster_cull(const __grid_constant__ Frame f) {
    wait_for_predecessor();
    __shared__ uint32_t s_wsum[8], s_base, s_stats[2];
    const uint32_t view = blockIdx.y, tid = threadIdx.x, lane = lane_id(), warp = tid >> 5;
    const Cam cam = load_cam(f, view);
    uint32_t *counters = f.counters + view * C_COUNT;
    uint4 *list = f.cluster_list + (size_t)view * f.list_cap;
    ViewBounds vb = {{0.f, 0.f, 0.f}, 0.f};
    if (lane == 0) { vb = view_bounds(cam); }
    vb.norm[0] = __shfl_sync(0xFFFFFFFFu, vb.norm[0], 0); vb.norm[1] = __shfl_sync(0xFFFFFFFFu, vb.norm[1], 0);
    vb.norm[2] = __shfl_sync(0xFFFFFFFFu, vb.norm[2], 0); vb.sigma = __shfl_sync(0xFFFFFFFFu, vb.sigma, 0);
    if (tid < 2) { s_stats[tid] = 0; }
    const uint32_t c_first = blockIdx.x * (CULL_ROUNDS * 256u) + tid;
    uint32_t alive = 0, near = 0, cull = 0;   // alive: bit k = the cluster of round k survives
#pragma unroll CULL_UNROLL
    for (uint32_t k = 0; k < CULL_ROUNDS; k++) {
        const uint32_t c = c_first + k * 256u;
        if (c < f.n_clusters) {
            const uint4 h0 = __ldg(f.cl_hdr + 2 * (size_t)c), h1 = __ldg(f.cl_hdr + 2 * (size_t)c + 1);
            const uint32_t n_tris = __ldg(f.cl_hdr + 2 * (size_t)c + 3).w - h1.w;
            const uint32_t verdict = f.cluster_cull ? cluster_verdict(f, cam, vb, __uint_as_float(h0.x), __uint_as_float(h0.y), __uint_as_float(h0.z), __uint_as_float(h0.w), __uint_as_float(h1.x)) : 0u;
            alive |= (verdict == 0u ? 1u : 0u) << k;
            near += verdict == 1u ? n_tris : 0u; cull += verdict == 2u ? n_tris : 0u;
        }
    }
    // list slots: block-wide exclusive scan of the survivor counts, one global atomic per CTA
    const uint32_t mine = (uint32_t)__popc(alive);
    uint32_t incl = mine;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const uint32_t v = __shfl_up_sync(0xFFFFFFFFu, incl, d); if (lane >= (uint32_t)d) { incl += v; } }
    if (lane == 31) { s_wsum[warp] = incl; }
    near = __reduce_add_sync(0xFFFFFFFFu, near); cull = __reduce_add_sync(0xFFFFFFFFu, cull);
    __syncthreads();
    if (lane == 0) { if (near) { atomicAdd(&s_stats[0], near); } if (cull) { atomicAdd(&s_stats[1], cull); } }
    if (tid == 0) {
        uint32_t run = 0;
#pragma unroll
        for (int w = 0; w < 8; w++) { const uint32_t n = s_wsum[w]; s_wsum[w] = run; run += n; }
        s_base = run ? atomicAdd(counters + C_CLUSTERS, run) : 0u;
    }
    __syncthreads();
    uint32_t at = s_base + s_wsum[warp] + incl - mine;
#pragma unroll 2
    for (uint32_t k = 0; k < CULL_ROUNDS; k++) {
        if (alive & (1u << k)) {
            const uint32_t c = c_first + k * 256u;
            const uint4 h1 = __ldg(f.cl_hdr + 2 * (size_t)c + 1), nx = __ldg(f.cl_hdr + 2 * (size_t)c + 3);
            list[at++] = make_uint4(h1.z, h1.w, h1.y, (nx.z - h1.z) | ((nx.w - h1.w) << 16));
        }
    }
    if (tid == 0) {
        if (s_stats[0]) { atomicAdd(counters + C_NEAR, s_stats[0]); }
        if (s_stats[1]) { atomicAdd(counters + C_CULLED, s_stats[1]); }
    }
}

// K1 + the front of K2a over the surviving clusters, one WARP per group of FRONT_GROUP clusters and no block-wide step
// anywhere: a warp's chain of dependent loads (list entries -> vertices and triangle words -> queue space) overlaps with
// those of the 31 other warps of its SM partition, and the next group's list entries are fetched while this one is processed.
//   1. the group's vertices, densely over the lanes (the owner of a flat index is found with three compares): vertex stage
//      (render.cpp:285-289) into the warp's shared-memory staging — raster-space vertices never travel to HBM;
//   2. the front tests (render.cpp:306-317), densely over the group's triangle words; candidates are packed into a list;
//   3. the candidates, densely: exact box and row ownership; a 40-byte record for the direct walk into queue space the warp
//      reserves WALK_CHUNK slots at a time (one global atomic per chunk; what is left of a chunk is padded with holes),
//      or a work item for K2b (straddlers and larger boxes).
__global__ void __launch_bounds__(256, FRONT_CTAS) cluster_front(const __grid_constant__ Frame f) {
    wait_for_predecessor();
    __shared__ FrontWarp sh_all[8];
    const uint32_t view = blockIdx.y, tid = threadIdx.x, lane = lane_id();
    FrontWarp &sh = sh_all[tid >> 5];
    const Cam cam = load_cam(f, view);
    uint32_t *counters = f.counters + view * C_COUNT;
    const uint32_t n_cl = min(counters[C_CLUSTERS], f.list_cap);   // list slots written by cluster_cull (empty ones included)
    const uint4 *list = f.cluster_list + (size_t)view * f.list_cap;
    WalkRecord *queue = f.walk_q + (size_t)view * f.walk_cap;
    FrontCounts n = {0u, 0u, 0u, 0u};
    uint32_t q_pos = 0, q_end = 0;   // the warp's reserved queue range [q_pos, q_end) (uniform over the lanes)
    const uint32_t n_groups = (n_cl + FRONT_GROUP - 1u) / FRONT_GROUP, warps = gridDim.x * 8u;
    uint32_t g = blockIdx.x * 8u + (tid >> 5);
    // lanes 0 .. FRONT_GROUP - 1 hold the list entries of the group's clusters
    uint4 e = make_uint4(0u, 0u, 0u, 0u);
    if (g < n_groups && lane < FRONT_GROUP && g * FRONT_GROUP + lane < n_cl) { e = __ldg(list + g * FRONT_GROUP + lane); }

    for (; g < n_groups; g += warps) {
        // the group's layout: exclusive prefix sums of the clusters' vertex and triangle counts (lanes >= FRONT_GROUP hold zeros)
        const uint32_t nv = e.w & 0xFFFFu, nt = e.w >> 16;
        uint32_t vpre = nv, tpre = nt;
#pragma unroll
        for (int d = 1; d < (int)FRONT_GROUP; d <<= 1) {
            const uint32_t a = __shfl_up_sync(0xFFFFFFFFu, vpre, d), b = __shfl_up_sync(0xFFFFFFFFu, tpre, d);
            if (lane >= (uint32_t)d) { vpre += a; tpre += b; }
        }
        const uint32_t v_tot = __shfl_sync(0xFFFFFFFFu, vpre, FRONT_GROUP - 1), t_tot = __shfl_sync(0xFFFFFFFFu, tpre, FRONT_GROUP - 1);
        vpre -= nv; tpre -= nt;   // exclusive
        uint32_t vstart[FRONT_GROUP], tstart[FRONT_GROUP], voff[FRONT_GROUP], toff[FRONT_GROUP], t0[FRONT_GROUP];
#pragma unroll
        for (int k = 0; k < (int)FRONT_GROUP; k++) {
            vstart[k] = __shfl_sync(0xFFFFFFFFu, vpre, k); tstart[k] = __shfl_sync(0xFFFFFFFFu, tpre, k);
            voff[k] = __shfl_sync(0xFFFFFFFFu, e.x, k); toff[k] = __shfl_sync(0xFFFFFFFFu, e.y, k); t0[k] = __shfl_sync(0xFFFFFFFFu, e.z, k);
        }
        // the next group's entries travel while this one is processed
        const uint32_t g_next = g + warps;
        e = make_uint4(0u, 0u, 0u, 0u);
        if (g_next < n_groups && lane < FRONT_GROUP && g_next * FRONT_GROUP + lane < n_cl) { e = __ldg(list + g_next * FRONT_GROUP + lane); }

        // owner of a flat index: three compares against the starts
        auto owner = [&](uint32_t j, const uint32_t (&start)[FRONT_GROUP]) {
            uint32_t k = 0;
#pragma unroll
            for (int q = 1; q < (int)FRONT_GROUP; q++) { k += j >= start[q] ? 1u : 0u; }
            return k;
        };
        auto pick = [&](const uint32_t (&a)[FRONT_GROUP], uint32_t k) {
            uint32_t r = a[0];
#pragma unroll
            for (int q = 1; q < (int)FRONT_GROUP; q++) { r = k == (uint32_t)q ? a[q] : r; }
            return r;
        };

        // ---- 1. vertex stage, and the triangle words requested alongside -----------------------------------------------
        constexpr int VP = FRONT_VERTS / 32, TP = FRONT_TRIS / 32;
        float px[VP], py[VP], pz[VP];
#pragma unroll
        for (int p = 0; p < VP; p++) {
            const uint32_t j = lane + 32u * p;
            if (j < v_tot) { const uint32_t k = owner(j, vstart), at = pick(voff, k) + (j - pick(vstart, k)); px[p] = __ldg(f.cl_px + at); py[p] = __ldg(f.cl_py + at); pz[p] = __ldg(f.cl_pz + at); }
        }
        uint32_t tw[TP], tk[TP];
#pragma unroll
        for (int p = 0; p < TP; p++) {
            const uint32_t j = lane + 32u * p;
            tw[p] = 0u; tk[p] = 0u;
            if (j < t_tot) { tk[p] = owner(j, tstart); tw[p] = __ldg(f.cl_tri + pick(toff, tk[p]) + (j - pick(tstart, tk[p]))); }
        }
#pragma unroll
        for (int p = 0; p < VP; p++) {
            const uint32_t j = lane + 32u * p;
            if (j < v_tot) {
                const float3 r = project(xform(cam, px[p], py[p], pz[p], 1.0f), f.factor, f.half_w, f.half_h);
                sh.rv[j] = make_float4(r.x, r.y, r.z, 0.f);
            }
        }
        __syncwarp();

        // ---- 2. front tests; candidates packed into the warp's list ---------------------------------------------------------
        uint32_t n_cand = 0;
#pragma unroll
        for (int p = 0; p < TP; p++) {
            const uint32_t j = lane + 32u * p;
            uint32_t cand = 0;
            if (j < t_tot) {
                const uint32_t o = pick(vstart, tk[p]);
                cand = front_test(f, sh.rv[o + (tw[p] & 255u)], sh.rv[o + ((tw[p] >> 8) & 255u)], sh.rv[o + ((tw[p] >> 16) & 255u)], n);
            }
            const uint32_t m = __ballot_sync(0xFFFFFFFFu, cand != 0u);
            if (cand) { sh.cand[n_cand + __popc(m & ((1u << lane) - 1u))] = (uint16_t)(j | (cand == 2u ? 0x8000u : 0u)); }
            n_cand += (uint32_t)__popc(m);
        }
        __syncwarp();

        // ---- 3. routing of the candidates, densely ---------------------------------------------------------------------------
        for (uint32_t cb = 0; cb < n_cand; cb += 32u) {
            uint32_t code = 0, item = 0;   // code: 1 work item for K2b, 3 direct walk
            float4 r0 = make_float4(0.f, 0.f, 0.f, 0.f), r1 = r0, r2 = r0;
            if (cb + lane < n_cand) {
                const uint32_t c = sh.cand[cb + lane], j = c & 0x7FFFu, k = owner(j, tstart);
                const uint32_t local = j - pick(tstart, k), w = __ldg(f.cl_tri + pick(toff, k) + local), o = pick(vstart, k);
                item = pick(t0, k) + local;   // the original triangle index is the order key
                if (c & 0x8000u) { code = 1u; item |= ITEM_STRADDLE; }
                else {
                    r0 = sh.rv[o + (w & 255u)]; r1 = sh.rv[o + ((w >> 8) & 255u)]; r2 = sh.rv[o + ((w >> 16) & 255u)];
                    code = route_candidate(f, r0, r1, r2).route;
                    if (code == 0u) { n.n_cull++; }
                }
            }
            const uint32_t m_walk = __ballot_sync(0xFFFFFFFFu, code == 3u), m_work = __ballot_sync(0xFFFFFFFFu, code == 1u);
            const uint32_t n_walk = (uint32_t)__popc(m_walk);
            if (n_walk) {
                if (q_pos + n_walk > q_end) {   // (uniform) the chunk cannot take them: pad it with holes, reserve the next one
                    for (uint32_t h = q_pos + lane; h < q_end; h += 32u) { if (h < f.walk_cap) { queue[h].order = WALK_HOLE; } }
                    if (lane == 0) { q_pos = atomicAdd(counters + C_WALKQ, WALK_CHUNK); }
                    q_pos = __shfl_sync(0xFFFFFFFFu, q_pos, 0);
                    q_end = q_pos + WALK_CHUNK;
                }
                if (code == 3u) {
                    const uint32_t at = q_pos + (uint32_t)__popc(m_walk & ((1u << lane) - 1u));
                    if (at < f.walk_cap) { store_walk_record(queue + at, r0, r1, r2, item); }
                }
                q_pos += n_walk;
            }
            if (m_work) {
                uint32_t base_work = 0;
                if (lane == 0) { base_work = atomicAdd(counters + C_WORK, __popc(m_work)); }
                base_work = __shfl_sync(0xFFFFFFFFu, base_work, 0);
                if (code == 1u) { f.worklist[(size_t)view * f.T + base_work + (uint32_t)__popc(m_work & ((1u << lane) - 1u))] = item; }
            }
        }
        __syncwarp();   // the staging is rewritten by the next group
    }
    for (uint32_t h = q_pos + lane; h < q_end; h += 32u) { if (h < f.walk_cap) { queue[h].order = WALK_HOLE; } }   // the last chunk's rest
    // statistics: one global atomic per warp and counter
    n.n_near = __reduce_add_sync(0xFFFFFFFFu, n.n_near); n.n_clip = __reduce_add_sync(0xFFFFFFFFu, n.n_clip); n.n_cull = __reduce_add_sync(0xFFFFFFFFu, n.n_cull);
    if (lane == 0) {
        if (n.n_near) { atomicAdd(counters + C_NEAR, n.n_near); }
        if (n.n_clip) { atomicAdd(counters + C_CLIPPED, n.n_clip); }
        if (n.n_cull) { atomicAdd(counters + C_CULLED, n.n_cull); }
    }
}

// The direct walk over the front kernel's candidate queue: persistent CTAs take rounds of 256 records — always full but
// the last — and run walk_round on them.  Nothing but the walk lives here, so the kernel's warps keep the reduction path
// (one red.global.max.u64 per covered pixel) busy back to back.
__global__ void __launch_bounds__(256, 6) direct_walk(const __grid_constant__ Frame f) {
    wait_for_predecessor();
    __shared__ WalkShared wsh;
    __shared__ uint32_t s_round;
    const uint32_t view = blockIdx.y, tid = threadIdx.x;
    uint32_t *counters = f.counters + view * C_COUNT;
    const uint32_t n_q = counters[C_WALKQ];
    if (n_q > f.walk_cap) {   // the queue overflowed: the host regrows it and renders the frame again
        if (blockIdx.x == 0 && tid == 0) { atomicOr(counters + C_OVERFLOW, 8u); atomicOr(f.sticky + 0, 8u); atomicMax(f.sticky + 4, n_q); }
        return;
    }
    if (tid < 4) { wsh.stats[tid] = 0; }
    FrontCounts n = {0u, 0u, 0u, 0u};
    const WalkRecord *queue = f.walk_q + (size_t)view * f.walk_cap;
    while (true) {
        __syncthreads();
        if (tid == 0) { s_round = atomicAdd(counters + C_WALKHEAD, 1u); }
        __syncthreads();
        const uint32_t base = s_round * 256u;
        if (base >= n_q) { break; }
        bool valid = base + tid < n_q;
        uint32_t item = 0;
        float4 r0 = make_float4(0.f, 0.f, 0.f, 0.f), r1 = r0, r2 = r0;
        if (valid) {
            item = load_walk_record(queue + base + tid, r0, r1, r2);
            valid = item != WALK_HOLE;   // a slot reserved for a candidate that went elsewhere
        }
        walk_round(f, view, wsh, n, valid, item, r0, r1, r2);
    }
    publish_front_counts(f, view, wsh, n);
}

// K2b: dense setup over the compacted work list (persistent grid-stride; every lane has a survivor
// candidate, so the register-heavy gather/clip/setup code runs at full lane efficiency).
template <bool HAS_RV>
__global__ void __launch_bounds__(256, 2) triangle_setup(const __grid_constant__ Frame f) {
    wait_for_predecessor();
    __shared__ SetupShared sh;
    const uint32_t view = blockIdx.y, tid = threadIdx.x;
    const Cam cam = load_cam(f, view);
    const uint32_t n_work = f.counters[view * C_COUNT + C_WORK];
    for (uint32_t base = blockIdx.x * 256u; base < n_work; base += gridDim.x * 256u) {
        if (tid == 0) { sh.count = min(256u, n_work - base); }
        if (tid < 4) { sh.stats[tid] = 0; }
        if (base + tid < n_work) { sh.list[tid] = f.worklist[(size_t)view * f.T + base + tid]; }
        __syncthreads();
        process_items<HAS_RV>(f, cam, view, sh);
    }
}

// ------------------------------------------------------------------------------------------------
// K3 — sort-middle binning (count -> scan -> fill).  Entries are (order << 32 | slot) so that each
// tile can restore the reference's processing order with one sort.
// ------------------------------------------------------------------------------------------------
// Triangles over more than BIG_TILES tiles: one CTA per triangle, threads over its tiles.
__device__ __forceinline__ void bin_big_body(const Frame &f, uint32_t view) {
    const uint32_t n = min(f.counters[view * C_COUNT + C_BIG], f.big_cap);
    for (uint32_t b = blockIdx.x; b < n; b += gridDim.x) {
        const uint32_t slot = f.big_list[(size_t)view * f.big_cap + b];
        const Head h = unpack_head(f.head[(size_t)view * f.setup_cap + slot]);
        const TileRange r = tile_range(f, h.xmin, h.xmax, h.ymin, h.ymax);
        const uint32_t nx = r.tx1 - r.tx0 + 1u, ntiles = nx * (r.a1 - r.a0 + 1u);
        const SetupVis *vp = f.vis + (size_t)view * f.setup_cap + slot;
        for (uint32_t i = threadIdx.x; i < ntiles; i += blockDim.x) {
            const uint32_t a = r.a0 + i / nx, tx = r.tx0 + i % nx;
            if (!owns_row(f, a)) { continue; }
            const uint32_t ya = a * TILE_H, ylo_t = max(ya, f.y0), yhi_t = min(ya + TILE_H, f.y1);
            if (tile_outside_triangle(*vp, tx * TILE_W, ylo_t, yhi_t)) { continue; }
            bin_one(f, view, local_row(f, a) * f.tiles_x + tx, slot);
        }
    }
}

// After all binning: total and longest tile list, overflow bits, and the cross-submission record the host
// reads back (one CTA per view: the last one to finish post_setup).
__device__ __forceinline__ void finalize_body(const Frame &f, uint32_t view, uint32_t *s_sum, uint32_t *s_max) {
    const uint32_t tid = threadIdx.x;
    uint32_t sum = 0, mx = 0;
    // (the counts are fetched eight at a time: one CTA walks the whole table, and a dependent L2 round trip per
    // iteration was 10 us of every frame)
    for (uint32_t t0 = 0; t0 < f.n_tiles; t0 += 8u * 256u) {
      uint32_t cs[8];
#pragma unroll
      for (int k = 0; k < 8; k++) { const uint32_t t = t0 + k * 256u + tid; cs[k] = t < f.n_tiles ? __ldcg(f.tile_count + view * f.tile_stride + t) : 0u; }
#pragma unroll
      for (int k = 0; k < 8; k++) {
        const uint32_t t = t0 + k * 256u + tid, c = cs[k];
        if (t >= f.n_tiles) { continue; }
        sum += c; mx = max(mx, c);
        // the tile kernel's work queue: one item per RASTER_CHUNK entries of a non-empty bin list
        const uint32_t n = min(c, f.tile_cap), chunks = (n + RASTER_CHUNK - 1u) / RASTER_CHUNK;
        if (chunks) {
            const uint32_t base = atomicAdd(f.counters + view * C_COUNT + C_ITEMS, chunks);
            for (uint32_t k = 0; k < chunks && base + k < f.items_cap; k++) {
                f.raster_items[(size_t)view * f.items_cap + base + k] = make_uint2(t, k * RASTER_CHUNK);
            }
        }
      }
    }
    atomicAdd(s_sum, sum);
    atomicMax(s_max, mx);
    __syncthreads();
    if (tid == 0) {
        uint32_t *c = f.counters + view * C_COUNT;
        const uint32_t overflow = __ldcg(c + C_OVERFLOW) | (*s_max > f.tile_cap ? 2u : 0u);
        c[C_ENTRIES] = *s_sum;
        c[C_OVERFLOW] = overflow;
        if (overflow) { atomicOr(f.sticky + 0, overflow); }
        atomicMax(f.sticky + 1, __ldcg(c + C_SETUPS));
        atomicMax(f.sticky + 2, *s_max);
        atomicMax(f.sticky + 3, __ldcg(c + C_BIG));
    }
}

// ------------------------------------------------------------------------------------------------
// Fused geometry for small scenes: one 256-thread CTA per view runs reset, vertex stage and setup back
// to back (block barriers instead of kernel boundaries).  No binning at all: with at most SORT_CAP
// surviving triangles every raster CTA scans the setup list itself (Frame::direct_bin).  The per-frame
// work of a 51-triangle scene is launch latency, not arithmetic.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) geometry_small(const __grid_constant__ Frame f) {
    __shared__ SetupShared sh;
    const uint32_t view = blockIdx.x, tid = threadIdx.x;
    const Cam cam = load_cam(f, view);
    if (tid < C_COUNT) { f.counters[view * C_COUNT + tid] = 0; }
    for (uint32_t i4 = tid * 4u; i4 < f.Vpad; i4 += 1024u) { vertex_body(f, cam, view, i4); }
    __syncthreads();
    for (uint32_t chunk = 0; chunk * 256u < f.T; chunk++) {
        classify_body(f, view, chunk, sh);
        process_items<true>(f, cam, view, sh);
    }
    __syncthreads();
    if (tid == 0) {
        const uint32_t *c = f.counters + view * C_COUNT;
        if (c[C_OVERFLOW]) { atomicOr(f.sticky + 0, c[C_OVERFLOW]); }
        atomicMax(f.sticky + 1, c[C_SETUPS]);
    }
    if (f.coltab && tid < 32u) {
        // the first SPAN_MAX survivors (in slot order) with a box of SPAN_MIN pixels or more get a checkpoint table
        const uint32_t n = f.counters[view * C_COUNT + C_OVERFLOW] ? 0u
                         : min(f.counters[view * C_COUNT + C_SETUPS], min(f.setup_cap, (uint32_t)SORT_CAP));
        uint32_t count = 0;
        for (uint32_t base = 0; base < n && count < SPAN_MAX; base += 32u) {
            const uint32_t slot = base + tid;
            bool q = false;
            if (slot < n) {
                const Head h = unpack_head(f.head[(size_t)view * f.setup_cap + slot]);
                q = h.xmax - h.xmin >= SPAN_MIN || h.ymax - h.ymin >= SPAN_MIN;
            }
            const uint32_t m = __ballot_sync(0xFFFFFFFFu, q);
            const uint32_t idx = count + __popc(m & ((1u << tid) - 1u));
            if (q && idx < SPAN_MAX) { f.span_slots[view * SPAN_MAX + idx] = slot; }
            count += __popc(m);
        }
        if (tid == 0) { f.counters[view * C_COUNT + C_SPANS] = min(count, SPAN_MAX); }
    }
}

// Small scenes, once per frame: the checkpoint tables of the (at most SPAN_MAX) largest survivors.  One thread per
// (span, component, pixel row): the row's start weight by the exact jump from the triangle's wstart (render.cpp:378-379),
// then the reference's own walk along the row (render.cpp:374) — true additions from xmin to xmax — dropping the
// weight at the first walked pixel of every tile column.  Every tile's stage A then loads what it would otherwise
// reach with two exact jumps per (row, component); the values are the same bits.  Threads of a warp are consecutive
// rows, so every store (and every later load) is one coalesced line.
__global__ void __launch_bounds__(128) span_walk(const __grid_constant__ Frame f) {
    const uint32_t view = blockIdx.z, k = blockIdx.y / 3u, c = blockIdx.y % 3u, y = blockIdx.x * 128u + threadIdx.x;
    if (k >= f.counters[view * C_COUNT + C_SPANS] || y >= f.H) { return; }
    const uint32_t a = y / TILE_H;   // rows of tile rows this submission does not rasterise are never read
    if (!owns_row(f, a) || a * TILE_H >= f.y1 || (a + 1u) * TILE_H <= f.y0) { return; }
    const uint32_t slot = f.span_slots[view * SPAN_MAX + k];
    const SetupVis *v = f.vis + (size_t)view * f.setup_cap + slot;
    const uint32_t xmin = v->xmin, xmax = v->xmax, ymin = v->ymin, ymax = v->ymax;
    if (y < ymin || y > ymax) { return; }
    const float d = v->dx[c];
    float w = walk_near(v->wstart[c], v->dy[c], y - ymin);
    const uint32_t t0 = xmin / TILE_W, t1 = xmax / TILE_W;
    float *tab = f.coltab + ((((size_t)view * SPAN_MAX + k) * f.tiles_x + t0) * 3u + c) * f.span_h + y;
    uint32_t x = xmin;
    for (uint32_t t = t0; ; t++) {
        *tab = w;
        if (t == t1) { break; }
        const uint32_t next = (t + 1u) * TILE_W;
        if (next - x == (uint32_t)TILE_W) {
#pragma unroll 16
            for (int j = 0; j < TILE_W; j++) { w = add_rn(w, d); }
        } else {
            for (uint32_t j = x; j < next; j++) { w = add_rn(w, d); }
        }
        x = next;
        tab += 3u * f.span_h;
    }
}

// ------------------------------------------------------------------------------------------------
// K4 — per-tile rasteriser
// ------------------------------------------------------------------------------------------------

struct RasterShared {
    union {                                               // 32 KB
        struct {
            float segstart[BATCH][TILE_H][SEGS_PER_ROW][3];   // big triangles: exact weights at each 8-pixel segment start
            SetupVis batch[BATCH];
            uint32_t bigq[RASTER_THREADS];                    // big triangles found in the current 256-entry chunk
            uint32_t span[BATCH];                             // the batch triangles' checkpoint tables (span_walk), NO_TRI = none
        } big;
        uint4 state[TILE_W * TILE_H];                     // later: per-pixel winners (w0, w1, w2, slot) for shading
    } u;
    union {                                               // 16 KB
        unsigned long long keys[TILE_W * TILE_H];         // small triangles: depth << 32 | ~order, atomicMax
        uint32_t colour[TILE_H][TILE_W];                  // later: the colour tile, source of the bulk write-out
    } k;
    uint16_t slots[SORT_CAP];                             // 7.5 KB: this tile's triangles when collected in-kernel (direct_bin)
    uint32_t n_list, n_big, any_small;
};
// four tile_raster CTAs per SM: 4 x (dynamic + 1 KB reserved) must fit the 228 KB of an SM
static_assert(sizeof(RasterShared) <= 56 * 1024, "RasterShared must leave room for four CTAs per SM");
static_assert(SORT_CAP < 0x8000, "list entries are 15-bit slots plus the WON flag");

__device__ __forceinline__ uint32_t next_pow2_8(uint32_t i) {  // render.cpp:115-122 for its domain 1 <= i <= 256
    // i--; i |= i >> 1; i |= i >> 2; i |= i >> 4; return i + 1;  ==  one past the smeared top bit of i - 1
    return 1u << (32 - __clz((int)(i - 1u)));
}

// render.cpp:363-372 + getColor (:339-359) + getTextureColor (:124-132) for one winning pixel
__device__ __forceinline__ uint32_t shade_math(const Frame &f, float rz0, float rz1, float rz2, const SetupShade &s,
                                               float w0, float w1, float w2) {
    const float ooz = (rz0 * w0 + rz1 * w1) + rz2 * w2;
    float b0, b1, b2;
    div3_rn(w0, w1, w2, ooz, b0, b1, b2);   // w / ooz (render.cpp:365), one reciprocal refinement for the three
    const float3 c0 = make_float3(s.cv[0], s.cv[1], s.cv[2]), c1 = make_float3(s.cv[3], s.cv[4], s.cv[5]),
                 c2 = make_float3(s.cv[6], s.cv[7], s.cv[8]);
    const float3 n0 = make_float3(s.n[0], s.n[1], s.n[2]), n1 = make_float3(s.n[3], s.n[4], s.n[5]),
                 n2 = make_float3(s.n[6], s.n[7], s.n[8]);
    const float3 pu = unit3(add3(add3(scale3(c0, b0), scale3(c1, b1)), scale3(c2, b2)));
    const float3 point = make_float3(-pu.x, -pu.y, -pu.z);
    const float3 normal = unit3(add3(add3(scale3(n0, b0), scale3(n1, b1)), scale3(n2, b2)));
    const float3 halfway = unit3(add3(point, normal));
    const float shade = dot3(halfway, normal);
    float3 base;
    if (s.kind == 0) {
        const float3 k0 = make_float3(s.pay[0], s.pay[1], s.pay[2]), k1 = make_float3(s.pay[3], s.pay[4], s.pay[5]),
                     k2 = make_float3(s.pay[6], s.pay[7], s.pay[8]);
        base = add3(add3(scale3(k0, b0), scale3(k1, b1)), scale3(k2, b2));
    } else {
        const float u = (s.pay[0] * b0 + s.pay[2] * b1) + s.pay[4] * b2;
        const float v = (s.pay[1] * b0 + s.pay[3] * b1) + s.pay[5] * b2;
        const float level_x = ooz / fabsf(s.tpp[0] - u * s.pay[6]);
        const float level_y = ooz / fabsf(s.tpp[1] - v * s.pay[7]);
        const uint32_t lx = next_pow2_8((uint32_t)fmaxf(fminf(level_x, 256.f), 1.f));
        const uint32_t ly = next_pow2_8((uint32_t)fmaxf(fminf(level_y, 256.f), 1.f));
        // fmodf(t, 1) == t - truncf(t) exactly for finite t (the fractional bits are representable)
        const uint32_t x = (uint32_t)((u - truncf(u)) * (float)lx) + (511u & ~(2u * lx - 1u));
        const uint32_t y = (uint32_t)((v - truncf(v)) * (float)ly) + (511u & ~(2u * ly - 1u));
        const uint32_t idx = (x + (y << 9)) & 0x3FFFFu;  // stays inside the atlas even for hostile uv
        const uint32_t rgb = __ldg(f.texels + ((size_t)s.texture << 18) + idx);   // s.texture < n_tex (make_setup)
        base = make_float3((float)(rgb >> 16), (float)((rgb >> 8) & 255u), (float)(rgb & 255u));
    }
    const uint32_t r = (uint32_t)(int)(shade * base.x) & 255u, g = (uint32_t)(int)(shade * base.y) & 255u,
                   b = (uint32_t)(int)(shade * base.z) & 255u;
    return (((r << 8) + g) << 8) + b;  // RGB(), render.cpp:8
}

// the same, from a setup record
__device__ __forceinline__ uint32_t shade_pixel(const Frame &f, uint32_t view, uint32_t slot, float w0, float w1, float w2) {
    const SetupVis *vp = f.vis + (size_t)view * f.setup_cap + slot;
    const float rz0 = vp->rvz[0], rz1 = vp->rvz[1], rz2 = vp->rvz[2];
    const uint4 *sp = reinterpret_cast<const uint4 *>(f.shade + (size_t)view * f.setup_cap + slot);
    SetupShade s;
    uint4 *sd = reinterpret_cast<uint4 *>(&s);
#pragma unroll
    for (int i = 0; i < 8; i++) { sd[i] = sp[i]; }
    return shade_math(f, rz0, rz1, rz2, s, w0, w1, w2);
}

__device__ __forceinline__ uint32_t swizzled(uint32_t row, uint32_t seg, uint32_t j) {
    return row * TILE_W + seg * SEG + (j ^ (seg & 7u));  // spreads a thread's 8-pixel run over the 16-byte bank groups
}

// Output row (inside the submission's output, signed: a band may start inside a tile) of a tile's first pixel row.
__device__ __forceinline__ int32_t tile_first_out_row(const Frame &f, uint32_t ty0, uint32_t tile_a) {
    return f.row_stride == 1u ? (int32_t)ty0 - (int32_t)f.y0 : (int32_t)(div_stride(f, tile_a) * TILE_H);
}

// One TMA tensor store for a whole tile: the box (TILE_W pixels x TILE_H rows, contiguous in shared memory) goes to
// {x, row, view} of the output tensor; whatever lies outside the tensor (band edges, a partial last tile) is clipped
// by the copy engine.  Called by all threads after the tile is complete in shared memory; one thread issues it.
__device__ __forceinline__ void tensor_store_tile(const Frame &f, const void *tile_smem, int32_t x, int32_t row, int32_t view) {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> visible to the async proxy
    __syncthreads();
    if (threadIdx.x == 0) {
        const uint32_t src = (uint32_t)__cvta_generic_to_shared(tile_smem);
        asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%1, %2, %3}], [%4];"
                     :: "l"(reinterpret_cast<unsigned long long>(&f.out_map)), "r"(x), "r"(row), "r"(view), "r"(src) : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    }
}

// Write-out of a finished tile whose rows lie in shared memory `pitch` bytes apart, `bpp` bytes per pixel (4: 32-bit pixels,
// 3: packed 24-bit transport).  One TMA tensor store for the tile (its map counts bytes for the packed format, pixels
// otherwise), else one bulk copy per row, else plain stores — 32-bit ones, or bytes for packed rows, which are not word
// aligned in the output.  All threads call.
__device__ __forceinline__ void write_tile(const Frame &f, uint32_t view, uint32_t tx0, uint32_t ty0, uint32_t tile_a,
                                           const void *tile, uint32_t pitch, uint32_t bpp) {
    const uint32_t tid = threadIdx.x, unit = bpp == 4u ? 4u : 1u;   // unit: bytes per plain store and per tensor-map element
    const uint32_t row_bytes = min((uint32_t)TILE_W, f.W - tx0) * bpp;
    uint8_t *out = reinterpret_cast<uint8_t *>(f.out) + (size_t)view * f.out_view_stride * bpp;
    const uint8_t *src = static_cast<const uint8_t *>(tile);
    if (f.use_tmap) {
        tensor_store_tile(f, tile, (int32_t)(tx0 * bpp / unit), tile_first_out_row(f, ty0, tile_a), (int32_t)view);
    } else if (f.use_tma) {
        // make the generic-proxy writes to the tile visible to the async (TMA) proxy
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncthreads();
        // the bulk copy takes uniform operands, so a warp issues its lanes' copies one after the other: four rows per
        // warp on all eight warps instead of 32 rows on one
        constexpr uint32_t ROWS_PER_WARP = TILE_H / (RASTER_THREADS / 32);
        static_assert(ROWS_PER_WARP * (RASTER_THREADS / 32) == TILE_H, "tile rows split evenly over the warps");
        const uint32_t srow = (tid >> 5) * ROWS_PER_WARP + (tid & 31u);
        if ((tid & 31u) < ROWS_PER_WARP) {
            const uint32_t yy = ty0 + srow;
            if (yy >= f.y0 && yy < f.y1) {
                uint8_t *dst = out + (out_row(f, yy, tile_a) * f.W + tx0) * bpp;
                const uint32_t s = (uint32_t)__cvta_generic_to_shared(src + srow * pitch);
                asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" :: "l"(dst), "r"(s), "r"(row_bytes) : "memory");
            }
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        }
    } else {
        __syncthreads();
        const uint32_t per_row = TILE_W * bpp / unit;
        for (uint32_t i = tid; i < TILE_H * per_row; i += RASTER_THREADS) {
            const uint32_t pr = i / per_row, off = (i % per_row) * unit, yy = ty0 + pr;
            if (off < row_bytes && yy >= f.y0 && yy < f.y1) {
                uint8_t *dst = out + (out_row(f, yy, tile_a) * f.W + tx0) * bpp + off;
                if (unit == 4u) { *reinterpret_cast<uint32_t *>(dst) = *reinterpret_cast<const uint32_t *>(src + pr * pitch + off); }
                else { *dst = src[pr * pitch + off]; }
            }
        }
    }
}

// Per-triangle walk of a small triangle inside one tile, exactly as the reference walks it
// (render.cpp:360-382): rows from the triangle's own ymin, pixels from its own xmin, true additions only.
// PASS 1 publishes depth keys with atomicMax; PASS 2 (after every key is final) lets the winner of each
// pixel drop its weights for shading.  Keys are depth << 32 | ~order: larger 1/z wins, on equal depth the
// earlier triangle in the reference's processing order wins (strict '>' at render.cpp:364).
template <int PASS>
__device__ __forceinline__ bool walk_small(const Frame &f, uint32_t view, uint32_t slot, const Head &h, uint32_t tx0,
                                           uint32_t ty0, uint32_t ylo_t, uint32_t yhi_t, RasterShared &sh) {
    const VisCore v = load_vis(f.vis + (size_t)view * f.setup_cap + slot).c;
    float wy0 = v.ws[0], wy1 = v.ws[1], wy2 = v.ws[2];
    const unsigned long long key_lo = (unsigned long long)(~h.order);
    const uint32_t y_end = min(h.ymax, yhi_t - 1u), x_end = min(h.xmax, tx0 + TILE_W - 1u);
    bool won = false;
    for (uint32_t y = h.ymin; y <= y_end; y++) {
        if (y >= ylo_t) {
            float w0 = wy0, w1 = wy1, w2 = wy2;
            for (uint32_t x = h.xmin; x <= x_end; x++) {
                if (x >= tx0 && w0 >= 0 && w1 >= 0 && w2 >= 0) {                      // render.cpp:362
                    const float ooz = (v.rz[0] * w0 + v.rz[1] * w1) + v.rz[2] * w2;  // render.cpp:363
                    if (ooz > 0.f) {                                                 // depth buffer starts at 0, strict '>'
                        const uint32_t idx = (y - ty0) * TILE_W + (x - tx0);
                        const unsigned long long key = ((unsigned long long)__float_as_uint(ooz) << 32) | key_lo;
                        if (PASS == 1) {
                            if (key > sh.k.keys[idx]) { atomicMax(&sh.k.keys[idx], key); won = true; }
                        } else if (sh.k.keys[idx] == key) {
                            const uint32_t pc = x - tx0;
                            sh.u.state[(y - ty0) * TILE_W + (pc & ~7u) + ((pc & 7u) ^ ((pc >> 3) & 7u))] =
                                make_uint4(__float_as_uint(w0), __float_as_uint(w1), __float_as_uint(w2), slot);
                        }
                    }
                }
                w0 = add_rn(w0, v.dx[0]); w1 = add_rn(w1, v.dx[1]); w2 = add_rn(w2, v.dx[2]);     // render.cpp:374
            }
        }
        wy0 = add_rn(wy0, v.dy[0]); wy1 = add_rn(wy1, v.dy[1]); wy2 = add_rn(wy2, v.dy[2]);       // render.cpp:378
    }
    return won;
}

// One tile (TILE_W x TILE_H pixels).  DIRECT (small scenes): the CTA collects the tile's triangles from the survivor
// list itself, resolves visibility, shades and writes the colour tile.  !DIRECT (general path): the CTA resolves
// entries [e0, e1) of the tile's bin list — recorded triangles too large for the flat walk — and merges its winners
// into the visibility buffer with 64-bit atomicMax, so that a long list can be shared by several CTAs.
template <bool DIRECT>
__device__ __forceinline__ void raster_one_tile(const Frame &f, RasterShared &sh, uint32_t view, uint32_t tile_x, uint32_t tile_y,
                                                uint32_t e0, uint32_t e1) {
    const uint32_t tid = threadIdx.x;
    const uint32_t tile = tile_y * f.tiles_x + tile_x;               // tile_y: local row index
    const uint32_t tile_a = abs_row(f, tile_y);                      // absolute tile row
    const uint32_t tx0 = tile_x * TILE_W, ty0 = tile_a * TILE_H;
    const uint32_t row = tid / SEGS_PER_ROW, seg = tid % SEGS_PER_ROW;
    const uint32_t y = ty0 + row, sx0 = tx0 + seg * SEG;
    const uint32_t ylo_t = max(ty0, f.y0), yhi_t = min(ty0 + TILE_H, f.y1);   // rows [ylo_t, yhi_t) of this tile are in the band

    // A capacity overflow anywhere upstream makes the lists incomplete: the host regrows the
    // buffers and renders the frame again, so this launch only has to stay in bounds.
    if (f.counters[view * C_COUNT + C_OVERFLOW] != 0) { return; }

    // ---- this tile's triangle list (unordered: depth keys carry the order) ---------------------
    if (tid == 0) { sh.n_list = 0; sh.n_big = 0; sh.any_small = 0; }
    if (DIRECT) {   // in-tile keys are only used when small triangles are walked in the tile (small scenes)
#pragma unroll
        for (int i = 0; i < (TILE_W * TILE_H) / RASTER_THREADS; i++) { sh.k.keys[i * RASTER_THREADS + tid] = 0ull; }
    }
    __syncthreads();
    uint32_t n;
    using Entry = typename std::conditional<DIRECT, uint16_t, uint32_t>::type;   // in-kernel list (shared) / bin list (global)
    constexpr Entry WON = DIRECT ? (Entry)0x8000u : (Entry)0x80000000u;
    Entry *list;
    if (DIRECT) {
        // small scene: collect straight from the survivors' heads (bbox overlap clamped to the band, plus the
        // conservative outside test); at most SORT_CAP survivors exist by construction of this mode
        const uint32_t n_setups = min(f.counters[view * C_COUNT + C_SETUPS], min(f.setup_cap, (uint32_t)SORT_CAP));
        for (uint32_t slot = tid; slot < n_setups; slot += RASTER_THREADS) {
            const Head h = unpack_head(f.head[(size_t)view * f.setup_cap + slot]);
            if (h.xmax >= tx0 && h.xmin < tx0 + TILE_W && h.ymax >= ylo_t && h.ymin < yhi_t) {
                if (!tile_outside_triangle(f.vis[(size_t)view * f.setup_cap + slot], tx0, ylo_t, yhi_t)) {
                    sh.slots[atomicAdd(&sh.n_list, 1u)] = (uint16_t)slot;
                }
            }
        }
        __syncthreads();
        n = sh.n_list;
        list = reinterpret_cast<Entry *>(sh.slots);
    } else {
        n = e1 - e0;
        list = reinterpret_cast<Entry *>(f.entries + ((size_t)view * f.tile_stride + tile) * f.tile_cap + e0);
    }

    if (DIRECT && n == 0u) {
        // nothing reaches this tile: it is background (render.cpp:282) — straight to the write-out
#pragma unroll
        for (int j = 0; j < SEG; j++) { sh.k.colour[row][seg * SEG + j] = kBackground; }
    } else {
    float depth[SEG], bw0[SEG], bw1[SEG], bw2[SEG];
    uint32_t win[SEG];
#pragma unroll
    for (int j = 0; j < SEG; j++) { depth[j] = 0.f; bw0[j] = bw1[j] = bw2[j] = 0.f; win[j] = NO_TRI; }

    // ---- phase 1: visibility.  256 list entries at a time: small triangles are walked by one thread each
    // (depth keys in shared memory), big ones are queued and then walked by the whole CTA, eight at a time,
    // every thread owning 8 pixels whose depth/winner/weights stay in registers.
    for (uint32_t cbase = 0; cbase < n; cbase += RASTER_THREADS) {
        const uint32_t i = cbase + tid;
        if (i < n) {
            const uint32_t slot = list[i];
            const Head h = unpack_head(f.head[(size_t)view * f.setup_cap + slot]);
            if (is_small_bbox(h.xmin, h.xmax, h.ymin, h.ymax)) {
                sh.any_small = 1u;
                if (walk_small<1>(f, view, slot, h, tx0, ty0, ylo_t, yhi_t, sh)) { list[i] = (Entry)(slot | WON); }
            } else {
                sh.u.big.bigq[atomicAdd(&sh.n_big, 1u)] = slot;
            }
        }
        __syncthreads();
        const uint32_t nbig = sh.n_big;
        for (uint32_t base = 0; base < nbig; base += BATCH) {
            const uint32_t nb = min((uint32_t)BATCH, nbig - base);
            if (tid < nb * 4u) {   // stage the batch's coverage records
                const uint32_t b = tid >> 2, q = tid & 3u;
                reinterpret_cast<uint4 *>(&sh.u.big.batch[b])[q] =
                    reinterpret_cast<const uint4 *>(f.vis + (size_t)view * f.setup_cap + sh.u.big.bigq[base + b])[q];
            } else if (tid >= 32u && tid < 32u + nb) {   // ... and find their checkpoint tables, if they have one
                uint32_t span = NO_TRI;   // DIRECT: index of the triangle's checkpoint table; queue path: offset of its row-start block
                const uint32_t slot = sh.u.big.bigq[base + tid - 32u];
                if (DIRECT && f.coltab) {
                    const uint32_t n_span = f.counters[view * C_COUNT + C_SPANS];
                    for (uint32_t k = 0; k < n_span; k++) { if (f.span_slots[view * SPAN_MAX + k] == slot) { span = k; } }
                } else if (!DIRECT && f.rowtab) {
                    span = f.rowbase[(size_t)view * f.setup_cap + slot];
                }
                sh.u.big.span[tid - 32u] = span;
            }
            __syncthreads();
            // stage A: exact weights at the first walked pixel of every (triangle, row, segment).  One work item per
            // (triangle, component, row), a warp holding the 32 rows of one (triangle, component) — neighbouring rows take
            // nearly the same path through the exact jump, so a warp does not serialise over components.  Each item goes
            // from the triangle's wstart down to its row (render.cpp:378-379), then along the row to the tile's first
            // column (render.cpp:374) — true steps when the target is near, the exact jump otherwise — and then takes
            // true steps through the tile, dropping the value at every 8-pixel segment boundary.
            for (uint32_t item = tid; item < nb * (TILE_H * 3u); item += RASTER_THREADS) {
                const uint32_t b = item / (TILE_H * 3u), rc = item % (TILE_H * 3u), c = rc / TILE_H, r = rc % TILE_H;
                const SetupVis &v = sh.u.big.batch[b];
                const uint32_t yy = ty0 + r;
                if (yy < v.ymin || yy > v.ymax) { continue; }
                const uint32_t xs = max(tx0, (uint32_t)v.xmin), xe = min(tx0 + TILE_W - 1u, (uint32_t)v.xmax);
                if (xs > xe) { continue; }
                const float d = v.dx[c];
                const uint32_t span = sh.u.big.span[b];
                float w;
                if (span == NO_TRI) {
                    w = weight_at(v.wstart[c], v.dy[c], yy - v.ymin, d, xs - v.xmin);
                } else if (DIRECT) {   // walked once for the whole frame by span_walk: the same bits, one load
                    w = f.coltab[((((size_t)view * SPAN_MAX + span) * f.tiles_x + tile_x) * 3u + c) * f.span_h + yy];
                } else {               // row start walked once by post_setup, then along the row
                    const uint32_t h = (uint32_t)v.ymax - v.ymin + 1u;
                    w = walk_near(f.rowtab[(size_t)view * f.rowtab_cap + span + c * h + (yy - v.ymin)], d, xs - v.xmin);
                }
                uint32_t x = xs, k = (xs - tx0) / SEG;
                while (true) {
                    sh.u.big.segstart[b][r][k][c] = w;
                    const uint32_t next = tx0 + (k + 1u) * SEG;
                    if (next > xe) { break; }
                    if (next - x == (uint32_t)SEG) {   // a whole segment: eight dependent additions, no loop control
#pragma unroll
                        for (int j = 0; j < SEG; j++) { w = add_rn(w, d); }
                        x = next;
                    } else {
                        for (; x < next; x++) { w = add_rn(w, d); }
                    }
                    k++;
                }
            }
            __syncthreads();
            // stage B: every thread walks its 8 pixels through the batch
            for (uint32_t b = 0; b < nb; b++) {
                const SetupVis &v = sh.u.big.batch[b];
                if (y < v.ymin || y > v.ymax) { continue; }
                const uint32_t xa = max(sx0, (uint32_t)v.xmin), xb = min(sx0 + SEG - 1u, (uint32_t)v.xmax);
                if (xa > xb) { continue; }
                const float d0 = v.dx[0], d1 = v.dx[1], d2 = v.dx[2];
                float w0 = sh.u.big.segstart[b][row][seg][0], w1 = sh.u.big.segstart[b][row][seg][1],
                      w2 = sh.u.big.segstart[b][row][seg][2];
                const float rz0 = v.rvz[0], rz1 = v.rvz[1], rz2 = v.rvz[2];
                const uint32_t slot = sh.u.big.bigq[base + b], order = v.order;
#pragma unroll
                for (int j = 0; j < SEG; j++) {
                    const uint32_t x = sx0 + j;
                    if (x >= xa && x <= xb) {
                        if (w0 >= 0 && w1 >= 0 && w2 >= 0) {                         // render.cpp:362
                            const float ooz = (rz0 * w0 + rz1 * w1) + rz2 * w2;      // render.cpp:363
                            bool better = ooz > depth[j];                            // render.cpp:364
                            if (ooz == depth[j] && ooz > 0.f) {
                                // exact depth tie between two triangles: the reference keeps the earlier one
                                better = order < f.head[(size_t)view * f.setup_cap + win[j]].z;
                            }
                            if (better) { depth[j] = ooz; bw0[j] = w0; bw1[j] = w1; bw2[j] = w2; win[j] = slot; }
                        }
                        w0 = add_rn(w0, d0); w1 = add_rn(w1, d1); w2 = add_rn(w2, d2);   // render.cpp:374
                    }
                }
            }
            __syncthreads();  // batch / segstart are rewritten by the next iteration
        }
        if (tid == 0) { sh.n_big = 0; }
        __syncthreads();
    }

    if (!DIRECT) {
        // general path: a candidate takes the pixel where its key beats what the flat walks and the other CTAs working
        // on this tile have published.  Shading (shade_tiles) finds the triangle through the key's order and re-derives
        // the weights at the pixel with the exact jump, so nothing but the key has to be stored.
        if (y >= ylo_t && y < yhi_t) {
            const size_t orow = out_row(f, y, tile_a);
            unsigned long long *krow = f.keys + (size_t)view * f.key_view_stride + key_at(f, orow, 0u);
#pragma unroll
            for (int j = 0; j < SEG; j++) {
                const uint32_t x = sx0 + j;
                if (win[j] != NO_TRI && x < f.W) {
                    const unsigned long long key = ((unsigned long long)__float_as_uint(depth[j]) << 32) |
                                                   (unsigned long long)(~f.head[(size_t)view * f.setup_cap + win[j]].z);
                    // the best candidate so far also leaves its exact weights: three aligned 64-bit words {weight, slot},
                    // each single-copy atomic on its own, so a reader sees every word whole and can tell from the three
                    // tags whether all of them belong to the triangle that holds the key.  A later, better candidate (this
                    // tile's list may be shared by several CTAs) overwrites them in any order; shading checks the tags and
                    // falls back to the exact jump on any mismatch.
                    if (atomicMax(krow + KEY_STEP * x, key) < key) {
                        unsigned long long *ps = f.pstate + 3u * ((size_t)view * f.out_view_stride + orow * f.W + x);
                        const unsigned long long tag = (unsigned long long)win[j] << 32;
                        ps[0] = tag | __float_as_uint(bw0[j]); ps[1] = tag | __float_as_uint(bw1[j]); ps[2] = tag | __float_as_uint(bw2[j]);
                    }
                }
            }
        }
        return;
    }

    // ---- phase 2: per-pixel winners into shared memory (pixel-per-lane layout for coherent shading) ----
    const bool any_small = sh.any_small != 0;
    if (any_small) {
#pragma unroll
        for (int j = 0; j < SEG; j++) { sh.u.state[swizzled(row, seg, j)] = make_uint4(0u, 0u, 0u, NO_TRI); }
        __syncthreads();
        for (uint32_t i = tid; i < n; i += RASTER_THREADS) {   // small triangles that ever led a pixel drop their weights where they won
            const uint32_t e = list[i];
            if (e & WON) {
                const uint32_t slot = e & (uint32_t)(Entry)~WON;
                walk_small<2>(f, view, slot, unpack_head(f.head[(size_t)view * f.setup_cap + slot]), tx0, ty0, ylo_t, yhi_t, sh);
            }
        }
        __syncthreads();
#pragma unroll
        for (int j = 0; j < SEG; j++) {   // a big-triangle candidate wins where its key beats the small ones'
            if (win[j] != NO_TRI) {
                const unsigned long long key = ((unsigned long long)__float_as_uint(depth[j]) << 32) |
                                               (unsigned long long)(~f.head[(size_t)view * f.setup_cap + win[j]].z);
                if (key > sh.k.keys[row * TILE_W + seg * SEG + j]) {
                    sh.u.state[swizzled(row, seg, j)] =
                        make_uint4(__float_as_uint(bw0[j]), __float_as_uint(bw1[j]), __float_as_uint(bw2[j]), win[j]);
                }
            }
        }
    } else {
        __syncthreads();  // big-triangle staging (aliased with state) is dead from here on
#pragma unroll
        for (int j = 0; j < SEG; j++) {
            sh.u.state[swizzled(row, seg, j)] =
                make_uint4(__float_as_uint(bw0[j]), __float_as_uint(bw1[j]), __float_as_uint(bw2[j]), win[j]);
        }
    }
    __syncthreads();
    // ---- phase 3: deferred shading, one pixel per lane -------------------------------------------
#pragma unroll 1
    for (uint32_t it = 0; it < (TILE_W * TILE_H) / RASTER_THREADS; it++) {
        const uint32_t p = it * RASTER_THREADS + tid, pr = p / TILE_W, pc = p % TILE_W;
        const uint4 st = sh.u.state[swizzled(pr, pc / SEG, pc % SEG)];
        uint32_t rgb = kBackground;
        if (st.w != NO_TRI) {
            rgb = shade_pixel(f, view, st.w, __uint_as_float(st.x), __uint_as_float(st.y), __uint_as_float(st.z));
        }
        sh.k.colour[pr][pc] = rgb;
    }
    }   // tile with triangles

    // ---- write-out -------------------------------------------------------------------------
    if (f.out_packed24) {
        // host transport format: 3 bytes per pixel.  Pack each row of 64 pixels into 48 words (reusing the dead per-pixel
        // state), then write out 192-byte rows.
        __syncthreads();
        constexpr uint32_t PW = TILE_W * 3u / 4u;                       // packed words per tile row
        uint32_t *packed = reinterpret_cast<uint32_t *>(sh.u.state);   // [TILE_H][PW]
        for (uint32_t g = tid; g < TILE_H * (TILE_W / 4); g += RASTER_THREADS) {
            const uint32_t pr = g / (TILE_W / 4), q = g % (TILE_W / 4);
            const uint4 p = *reinterpret_cast<const uint4 *>(&sh.k.colour[pr][q * 4]);
            uint32_t *o = packed + pr * PW + q * 3u;
            o[0] = p.x | (p.y << 24);
            o[1] = (p.y >> 8) | (p.z << 16);
            o[2] = (p.z >> 16) | (p.w << 8);
        }
        write_tile(f, view, tx0, ty0, tile_a, packed, PW * 4u, 3u);
    } else {
        write_tile(f, view, tx0, ty0, tile_a, &sh.k.colour[0][0], TILE_W * 4u, 4u);
    }
}

__global__ void __launch_bounds__(RASTER_THREADS, RASTER_CTAS) tile_raster(const __grid_constant__ Frame f) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    raster_one_tile<true>(f, *reinterpret_cast<RasterShared *>(smem_raw), blockIdx.z, blockIdx.x, blockIdx.y + f.raster_row0, 0u, 0u);
}

// General path: persistent CTAs pop (tile, chunk of its bin list) items from the queue post_setup built.  A tile with
// a long list is shared by as many CTAs as it has chunks, so the busiest tile no longer sets the kernel's duration.
constexpr int QUEUE_CTAS = 4;   // tile_raster_queue CTAs per SM
__global__ void __launch_bounds__(RASTER_THREADS, QUEUE_CTAS) tile_raster_queue(const __grid_constant__ Frame f) {
    wait_for_predecessor();
    extern __shared__ __align__(128) unsigned char smem_raw[];
    RasterShared &sh = *reinterpret_cast<RasterShared *>(smem_raw);
    const uint32_t view = blockIdx.y;
    uint32_t *c = f.counters + view * C_COUNT;
    const uint32_t n_items = min(c[C_ITEMS], f.items_cap);
    if (n_items == 0u) { return; }   // no triangle over 128 pixels this frame: not even the queue counter is touched
    while (true) {
        __syncthreads();   // the previous item's shared-memory state is dead
        if (threadIdx.x == 0) { sh.n_list = atomicAdd(c + C_QHEAD, 1u); }
        __syncthreads();
        const uint32_t i = sh.n_list;
        if (i >= n_items) { return; }
        __syncthreads();
        const uint2 item = f.raster_items[(size_t)view * f.items_cap + i];   // {tile, first entry}
        const uint32_t n = min(f.tile_count[view * f.tile_stride + item.x], f.tile_cap);
        raster_one_tile<false>(f, sh, view, item.x % f.tiles_x, item.x / f.tiles_x, item.y, min(n, item.y + RASTER_CHUNK));
    }
}

// ------------------------------------------------------------------------------------------------
// Flat path for small triangles (general, binned mode).  Dense fields put thousands of tiny triangles into
// the busiest tiles; a tile CTA would then run as long as its list.  Instead every small survivor is walked by
// one thread over its whole bounding box (no tiles, no binning, no duplication), publishing 64-bit depth keys
// with atomicMax in global memory (L2-resident), exactly like walk_small does in shared memory.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) post_setup(const __grid_constant__ Frame f) {
    wait_for_predecessor();
    constexpr uint32_t FLAT_ROUND = 64, FLAT_CK = 16;   // survivors per round; row-start checkpoints per survivor, one every 8 rows
    __shared__ uint32_t s_sum, s_max, s_last, s_round, s_warp[8], s_pref[257];
    __shared__ float s_ck[FLAT_ROUND][FLAT_CK][3];
    __shared__ uint4 s_head[FLAT_ROUND], s_rec[FLAT_ROUND][4];   // the round's survivors, staged once (the items are latency-bound otherwise)
    const uint32_t view = blockIdx.y;
    if (f.counters[view * C_COUNT + C_SETUPS] == 0u && f.counters[view * C_COUNT + C_BIG] == 0u) {
        // no recorded triangle at all (every survivor took the record-free direct walk): nothing to bin, nothing to walk, all
        // tile lists empty — one thread closes the frame's geometry, and 591 CTAs skip their two global atomics
        if (blockIdx.x == 0 && threadIdx.x == 0) {
            uint32_t *c = f.counters + view * C_COUNT;
            const uint32_t overflow = c[C_OVERFLOW];
            c[C_ENTRIES] = 0;
            if (overflow) { atomicOr(f.sticky + 0, overflow); }
        }
        return;
    }
    bin_big_body(f, view);   // K3 for the triangles the setup kernel left to a whole CTA
    if (f.rowtab) {
        // row starts of the tile-path triangles: one thread per triangle takes a block of the table and walks its own
        // rows with true additions (three independent chains).  Every (tile, triangle) pair of the tile kernel would
        // otherwise pay an exact jump per (row, component) for the same values.
        const uint32_t n_all = min(f.counters[view * C_COUNT + C_SETUPS], f.setup_cap);
        for (uint32_t slot = blockIdx.x * blockDim.x + threadIdx.x; slot < n_all; slot += gridDim.x * blockDim.x) {
            const Head hd = unpack_head(f.head[(size_t)view * f.setup_cap + slot]);
            uint32_t base = NO_TRI;
            if (!is_flat_bbox(f, hd.xmin, hd.xmax, hd.ymin, hd.ymax)) {
                const uint32_t h = hd.ymax - hd.ymin + 1u;
                base = atomicAdd(f.counters + view * C_COUNT + C_ROWTAB, 3u * h);
                if (base > f.rowtab_cap || 3u * h > f.rowtab_cap - base) { base = NO_TRI; }   // table full: this one keeps jumping
            }
            f.rowbase[(size_t)view * f.setup_cap + slot] = base;
            if (base == NO_TRI) { continue; }
            const VisCore v = load_vis(f.vis + (size_t)view * f.setup_cap + slot).c;
            float w0 = v.ws[0], w1 = v.ws[1], w2 = v.ws[2];
            const uint32_t h = hd.ymax - hd.ymin + 1u;
            float *t = f.rowtab + (size_t)view * f.rowtab_cap + base;
            for (uint32_t r = 0; r < h; r++) {
                t[r] = w0; t[h + r] = w1; t[2u * h + r] = w2;
                w0 = add_rn(w0, v.dy[0]); w1 = add_rn(w1, v.dy[1]); w2 = add_rn(w2, v.dy[2]);
            }
        }
    }
    // Flat walk of the recorded triangles under flat_max x flat_max pixels: FLAT_ROUND survivors per CTA and round, one
    // work item per (triangle, box row) found by binary search in the prefix sums of the rows, so that every lane walks
    // one row whatever the mix of box sizes.  Exactly the reference's own additions (render.cpp:374-379).  Rounds are
    // small and handed out by an atomic counter: their cost varies by orders of magnitude with the box sizes, and a
    // static deal of 256-survivor rounds left two thirds of the CTAs without work on the clipping-stress scene.
    unsigned long long *keys = f.keys + (size_t)view * f.key_view_stride;
    const uint32_t n = min(f.counters[view * C_COUNT + C_SETUPS], f.setup_cap);
    const uint32_t tid = threadIdx.x, lane = lane_id(), warp = tid >> 5;
    while (true) {
        if (tid == 0) { s_round = atomicAdd(f.counters + view * C_COUNT + C_FLATQ, 1u); }
        __syncthreads();
        const uint32_t g0 = s_round * FLAT_ROUND;
        if (g0 >= n) { break; }
        uint32_t rows = 0;
        if (g0 + (tid >> 2) < n) {   // 64-byte coverage records of the round: one coalesced 4 KB read
            s_rec[tid >> 2][tid & 3u] = reinterpret_cast<const uint4 *>(f.vis + (size_t)view * f.setup_cap + g0 + (tid >> 2))[tid & 3u];
        }
        if (tid < FLAT_ROUND && g0 + tid < n) {
            const uint4 head = f.head[(size_t)view * f.setup_cap + g0 + tid];
            s_head[tid] = head;
            const Head h = unpack_head(head);
            const uint32_t ylo = max(h.ymin, f.y0), yhi = min(h.ymax, f.y1 - 1u);
            if (is_flat_bbox(f, h.xmin, h.xmax, h.ymin, h.ymax) && ylo <= yhi) { rows = owned_pixel_rows(f, ylo, yhi).count; }
        }
        uint32_t incl = rows;   // block-wide inclusive scan
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const uint32_t v = __shfl_up_sync(0xFFFFFFFFu, incl, d); if (lane >= (uint32_t)d) { incl += v; } }
        if (lane == 31) { s_warp[warp] = incl; }
        __syncthreads();
        uint32_t before = 0;
#pragma unroll
        for (int w = 0; w < 8; w++) { if ((uint32_t)w < warp) { before += s_warp[w]; } }
        s_pref[tid + 1] = before + incl;
        if (tid == 0) { s_pref[0] = 0; }
        __syncthreads();
        const uint32_t total = s_pref[256];
        // row starts (render.cpp:378-379) by true additions, once per (survivor, component): every 8th one is kept, an
        // item then needs at most 7 more additions instead of an exact jump per component
        for (uint32_t idx = tid; idx < FLAT_ROUND * 3u; idx += 256u) {
            const uint32_t sv = idx / 3u, c = idx % 3u;
            if (s_pref[sv + 1u] == s_pref[sv]) { continue; }
            const SetupVis *v = reinterpret_cast<const SetupVis *>(&s_rec[sv][0]);
            const uint32_t last = min(min((uint32_t)v->ymax, f.y1 - 1u) - v->ymin, FLAT_CK * 8u - 1u);
            const float d = v->dy[c];
            float w = v->wstart[c];
            for (uint32_t r = 0; ; r++) {
                if ((r & 7u) == 0u) { s_ck[sv][r >> 3][c] = w; }
                if (r == last) { break; }
                w = add_rn(w, d);
            }
        }
        __syncthreads();
        for (uint32_t i = tid; i < total; i += 256u) {
            uint32_t lo = 0, hi = 256;   // largest j with s_pref[j] <= i
            while (hi - lo > 1u) { const uint32_t mid = (lo + hi) >> 1; if (s_pref[mid] <= i) { lo = mid; } else { hi = mid; } }
            const Head h = unpack_head(s_head[lo]);
            const uint32_t y = owned_row_at(f, owned_pixel_rows(f, max(h.ymin, f.y0), min(h.ymax, f.y1 - 1u)), i - s_pref[lo]), a = y / TILE_H;
            const VisCore v = load_vis(reinterpret_cast<const SetupVis *>(&s_rec[lo][0])).c;
            const uint32_t ck = min((y - h.ymin) >> 3, FLAT_CK - 1u), more = y - h.ymin - 8u * ck;   // more <= 7 for boxes under 128 rows
            const float w0 = walk_near(s_ck[lo][ck][0], v.dy[0], more);   // render.cpp:378
            const float w1 = walk_near(s_ck[lo][ck][1], v.dy[1], more);
            const float w2 = walk_near(s_ck[lo][ck][2], v.dy[2], more);
            unsigned long long *krow = keys + key_at(f, out_row(f, y, a), 0u);
            publish_row(krow, h.xmin, h.xmax, make_float3(w0, w1, w2), make_float3(v.dx[0], v.dx[1], v.dx[2]),
                        make_float3(v.rz[0], v.rz[1], v.rz[2]), (unsigned long long)(~h.order));
        }
        __syncthreads();   // s_pref and s_round are rewritten by the next round
    }
    // the last CTA of the view to get here closes the frame's geometry (tile statistics, overflow record)
    if (threadIdx.x == 0) { s_sum = 0; s_max = 0; }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) { s_last = atomicAdd(f.counters + view * C_COUNT + C_DONE, 1u) == gridDim.x - 1u ? 1u : 0u; }
    __syncthreads();
    if (s_last) {
        __threadfence();
        finalize_body(f, view, &s_sum, &s_max);
    }
}

// Deferred shading of the general path (visibility buffer -> colour).  One CTA per 32 x 16 block of output pixels:
//   1. read the block's depth keys, clear them for the next frame (so no separate reset pass exists), compact the
//      covered pixels into a list and find the block's distinct triangles with a shared-memory hash set (the key's
//      low word is ~order) — background pixels cost nothing beyond this;
//   2. one distinct triangle per lane: an unclipped triangle under 16 x 16 pixels has no record, so its three corners
//      are gathered and set up right here (the same make_setup the recorded path runs, hence the same bits);
//      attributes and normals of triangles that win no pixel are never read.  Recorded triangles are copied from
//      their records (found through slot_of).  The setups are staged in shared memory, 256 per pass;
//   3. one covered pixel per lane: small winners replay their own walk to the pixel (<= 15 + 15 true additions,
//      render.cpp:374-379), winners of the tile path get there with the exact jump; shade (render.cpp:363-372);
//   4. the colour block goes out in 16-byte (or 12-byte, 24-bit transport) pieces.
// (32 x 32 blocks were measured and lose: profiles/r02_experiments.md)
constexpr uint32_t SHADE_B = 32;                              // block width in pixels
constexpr uint32_t SHADE_BH = 16;                             // block height in pixels
constexpr uint32_t SHADE_THREADS = SHADE_B * SHADE_BH / 4;    // four pixels per thread when the keys are read
constexpr uint32_t SHADE_PIX = SHADE_B * SHADE_BH;
constexpr uint32_t SHADE_TAB = 2 * SHADE_PIX;                 // hash slots (load factor <= 0.5)
constexpr uint32_t SHADE_TAB_SHIFT = 22;                      // 32 - log2(SHADE_TAB)
constexpr int SHADE_CTAS = 8;                                 // shade_tiles CTAs per SM the launch bounds ask for
constexpr uint32_t SHADE_TRIS = 96;   // triangle setups staged per pass (one per thread; sized so that the CTAs fit an SM's shared memory)
constexpr uint32_t SHADE_WORDS = 47;      // words per staged setup (odd: distinct triangles fall into distinct banks)
constexpr uint32_t SHADE_EMPTY = 0xFFFFFFFFu;

struct ShadeShared {
    __align__(16) uint32_t colour[SHADE_BH][SHADE_B];
    uint32_t tab[SHADE_TAB];              // hash set of orders; after numbering: slot -> triangle number
    uint32_t tri_order[SHADE_PIX];        // triangle number -> order
    uint16_t pix[SHADE_PIX];              // covered pixel list: position in the block ...
    uint16_t pslot[SHADE_PIX];            // ... and its triangle's hash slot
    uint32_t setup[SHADE_TRIS][SHADE_WORDS];   // ws[3] dx[3] dy[3] rz[3] | xmin|ymin<<16 | big | SetupShade[32]
    uint32_t count, n_tri;
};

template <bool HAS_RV>
__global__ void __launch_bounds__(SHADE_THREADS, SHADE_CTAS) shade_tiles(const __grid_constant__ Frame f, uint32_t row0, uint32_t nrows) {
    wait_for_predecessor();
    extern __shared__ __align__(128) unsigned char smem_raw[];
    ShadeShared &sh = *reinterpret_cast<ShadeShared *>(smem_raw);
    const uint32_t view = blockIdx.z, tid = threadIdx.x, lane = lane_id();
    const uint32_t bx0 = blockIdx.x * SHADE_B, br0 = blockIdx.y * SHADE_BH;       // block origin: pixel column, row within [row0, row0 + nrows)
    const bool broken = f.counters[view * C_COUNT + C_OVERFLOW] != 0;            // incomplete lists: the host renders the frame again
    if (tid == 0) { sh.count = 0; sh.n_tri = 0; }
    const size_t vbase = (size_t)view * f.out_view_stride;
    // ---- 1. keys -> compacted list of covered pixels + distinct triangles ---------------------------
    // A thread reads (and clears) the keys of one column of 4 rows — one 32-byte sector of the key plane where the block
    // starts on a multiple of 4 output rows (always, except in bands that begin inside a tile row).
    const uint32_t pr = tid >> 3, pc = (tid & 7u) * 4u;   // write-out (step 4): block row pr, columns pc .. pc + 3
    const uint32_t kr = (tid >> 5) * 4u, kc = tid & 31u;   // keys: block rows kr .. kr + 3 of block column kc
    uint32_t ord[4] = {0u, 0u, 0u, 0u}, mask = 0;
    if (bx0 + kc < f.W && br0 + kr < nrows) {
        unsigned long long *plane = f.keys + (size_t)view * f.key_view_stride;
        const size_t r_first = (size_t)row0 + br0 + kr;
        if ((r_first & 3u) == 0u && br0 + kr + 3u < nrows) {
            ulonglong2 *kp = reinterpret_cast<ulonglong2 *>(plane + key_at(f, r_first, bx0 + kc));
            const ulonglong2 lo = kp[0], hi = kp[1];
            const unsigned long long key[4] = {lo.x, lo.y, hi.x, hi.y};
#pragma unroll
            for (int k = 0; k < 4; k++) { if (key[k] != 0ull) { ord[k] = ~(uint32_t)key[k]; mask |= 1u << k; } }
            if (mask & 3u) { kp[0] = make_ulonglong2(0ull, 0ull); }
            if (mask & 12u) { kp[1] = make_ulonglong2(0ull, 0ull); }
        } else {
#pragma unroll
            for (int k = 0; k < 4; k++) {
                if (br0 + kr + k < nrows) {
                    unsigned long long *kp = plane + key_at(f, r_first + k, bx0 + kc);
                    const unsigned long long key = *kp;
                    if (key != 0ull) { *kp = 0ull; ord[k] = ~(uint32_t)key; mask |= 1u << k; }
                }
            }
        }
    }
    if (broken) { mask = 0; }
    *reinterpret_cast<uint4 *>(&sh.colour[pr][pc]) = make_uint4(kBackground, kBackground, kBackground, kBackground);
    const bool any = __syncthreads_or(mask != 0u);
    if (any) {
#pragma unroll
        for (int k = 0; k < (int)(SHADE_TAB / SHADE_THREADS); k++) { sh.tab[k * SHADE_THREADS + tid] = SHADE_EMPTY; }
        __syncthreads();
        // warp-aggregated append (a warp's pixels stay together in the list, column by column: neighbours share triangles)
        const uint32_t n = __popc(mask);
        uint32_t incl = n;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const uint32_t v = __shfl_up_sync(0xFFFFFFFFu, incl, d); if (lane >= (uint32_t)d) { incl += v; } }
        const uint32_t total = __shfl_sync(0xFFFFFFFFu, incl, 31);
        uint32_t base = 0;
        if (lane == 31 && total) { base = atomicAdd(&sh.count, total); }
        uint32_t j = __shfl_sync(0xFFFFFFFFu, base, 31) + incl - n;
        uint32_t last_order = SHADE_EMPTY, last_slot = 0;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            if (mask & (1u << k)) {
                uint32_t h = last_slot;
                if (ord[k] != last_order) {   // insert into the hash set (linear probing)
                    h = (ord[k] * 2654435761u) >> SHADE_TAB_SHIFT;
                    while (true) {
                        const uint32_t prev = atomicCAS(&sh.tab[h], SHADE_EMPTY, ord[k]);
                        if (prev == SHADE_EMPTY || prev == ord[k]) { break; }
                        h = (h + 1u) & (SHADE_TAB - 1u);
                    }
                    last_order = ord[k]; last_slot = h;
                }
                sh.pix[j] = (uint16_t)((kr + k) * SHADE_B + kc); sh.pslot[j] = (uint16_t)h; j++;
            }
        }
        __syncthreads();
        // number the distinct triangles
#pragma unroll
        for (int k = 0; k < (int)(SHADE_TAB / SHADE_THREADS); k++) {
            const uint32_t slot = k * SHADE_THREADS + tid, o = sh.tab[slot];
            const uint32_t m = __ballot_sync(0xFFFFFFFFu, o != SHADE_EMPTY);   // one shared-memory atomic per warp, not per triangle
            uint32_t first = 0;
            if (lane == 0 && m) { first = atomicAdd(&sh.n_tri, (uint32_t)__popc(m)); }
            first = __shfl_sync(0xFFFFFFFFu, first, 0);
            if (o != SHADE_EMPTY) { const uint32_t id = first + (uint32_t)__popc(m & ((1u << lane) - 1u)); sh.tri_order[id] = o; sh.tab[slot] = id; }
        }
        __syncthreads();
        const uint32_t count = sh.count, n_tri = sh.n_tri;
        const Cam cam = load_cam(f, view);
#pragma unroll 1
        for (uint32_t tb = 0; tb < n_tri; tb += SHADE_TRIS) {
            // ---- 2. setups of this pass's triangles ------------------------------------------------
            if (tid < SHADE_TRIS && tb + tid < n_tri) {
                const uint32_t order = sh.tri_order[tb + tid];
                uint32_t *dst = sh.setup[tid];
                bool direct = false;
                Corner d0, d1, d2;
                if (f.direct_small && order < f.T) {
                    // all gathers of the triangle are issued before anything is decided: two dependent round trips
                    // (indices, then vertices + attributes) instead of three
                    const uint32_t i0 = __ldg(f.vi0 + order), i1 = __ldg(f.vi1 + order), i2 = __ldg(f.vi2 + order);
                    const uint32_t a0 = __ldg(f.ai0 + order), a1 = __ldg(f.ai1 + order), a2 = __ldg(f.ai2 + order);
                    d0 = gather_corner<HAS_RV>(f, cam, view, i0, a0); d1 = gather_corner<HAS_RV>(f, cam, view, i1, a1); d2 = gather_corner<HAS_RV>(f, cam, view, i2, a2);
                    direct = is_record_free(f, d0.rv.z, d1.rv.z, d2.rv.z, bounds_of(f, d0.rv.x, d0.rv.y, d1.rv.x, d1.rv.y, d2.rv.x, d2.rv.y));
                }
                if (direct) {
                    SetupVis v;
                    SetupShade s;
                    make_setup(d0, d1, d2, order, f, v, s);
#pragma unroll
                    for (int k = 0; k < 3; k++) {
                        dst[k] = __float_as_uint(v.wstart[k]); dst[3 + k] = __float_as_uint(v.dx[k]);
                        dst[6 + k] = __float_as_uint(v.dy[k]); dst[9 + k] = __float_as_uint(v.rvz[k]);
                    }
                    dst[12] = (uint32_t)v.xmin | ((uint32_t)v.ymin << 16);
                    dst[13] = 0u;
                    const uint32_t *sw = reinterpret_cast<const uint32_t *>(&s);
#pragma unroll
                    for (int k = 0; k < 32; k++) { dst[14 + k] = sw[k]; }
                } else {
                    const uint32_t slot = f.slot_of[(size_t)view * 2u * f.T + order];
                    const VisRecord r = load_vis(f.vis + (size_t)view * f.setup_cap + slot);
                    const Head &h = r.head;
#pragma unroll
                    for (int k = 0; k < 3; k++) {
                        dst[k] = __float_as_uint(r.c.ws[k]); dst[3 + k] = __float_as_uint(r.c.dx[k]);
                        dst[6 + k] = __float_as_uint(r.c.dy[k]); dst[9 + k] = __float_as_uint(r.c.rz[k]);
                    }
                    dst[12] = h.xmin | (h.ymin << 16);
                    dst[13] = is_flat_bbox(f, h.xmin, h.xmax, h.ymin, h.ymax) ? 0u : 1u + slot;   // tile path: tag of its pstate entries
                    const uint4 *sp = reinterpret_cast<const uint4 *>(f.shade + (size_t)view * f.setup_cap + slot);
#pragma unroll
                    for (int k = 0; k < 8; k++) { const uint4 q = sp[k]; dst[14 + 4 * k] = q.x; dst[15 + 4 * k] = q.y; dst[16 + 4 * k] = q.z; dst[17 + 4 * k] = q.w; }
                }
            }
            __syncthreads();
            // ---- 3. shade, one covered pixel per lane ---------------------------------------------
#pragma unroll 1
            for (uint32_t i = tid; i < count; i += SHADE_THREADS) {
                const uint32_t id = sh.tab[sh.pslot[i]] - tb;
                if (id >= SHADE_TRIS) { continue; }
                const uint32_t *src = sh.setup[id];
                const uint32_t p = sh.pix[i], qr = p / SHADE_B, qc = p % SHADE_B;
                const uint32_t px = bx0 + qc, py = pixel_y(f, row0 + br0 + qr);
                float w0, w1, w2;
                if (src[13] == 0u) {
                    const uint32_t xy = src[12];
                    w0 = __uint_as_float(src[0]); w1 = __uint_as_float(src[1]); w2 = __uint_as_float(src[2]);
                    const float dy0 = __uint_as_float(src[6]), dy1 = __uint_as_float(src[7]), dy2 = __uint_as_float(src[8]);
                    const uint32_t ny = py - (xy >> 16), nx = px - (xy & 0xFFFFu);
                    if (ny < SMALL_MAX && nx < SMALL_MAX) {
                        for (uint32_t k = 0; k < ny; k++) { w0 = add_rn(w0, dy0); w1 = add_rn(w1, dy1); w2 = add_rn(w2, dy2); }       // render.cpp:378
                        const float dx0 = __uint_as_float(src[3]), dx1 = __uint_as_float(src[4]), dx2 = __uint_as_float(src[5]);
                        for (uint32_t k = 0; k < nx; k++) { w0 = add_rn(w0, dx0); w1 = add_rn(w1, dx1); w2 = add_rn(w2, dx2); }   // render.cpp:374
                    } else {   // a flat-walked box larger than 16 x 16: same values, by the exact jump where the way is long
                        w0 = weight_at(w0, dy0, ny, __uint_as_float(src[3]), nx);
                        w1 = weight_at(w1, dy1, ny, __uint_as_float(src[4]), nx);
                        w2 = weight_at(w2, dy2, ny, __uint_as_float(src[5]), nx);
                    }
                } else if (const unsigned long long *ps = f.pstate + 3u * (vbase + (size_t)(row0 + br0 + qr) * f.W + px), p0 = ps[0], p1 = ps[1], p2 = ps[2];
                           (uint32_t)(p0 >> 32) + 1u == src[13] && (uint32_t)(p1 >> 32) + 1u == src[13] && (uint32_t)(p2 >> 32) + 1u == src[13]) {
                    w0 = __uint_as_float((uint32_t)p0); w1 = __uint_as_float((uint32_t)p1); w2 = __uint_as_float((uint32_t)p2);   // left by the tile kernel, all three words the winner's
                } else {   // (another CTA's candidate raced the winner's note) exact jump down the rows, then along the row
                    const uint32_t xy = src[12], ny = py - (xy >> 16), nx = px - (xy & 0xFFFFu);
                    w0 = weight_at(__uint_as_float(src[0]), __uint_as_float(src[6]), ny, __uint_as_float(src[3]), nx);
                    w1 = weight_at(__uint_as_float(src[1]), __uint_as_float(src[7]), ny, __uint_as_float(src[4]), nx);
                    w2 = weight_at(__uint_as_float(src[2]), __uint_as_float(src[8]), ny, __uint_as_float(src[5]), nx);
                }
                SetupShade s;
                uint32_t *sw = reinterpret_cast<uint32_t *>(&s);
#pragma unroll
                for (int k = 0; k < 32; k++) { sw[k] = src[14 + k]; }
                sh.colour[qr][qc] = shade_math(f, __uint_as_float(src[9]), __uint_as_float(src[10]), __uint_as_float(src[11]), s, w0, w1, w2);
            }
            __syncthreads();
        }
    }
    // ---- 4. write-out: 4 consecutive pixels per thread --------------------------------------------
    const uint32_t x0 = bx0 + pc;
    if (br0 + pr >= nrows || x0 >= f.W) { return; }
    const uint4 c = *reinterpret_cast<const uint4 *>(&sh.colour[pr][pc]);
    const uint32_t rgb[4] = {c.x, c.y, c.z, c.w};
    const size_t base = vbase + (size_t)(row0 + br0 + pr) * f.W + x0;
    if (f.n_peers) {
        // fused assembly: this row goes to its absolute place in every rank's frame (one 16-byte store per
        // destination; remote ones travel over NVLink while the CTA's other warps are still shading)
        const uint32_t py = pixel_y(f, row0 + br0 + pr);
        if (py < f.H) {
            const size_t at = ((size_t)view * f.H + py) * f.W + x0;
            const bool wide = x0 + 3u < f.W && (at & 3u) == 0;
            for (uint32_t k = 0; k < f.n_peers; k++) {
                uint32_t *o = f.peer_out[k] + at;
                if (wide) { *reinterpret_cast<uint4 *>(o) = make_uint4(rgb[0], rgb[1], rgb[2], rgb[3]); }
                else { for (int q = 0; q < 4 && x0 + q < f.W; q++) { o[q] = rgb[q]; } }
            }
        }
        return;
    }
    if (f.out_packed24) {
        uint8_t *o = reinterpret_cast<uint8_t *>(f.out) + base * 3u;
        if (x0 + 3u < f.W && (reinterpret_cast<uintptr_t>(o) & 3u) == 0) {
            uint32_t *o32 = reinterpret_cast<uint32_t *>(o);
            o32[0] = rgb[0] | (rgb[1] << 24); o32[1] = (rgb[1] >> 8) | (rgb[2] << 16); o32[2] = (rgb[2] >> 16) | (rgb[3] << 8);
        } else {
            for (int k = 0; k < 4 && x0 + k < f.W; k++) { o[3 * k] = rgb[k] & 255u; o[3 * k + 1] = (rgb[k] >> 8) & 255u; o[3 * k + 2] = rgb[k] >> 16; }
        }
    } else {
        uint32_t *o = f.out + base;
        if (x0 + 3u < f.W && (reinterpret_cast<uintptr_t>(o) & 15u) == 0) {
            *reinterpret_cast<uint4 *>(o) = make_uint4(rgb[0], rgb[1], rgb[2], rgb[3]);
        } else {
            for (int k = 0; k < 4 && x0 + k < f.W; k++) { o[k] = rgb[k]; }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------------------
static int g_sm_count = 148;

cudaError_t configure_kernels() {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) { return e; }
    cudaDeviceGetAttribute(&g_sm_count, cudaDevAttrMultiProcessorCount, dev);
    e = cudaFuncSetAttribute(tile_raster, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(RasterShared));
    if (e != cudaSuccess) { return e; }
    e = cudaFuncSetAttribute(tile_raster, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) { return e; }
    e = cudaFuncSetAttribute(tile_raster_queue, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(RasterShared));
    if (e != cudaSuccess) { return e; }
    e = cudaFuncSetAttribute(tile_raster_queue, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) { return e; }
    // both keep ~40 KB of static shared memory per CTA: without the carve-out hint the driver may leave too little for 4-6 CTAs per SM
    e = cudaFuncSetAttribute(cluster_front, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) { return e; }
    e = cudaFuncSetAttribute(direct_walk, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) { return e; }
    e = cudaFuncSetAttribute(shade_tiles<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(ShadeShared));
    if (e != cudaSuccess) { return e; }
    e = cudaFuncSetAttribute(shade_tiles<true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) { return e; }
    e = cudaFuncSetAttribute(shade_tiles<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(ShadeShared));
    if (e != cudaSuccess) { return e; }
    e = cudaFuncSetAttribute(shade_tiles<false>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) { return e; }
    return cudaFuncSetAttribute(triangle_classify, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
}

static inline uint32_t ceil_div(uint32_t a, uint32_t b) { return (a + b - 1) / b; }

static inline void mark(const LaunchMarks *m, const char *kernel) { if (m) { m->fn(m->ctx, kernel); } }

// Launch with programmatic stream serialization (see wait_for_predecessor): `after_kernel` = the previous operation in the
// stream is one of this path's kernels.
template <typename... KArgs, typename... Args>
static void launch_chain(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, bool after_kernel, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    // (not on the legacy / per-thread default streams: their implicit synchronisation and the programmatic edge do not mix)
    const bool real_stream = s != nullptr && s != cudaStreamLegacy && s != cudaStreamPerThread;
    cfg.attrs = attr; cfg.numAttrs = (after_kernel && real_stream) ? 1u : 0u;
    cudaLaunchKernelEx(&cfg, kernel, args...);
}

int launch_geometry(const Frame &f, cudaStream_t s, const LaunchMarks *m) {
    int launches = 0;
    const uint32_t persistent = (uint32_t)g_sm_count * 4u;
    if (f.cl_hdr) {
        // spatial pre-partition: vertex stage + front + direct walk in one kernel over the clusters; the frame's counters
        // and tile histograms (zeroed by vertex_stage on the other path) are cleared by one small memset
        cudaMemsetAsync(f.counters, 0, ((size_t)(f.tile_count - f.counters) + (size_t)f.n_views * f.tile_stride) * sizeof(uint32_t), s);   // (the histograms follow the counters)
        const bool chain = true;
        launch_chain(cluster_cull, dim3(max(1u, ceil_div(f.n_clusters, CULL_ROUNDS * 256u)), f.n_views), dim3(256), 0, s, false, f); launches++; mark(m, "cluster_cull");
        launch_chain(cluster_front, dim3((uint32_t)g_sm_count * (uint32_t)FRONT_CTAS, f.n_views), dim3(256), 0, s, chain, f); launches++; mark(m, "cluster_front");
        launch_chain(direct_walk, dim3((uint32_t)g_sm_count * 6u, f.n_views), dim3(256), 0, s, chain, f); launches++; mark(m, "direct_walk");
    } else {
        vertex_stage<<<dim3(max(1u, ceil_div(f.Vpad / 4, 256)), f.n_views), 256, 0, s>>>(f); launches++; mark(m, "vertex_stage");
        triangle_classify<<<dim3(max(1u, ceil_div(f.T, CLS_PER_CTA)), f.n_views), 256, 0, s>>>(f); launches++; mark(m, "triangle_classify");
    }
    const dim3 setup_grid(min((uint32_t)g_sm_count * 2u, max(1u, ceil_div(f.T, 256))), f.n_views);
    const bool chain2 = true;
    if (f.rv) { launch_chain(triangle_setup<true>, setup_grid, dim3(256), 0, s, chain2, f); } else { launch_chain(triangle_setup<false>, setup_grid, dim3(256), 0, s, chain2, f); }
    launches++; mark(m, "triangle_setup");
    // cooperative binning of the big triangles, flat visibility pass over the recorded small ones (clipped or spawned),
    // and — by the last CTA to finish — the frame's tile statistics and overflow record
    launch_chain(post_setup, dim3(persistent, f.n_views), dim3(256), 0, s, chain2, f); launches++; mark(m, "post_setup");
    return launches;
}

int launch_raster(const Frame &f, cudaStream_t s, const LaunchMarks *m) {
    if (f.direct_bin) {
        tile_raster<<<dim3(f.tiles_x, f.raster_rows, f.n_views), RASTER_THREADS, sizeof(RasterShared), s>>>(f); mark(m, "tile_raster");
        return 1;
    }
    // general path: the queue holds every non-empty tile of the submission, so the tile kernel runs once per frame, with
    // the first band; the bands only cut the shading pass (the host path copies band k while band k + 1 is shaded)
    int launches = 0;
    if (f.raster_row0 == 0u) {
        launch_chain(tile_raster_queue, dim3((uint32_t)g_sm_count * (uint32_t)QUEUE_CTAS, f.n_views), dim3(RASTER_THREADS), sizeof(RasterShared), s, true, f); mark(m, "tile_raster_queue");
        launches++;
    }
    uint32_t row0, nrows;
    if (f.row_stride == 1u) {
        const uint32_t ya = (f.tile_row0 + f.raster_row0) * TILE_H, yb = ya + f.raster_rows * TILE_H;
        const uint32_t lo = max(ya, f.y0), hi = min(yb, f.y1);
        row0 = lo - f.y0; nrows = hi > lo ? hi - lo : 0u;
    } else {
        row0 = f.raster_row0 * TILE_H; nrows = f.raster_rows * TILE_H;
    }
    if (nrows) {
        const dim3 grid(ceil_div(f.W, SHADE_B), ceil_div(nrows, SHADE_BH), f.n_views);
        if (f.rv) { launch_chain(shade_tiles<true>, grid, dim3(SHADE_THREADS), sizeof(ShadeShared), s, true, f, row0, nrows); }
        else { launch_chain(shade_tiles<false>, grid, dim3(SHADE_THREADS), sizeof(ShadeShared), s, true, f, row0, nrows); }
        mark(m, "shade_tiles");
        launches++;
    }
    return launches;
}

int launch_geometry_small(const Frame &f, cudaStream_t s, const LaunchMarks *m) {
    geometry_small<<<f.n_views, 256, 0, s>>>(f); mark(m, "geometry_small");
    if (!f.coltab) { return 1; }
    span_walk<<<dim3(ceil_div(f.H, 128u), SPAN_MAX * 3u, f.n_views), 128, 0, s>>>(f); mark(m, "span_walk");
    return 2;
}

// the vertex stage alone (raster-vertex dumps when the frame itself went through the cluster front)
void launch_vertex_stage(const Frame &f, cudaStream_t s) {
    vertex_stage<<<dim3(max(1u, ceil_div(f.Vpad / 4, 256)), f.n_views), 256, 0, s>>>(f);
}

// test hook: the device build of walk_jump on arrays (tests compare it with sequential adds)
__global__ void walk_jump_kernel(const float *s, const float *d, const uint32_t *n, float *out, uint32_t count) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) { out[i] = walk_jump(s[i], d[i], n[i]); }
}

// test hook: exact_math.cuh against the compiler's IEEE operators.  mode 0: inv_sqrt_rn over every binary32 bit pattern
// in [lo_bits, hi_bits]; mode 1: div3_rn over `count` pseudo-random operand sets (seeded), a quarter of them
// with extreme mantissas.  result[0] = mismatches, result[1..4] = the first mismatch's operands / values (bit patterns).
__device__ __forceinline__ uint32_t mix32(uint32_t x) { x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16; return x; }
__global__ void exact_math_kernel(uint32_t mode, unsigned long long lo, unsigned long long count, uint32_t seed,
                                  unsigned long long *result) {
    for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < count;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        if (mode == 0) {
            const float x = __uint_as_float((uint32_t)(lo + i));
            const uint32_t got = __float_as_uint(inv_sqrt_rn(x)), want = __float_as_uint(__frcp_rn(__fsqrt_rn(x)));
            if (got != want && !(got > 0x7f800000u && want > 0x7f800000u)) {
                if (atomicAdd(result, 1ull) == 0ull) { result[1] = __float_as_uint(x); result[2] = got; result[3] = want; }
            }
        } else if (mode == 2) {
            // div2_rn_signed: operands of either sign, zeros, extreme mantissas, exponents beyond the guarded range
            uint32_t h = mix32((uint32_t)i ^ seed), g = mix32((uint32_t)(i >> 32) + h + 0x9e3779b9u);
            uint32_t op[3];
#pragma unroll
            for (int k = 0; k < 3; k++) {
                g = mix32(g + 0x85ebca6bu * (k + 1)); h = mix32(h ^ g);
                uint32_t mant = g & 0x7FFFFFu;
                const uint32_t sel = (h >> 8) & 15u;
                if (sel == 0) { mant = 0x7FFFFFu; } else if (sel == 1) { mant = 0u; } else if (sel == 2) { mant = 0x7FFFFEu; } else if (sel == 3) { mant = 1u; }
                const uint32_t e = 127u - 62u + (h >> 24) % 124u;
                op[k] = (e << 23) | mant | ((h & 1u) << 31);
            }
            if (((h >> 3) & 63u) == 0u) { op[(h >> 12) % 3u] &= 0x80000000u; }     // signed zeros take the fallback
            const float a0 = __uint_as_float(op[0]), a1 = __uint_as_float(op[1]), b = __uint_as_float(op[2]);
            float q0, q1;
            div2_rn_signed(a0, a1, b, q0, q1);
            const float w0 = a0 / b, w1 = a1 / b;
            const bool ok = (__float_as_uint(q0) == __float_as_uint(w0) || (q0 != q0 && w0 != w0)) && (__float_as_uint(q1) == __float_as_uint(w1) || (q1 != q1 && w1 != w1));
            if (!ok) {
                if (atomicAdd(result, 1ull) == 0ull) { result[1] = op[0]; result[2] = op[2]; result[3] = __float_as_uint(q0); result[4] = __float_as_uint(w0); }
            }
        } else {
            uint32_t h = mix32((uint32_t)i ^ seed) , g = mix32((uint32_t)(i >> 32) + h + 0x9e3779b9u);
            uint32_t op[4];
#pragma unroll
            for (int k = 0; k < 4; k++) {
                g = mix32(g + 0x85ebca6bu * (k + 1)); h = mix32(h ^ g);
                uint32_t mant = g & 0x7FFFFFu;
                const uint32_t sel = (h >> 8) & 15u;
                if (sel == 0) { mant = 0x7FFFFFu; } else if (sel == 1) { mant = 0u; } else if (sel == 2) { mant = 0x7FFFFEu; } else if (sel == 3) { mant = 1u; }
                const uint32_t e = 127u - 62u + (h >> 24) % 124u;   // a little beyond the guarded range on both sides
                op[k] = (e << 23) | mant;
            }
            if (((h >> 3) & 63u) == 0u) { op[(h >> 12) & 3u] = 0u; }     // zeros take the fallback
            const float a0 = __uint_as_float(op[0]), a1 = __uint_as_float(op[1]), a2 = __uint_as_float(op[2]), b = __uint_as_float(op[3]);
            float q0, q1, q2;
            div3_rn(a0, a1, a2, b, q0, q1, q2);
            const float w0 = a0 / b, w1 = a1 / b, w2 = a2 / b;
            const bool ok = __float_as_uint(q0) == __float_as_uint(w0) && __float_as_uint(q1) == __float_as_uint(w1) &&
                            __float_as_uint(q2) == __float_as_uint(w2);
            if (!ok && !(b == 0.f)) {
                if (atomicAdd(result, 1ull) == 0ull) { result[1] = op[0]; result[2] = op[3]; result[3] = __float_as_uint(q0); result[4] = __float_as_uint(w0); }
            }
        }
    }
}

void launch_exact_math(uint32_t mode, unsigned long long lo, unsigned long long count, uint32_t seed, unsigned long long *result,
                       cudaStream_t st) {
    exact_math_kernel<<<(uint32_t)g_sm_count * 8u, 256, 0, st>>>(mode, lo, count, seed, result);
}

void launch_walk_jump(const float *s, const float *d, const uint32_t *n, float *out, uint32_t count, cudaStream_t st) {
    walk_jump_kernel<<<(count + 255) / 256, 256, 0, st>>>(s, d, n, out, count);
}

}  // namespace s3r
