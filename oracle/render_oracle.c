/*
 * oracle/render_oracle.c — TEST INFRASTRUCTURE (CPU parity checker); see render_oracle.h.
 *
 * Plain-C restatement of the reference's frame algorithm.  Each function cites the
 * reference lines it follows (paths relative to /root/reference).  Scalar binary32 arithmetic,
 * written out component by component in the evaluation order the reference source has under
 * the simd semantics of oracle/shim/simd/simd.h; build with -ffp-contract=off.
 */
#define _POSIX_C_SOURCE 200112L
#include "render_oracle.h"

#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

/* render-cpp/render.cpp:81-97.  scale = near * tanf(fov / 2) as evaluated at load time by the
 * reference build (value read back from oracle/_ref/render_ref.so's config static). */
static const float kNear = 0.1f;
static const float kScale = 0x1.0a2c9ap-5f;
static const float kSpeed = 0.1f;
static const float kRotationSpeed = 0.3f;
static const uint32_t kBackground = 0x001E1E1Eu;

typedef struct { float x, y, z; } v3;

static v3 v3_make(float x, float y, float z) { v3 r = {x, y, z}; return r; }
static v3 v3_add(v3 a, v3 b) { return v3_make(a.x + b.x, a.y + b.y, a.z + b.z); }
static v3 v3_scale(v3 a, float s) { return v3_make(a.x * s, a.y * s, a.z * s); }
static float v3_dot(v3 a, v3 b) { return (a.x * b.x + a.y * b.y) + a.z * b.z; }
static v3 v3_cross(v3 a, v3 b) {
    return v3_make(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}
static v3 v3_unit(v3 a) { return v3_scale(a, 1.0f / sqrtf(v3_dot(a, a))); }
static v3 v3_load(const float *p) { return v3_make(p[0], p[1], p[2]); }
static void v3_store(float *p, v3 a) { p[0] = a.x; p[1] = a.y; p[2] = a.z; }

/* ---------------------------------------------------------------------------------------------
 * Scene loading — render-cpp/render.cpp:177-209 (section headers [count, ignored]; odd index
 * counts are followed by 8 bytes of padding).
 * ------------------------------------------------------------------------------------------- */
int oracle_scene_load(OracleScene *scene, const char *path) {
    memset(scene, 0, sizeof(*scene));
    FILE *fp = fopen(path, "rb");
    if (!fp) { return -1; }
    fseek(fp, 0, SEEK_END);
    long size = ftell(fp);
    fseek(fp, 0, SEEK_SET);
    /* 16-byte aligned so float4 / u64 views are aligned */
    uint8_t *raw = NULL;
    if (posix_memalign((void **)&raw, 64, (size_t)size + 64) != 0) { fclose(fp); return -2; }
    if (fread(raw, 1, (size_t)size, fp) != (size_t)size) { fclose(fp); free(raw); return -3; }
    fclose(fp);
    size_t off = 0;
    uint64_t n;
    memcpy(&n, raw + off, 8); off += 16;
    scene->vertex_count = n;
    scene->vertices = (const float *)(raw + off); off += n * 16;
    memcpy(&n, raw + off, 8); off += 16;
    scene->index_count = n;
    scene->vertex_indices = (const uint64_t *)(raw + off); off += (n + (n & 1)) * 8;
    memcpy(&n, raw + off, 8); off += 16;
    scene->attribute_count = n;
    scene->attributes = raw + off; off += n * 48;
    memcpy(&n, raw + off, 8); off += 16;
    scene->attribute_indices = (const uint64_t *)(raw + off); off += (n + (n & 1)) * 8;
    memcpy(&n, raw + off, 8); off += 16;
    scene->texel_count = n;
    scene->texels = (const uint32_t *)(raw + off); off += n * 4;
    scene->owned = raw;
    return off <= (size_t)size ? 0 : -4;
}

void oracle_scene_free(OracleScene *scene) {
    free(scene->owned);
    memset(scene, 0, sizeof(*scene));
}

/* ---------------------------------------------------------------------------------------------
 * Camera — render-cpp/render.cpp:51-65 (initial state), :134-156 (update_camera)
 * ------------------------------------------------------------------------------------------- */
void oracle_camera_reset(OracleCamera *cam) {
    memset(cam, 0, sizeof(*cam));
    cam->axis_x[0] = 1.f; cam->axis_y[1] = 1.f; cam->axis_z[2] = 1.f;
    cam->matrix[0] = 1.f; cam->matrix[5] = 1.f; cam->matrix[10] = 1.f;
}

/* simd_act: v + q.w * t + cross(q.xyz, t), t = 2 * cross(q.xyz, v) */
static v3 quat_act(v3 qv, float qw, v3 v) {
    v3 t = v3_scale(v3_cross(qv, v), 2.f); /* 2.f * c == c * 2.f in binary32 */
    return v3_add(v3_add(v, v3_scale(t, qw)), v3_cross(qv, t));
}

void oracle_camera_update(OracleCamera *cam, const OracleInput *in) {
    int changed = 0;
    v3 pos = v3_load(cam->position), ax = v3_load(cam->axis_x), ay = v3_load(cam->axis_y), az = v3_load(cam->axis_z);
    if (in->left > 0 || in->right > 0 || in->up > 0 || in->down > 0) { /* :136-139 */
        changed = 1;
        float sx = in->right - in->left, sz = in->down - in->up;
        v3 step = v3_add(v3_scale(ax, sx), v3_scale(az, sz));
        pos = v3_add(pos, v3_scale(step, kSpeed));
    }
    if (in->mouse_x != cam->mouse[0] || in->mouse_y != cam->mouse[1]) { /* :140-150 */
        changed = 1;
        float mx = cam->mouse[0] - in->mouse_x, my = cam->mouse[1] - in->mouse_y, mz = 100 / kRotationSpeed;
        v3 z = v3_unit(v3_add(v3_add(v3_scale(ax, mx), v3_scale(ay, my)), v3_scale(az, mz)));
        v3 qv;
        float qw;
        if (v3_dot(az, z) >= 0.f) { /* simd_quaternion(from, to), acute branch */
            v3 half = v3_unit(v3_add(az, z));
            qv = v3_cross(az, half);
            qw = v3_dot(az, half);
        } else { /* obtuse: two half rotations (unreachable at 0.3 deg/pt, kept for completeness) */
            v3 half = v3_unit(v3_add(az, z));
            if (!(v3_dot(half, half) > 0.f)) {
                v3 pick = fabsf(az.x) < fabsf(az.y) ? v3_make(1, 0, 0) : v3_make(0, 1, 0);
                half = v3_unit(v3_cross(az, pick));
            }
            v3 pv = v3_cross(half, z), sv = v3_cross(az, half);
            float pw = v3_dot(half, z), sw = v3_dot(az, half);
            qv = v3_add(v3_add(v3_scale(sv, pw), v3_scale(pv, sw)), v3_cross(pv, sv));
            qw = pw * sw - v3_dot(pv, sv);
        }
        ax = v3_unit(quat_act(qv, qw, ax));
        ay = v3_unit(quat_act(qv, qw, ay));
        az = z;
        cam->mouse[0] = in->mouse_x;
        cam->mouse[1] = in->mouse_y;
    }
    if (changed || !cam->started) { /* :151-155; first frame forces the rebuild (:270) */
        v3_store(cam->matrix + 0, ax); cam->matrix[3] = -v3_dot(ax, pos);
        v3_store(cam->matrix + 4, ay); cam->matrix[7] = -v3_dot(ay, pos);
        v3_store(cam->matrix + 8, az); cam->matrix[11] = -v3_dot(az, pos);
    }
    cam->started = 1;
    v3_store(cam->position, pos); v3_store(cam->axis_x, ax); v3_store(cam->axis_y, ay); v3_store(cam->axis_z, az);
}

float oracle_factor(uint32_t height) { return kNear * (float)height / (2 * kScale); } /* :279 */

/* simd_mul(float4x3, float4) = ((c0*x + c1*y) + c2*z) + c3*w, columns c_k = (r0[k], r1[k], r2[k]) */
static v3 transform(const float *m, float x, float y, float z, float w) {
    return v3_make(((m[0] * x + m[1] * y) + m[2] * z) + m[3] * w,
                   ((m[4] * x + m[5] * y) + m[6] * z) + m[7] * w,
                   ((m[8] * x + m[9] * y) + m[10] * z) + m[11] * w);
}

/* render.cpp:288 — (v.x, -v.y, 0) * factor / -v.z + (W/2, H/2, -v.z) */
static v3 project(v3 cv, float factor, float half_w, float half_h) {
    float nz = -cv.z;
    return v3_make(cv.x * factor / nz + half_w, -cv.y * factor / nz + half_h, 0.f * factor / nz + nz);
}

void oracle_vertex_stage(const OracleScene *s, const float *m, uint32_t width, uint32_t height,
                         float *cvs, float *rvs) {
    float factor = oracle_factor(height), hw = (float)width / 2, hh = (float)height / 2;
    for (uint64_t i = 0; i < s->vertex_count; i++) {
        const float *p = s->vertices + 4 * i;
        v3 cv = transform(m, p[0], p[1], p[2], p[3]);
        v3_store(cvs + 3 * i, cv);
        v3_store(rvs + 3 * i, project(cv, factor, hw, hh));
    }
}

float oracle_walk(float start, float delta, uint32_t n) {
    volatile float w = start; /* volatile: keep every intermediate in binary32 */
    for (uint32_t i = 0; i < n; i++) { w = w + delta; }
    return w;
}

/* ---------------------------------------------------------------------------------------------
 * Per-corner working record — render-cpp/render.cpp:26-31 (data_t), :11-24 (colour attribute).
 * The 16-byte payload is kept as raw words: colour = floats 0..2, texture = {index, -, u, v}.
 * ------------------------------------------------------------------------------------------- */
typedef struct {
    v3 cv, rv, n;
    uint32_t payload[4];
    uint32_t kind;
} corner_t;

static float word_f(uint32_t w) { float f; memcpy(&f, &w, 4); return f; }
static uint32_t f_word(float f) { uint32_t w; memcpy(&w, &f, 4); return w; }

typedef struct {
    v3 *cv, *rv, *n;      /* scratch: 2V, 2V, 2A */
    uint32_t *payload;    /* 2A x 4 */
    uint32_t *kind;       /* 2A */
    uint64_t *vi, *ai;    /* 2 * aligned I */
    uint64_t v_cap, a_cap, i_cap;
    uint32_t *spawn_parent; /* parent triangle of the k-th appended triangle */
    uint64_t spawn_n;
} scratch_t;

static corner_t gather(const scratch_t *sc, uint64_t vi, uint64_t ai) {
    corner_t c;
    c.cv = sc->cv[vi]; c.rv = sc->rv[vi]; c.n = sc->n[ai];
    memcpy(c.payload, sc->payload + 4 * ai, 16);
    c.kind = sc->kind[ai];
    return c;
}

static v3 lerp3(v3 a, v3 b, float one_minus_t, float t) { /* x*(1-a) + y*a */
    return v3_add(v3_scale(a, one_minus_t), v3_scale(b, t));
}

/* render-cpp/render.cpp:212-262.  Returns 1 when a triangle was appended. */
static int clip_near(corner_t *d, scratch_t *sc, uint64_t *v_count, uint64_t *a_count, uint64_t *i_count,
                     const uint64_t *vi, const uint64_t *ai, float factor, float half_w, float half_h,
                     uint32_t parent, int *overflow) {
    corner_t made[3];
    memset(made, 0, sizeof(made));
    uint32_t cur = 0, nxt = 0, pre = 0;
    int two_in_front = 0;
    for (uint32_t i = 0; i < 3; i++) {
        uint32_t j = (i + 1) % 3;
        int fi = d[i].rv.z > kNear, fj = d[j].rv.z > kNear;
        if (fi == fj) {
            cur = i; nxt = j; pre = (i + 2) % 3;
            two_in_front = fi;
        } else {
            float t = (kNear - d[i].rv.z) / (d[j].rv.z - d[i].rv.z);
            float u = 1 - t;
            corner_t c;
            memset(&c, 0, sizeof(c));
            c.cv = lerp3(d[i].cv, d[j].cv, u, t);
            c.rv = v3_make(c.cv.x * factor / kNear + half_w, -c.cv.y * factor / kNear + half_h,
                           0.f * factor / kNear + kNear);
            c.kind = d[0].kind; /* :225 — the kind always comes from corner 0 */
            if (c.kind == 0) {
                v3 a = v3_make(word_f(d[i].payload[0]), word_f(d[i].payload[1]), word_f(d[i].payload[2]));
                v3 b = v3_make(word_f(d[j].payload[0]), word_f(d[j].payload[1]), word_f(d[j].payload[2]));
                v3 col = lerp3(a, b, u, t);
                c.payload[0] = f_word(col.x); c.payload[1] = f_word(col.y); c.payload[2] = f_word(col.z);
            } else if (c.kind == 1) {
                c.payload[0] = d[i].payload[0]; /* texture index of the edge's first endpoint, :233 */
                c.payload[2] = f_word(word_f(d[i].payload[2]) * u + word_f(d[j].payload[2]) * t);
                c.payload[3] = f_word(word_f(d[i].payload[3]) * u + word_f(d[j].payload[3]) * t);
            }
            c.n = lerp3(d[i].n, d[j].n, u, t);
            made[i] = c;
        }
    }
    if (!two_in_front) { /* one corner in front: shrink in place, :258-261 */
        d[cur] = made[pre];
        d[nxt] = made[nxt];
        return 0;
    }
    /* two in front: in place (cur, nxt, made[nxt]); append (cur, made[nxt], made[pre]), :239-257 */
    d[pre] = made[nxt];
    if (*v_count + 2 > sc->v_cap || *a_count + 2 > sc->a_cap || *i_count + 3 > sc->i_cap) {
        *overflow = 1; /* the reference writes out of bounds here (H13); we drop the spawn instead */
        return 0;
    }
    const corner_t *add[2] = {&made[nxt], &made[pre]};
    for (int k = 0; k < 2; k++) {
        sc->cv[*v_count + k] = add[k]->cv;
        sc->rv[*v_count + k] = add[k]->rv;
        sc->n[*a_count + k] = add[k]->n;
        memcpy(sc->payload + 4 * (*a_count + k), add[k]->payload, 16);
        sc->kind[*a_count + k] = add[k]->kind;
    }
    sc->vi[*i_count] = vi[cur]; sc->vi[*i_count + 1] = *v_count; sc->vi[*i_count + 2] = *v_count + 1;
    sc->ai[*i_count] = ai[cur]; sc->ai[*i_count + 1] = *a_count; sc->ai[*i_count + 2] = *a_count + 1;
    sc->spawn_parent[sc->spawn_n++] = parent;
    *v_count += 2; *a_count += 2; *i_count += 3;
    return 1;
}

static float edge(v3 a, v3 b, float cx, float cy) { /* EDGE_FUNCTION, render.cpp:9 */
    return (cx - a.x) * (a.y - b.y) + (cy - a.y) * (b.x - a.x);
}

static uint32_t next_pow2(uint32_t i) { /* render.cpp:115-122 */
    i--; i |= i >> 1; i |= i >> 2; i |= i >> 4;
    return i + 1;
}

/* render.cpp:124-131 */
static v3 sample_ripmap(const uint32_t *atlas, float u, float v, float level_x, float level_y) {
    uint32_t lx = next_pow2((uint32_t)fmaxf(fminf(level_x, 256.f), 1.f));
    uint32_t ly = next_pow2((uint32_t)fmaxf(fminf(level_y, 256.f), 1.f));
    uint32_t x = (uint32_t)(fmodf(u, 1) * (float)lx) + (511 & ~(2 * lx - 1));
    uint32_t y = (uint32_t)(fmodf(v, 1) * (float)ly) + (511 & ~(2 * ly - 1));
    uint32_t rgb = atlas[x + (y << 9)];
    return v3_make((float)(rgb >> 16), (float)((rgb >> 8) & 255), (float)(rgb & 255));
}

static uint32_t pack_rgb(v3 c) { /* RGB(), render.cpp:8: each channel through (uint8_t) */
    uint32_t r = (uint32_t)(int32_t)c.x & 255u, g = (uint32_t)(int32_t)c.y & 255u, b = (uint32_t)(int32_t)c.z & 255u;
    return (((r << 8) + g) << 8) + b;
}

int oracle_render(const OracleScene *s, const float *m, uint32_t width, uint32_t height, uint32_t *pixels,
                  float *depth_out, OracleStats *stats, OracleSetup *setups, size_t setup_cap, size_t *setup_count,
                  uint32_t *winner) {
    OracleStats st;
    memset(&st, 0, sizeof(st));
    size_t n_setups = 0;
    const uint64_t V = s->vertex_count, A = s->attribute_count, I = s->index_count;
    const uint64_t I_al = I + (I & 1);
    const size_t npix = (size_t)width * height;
    float *depth = depth_out ? depth_out : (float *)malloc(npix * sizeof(float));
    scratch_t sc;
    sc.v_cap = 2 * V; sc.a_cap = 2 * A; sc.i_cap = 2 * I_al;
    sc.cv = (v3 *)malloc((sc.v_cap + 1) * sizeof(v3));
    sc.rv = (v3 *)malloc((sc.v_cap + 1) * sizeof(v3));
    sc.n = (v3 *)malloc((sc.a_cap + 1) * sizeof(v3));
    sc.payload = (uint32_t *)malloc((sc.a_cap + 1) * 16);
    sc.kind = (uint32_t *)malloc((sc.a_cap + 1) * 4);
    sc.vi = (uint64_t *)malloc((sc.i_cap + 1) * 8);
    sc.ai = (uint64_t *)malloc((sc.i_cap + 1) * 8);
    sc.spawn_parent = (uint32_t *)malloc((sc.i_cap / 3 + 2) * 4);
    sc.spawn_n = 0;
    memcpy(sc.vi, s->vertex_indices, I * 8);
    memcpy(sc.ai, s->attribute_indices, I * 8);

    const float factor = oracle_factor(height);
    const float fw = (float)width, fh = (float)height, half_w = fw / 2, half_h = fh / 2;

    /* clears, render.cpp:281-282 */
    for (size_t i = 0; i < npix; i++) { depth[i] = 0.f; pixels[i] = kBackground; }
    if (winner) { for (size_t i = 0; i < npix; i++) { winner[i] = 0xFFFFFFFFu; } }

    /* vertex + normal loops, render.cpp:285-292 */
    for (uint64_t i = 0; i < V; i++) {
        const float *p = s->vertices + 4 * i;
        sc.cv[i] = transform(m, p[0], p[1], p[2], p[3]);
        sc.rv[i] = project(sc.cv[i], factor, half_w, half_h);
    }
    for (uint64_t i = 0; i < A; i++) {
        const uint8_t *rec = s->attributes + 48 * i;
        float nrm[4];
        memcpy(nrm, rec, 16);
        sc.n[i] = transform(m, nrm[0], nrm[1], nrm[2], nrm[3]);
        memcpy(sc.payload + 4 * i, rec + 16, 16);
        memcpy(sc.kind + i, rec + 32, 4);
    }

    uint64_t i_count = I, v_count = V, a_count = A;
    for (uint32_t index = 0; index < i_count; index += 3) { /* render.cpp:297 */
        st.triangles_in++;
        const uint64_t vi[3] = {sc.vi[index], sc.vi[index + 1], sc.vi[index + 2]};
        const uint64_t ai[3] = {sc.ai[index], sc.ai[index + 1], sc.ai[index + 2]};
        corner_t d[3] = {gather(&sc, vi[0], ai[0]), gather(&sc, vi[1], ai[1]), gather(&sc, vi[2], ai[2])};

        if (fmaxf(fmaxf(d[0].rv.z, d[1].rv.z), d[2].rv.z) <= kNear) { st.near_rejected++; continue; }
        if (fminf(fminf(d[0].rv.z, d[1].rv.z), d[2].rv.z) < kNear) {
            st.clipped++;
            st.spawned += (uint64_t)clip_near(d, &sc, &v_count, &a_count, &i_count, vi, ai, factor, half_w, half_h,
                                              index / 3, &st.scratch_overflow);
        }
        const float max_x = fmaxf(fmaxf(d[0].rv.x, d[1].rv.x), d[2].rv.x);
        const float max_y = fmaxf(fmaxf(d[0].rv.y, d[1].rv.y), d[2].rv.y);
        if (max_x < 0 || max_y < 0) { st.offscreen++; continue; }
        const float min_x = fminf(fminf(d[0].rv.x, d[1].rv.x), d[2].rv.x);
        const float min_y = fminf(fminf(d[0].rv.y, d[1].rv.y), d[2].rv.y);
        if (min_x >= fw || min_y >= fh) { st.offscreen++; continue; }

        const float area = edge(d[0].rv, d[1].rv, d[2].rv.x, d[2].rv.y);
        if (area < 10) { st.small_or_backfacing++; continue; }
        st.rasterized++;
        const float inv_area = 1 / area;
        const uint32_t xmin = (uint32_t)fmaxf(0, min_x), xmax = (uint32_t)fminf(fw - 1, max_x);
        const uint32_t ymin = (uint32_t)fmaxf(0, min_y), ymax = (uint32_t)fminf(fh - 1, max_y);
        const float px = (float)xmin + 0.5f, py = (float)ymin + 0.5f;
        const float ws[3] = {edge(d[1].rv, d[2].rv, px, py) * inv_area, edge(d[2].rv, d[0].rv, px, py) * inv_area,
                             edge(d[0].rv, d[1].rv, px, py) * inv_area};
        const float dx[3] = {(d[1].rv.y - d[2].rv.y) * inv_area, (d[2].rv.y - d[0].rv.y) * inv_area,
                             (d[0].rv.y - d[1].rv.y) * inv_area};
        const float dy[3] = {(d[2].rv.x - d[1].rv.x) * inv_area, (d[0].rv.x - d[2].rv.x) * inv_area,
                             (d[1].rv.x - d[0].rv.x) * inv_area};
        const float rvz[3] = {1 / d[0].rv.z, 1 / d[1].rv.z, 1 / d[2].rv.z};
        v3 cvz[3], nz[3], pay[3];
        for (int k = 0; k < 3; k++) {
            cvz[k] = v3_scale(d[k].cv, rvz[k]);
            nz[k] = v3_scale(d[k].n, rvz[k]);
        }
        const uint32_t kind = d[0].kind; /* :340 */
        uint32_t tex_index = 0;
        float dz[2] = {0, 0}, tpp[2] = {0, 0};
        const uint32_t *atlas = NULL;
        if (kind == 0) {
            for (int k = 0; k < 3; k++) {
                pay[k] = v3_scale(v3_make(word_f(d[k].payload[0]), word_f(d[k].payload[1]), word_f(d[k].payload[2])), rvz[k]);
            }
        } else {
            tex_index = d[0].payload[0];
            atlas = s->texels + ((size_t)(int32_t)tex_index << 18); /* :347 */
            for (int k = 0; k < 3; k++) {
                pay[k] = v3_make(word_f(d[k].payload[2]) * rvz[k], word_f(d[k].payload[3]) * rvz[k], 0.f);
            }
            dz[0] = (rvz[0] * dx[0] + rvz[1] * dx[1]) + rvz[2] * dx[2]; /* simd_dot(rvz, dx), :349 */
            dz[1] = (rvz[0] * dy[0] + rvz[1] * dy[1]) + rvz[2] * dy[2];
            tpp[0] = (pay[0].x * dx[0] + pay[1].x * dx[1]) + pay[2].x * dx[2]; /* :350-352 */
            tpp[1] = (pay[0].y * dy[0] + pay[1].y * dy[1]) + pay[2].y * dy[2];
        }
        /* in place: own index; appended: T + parent index (appended triangles run in parent order) */
        const uint32_t tri = index / 3, t_in = (uint32_t)(I / 3);
        const uint32_t order = tri < t_in ? tri : t_in + sc.spawn_parent[tri - t_in];
        if (setups && n_setups < setup_cap) {
            OracleSetup *o = &setups[n_setups];
            memset(o, 0, sizeof(*o));
            o->order = order;
            o->xmin = xmin; o->xmax = xmax; o->ymin = ymin; o->ymax = ymax; o->area = area;
            for (int k = 0; k < 3; k++) {
                o->wstart[k] = ws[k]; o->dx[k] = dx[k]; o->dy[k] = dy[k]; o->rvz[k] = rvz[k];
                v3_store(o->cv[k], cvz[k]); v3_store(o->n[k], nz[k]); v3_store(o->payload[k], pay[k]);
            }
            o->kind = kind; o->texture = tex_index;
            o->dz[0] = dz[0]; o->dz[1] = dz[1]; o->tpp[0] = tpp[0]; o->tpp[1] = tpp[1];
        }
        n_setups++;

        /* pixel loops, render.cpp:360-382: incremental barycentric walk */
        float w[3] = {ws[0], ws[1], ws[2]}, wy[3] = {ws[0], ws[1], ws[2]};
        for (uint32_t y = ymin; y <= ymax; y++) {
            uint32_t *prow = pixels + (size_t)y * width;
            uint32_t *wrow = winner ? winner + (size_t)y * width : NULL;
            float *drow = depth + (size_t)y * width;
            for (uint32_t x = xmin; x <= xmax; x++) {
                st.bbox_pixels++;
                if (w[0] >= 0 && w[1] >= 0 && w[2] >= 0) {
                    st.covered_pixels++;
                    const float ooz = (rvz[0] * w[0] + rvz[1] * w[1]) + rvz[2] * w[2];
                    if (ooz > drow[x]) {
                        st.shaded_pixels++;
                        drow[x] = ooz;
                        if (wrow) { wrow[x] = order; }
                        const float b0 = w[0] / ooz, b1 = w[1] / ooz, b2 = w[2] / ooz;
                        v3 p = v3_add(v3_add(v3_scale(cvz[0], b0), v3_scale(cvz[1], b1)), v3_scale(cvz[2], b2));
                        v3 pu = v3_unit(p);
                        v3 point = v3_make(-pu.x, -pu.y, -pu.z);
                        v3 normal = v3_unit(v3_add(v3_add(v3_scale(nz[0], b0), v3_scale(nz[1], b1)), v3_scale(nz[2], b2)));
                        v3 halfway = v3_unit(v3_add(point, normal));
                        const float shade = v3_dot(halfway, normal);
                        v3 base;
                        if (kind == 0) {
                            base = v3_add(v3_add(v3_scale(pay[0], b0), v3_scale(pay[1], b1)), v3_scale(pay[2], b2));
                        } else {
                            const float u = (pay[0].x * b0 + pay[1].x * b1) + pay[2].x * b2;
                            const float v = (pay[0].y * b0 + pay[1].y * b1) + pay[2].y * b2;
                            const float lx = ooz / fabsf(tpp[0] - u * dz[0]);
                            const float ly = ooz / fabsf(tpp[1] - v * dz[1]);
                            base = sample_ripmap(atlas, u, v, lx, ly);
                        }
                        prow[x] = pack_rgb(v3_make(shade * base.x, shade * base.y, shade * base.z));
                    }
                }
                w[0] += dx[0]; w[1] += dx[1]; w[2] += dx[2];
            }
            wy[0] += dy[0]; wy[1] += dy[1]; wy[2] += dy[2];
            w[0] = wy[0]; w[1] = wy[1]; w[2] = wy[2];
        }
    }

    free(sc.spawn_parent);
    free(sc.cv); free(sc.rv); free(sc.n); free(sc.payload); free(sc.kind); free(sc.vi); free(sc.ai);
    if (!depth_out) { free(depth); }
    if (stats) { *stats = st; }
    if (setup_count) { *setup_count = n_setups; }
    return st.scratch_overflow ? 1 : 0;
}
