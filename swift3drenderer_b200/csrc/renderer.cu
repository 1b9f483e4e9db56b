// renderer.cu — C++ host layer and the extern "C" boundary (include/render.h, include/s3r_b200.h).
//
// Owns: scene conversion data.bin -> HBM layout, per-view frame scratch with capacity regrowth,
// host camera stepping (update_camera, render-cpp/render.cpp:134-156), frame orchestration on a
// CUDA stream, the synchronous drop-in updateAndRender (render-cpp/render.cpp:264-384) with
// data.bin discovery via dladdr (render.cpp:161-176).  There is no CPU rendering path in here.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>
#include <limits.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <exception>
#include <mutex>
#include <string>
#include <thread>
#include <functional>
#include <vector>

#include "../../include/render.h"
#include "../../include/s3r_b200.h"
#include "cluster.hpp"
#include "hostcopy.hpp"
#include "pipeline.cuh"

using namespace s3r;

static thread_local std::string g_error;

static int fail(int code, const std::string &msg) {
    g_error = msg;
    return code;
}

#define CUDA_TRY(expr)                                                                                   \
    do {                                                                                                 \
        cudaError_t e_ = (expr);                                                                         \
        if (e_ != cudaSuccess) {                                                                         \
            return fail(S3R_E_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e_));                 \
        }                                                                                                \
    } while (0)

// A device allocation owned by its holder: grown by ensure(), freed with the holder (on the current device).
template <typename T>
struct DevBuf {
    T *p = nullptr;
    size_t n = 0;
    DevBuf() = default;
    DevBuf(DevBuf &&o) noexcept { *this = std::move(o); }
    DevBuf &operator=(DevBuf &&o) noexcept { std::swap(p, o.p); std::swap(n, o.n); return *this; }
    ~DevBuf() { if (p) { cudaFree(p); } }
    cudaError_t ensure(size_t count) {
        if (count <= n) { return cudaSuccess; }
        if (p) { cudaFree(p); p = nullptr; n = 0; }
        cudaError_t e = cudaMalloc(&p, std::max<size_t>(count, 1) * sizeof(T));
        if (e == cudaSuccess) { n = count; }
        return e;
    }
};

// Registrations of caller frame buffers (cudaHostRegister with `flags`), so that their device->host copies run at full
// PCIe rate.  A buffer seen before is looked up; a new one (or a resize, main.swift:156-165) first drops the registrations
// it overlaps, and a ninth drops them all.  pin() returns false when the registration fails: copy through staging.
struct HostPins {
    struct Pin { const void *ptr; size_t bytes; };
    unsigned flags;
    std::vector<Pin> pins;
    explicit HostPins(unsigned f) : flags(f) {}
    bool pin(const void *ptr, size_t bytes) {
        for (auto &p : pins) {
            if (p.ptr == ptr && p.bytes >= bytes) { return true; }
        }
        for (size_t i = 0; i < pins.size();) {
            const char *a = static_cast<const char *>(pins[i].ptr), *b = static_cast<const char *>(ptr);
            if (a < b + bytes && b < a + pins[i].bytes) {
                cudaHostUnregister(const_cast<void *>(pins[i].ptr));
                pins.erase(pins.begin() + (long)i);
            } else {
                i++;
            }
        }
        if (pins.size() >= 8) { clear(); }
        if (cudaHostRegister(const_cast<void *>(ptr), bytes, flags) != cudaSuccess) {
            cudaGetLastError();  // clear; fall back to a pageable copy
            return false;
        }
        pins.push_back(Pin{ptr, bytes});
        return true;
    }
    void clear() {
        for (auto &p : pins) { cudaHostUnregister(const_cast<void *>(p.ptr)); }
        pins.clear();
    }
};

// Per-view scratch of the loaded scene's submissions: capacities and buffers, sized by ensure_scratch and dropped as a
// whole when a scene is loaded.
struct FrameScratch {
    uint32_t views_cap = 0, tile_stride = 0;
    uint32_t setup_cap = 0, tile_cap = 0, big_cap = 0, items_cap = 0;
    uint32_t walk_cap = 0;
    DevBuf<uint4> cluster_list;
    DevBuf<uint8_t> walk_q;            // candidate queue of the direct walk: 40-byte records (front kernel -> walk kernel)
    DevBuf<float4> rv;
    DevBuf<SetupVis> vis;
    DevBuf<SetupShade> shade;
    DevBuf<uint4> head;
    DevBuf<uint32_t> slot_of;
    DevBuf<unsigned long long> keys;   // general path: per-pixel depth keys ...
    DevBuf<uint2> raster_items;        // ... and the tile kernel's work queue
    DevBuf<unsigned long long> pstate; // weights of the tile kernel's winners: 3 tagged words per pixel
    DevBuf<uint32_t> worklist;
    DevBuf<uint32_t> counters, big_list;   // counters: [views_cap][C_COUNT] followed by the tile histograms [views_cap][tile_stride]
    DevBuf<uint32_t> entries;
    DevBuf<float> cams;
    DevBuf<float> coltab;     // small scenes: tile-column checkpoints of the largest survivors (span_walk)
    DevBuf<uint32_t> span_slots;
    DevBuf<float> rowtab;     // general path: row-start blocks of the tile-path triangles (post_setup)
    DevBuf<uint32_t> rowbase;
};

struct S3RRenderer {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool has_scene = false;
    uint64_t V = 0, Vpad = 0, I = 0, T = 0, A = 0, n_texels = 0;
    DevBuf<float> pos_x, pos_y, pos_z;
    DevBuf<uint32_t> vi[3], ai[3];
    DevBuf<uint4> attr;
    DevBuf<uint32_t> texels;
    // spatial pre-partition of the triangle stream (cluster.hpp), built at load
    DevBuf<uint4> cl_hdr;
    DevBuf<float> cl_px, cl_py, cl_pz;
    DevBuf<uint32_t> cl_tri;
    uint32_t n_clusters = 0;
    int opt_clusters = 2, opt_cluster_cull = 1;   // clusters: 0 off, 1 on, 2 on for partitioned submissions
    Frame last_frame;   // parameter block of the last submission (raster-vertex dumps on the cluster path)
    FrameScratch scratch;
    uint32_t views_per_chunk = 256;
    int opt_flat_max = 128;
    int64_t rowtab_limit = -1;         // test hook "rowtab_capacity": floats of row-start table per view (< 0: no limit)
    DevBuf<uint32_t> sticky;
    uint32_t *sticky_host = nullptr;   // pinned mirror of `sticky`
    float factor_override = 0.f;   // drop-in path: the reference's stale-factor rule (render.cpp:276-279)
    DevBuf<uint32_t> frame;   // internal device framebuffer for host renders (u32 pixels, or 3 bytes/pixel when packed)
    // submission ring: pinned camera staging + events, so the host can run RING chunks ahead
    static constexpr int RING = 16;
    float *cams_pinned = nullptr;     // RING x views_cap x 12
    size_t cams_pinned_views = 0;
    cudaEvent_t ev_cams[RING] = {}, ev_t0[RING] = {}, ev_t1[RING] = {}, ev_t2[RING] = {};
    bool slot_used[RING] = {}, slot_timed[RING] = {};
    // per-kernel timing (option "timing"): an event after every kernel launch of a timed submission
    static constexpr int MAX_MARKS = 40;
    cudaEvent_t ev_mark[RING][MAX_MARKS] = {};
    const char *mark_name[RING][MAX_MARKS] = {};
    int n_marks[RING] = {};
    struct KernelAcc { const char *name; double ms; uint64_t launches; };
    std::vector<KernelAcc> kernel_acc;
    uint64_t chunk_counter = 0;
    int opt_timing = 0;          // 0 off, n > 0: every n-th submission is timed (events after every launch cost launch overlap)
    uint64_t timing_phase = 0;
    double geometry_ms = 0, raster_ms = 0;
    uint64_t timed_chunks = 0;
    // last render (for finish / dumps)
    uint32_t last_views = 0, last_W = 0, last_H = 0;
    cudaStream_t last_stream = nullptr;   // stream of the last s3r_render_device submission
    uint64_t launches = 0;
    int opt_tma = 1, opt_pin_host = 0;   // pinning caller memory is opt-in: see s3r_render_host
    // staged host output (default path of s3r_render_host)
    cudaStream_t copy_stream = nullptr, aux_stream = nullptr;
    cudaEvent_t ev_geometry = nullptr;
    static constexpr int MAX_SLICES = 64;
    cudaEvent_t ev_raster[MAX_SLICES] = {}, ev_copy[MAX_SLICES] = {};
    uint8_t *staging = nullptr;
    size_t staging_bytes = 0;
    HostCopier *copier = nullptr;
    int opt_copy_threads = 0, opt_host_bands = 12, opt_pack24 = 1, opt_fused_small = 1, opt_direct_small = 1, opt_spans = 1, opt_tmap = 1, opt_band_taper = 1;
    HostPins pins{cudaHostRegisterDefault};
    // fused frame assembly
    std::vector<void *> own_frames, opened_frames;
    uint32_t *peer_out[MAX_PEERS] = {};
    uint32_t n_peers = 0;
};

// --------------------------------------------------------------------------------------------------
// lifetime
// --------------------------------------------------------------------------------------------------
extern "C" const char *s3r_last_error(void) { return g_error.c_str(); }

static int create_device_objects(S3RRenderer *r) {
    CUDA_TRY(cudaStreamCreateWithFlags(&r->stream, cudaStreamNonBlocking));
    for (int i = 0; i < S3RRenderer::RING; i++) {
        CUDA_TRY(cudaEventCreateWithFlags(&r->ev_cams[i], cudaEventDisableTiming));
        CUDA_TRY(cudaEventCreate(&r->ev_t0[i])); CUDA_TRY(cudaEventCreate(&r->ev_t1[i])); CUDA_TRY(cudaEventCreate(&r->ev_t2[i]));
        for (int k = 0; k < S3RRenderer::MAX_MARKS; k++) { CUDA_TRY(cudaEventCreate(&r->ev_mark[i][k])); }
    }
    CUDA_TRY(cudaStreamCreateWithFlags(&r->copy_stream, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&r->aux_stream, cudaStreamNonBlocking));
    CUDA_TRY(cudaEventCreateWithFlags(&r->ev_geometry, cudaEventDisableTiming));
    for (int i = 0; i < S3RRenderer::MAX_SLICES; i++) {
        CUDA_TRY(cudaEventCreateWithFlags(&r->ev_raster[i], cudaEventDisableTiming));
        CUDA_TRY(cudaEventCreateWithFlags(&r->ev_copy[i], cudaEventDisableTiming));
    }
    CUDA_TRY(configure_kernels());
    return S3R_OK;
}

extern "C" int s3r_create(S3RRenderer **out, int device) {
    if (!out) { return fail(S3R_E_ARG, "out is null"); }
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        return fail(S3R_E_CUDA, std::string("no CUDA device: ") + cudaGetErrorString(e) +
                                    " (this library has no CPU fallback)");
    }
    if (device < 0 || device >= count) { return fail(S3R_E_ARG, "device index out of range"); }
    CUDA_TRY(cudaSetDevice(device));
    S3RRenderer *r = new S3RRenderer();
    r->device = device;
    const int rc = create_device_objects(r);
    if (rc) { s3r_destroy(r); return rc; }   // (s3r_destroy skips what was not created)
    if (const char *env = getenv("S3R_COPY_THREADS")) { r->opt_copy_threads = atoi(env); }
    if (const char *env = getenv("S3R_HOST_BANDS")) { r->opt_host_bands = std::max(1, atoi(env)); }
    if (const char *env = getenv("S3R_BAND_TAPER")) { r->opt_band_taper = atoi(env) != 0; }
    if (const char *env = getenv("S3R_PACK24")) { r->opt_pack24 = atoi(env) != 0; }
    *out = r;
    return S3R_OK;
}

// The renderer's device buffers are freed by their destructors, on the device set here.
extern "C" void s3r_destroy(S3RRenderer *r) {
    if (!r) { return; }
    cudaSetDevice(r->device);
    cudaStreamSynchronize(r->stream);
    for (void *p : r->opened_frames) { cudaIpcCloseMemHandle(p); }
    for (void *p : r->own_frames) { cudaFree(p); }
    r->pins.clear();
    if (r->cams_pinned) { cudaFreeHost(r->cams_pinned); }
    delete r->copier;
    if (r->sticky_host) { cudaFreeHost(r->sticky_host); }
    if (r->staging) { cudaFreeHost(r->staging); }
    for (int i = 0; i < S3RRenderer::MAX_SLICES; i++) {
        if (r->ev_raster[i]) { cudaEventDestroy(r->ev_raster[i]); cudaEventDestroy(r->ev_copy[i]); }
    }
    if (r->copy_stream) { cudaStreamDestroy(r->copy_stream); }
    if (r->aux_stream) { cudaStreamDestroy(r->aux_stream); }
    if (r->ev_geometry) { cudaEventDestroy(r->ev_geometry); }
    for (int i = 0; i < S3RRenderer::RING; i++) {
        if (r->ev_cams[i]) { cudaEventDestroy(r->ev_cams[i]); cudaEventDestroy(r->ev_t0[i]); cudaEventDestroy(r->ev_t1[i]); cudaEventDestroy(r->ev_t2[i]); }
        for (int k = 0; k < S3RRenderer::MAX_MARKS; k++) { if (r->ev_mark[i][k]) { cudaEventDestroy(r->ev_mark[i][k]); } }
    }
    if (r->stream) { cudaStreamDestroy(r->stream); }
    delete r;
}

// --------------------------------------------------------------------------------------------------
// scene: data.bin (render-cpp/render.cpp:177-209) -> HBM layout (pipeline.cuh)
// --------------------------------------------------------------------------------------------------
extern "C" int s3r_load_scene_arrays(S3RRenderer *r, const float *vertices, uint64_t V, const uint64_t *vidx,
                                     const uint64_t *aidx, uint64_t I, const void *attributes, uint64_t A,
                                     const uint32_t *texels, uint64_t n_texels) {
    if (!r) { return fail(S3R_E_ARG, "renderer is null"); }
    if (I % 3) { return fail(S3R_E_SCENE, "index count is not a multiple of 3"); }
    if (V >= 0xFFFFFFFFull || A >= 0xFFFFFFFFull || I >= 0xFFFFFFFFull) {
        return fail(S3R_E_SCENE, "counts exceed the reference's uint32 loop counters (render.cpp:285,290,297)");
    }
    if (n_texels & 0x3FFFFull) { return fail(S3R_E_SCENE, "texel count is not a multiple of 512*512"); }
    CUDA_TRY(cudaSetDevice(r->device));
    CUDA_TRY(cudaStreamSynchronize(r->stream));
    const uint64_t T = I / 3, Vpad = (V + 3) & ~3ull;
    std::vector<float> px(std::max<uint64_t>(Vpad, 4), 0.f), py(px.size(), 0.f), pz(px.size(), -1.f);
    for (uint64_t i = 0; i < V; i++) {
        if (vertices[4 * i + 3] != 1.0f) { return fail(S3R_E_SCENE, "vertex w != 1"); }
        px[i] = vertices[4 * i]; py[i] = vertices[4 * i + 1]; pz[i] = vertices[4 * i + 2];
    }
    std::vector<uint32_t> v[3], a[3];
    for (int k = 0; k < 3; k++) { v[k].resize(std::max<uint64_t>(T, 1)); a[k].resize(std::max<uint64_t>(T, 1)); }
    for (uint64_t t = 0; t < T; t++) {
        for (int k = 0; k < 3; k++) {
            const uint64_t vv = vidx[3 * t + k], aa = aidx[3 * t + k];
            if (vv >= V || aa >= A) { return fail(S3R_E_SCENE, "index out of range"); }
            v[k][t] = (uint32_t)vv; a[k][t] = (uint32_t)aa;
        }
    }
    const uint32_t n_tex = (uint32_t)(n_texels >> 18);
    std::vector<uint4> at(std::max<uint64_t>(2 * A, 2));
    const uint8_t *rec = static_cast<const uint8_t *>(attributes);
    for (uint64_t i = 0; i < A; i++) {
        uint32_t w[12];
        memcpy(w, rec + 48 * i, 48);
        float nw;
        memcpy(&nw, &w[3], 4);
        if (nw != 0.0f) { return fail(S3R_E_SCENE, "normal w != 0"); }
        if (w[8] > 1) { return fail(S3R_E_SCENE, "attribute kind not in {0, 1}"); }
        if (w[8] == 1 && w[4] >= n_tex) { return fail(S3R_E_SCENE, "texture index out of range"); }
        at[2 * i] = make_uint4(w[0], w[1], w[2], w[8]);
        at[2 * i + 1] = make_uint4(w[4], w[5], w[6], w[7]);
    }
    CUDA_TRY(r->pos_x.ensure(px.size())); CUDA_TRY(r->pos_y.ensure(px.size())); CUDA_TRY(r->pos_z.ensure(px.size()));
    CUDA_TRY(cudaMemcpy(r->pos_x.p, px.data(), px.size() * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(r->pos_y.p, py.data(), py.size() * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(r->pos_z.p, pz.data(), pz.size() * 4, cudaMemcpyHostToDevice));
    for (int k = 0; k < 3; k++) {
        CUDA_TRY(r->vi[k].ensure(v[k].size())); CUDA_TRY(r->ai[k].ensure(a[k].size()));
        CUDA_TRY(cudaMemcpy(r->vi[k].p, v[k].data(), v[k].size() * 4, cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMemcpy(r->ai[k].p, a[k].data(), a[k].size() * 4, cudaMemcpyHostToDevice));
    }
    r->n_clusters = 0;
    if (T > 0) {   // clusters of consecutive, spatially close triangles for the general path's front kernel
        ClusterSet cs;
        build_clusters(px.data(), py.data(), pz.data(), v[0].data(), v[1].data(), v[2].data(), T, cs);
        CUDA_TRY(r->cl_hdr.ensure(cs.hdr.size() * 2)); CUDA_TRY(r->cl_px.ensure(cs.px.size())); CUDA_TRY(r->cl_py.ensure(cs.px.size()));
        CUDA_TRY(r->cl_pz.ensure(cs.px.size())); CUDA_TRY(r->cl_tri.ensure(cs.tri.size()));
        CUDA_TRY(cudaMemcpy(r->cl_hdr.p, cs.hdr.data(), cs.hdr.size() * sizeof(ClusterHeader), cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMemcpy(r->cl_px.p, cs.px.data(), cs.px.size() * 4, cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMemcpy(r->cl_py.p, cs.py.data(), cs.py.size() * 4, cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMemcpy(r->cl_pz.p, cs.pz.data(), cs.pz.size() * 4, cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMemcpy(r->cl_tri.p, cs.tri.data(), cs.tri.size() * 4, cudaMemcpyHostToDevice));
        r->n_clusters = cs.n_clusters;
    }
    CUDA_TRY(r->attr.ensure(at.size()));
    CUDA_TRY(cudaMemcpy(r->attr.p, at.data(), at.size() * sizeof(uint4), cudaMemcpyHostToDevice));
    CUDA_TRY(r->texels.ensure(std::max<uint64_t>(n_texels, 1)));
    if (n_texels) { CUDA_TRY(cudaMemcpy(r->texels.p, texels, n_texels * 4, cudaMemcpyHostToDevice)); }
    r->V = V; r->Vpad = px.size(); r->I = I; r->T = T; r->A = A; r->n_texels = n_texels;
    r->has_scene = true;
    r->scratch = FrameScratch();   // sized for the new scene by the next render
    return S3R_OK;
}

extern "C" int s3r_load_scene_file(S3RRenderer *r, const char *path) {
    if (!r || !path) { return fail(S3R_E_ARG, "null argument"); }
    // The file is mapped, not read: a 20 M-triangle data.bin is 4 GB, and the sections are converted straight from the
    // page cache.  Every section length is checked against what is left of the file BEFORE it is multiplied by the
    // record size, so a hostile header cannot wrap the arithmetic.
    const int fd = open(path, O_RDONLY);
    if (fd < 0) { return fail(S3R_E_IO, std::string("cannot open ") + path); }
    struct stat st;
    if (fstat(fd, &st) != 0 || st.st_size < 0) { close(fd); return fail(S3R_E_IO, std::string("cannot stat ") + path); }
    const size_t size = (size_t)st.st_size;
    if (size < 5 * 16) { close(fd); return fail(S3R_E_IO, "truncated file (five section headers expected)"); }
    void *map = mmap(nullptr, size, PROT_READ, MAP_PRIVATE, fd, 0);
    close(fd);
    if (map == MAP_FAILED) { return fail(S3R_E_IO, std::string("cannot map ") + path); }
    madvise(map, size, MADV_SEQUENTIAL);
    const uint8_t *b = static_cast<const uint8_t *>(map);
    size_t off = 0;
    // one section: header {count, ignored} (render.cpp:178-179), then `padded(count)` records of `elem` bytes
    auto section = [&](uint64_t &n, size_t elem, bool pad_odd, const uint8_t *&data) -> bool {
        if (size - off < 16) { return false; }
        memcpy(&n, b + off, 8);
        off += 16;
        const uint64_t records = n + (pad_odd ? (n & 1) : 0);   // n < 2^64 - 1 is implied by the division below
        if (n == UINT64_MAX || records > (size - off) / elem) { return false; }
        data = b + off;
        off += (size_t)records * elem;
        return true;
    };
    uint64_t V = 0, I = 0, A = 0, I2 = 0, NT = 0;
    const uint8_t *vertices = nullptr, *vidx = nullptr, *attrs = nullptr, *aidx = nullptr, *texels = nullptr;
    int rc = S3R_OK;
    if (!section(V, 16, false, vertices)) { rc = fail(S3R_E_IO, "truncated vertex section"); }
    else if (!section(I, 8, true, vidx)) { rc = fail(S3R_E_IO, "truncated index section"); }
    else if (!section(A, 48, false, attrs)) { rc = fail(S3R_E_IO, "truncated attribute section"); }
    else if (!section(I2, 8, true, aidx)) { rc = fail(S3R_E_IO, "truncated attribute-index section"); }
    else if (I2 != I) { rc = fail(S3R_E_SCENE, "index streams differ in length"); }
    else if (!section(NT, 4, false, texels)) { rc = fail(S3R_E_IO, "truncated texture section"); }
    else {
        try {
            rc = s3r_load_scene_arrays(r, reinterpret_cast<const float *>(vertices), V, reinterpret_cast<const uint64_t *>(vidx),
                                       reinterpret_cast<const uint64_t *>(aidx), I, attrs, A, reinterpret_cast<const uint32_t *>(texels), NT);
        } catch (const std::exception &e) {   // allocation failure while converting: report, do not unwind through extern "C"
            rc = fail(S3R_E_IO, std::string("scene conversion failed: ") + e.what());
        }
    }
    munmap(map, size);
    return rc;
}

// Test hook, callable without a GPU: the spatial pre-partition (cluster.hpp) of a triangle stream.  counts_out =
// {clusters, cluster vertices, triangles}; the arrays are filled when they are non-null and large enough.
extern "C" int s3r_debug_clusters(const float *vertices, uint64_t V, const uint64_t *vidx, uint64_t I, void *hdr_out, uint64_t hdr_cap,
                                  float *pos_out, uint64_t v_cap, uint32_t *tri_out, uint64_t counts_out[3]) {
    if (!vertices || !vidx || !counts_out || I % 3) { return fail(S3R_E_ARG, "bad cluster request"); }
    const uint64_t T = I / 3;
    try {
        std::vector<float> px(V), py(V), pz(V);
        for (uint64_t i = 0; i < V; i++) { px[i] = vertices[4 * i]; py[i] = vertices[4 * i + 1]; pz[i] = vertices[4 * i + 2]; }
        std::vector<uint32_t> v[3];
        for (int k = 0; k < 3; k++) { v[k].resize(T); }
        for (uint64_t t = 0; t < T; t++) {
            for (int k = 0; k < 3; k++) {
                if (vidx[3 * t + k] >= V) { return fail(S3R_E_SCENE, "index out of range"); }
                v[k][t] = (uint32_t)vidx[3 * t + k];
            }
        }
        ClusterSet cs;
        build_clusters(px.data(), py.data(), pz.data(), v[0].data(), v[1].data(), v[2].data(), T, cs);
        counts_out[0] = cs.n_clusters; counts_out[1] = cs.px.size(); counts_out[2] = cs.tri.size();
        if (hdr_out && hdr_cap >= cs.hdr.size()) { memcpy(hdr_out, cs.hdr.data(), cs.hdr.size() * sizeof(ClusterHeader)); }
        if (pos_out && v_cap >= cs.px.size()) {
            memcpy(pos_out, cs.px.data(), cs.px.size() * 4); memcpy(pos_out + v_cap, cs.py.data(), cs.px.size() * 4);
            memcpy(pos_out + 2 * v_cap, cs.pz.data(), cs.px.size() * 4);
        }
        if (tri_out) { memcpy(tri_out, cs.tri.data(), cs.tri.size() * 4); }
    } catch (const std::exception &e) {
        return fail(S3R_E_IO, std::string("clustering failed: ") + e.what());
    }
    return S3R_OK;
}

extern "C" int s3r_scene_counts(const S3RRenderer *r, uint64_t *v, uint64_t *i, uint64_t *a, uint64_t *t) {
    if (!r || !r->has_scene) { return fail(S3R_E_NOSCENE, "no scene loaded"); }
    if (v) { *v = r->V; } if (i) { *i = r->I; } if (a) { *a = r->A; } if (t) { *t = r->n_texels; }
    return S3R_OK;
}

// --------------------------------------------------------------------------------------------------
// camera — render-cpp/render.cpp:51-65 (initial state), :134-156 (update_camera); scalar binary32
// in the reference's evaluation order (simd semantics as pinned by the oracle shim).
// --------------------------------------------------------------------------------------------------
namespace {
struct V3 { float x, y, z; };
inline V3 mk(float x, float y, float z) { return V3{x, y, z}; }
inline V3 add(V3 a, V3 b) { return mk(a.x + b.x, a.y + b.y, a.z + b.z); }
inline V3 mul(V3 a, float s) { return mk(a.x * s, a.y * s, a.z * s); }
inline float dot(V3 a, V3 b) { return (a.x * b.x + a.y * b.y) + a.z * b.z; }
inline V3 cross(V3 a, V3 b) { return mk(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x); }
inline V3 unit(V3 a) { return mul(a, 1.0f / sqrtf(dot(a, a))); }
inline V3 ld(const float *p) { return mk(p[0], p[1], p[2]); }
inline void st(float *p, V3 a) { p[0] = a.x; p[1] = a.y; p[2] = a.z; }
inline V3 rotate(V3 qv, float qw, V3 v) {  // simd_act
    const V3 t = mul(cross(qv, v), 2.f);
    return add(add(v, mul(t, qw)), cross(qv, t));
}
}  // namespace

extern "C" void s3r_camera_reset(S3RCamera *cam) {
    memset(cam, 0, sizeof(*cam));
    cam->axis_x[0] = cam->axis_y[1] = cam->axis_z[2] = 1.f;
    cam->matrix[0] = cam->matrix[5] = cam->matrix[10] = 1.f;
}

extern "C" void s3r_camera_update(S3RCamera *cam, const S3RInput *in) {
    const float speed = 0.1f, rotation_speed = 0.3f;  // render.cpp:94-95
    bool changed = false;
    V3 pos = ld(cam->position), X = ld(cam->axis_x), Y = ld(cam->axis_y), Z = ld(cam->axis_z);
    if (in->left > 0 || in->right > 0 || in->up > 0 || in->down > 0) {
        changed = true;
        const V3 step = add(mul(X, in->right - in->left), mul(Z, in->down - in->up));
        pos = add(pos, mul(step, speed));
    }
    if (in->mouse_x != cam->mouse[0] || in->mouse_y != cam->mouse[1]) {
        changed = true;
        const V3 z = unit(add(add(mul(X, cam->mouse[0] - in->mouse_x), mul(Y, cam->mouse[1] - in->mouse_y)),
                              mul(Z, 100 / rotation_speed)));
        V3 qv;
        float qw;
        if (dot(Z, z) >= 0.f) {
            const V3 half = unit(add(Z, z));
            qv = cross(Z, half);
            qw = dot(Z, half);
        } else {  // obtuse turn in one frame: two half rotations
            V3 half = unit(add(Z, z));
            if (!(dot(half, half) > 0.f)) {
                half = unit(cross(Z, fabsf(Z.x) < fabsf(Z.y) ? mk(1, 0, 0) : mk(0, 1, 0)));
            }
            const V3 pv = cross(half, z), sv = cross(Z, half);
            const float pw = dot(half, z), sw = dot(Z, half);
            qv = add(add(mul(sv, pw), mul(pv, sw)), cross(pv, sv));
            qw = pw * sw - dot(pv, sv);
        }
        X = unit(rotate(qv, qw, X));
        Y = unit(rotate(qv, qw, Y));
        Z = z;
        cam->mouse[0] = in->mouse_x;
        cam->mouse[1] = in->mouse_y;
    }
    if (changed || !cam->started) {
        st(cam->matrix + 0, X); cam->matrix[3] = -dot(X, pos);
        st(cam->matrix + 4, Y); cam->matrix[7] = -dot(Y, pos);
        st(cam->matrix + 8, Z); cam->matrix[11] = -dot(Z, pos);
    }
    cam->started = 1;
    st(cam->position, pos); st(cam->axis_x, X); st(cam->axis_y, Y); st(cam->axis_z, Z);
}

extern "C" float s3r_factor(uint32_t height) { return kNear * (float)height / (2 * kScale); }

// --------------------------------------------------------------------------------------------------
// frame scratch
// --------------------------------------------------------------------------------------------------
// Small scenes (2T <= SORT_CAP survivors at most) skip the bin arrays: one fused geometry CTA per view and
// in-kernel per-tile collection in the rasteriser.
static bool uses_direct_bin(const S3RRenderer *r) {
    return r->opt_fused_small && 2ull * r->T <= (uint64_t)SORT_CAP && r->scratch.setup_cap >= 2ull * r->T;
}

// The cluster front (batch_cull, cluster_cull, cluster_front, direct_walk) pays for itself when much of the scene can be
// rejected wholesale — above all on a screen partition, where a rank keeps 1/n of the clusters.  opt_clusters: 0 never,
// 1 always, 2 (default) for partitioned submissions only: on a whole frame of the benchmark field it rejects a quarter of
// the clusters and costs more than the raw-stream classify kernel it replaces.
static bool uses_clusters(const S3RRenderer *r, bool partitioned) {
    return r->n_clusters > 0 && (r->opt_clusters == 1 || (r->opt_clusters == 2 && partitioned));
}

// Sizes every per-view buffer a submission needs and points `f` at them.  `f` arrives with the submission's geometry
// (views, frame size, tiles, output and key-plane strides).  Capacities only grow here; finish_on and the
// "setup_capacity" hook change them, and a buffer whose size expression then grows is reallocated on the next call.
// banded: the tile rows are rasterised in several launches (host renders).
static int ensure_scratch(S3RRenderer *r, Frame &f, bool partitioned, bool banded, cudaStream_t s) {
    FrameScratch &b = r->scratch;
    const uint32_t T = (uint32_t)r->T;
    if (b.setup_cap == 0) {
        // survivors are usually a small share of 2T; start at T/4 (min 4096) and regrow on demand
        b.setup_cap = (uint32_t)std::min<uint64_t>(2ull * T + 16, std::max<uint64_t>(4096, T / 4));
        b.big_cap = std::max<uint32_t>(1024, b.setup_cap / 16u);
        b.tile_cap = 0;
    }
    if (b.tile_cap == 0) {
        // per-tile list capacity: 4x the average load, a power of two in [256, setup_cap]; regrown on overflow
        uint64_t want = 4ull * b.setup_cap / std::max<uint32_t>(f.n_tiles, 1u), cap = 256;
        while (cap < want) { cap <<= 1; }
        b.tile_cap = (uint32_t)std::min<uint64_t>(cap, std::max<uint32_t>(b.setup_cap, 256u));
    }
    b.views_cap = std::max(f.n_views, b.views_cap);
    b.tile_stride = std::max(((f.n_tiles + 1 + 63) / 64) * 64, b.tile_stride);
    const size_t vc = b.views_cap;
    // small scenes are launch-latency bound: one fused CTA per view and no bin arrays instead of eight
    // launches; 2T <= SORT_CAP guarantees every raster CTA can hold the whole survivor list
    f.direct_bin = uses_direct_bin(r) ? 1 : 0;
    const bool front = !f.direct_bin && uses_clusters(r, partitioned);
    if (!front) { CUDA_TRY(b.rv.ensure(vc * r->Vpad)); }   // the cluster front keeps raster-space vertices on chip
    f.rv = front ? nullptr : b.rv.p;
    CUDA_TRY(b.vis.ensure(vc * b.setup_cap));
    CUDA_TRY(b.shade.ensure(vc * b.setup_cap));
    CUDA_TRY(b.head.ensure(vc * b.setup_cap));
    if (!f.direct_bin) {
        CUDA_TRY(b.slot_of.ensure(vc * 2ull * std::max<uint64_t>(r->T, 1)));
    }
    CUDA_TRY(b.worklist.ensure(vc * std::max<uint64_t>(r->T, 1)));
    f.vis = b.vis.p; f.shade = b.shade.p; f.head = b.head.p; f.slot_of = b.slot_of.p; f.worklist = b.worklist.p; f.setup_cap = b.setup_cap;
    // per-view counters and, right behind them, the per-tile histograms: the cluster path clears both with one memset
    if (vc * (C_COUNT + (size_t)b.tile_stride) > b.counters.n) { CUDA_TRY(cudaStreamSynchronize(r->stream)); }
    CUDA_TRY(b.counters.ensure(vc * (C_COUNT + (size_t)b.tile_stride)));
    f.counters = b.counters.p;
    f.tile_count = b.counters.p + vc * C_COUNT;
    f.tile_stride = b.tile_stride;
    if (!r->sticky.p) {
        CUDA_TRY(r->sticky.ensure(8)); CUDA_TRY(cudaMemset(r->sticky.p, 0, 32));
        CUDA_TRY(cudaMallocHost(reinterpret_cast<void **>(&r->sticky_host), 32));
        memset(r->sticky_host, 0, 32);
    }
    f.sticky = r->sticky.p;
    // bin lists exist only for scenes that do not take the in-kernel collection path
    if (!f.direct_bin) {
        CUDA_TRY(b.entries.ensure(vc * (size_t)b.tile_stride * b.tile_cap));
        b.items_cap = b.tile_stride * (1u + b.tile_cap / RASTER_CHUNK);   // every non-empty tile + every full chunk
        CUDA_TRY(b.raster_items.ensure(vc * (size_t)b.items_cap));
    }
    f.entries = b.entries.p; f.tile_cap = b.tile_cap;
    f.raster_items = b.raster_items.p; f.items_cap = b.items_cap;
    CUDA_TRY(b.big_list.ensure(vc * b.big_cap));
    f.big_list = b.big_list.p; f.big_cap = b.big_cap;
    CUDA_TRY(b.cams.ensure(vc * 12));
    f.cams = b.cams.p;
    if (r->cams_pinned_views < vc) {
        CUDA_TRY(cudaStreamSynchronize(r->stream));
        if (r->cams_pinned) { cudaFreeHost(r->cams_pinned); }
        CUDA_TRY(cudaMallocHost(&r->cams_pinned, (size_t)S3RRenderer::RING * vc * 12 * sizeof(float)));
        r->cams_pinned_views = vc;
    }
    if (front) {
        f.cl_hdr = r->cl_hdr.p; f.cl_px = r->cl_px.p; f.cl_py = r->cl_py.p; f.cl_pz = r->cl_pz.p; f.cl_tri = r->cl_tri.p;
        f.n_clusters = r->n_clusters; f.cluster_cull = r->opt_cluster_cull;
        f.list_cap = r->n_clusters;
        CUDA_TRY(b.cluster_list.ensure(vc * f.list_cap));
        f.cluster_list = b.cluster_list.p;
        // candidates of the direct walk: a quarter of the triangles to begin with, regrown on overflow
        if (b.walk_cap == 0) { b.walk_cap = (uint32_t)std::min<uint64_t>(std::max<uint64_t>(r->T, 1), std::max<uint64_t>(4096, r->T / 4)); }
        CUDA_TRY(b.walk_q.ensure(vc * b.walk_cap * 40u));
        f.walk_q = reinterpret_cast<WalkRecord *>(b.walk_q.p); f.walk_cap = b.walk_cap;
    }
    if (!f.direct_bin) {   // general path: per-pixel keys and winners for the flat passes
        // keys are all zero between frames: allocation clears them, shade_tiles clears what a frame has set.  The old
        // plane may still be read by the submission before: wait for it before it is freed.
        if ((size_t)f.n_views * f.key_view_stride + 2 > b.keys.n) {
            CUDA_TRY(cudaStreamSynchronize(s));
            CUDA_TRY(b.keys.ensure((size_t)f.n_views * f.key_view_stride + 2));
            CUDA_TRY(cudaMemsetAsync(b.keys.p, 0, b.keys.n * sizeof(unsigned long long), s));
        }
        CUDA_TRY(b.pstate.ensure(3u * ((size_t)f.n_views * f.out_view_stride + 2)));
        f.pstate = b.pstate.p;
    }
    f.keys = b.keys.p;
    if (f.direct_bin && r->opt_spans && !banded) {
        // whole-frame launches of a small scene: the largest survivors' row walks are done once per frame (span_walk)
        // instead of by exact jumps in every tile.  The banded host path keeps the jumps: its first band must not wait.
        f.span_h = (f.H + 31u) & ~31u;
        const size_t per_view = (size_t)SPAN_MAX * f.tiles_x * 3u * f.span_h;
        if (per_view * vc * sizeof(float) <= (size_t)1 << 30) {
            CUDA_TRY(b.coltab.ensure(per_view * vc));
            CUDA_TRY(b.span_slots.ensure((size_t)SPAN_MAX * vc));
            f.coltab = b.coltab.p; f.span_slots = b.span_slots.p;
        }
    }
    if (!f.direct_bin && r->opt_spans) {
        // general path: 8 M floats of row-start blocks per view; a triangle that does not fit keeps its exact jumps
        f.rowtab_cap = (uint32_t)std::min<size_t>(8u << 20, ((size_t)256 << 20) / std::max<size_t>(vc, 1));   // <= 1 GB in all
        if (r->rowtab_limit >= 0) { f.rowtab_cap = (uint32_t)std::min<int64_t>(f.rowtab_cap, r->rowtab_limit); }
        CUDA_TRY(b.rowtab.ensure(std::max<size_t>(1, (size_t)f.rowtab_cap * vc)));   // (an empty table still exists: its triangles jump)
        CUDA_TRY(b.rowbase.ensure((size_t)b.setup_cap * vc));
        f.rowtab = b.rowtab.p; f.rowbase = b.rowbase.p;
    }
    return S3R_OK;
}

// Tensor map of a submission's output for tile_raster's one-store-per-tile write-out: {x, output row, view}, 32-bit
// pixels or (packed host transport) bytes with 3 per pixel.  cuTensorMapEncodeTiled comes from the driver through the
// runtime's entry-point query, so the library does not link libcuda.  false = use the bulk row copies.
static bool encode_out_map(CUtensorMap *map, void *base, uint32_t W, uint64_t rows, uint32_t views, uint64_t view_stride_px, bool packed24) {
    typedef CUresult (*EncodeFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                 const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                 CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    static EncodeFn encode = [] {
        void *fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) {
            cudaGetLastError();
            fn = nullptr;
        }
        return reinterpret_cast<EncodeFn>(fn);
    }();
    if (!encode || rows == 0) { return false; }
    const uint64_t bpp = packed24 ? 3 : 4;
    const cuuint64_t dims[3] = {packed24 ? (cuuint64_t)W * 3u : (cuuint64_t)W, rows, views};
    const cuuint64_t strides[2] = {(cuuint64_t)W * bpp, view_stride_px * bpp};   // bytes, dimensions 1 and 2
    const cuuint32_t box[3] = {packed24 ? (cuuint32_t)TILE_W * 3u : (cuuint32_t)TILE_W, (cuuint32_t)TILE_H, 1u};
    const cuuint32_t estr[3] = {1u, 1u, 1u};
    if (strides[0] % 16u || strides[1] % 16u) { return false; }
    return encode(map, packed24 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_UINT32, 3, base, dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// Band edges in tile rows for `nb` <= tiles_y raster launches: uniform — the copy workers expand 24-bit pixels about as
// fast as the link delivers them, so any larger band builds a backlog — except that (taper, host path) the last band
// is split 1/2, 1/4, 1/4: what is left to expand when the link goes idle is a quarter band instead of a whole one.
// Returns the number of edges (bands + 1); every band has at least one tile row.
static int band_edges(uint32_t tiles_y, int nb, bool taper, uint32_t *edge) {
    int n_edges = 0;
    for (int b = 0; b <= nb; b++) { edge[n_edges++] = (uint32_t)((uint64_t)tiles_y * b / nb); }
    if (taper && nb >= 3 && n_edges + 2 <= S3RRenderer::MAX_SLICES) {
        const uint32_t lo = edge[nb - 1], rows = tiles_y - lo;
        if (rows >= 2) {   // strictly increasing edges: 2 rows -> 1 + 1, 3 -> 2 + 1, 4 -> 2 + 1 + 1, 6 -> 3 + 1 + 2, ...
            const uint32_t a = lo + (rows + 1) / 2, b2 = a + (tiles_y - a) / 2;
            n_edges = nb;
            edge[n_edges++] = a;
            if (b2 > a && b2 < tiles_y) { edge[n_edges++] = b2; }
            edge[n_edges++] = tiles_y;
        }
    }
    return n_edges;
}

// Test hook (CPU-callable): the band edges s3r_render_host uses for `tiles_y` tile rows and `bands` requested bands.
extern "C" int s3r_debug_band_edges(uint32_t tiles_y, int bands, int taper, uint32_t *edges_out, int capacity) {
    if (!edges_out || tiles_y == 0 || bands < 1 || capacity < S3RRenderer::MAX_SLICES + 1) { return fail(S3R_E_ARG, "bad band request"); }
    const int nb = std::max(1, std::min<int>(std::min(bands, (int)S3RRenderer::MAX_SLICES - 2), (int)tiles_y));
    return band_edges(tiles_y, nb, taper != 0, edges_out);
}

// Collects the stage and per-kernel times of the timed submission that used ring slot `slot`.
static int retire_timed_slot(S3RRenderer *r, int slot) {
    if (!r->slot_timed[slot]) { return S3R_OK; }
    CUDA_TRY(cudaEventSynchronize(r->ev_t2[slot]));
    float g = 0, q = 0;
    cudaEventElapsedTime(&g, r->ev_t0[slot], r->ev_t1[slot]);
    cudaEventElapsedTime(&q, r->ev_t1[slot], r->ev_t2[slot]);
    r->geometry_ms += g; r->raster_ms += q; r->timed_chunks++;
    cudaEvent_t prev = r->ev_t0[slot];
    for (int k = 0; k < r->n_marks[slot]; k++) {
        float ms = 0;
        cudaEventElapsedTime(&ms, prev, r->ev_mark[slot][k]);
        prev = r->ev_mark[slot][k];
        const char *name = r->mark_name[slot][k];
        auto it = std::find_if(r->kernel_acc.begin(), r->kernel_acc.end(), [&](const S3RRenderer::KernelAcc &a) { return !strcmp(a.name, name); });
        if (it == r->kernel_acc.end()) { r->kernel_acc.push_back({name, 0.0, 0}); it = r->kernel_acc.end() - 1; }
        it->ms += ms; it->launches++;
    }
    r->n_marks[slot] = 0;
    r->slot_timed[slot] = false;
    return S3R_OK;
}

struct MarkCtx { S3RRenderer *r; int slot; cudaStream_t s; };
static void mark_kernel(void *ctx, const char *kernel) {
    MarkCtx *m = static_cast<MarkCtx *>(ctx);
    int &n = m->r->n_marks[m->slot];
    if (n < S3RRenderer::MAX_MARKS && cudaEventRecord(m->r->ev_mark[m->slot][n], m->s) == cudaSuccess) { m->r->mark_name[m->slot][n++] = kernel; }
}

// Called by a host render after band b's raster launch and the record of r->ev_raster[b]; end_row is the first pixel
// row (relative to y0) after band b.
typedef std::function<int(int b, uint32_t end_row)> BandFn;

// One submission of n_views views: pixel rows [y0, y1) of the W x H frame, or (row_stride > 1; y0 = 0, y1 = H) the tile
// rows a with a % row_stride == row_phase, compacted.  The tile rows are rasterised in raster_bands launches; with
// after_band (host renders), r->ev_raster[b] is recorded after band b and after_band runs.
static int render_chunk(S3RRenderer *r, const float *cams, uint32_t n_views, uint32_t W, uint32_t H, uint32_t y0, uint32_t y1,
                        uint32_t row_stride, uint32_t row_phase, uint32_t *dev_out, cudaStream_t s, int raster_bands = 1,
                        bool packed24 = false, const BandFn &after_band = nullptr) {
    Frame f;
    memset(&f, 0, sizeof(f));
    f.tiles_x = (W + TILE_W - 1) / TILE_W;
    f.row_stride = row_stride; f.row_phase = row_phase;
    if (row_stride == 1) {
        f.tile_row0 = y0 / TILE_H;
        f.tiles_y = (y1 - 1) / TILE_H - f.tile_row0 + 1;
    } else {   // interleaved tile rows of the whole frame
        const uint32_t rows = (H + TILE_H - 1) / TILE_H;
        f.tile_row0 = 0;
        f.tiles_y = rows > row_phase ? (rows - row_phase + row_stride - 1) / row_stride : 0;
    }
    f.n_tiles = f.tiles_x * f.tiles_y;
    f.n_views = n_views;
    f.W = W; f.H = H; f.y0 = y0; f.y1 = y1;
    f.out_view_stride = row_stride == 1 ? (unsigned long long)W * (y1 - y0) : (unsigned long long)W * f.tiles_y * TILE_H;
    f.key_view_stride = (unsigned long long)W * (((f.out_view_stride / W) + 3u) & ~3ull);   // key plane: columns of 4 output rows
    const bool partitioned = row_stride > 1 || y0 > 0 || y1 < H;
    int rc = ensure_scratch(r, f, partitioned, raster_bands > 1, s);
    if (rc) { return rc; }
    const int slot = (int)(r->chunk_counter++ % S3RRenderer::RING);
    if (r->slot_used[slot]) {  // the chunk that used this slot RING submissions ago
        CUDA_TRY(cudaEventSynchronize(r->ev_cams[slot]));
        int rc2 = retire_timed_slot(r, slot);
        if (rc2) { return rc2; }
    }
    if (n_views == 1) {
        // one view: the matrix travels in the kernels' parameter block (an H2D copy in front of the first kernel costs
        // more than the kernel launch itself)
        memcpy(f.cam0, cams, 12 * sizeof(float));
        f.cam_inline = 1;
        CUDA_TRY(cudaEventRecord(r->ev_cams[slot], s));   // (keeps the ring's retire logic uniform; an event record is not a copy)
        r->slot_used[slot] = true;
    } else {
        float *staging = r->cams_pinned + (size_t)slot * r->cams_pinned_views * 12;
        memcpy(staging, cams, (size_t)n_views * 12 * sizeof(float));
        CUDA_TRY(cudaMemcpyAsync(r->scratch.cams.p, staging, (size_t)n_views * 12 * sizeof(float), cudaMemcpyHostToDevice, s));
        CUDA_TRY(cudaEventRecord(r->ev_cams[slot], s));
        r->slot_used[slot] = true;
    }
    const bool timed = r->opt_timing > 0 && (r->timing_phase++ % (uint64_t)r->opt_timing) == 0;
    MarkCtx mark_ctx{r, slot, s};
    const LaunchMarks marks{mark_kernel, &mark_ctx};
    const LaunchMarks *mk = timed ? &marks : nullptr;
    r->n_marks[slot] = 0;

    f.pos_x = r->pos_x.p; f.pos_y = r->pos_y.p; f.pos_z = r->pos_z.p;
    f.vi0 = r->vi[0].p; f.vi1 = r->vi[1].p; f.vi2 = r->vi[2].p;
    f.ai0 = r->ai[0].p; f.ai1 = r->ai[1].p; f.ai2 = r->ai[2].p;
    f.attr = r->attr.p; f.texels = r->texels.p;
    f.V = (uint32_t)r->V; f.Vpad = (uint32_t)r->Vpad; f.T = (uint32_t)r->T; f.A = (uint32_t)r->A;
    f.n_tex = std::max<uint32_t>(1, (uint32_t)(r->n_texels >> 18));
    f.fw = (float)W; f.fh = (float)H; f.half_w = f.fw / 2; f.half_h = f.fh / 2;  // screen_size / 2, render.cpp:284,288
    f.factor = r->factor_override != 0.f ? r->factor_override : s3r_factor(H);
    f.band_lo = (float)y0; f.band_hi = (float)y1;
    f.out = dev_out;
    f.n_peers = r->n_peers;
    for (uint32_t k = 0; k < r->n_peers; k++) { f.peer_out[k] = r->peer_out[k]; }
    f.out_packed24 = packed24 ? 1 : 0;
    f.use_tma = r->opt_tma && (W % (packed24 ? 16 : 4) == 0) && ((reinterpret_cast<uintptr_t>(dev_out) & 15u) == 0);
    // (interleaved tile rows keep the row copies: rows past H stay unwritten; so do bands that start inside a tile row —
    // the store's start coordinate must not be negative)
    if (f.use_tma && r->opt_tmap && f.direct_bin && dev_out && row_stride == 1 && y0 % TILE_H == 0) {
        f.use_tmap = encode_out_map(&f.out_map, dev_out, W, (uint64_t)(f.out_view_stride / W), n_views, f.out_view_stride, packed24) ? 1 : 0;
    }
    if (timed) { CUDA_TRY(cudaEventRecord(r->ev_t0[slot], s)); }
    if (f.n_peers && (f.direct_bin || packed24)) { return fail(S3R_E_ARG, "peer frames need the general path (scene over 1920 triangles) and device output"); }
    f.direct_small = !f.direct_bin && r->opt_direct_small ? 1 : 0;
    f.flat_max = (uint32_t)r->opt_flat_max;
    f.rs_magic = row_stride > 1 ? (uint32_t)((1ull << 32) / row_stride) + 1u : 0u;
    r->launches += (uint64_t)(f.direct_bin ? launch_geometry_small(f, s, mk) : launch_geometry(f, s, mk));
    if (r->sticky_host) {
        // overflow record of this submission, read back on a side stream behind the geometry kernels: a 16-byte copy IN the
        // rendering stream would sit between post_setup and the raster kernels (10 us of every frame)
        CUDA_TRY(cudaEventRecord(r->ev_geometry, s));
        CUDA_TRY(cudaStreamWaitEvent(r->aux_stream, r->ev_geometry, 0));
        CUDA_TRY(cudaMemcpyAsync(r->sticky_host, r->sticky.p, 32, cudaMemcpyDeviceToHost, r->aux_stream));
    }
    if (timed) { CUDA_TRY(cudaEventRecord(r->ev_t1[slot], s)); }
    // (general path: the tile kernel runs with the first band over the whole frame, the bands cut the shading pass)
    const int nb = std::max(1, std::min<int>(raster_bands, (int)f.tiles_y));
    uint32_t edge[S3RRenderer::MAX_SLICES + 1];
    const int n_edges = band_edges(f.tiles_y, nb, r->opt_band_taper && after_band != nullptr, edge);
    for (int b = 0; b + 1 < n_edges; b++) {
        f.raster_row0 = edge[b];
        f.raster_rows = edge[b + 1] - edge[b];
        r->launches += (uint64_t)launch_raster(f, s, mk);
        if (after_band) {
            // the host path enqueues band b's device->host copy right here, before the next band's launch call,
            // so that the link starts as early as the GPU allows
            CUDA_TRY(cudaEventRecord(r->ev_raster[b], s));
            const uint32_t end_row = (f.tile_row0 + f.raster_row0 + f.raster_rows) * TILE_H;
            int rc2 = after_band(b, std::min(y1, std::max(y0, end_row)) - y0);
            if (rc2) { return rc2; }
        }
    }
    if (timed) { CUDA_TRY(cudaEventRecord(r->ev_t2[slot], s)); r->slot_timed[slot] = true; }
    CUDA_TRY(cudaGetLastError());
    r->last_frame = f;
    return S3R_OK;
}

// The device entry points: validation, stream choice and the view-chunk loop.  row_stride == 1: pixel rows [y0, y1);
// otherwise y0 = 0, y1 = H and the tile rows a with a % row_stride == row_phase.
static int render_device(S3RRenderer *r, const float *cams, uint32_t n_views, uint32_t W, uint32_t H, uint32_t y0, uint32_t y1,
                         uint32_t row_stride, uint32_t row_phase, uint32_t *dev_out, void *stream) {
    if (!r || !cams || (!dev_out && r->n_peers == 0)) { return fail(S3R_E_ARG, "null argument"); }
    if (!r->has_scene) { return fail(S3R_E_NOSCENE, "no scene loaded"); }
    if (W == 0 || H == 0 || W > 65535 || H > 65535 || y0 >= y1 || y1 > H || n_views == 0 || row_stride == 0 || row_phase >= row_stride) {
        return fail(S3R_E_ARG, "bad frame geometry");
    }
    const uint32_t tile_rows = (H + TILE_H - 1) / TILE_H;
    if (tile_rows <= row_phase) { return S3R_OK; }   // this phase owns no tile row
    CUDA_TRY(cudaSetDevice(r->device));
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : r->stream;
    r->last_stream = s;
    const size_t view_px = (size_t)W * (row_stride == 1 ? y1 - y0 : (tile_rows - row_phase + row_stride - 1) / row_stride * TILE_H);
    for (uint32_t v0 = 0; v0 < n_views; v0 += r->views_per_chunk) {
        const uint32_t nv = std::min(r->views_per_chunk, n_views - v0);
        int rc = render_chunk(r, cams + 12 * (size_t)v0, nv, W, H, y0, y1, row_stride, row_phase, dev_out + view_px * v0, s);
        if (rc) { return rc; }
        r->last_views = nv;
    }
    r->last_W = W; r->last_H = H;
    return S3R_OK;
}

extern "C" int s3r_render_device(S3RRenderer *r, const float *cams, uint32_t n_views, uint32_t W, uint32_t H,
                                 uint32_t y0, uint32_t y1, uint32_t *dev_out, void *stream) {
    return render_device(r, cams, n_views, W, H, y0, y1, 1, 0, dev_out, stream);
}

extern "C" int s3r_render_device_rows(S3RRenderer *r, const float *cams, uint32_t n_views, uint32_t W, uint32_t H,
                                      uint32_t row_stride, uint32_t row_phase, uint32_t *dev_out, void *stream) {
    return render_device(r, cams, n_views, W, H, 0, H, row_stride, row_phase, dev_out, stream);
}

extern "C" uint32_t s3r_tile_height(void) { return (uint32_t)TILE_H; }

// Waits for the renderer's work, reads the per-view counters back and regrows capacities.
// Returns 1 if something overflowed (the frame(s) of the last chunk must be rendered again).
static int finish_on(S3RRenderer *r, cudaStream_t s) {
    CUDA_TRY(cudaSetDevice(r->device));
    CUDA_TRY(cudaStreamSynchronize(s));
    CUDA_TRY(cudaStreamSynchronize(r->aux_stream));   // the overflow record's copy
    if (r->last_views == 0 || !r->sticky.p) { return S3R_OK; }
    uint32_t sticky[8];
    memcpy(sticky, r->sticky_host, sizeof(sticky));   // copied after the geometry of the last submission; the sync above covers it
    const uint32_t overflow = sticky[0], need_setups = sticky[1], need_entries = sticky[2], need_big = sticky[3], need_walk = sticky[4];
    if (!overflow) { return S3R_OK; }
    CUDA_TRY(cudaMemset(r->sticky.p, 0, sizeof(sticky)));
    memset(r->sticky_host, 0, sizeof(sticky));
    FrameScratch &b = r->scratch;   // (ensure_scratch regrows the buffers whose size these capacities set)
    if (overflow & 1u) {
        b.setup_cap = (uint32_t)std::min<uint64_t>(2ull * r->T + 16, (uint64_t)need_setups + need_setups / 2 + 1024);
        b.big_cap = std::max(b.big_cap, b.setup_cap / 16u);
    }
    if (overflow & 2u) { b.tile_cap = std::max(b.tile_cap, need_entries + need_entries / 2 + 64); }
    if (overflow & 4u) { b.big_cap = std::max(b.big_cap, need_big + need_big / 2 + 64); }
    if (overflow & 8u) {
        // (not bounded by T: the front reserves the queue in per-warp chunks of 64 and pads them with holes, so a scene whose
        // triangles nearly all take the direct walk needs more records than it has triangles)
        b.walk_cap = (uint32_t)std::min<uint64_t>(0xFFFFFFFFull, (uint64_t)need_walk + need_walk / 4 + 1024);
    }
    return 1;
}

extern "C" int s3r_finish(S3RRenderer *r) {
    if (!r) { return fail(S3R_E_ARG, "renderer is null"); }
    return finish_on(r, r->last_stream ? r->last_stream : r->stream);
}

// A registration made for a caller's buffer goes stale if the caller unmaps that memory and later
// gets the same virtual address back (free + malloc of a large block): the DMA would then land in
// the old, still-pinned physical pages.  Pixels always have a zero top byte (0x00RRGGBB), so a
// sentinel with a non-zero top byte written by the CPU before the copy and still present after it
// proves that the copy did not reach the memory the CPU sees.
static const uint32_t kSentinel = 0xA5C3A5C3u;

static void plant_sentinels(uint32_t *dst, size_t n) {
    dst[0] = kSentinel; dst[n / 2] = kSentinel; dst[n - 1] = kSentinel;
}
static bool sentinels_gone(const uint32_t *dst, size_t n) {
    return dst[0] != kSentinel && dst[n / 2] != kSentinel && dst[n - 1] != kSentinel;
}

static int ensure_staging(S3RRenderer *r, size_t bytes) {
    if (r->staging_bytes < bytes) {
        if (r->staging) { cudaFreeHost(r->staging); r->staging = nullptr; r->staging_bytes = 0; }
        CUDA_TRY(cudaMallocHost(reinterpret_cast<void **>(&r->staging), bytes));
        r->staging_bytes = bytes;
    }
    if (!r->copier) {
        int n = r->opt_copy_threads;
        if (n <= 0) {  // measured on the 16-core B200 host: 14 workers keep up with 24-bit PCIe transport
            const unsigned hc = std::thread::hardware_concurrency();
            n = (int)std::min<unsigned>(14, hc > 3 ? hc - 2 : 1);
        }
        r->copier = new HostCopier(n);
    }
    return S3R_OK;
}

extern "C" int s3r_render_host(S3RRenderer *r, const float *cams, uint32_t n_views, uint32_t W, uint32_t H,
                               uint32_t y0, uint32_t y1, uint32_t *host_out) {
    if (!r || !cams || !host_out) { return fail(S3R_E_ARG, "null argument"); }
    if (!r->has_scene) { return fail(S3R_E_NOSCENE, "no scene loaded"); }
    // SetupVis and the survivor heads pack box bounds in 16 bits: the same limits as s3r_render_device
    if (W == 0 || H == 0 || W > 65535 || H > 65535 || y0 >= y1 || y1 > H || n_views == 0) { return fail(S3R_E_ARG, "bad frame geometry"); }
    CUDA_TRY(cudaSetDevice(r->device));
    const size_t view_px = (size_t)W * (y1 - y0);
    // OPT-IN ("pin_host" option / S3R_PIN_HOST=1): cudaHostRegister the caller's frame buffer so the D2H
    // copy runs at full PCIe rate.  Only safe when the caller keeps that allocation mapped for as long
    // as it passes it (the reference's main loop does: one double buffer, re-allocated on resize only,
    // main.swift:156-165).  A registration that outlives its memory poisons every later CUDA call that
    // touches a host pointer in the recycled range, so it is never done behind the caller's back.
    const bool pinned = r->opt_pin_host && r->pins.pin(host_out, view_px * n_views * 4);
    for (uint32_t v0 = 0; v0 < n_views; v0 += r->views_per_chunk) {
        const uint32_t nv = std::min(r->views_per_chunk, n_views - v0);
        uint32_t *dst = host_out + view_px * v0;
        // 24-bit transport: the top byte of every pixel is zero, so only 3 bytes per pixel cross PCIe and
        // the copy threads expand them while moving staging -> caller buffer
        const bool packed = !pinned && r->opt_pack24;
        const size_t bpp = packed ? 3 : 4;
        const size_t chunk_bytes = view_px * nv * bpp;
        CUDA_TRY(r->frame.ensure(view_px * nv));
        if (!pinned) { int rc = ensure_staging(r, chunk_bytes + 64); if (rc) { return rc; } }
        bool rendered = false;
        for (int attempt = 0; attempt < 8 && !rendered; attempt++) {
            // ---- enqueue: geometry, banded raster, one D2H per band/slice on the copy stream -----
            // band-pipelined raster (small scenes) or shading (general path) and copy: band k crosses PCIe while band k + 1 renders
            const int bands = nv == 1 ? std::max(1, std::min(r->opt_host_bands, S3RRenderer::MAX_SLICES)) : 1;
            std::vector<CopySlice> slices;
            uint8_t *target = pinned ? reinterpret_cast<uint8_t *>(dst) : r->staging;
            if (pinned) { plant_sentinels(dst, view_px * nv); }
            int n_ev = 0;
            uint32_t row = 0;
            // band b's pixels of all nv views; several views have one band, copied in slices of about 4 MB
            const BandFn copy_band = [&](int b, uint32_t end_row) -> int {
                const size_t pa = (size_t)row * W * nv, pe = (size_t)end_row * W * nv;
                row = end_row;
                CUDA_TRY(cudaStreamWaitEvent(r->copy_stream, r->ev_raster[b], 0));
                const size_t n_sl = nv == 1 ? 1 : std::min<size_t>(S3RRenderer::MAX_SLICES, std::max<size_t>(1, chunk_bytes >> 22));
                for (size_t i = 0; i < n_sl; i++) {
                    const size_t a = pa + (((pe - pa) * i / n_sl) & ~(size_t)63);
                    const size_t e = i + 1 == n_sl ? pe : pa + (((pe - pa) * (i + 1) / n_sl) & ~(size_t)63);
                    if (e <= a) { continue; }
                    CUDA_TRY(cudaMemcpyAsync(target + a * bpp, reinterpret_cast<uint8_t *>(r->frame.p) + a * bpp, (e - a) * bpp,
                                             cudaMemcpyDeviceToHost, r->copy_stream));
                    CUDA_TRY(cudaEventRecord(r->ev_copy[n_ev], r->copy_stream));
                    slices.push_back(CopySlice{r->staging + a * bpp, reinterpret_cast<uint8_t *>(dst) + a * 4, e - a});
                    n_ev++;
                }
                return S3R_OK;
            };
            int rc = render_chunk(r, cams + 12 * (size_t)v0, nv, W, H, y0, y1, 1, 0, r->frame.p, r->stream, bands, packed, copy_band);
            if (rc) { return rc; }
            r->last_views = nv; r->last_W = W; r->last_H = H;
            // ---- drain: as each slice lands in staging the worker threads move it to the caller ----
            if (!pinned) { r->copier->begin(&slices, packed); }
            cudaError_t ce = cudaSuccess;
            for (int i = 0; i < n_ev; i++) {
                const cudaError_t e1 = cudaEventSynchronize(r->ev_copy[i]);
                if (e1 != cudaSuccess) { ce = e1; }
                if (!pinned) { r->copier->publish(i + 1); }
            }
            if (!pinned) { r->copier->wait(); }
            if (ce != cudaSuccess) { return fail(S3R_E_CUDA, std::string("device-to-host copy: ") + cudaGetErrorString(ce)); }
            rc = finish_on(r, r->stream);
            if (rc < 0) { return rc; }
            if (rc == 0) {
                if (pinned && !sentinels_gone(dst, view_px * nv)) {
                    // stale registration: drop every pin and copy again through the pageable path
                    r->pins.clear();
                    CUDA_TRY(cudaMemcpy(dst, r->frame.p, view_px * nv * 4, cudaMemcpyDeviceToHost));
                }
                rendered = true;
            }
        }
        if (!rendered) { return fail(S3R_E_CUDA, "frame scratch still overflowing after 8 regrowths"); }
    }
    return S3R_OK;
}

// --------------------------------------------------------------------------------------------------
// fused frame assembly over peer memory
// --------------------------------------------------------------------------------------------------
extern "C" int s3r_peer_frame_alloc(S3RRenderer *r, uint64_t bytes, void **dev_ptr, unsigned char handle_out[64]) {
    if (!r || !dev_ptr || !handle_out || bytes == 0) { return fail(S3R_E_ARG, "null argument"); }
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle is 64 bytes");
    CUDA_TRY(cudaSetDevice(r->device));
    void *p = nullptr;
    CUDA_TRY(cudaMalloc(&p, bytes));
    CUDA_TRY(cudaMemset(p, 0, bytes));
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) { cudaFree(p); return fail(S3R_E_CUDA, std::string("cudaIpcGetMemHandle: ") + cudaGetErrorString(e)); }
    memcpy(handle_out, &h, 64);
    r->own_frames.push_back(p);
    *dev_ptr = p;
    return S3R_OK;
}

extern "C" int s3r_peer_frame_open(S3RRenderer *r, const unsigned char handle[64], void **dev_ptr) {
    if (!r || !dev_ptr || !handle) { return fail(S3R_E_ARG, "null argument"); }
    CUDA_TRY(cudaSetDevice(r->device));
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, 64);
    void *p = nullptr;
    CUDA_TRY(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    r->opened_frames.push_back(p);
    *dev_ptr = p;
    return S3R_OK;
}

extern "C" int s3r_peer_frame_release(S3RRenderer *r, void *dev_ptr) {
    if (!r || !dev_ptr) { return fail(S3R_E_ARG, "null argument"); }
    CUDA_TRY(cudaSetDevice(r->device));
    CUDA_TRY(cudaDeviceSynchronize());
    for (uint32_t k = 0; k < r->n_peers; k++) { if (r->peer_out[k] == dev_ptr) { r->n_peers = 0; } }
    for (size_t i = 0; i < r->own_frames.size(); i++) {
        if (r->own_frames[i] == dev_ptr) { r->own_frames.erase(r->own_frames.begin() + (long)i); CUDA_TRY(cudaFree(dev_ptr)); return S3R_OK; }
    }
    for (size_t i = 0; i < r->opened_frames.size(); i++) {
        if (r->opened_frames[i] == dev_ptr) { r->opened_frames.erase(r->opened_frames.begin() + (long)i); CUDA_TRY(cudaIpcCloseMemHandle(dev_ptr)); return S3R_OK; }
    }
    return fail(S3R_E_ARG, "not a peer frame of this renderer");
}

extern "C" int s3r_set_peer_frames(S3RRenderer *r, void *const *dev_ptrs, uint32_t n) {
    if (!r || (n && !dev_ptrs) || n > (uint32_t)MAX_PEERS) { return fail(S3R_E_ARG, "bad peer frame list"); }
    for (uint32_t k = 0; k < n; k++) {
        if (!dev_ptrs[k]) { return fail(S3R_E_ARG, "null peer frame"); }
        // shade_tiles stores 16-byte pieces at 16-byte offsets from the base
        if (reinterpret_cast<uintptr_t>(dev_ptrs[k]) & 15u) { return fail(S3R_E_ARG, "peer frame is not 16-byte aligned"); }
        r->peer_out[k] = static_cast<uint32_t *>(dev_ptrs[k]);
    }
    r->n_peers = n;
    return S3R_OK;
}

extern "C" int s3r_copy_from_device(S3RRenderer *r, void *host_dst, const void *dev_src, uint64_t bytes) {
    if (!r || !host_dst || !dev_src) { return fail(S3R_E_ARG, "null argument"); }
    CUDA_TRY(cudaSetDevice(r->device));
    CUDA_TRY(cudaMemcpy(host_dst, dev_src, bytes, cudaMemcpyDeviceToHost));
    return S3R_OK;
}

// --------------------------------------------------------------------------------------------------
// introspection
// --------------------------------------------------------------------------------------------------
extern "C" int s3r_get_stats(S3RRenderer *r, uint32_t view, S3RStats *out) {
    if (!r || !out) { return fail(S3R_E_ARG, "null argument"); }
    if (view >= r->last_views) { return fail(S3R_E_ARG, "view out of range"); }
    CUDA_TRY(cudaSetDevice(r->device));
    uint32_t c[C_COUNT];
    CUDA_TRY(cudaMemcpy(c, r->scratch.counters.p + (size_t)view * C_COUNT, sizeof(c), cudaMemcpyDeviceToHost));
    memset(out, 0, sizeof(*out));
    out->triangles_in = (uint32_t)r->T;
    out->near_rejected = c[C_NEAR]; out->clipped = c[C_CLIPPED]; out->spawned = c[C_SPAWNED]; out->culled = c[C_CULLED];
    out->setups = c[C_SETUPS] + c[C_DIRECT]; out->bin_entries = c[C_ENTRIES]; out->big_triangles = c[C_BIG]; out->overflow = c[C_OVERFLOW];
    return S3R_OK;
}

extern "C" int s3r_dump_raster_vertices(S3RRenderer *r, uint32_t view, float *out, uint64_t cap) {
    if (!r || !out) { return fail(S3R_E_ARG, "null argument"); }
    if (view >= r->last_views || cap < r->V) { return fail(S3R_E_ARG, "view/capacity out of range"); }
    CUDA_TRY(cudaSetDevice(r->device));
    if (!r->last_frame.rv) {
        // the frame went through the cluster front, which keeps raster-space vertices in shared memory: run the vertex
        // stage alone over the original vertex stream with the same camera, factor and frame size
        CUDA_TRY(cudaStreamSynchronize(r->last_stream ? r->last_stream : r->stream));
        CUDA_TRY(r->scratch.rv.ensure((size_t)r->scratch.views_cap * r->Vpad));
        Frame f = r->last_frame;
        f.rv = r->scratch.rv.p; f.counters = nullptr; f.n_tiles = 0;
        launch_vertex_stage(f, r->stream);
        r->launches++;
        CUDA_TRY(cudaStreamSynchronize(r->stream));
    }
    CUDA_TRY(cudaMemcpy(out, r->scratch.rv.p + (size_t)view * r->Vpad, r->V * sizeof(float4), cudaMemcpyDeviceToHost));
    return S3R_OK;
}

extern "C" int s3r_dump_setups(S3RRenderer *r, uint32_t view, S3RSetupDump *out, uint64_t cap, uint64_t *count) {
    if (!r || !count) { return fail(S3R_E_ARG, "null argument"); }
    if (view >= r->last_views) { return fail(S3R_E_ARG, "view out of range"); }
    CUDA_TRY(cudaSetDevice(r->device));
    uint32_t n = 0;
    CUDA_TRY(cudaMemcpy(&n, r->scratch.counters.p + (size_t)view * C_COUNT + C_SETUPS, 4, cudaMemcpyDeviceToHost));
    n = std::min(n, r->scratch.setup_cap);
    *count = n;
    if (!out || n == 0) { return S3R_OK; }
    std::vector<SetupVis> v(n);
    std::vector<SetupShade> s(n);
    CUDA_TRY(cudaMemcpy(v.data(), r->scratch.vis.p + (size_t)view * r->scratch.setup_cap, n * sizeof(SetupVis), cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemcpy(s.data(), r->scratch.shade.p + (size_t)view * r->scratch.setup_cap, n * sizeof(SetupShade), cudaMemcpyDeviceToHost));
    std::vector<uint32_t> idx(n);
    for (uint32_t i = 0; i < n; i++) { idx[i] = i; }
    std::sort(idx.begin(), idx.end(), [&](uint32_t a, uint32_t b) { return v[a].order < v[b].order; });
    for (uint64_t k = 0; k < std::min<uint64_t>(n, cap); k++) {
        const SetupVis &a = v[idx[k]];
        const SetupShade &b = s[idx[k]];
        S3RSetupDump &o = out[k];
        memset(&o, 0, sizeof(o));
        o.order = a.order; o.xmin = a.xmin; o.xmax = a.xmax; o.ymin = a.ymin; o.ymax = a.ymax; o.area = b.area;
        for (int c = 0; c < 3; c++) {
            o.wstart[c] = a.wstart[c]; o.dx[c] = a.dx[c]; o.dy[c] = a.dy[c]; o.rvz[c] = a.rvz[c];
            for (int e = 0; e < 3; e++) { o.cv[c][e] = b.cv[3 * c + e]; o.n[c][e] = b.n[3 * c + e]; }
        }
        o.kind = b.kind; o.texture = b.texture;
        if (b.kind == 0) {
            for (int c = 0; c < 3; c++) { for (int e = 0; e < 3; e++) { o.payload[c][e] = b.pay[3 * c + e]; } }
        } else {
            for (int c = 0; c < 3; c++) { o.payload[c][0] = b.pay[2 * c]; o.payload[c][1] = b.pay[2 * c + 1]; }
            o.dz[0] = b.pay[6]; o.dz[1] = b.pay[7]; o.tpp[0] = b.tpp[0]; o.tpp[1] = b.tpp[1];
        }
    }
    return S3R_OK;
}

extern "C" int s3r_debug_walk(S3RRenderer *r, const float *start, const float *delta, const uint32_t *steps,
                              float *out, uint32_t count) {
    if (!r || !start || !delta || !steps || !out) { return fail(S3R_E_ARG, "null argument"); }
    CUDA_TRY(cudaSetDevice(r->device));
    DevBuf<float> s, d, o;
    DevBuf<uint32_t> n;
    CUDA_TRY(s.ensure(count)); CUDA_TRY(d.ensure(count)); CUDA_TRY(o.ensure(count)); CUDA_TRY(n.ensure(count));
    CUDA_TRY(cudaMemcpy(s.p, start, count * 4ull, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(d.p, delta, count * 4ull, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(n.p, steps, count * 4ull, cudaMemcpyHostToDevice));
    launch_walk_jump(s.p, d.p, n.p, o.p, count, r->stream);
    r->launches++;
    CUDA_TRY(cudaStreamSynchronize(r->stream));
    CUDA_TRY(cudaMemcpy(out, o.p, count * 4ull, cudaMemcpyDeviceToHost));
    return S3R_OK;
}

extern "C" int s3r_debug_exact_math(S3RRenderer *r, uint32_t mode, uint64_t first, uint64_t count, uint32_t seed, uint64_t result[5]) {
    if (!r || !result) { return fail(S3R_E_ARG, "null argument"); }
    CUDA_TRY(cudaSetDevice(r->device));
    DevBuf<unsigned long long> res;
    CUDA_TRY(res.ensure(5));
    CUDA_TRY(cudaMemset(res.p, 0, 5 * sizeof(unsigned long long)));
    launch_exact_math(mode, first, count, seed, res.p, r->stream);
    r->launches++;
    CUDA_TRY(cudaStreamSynchronize(r->stream));
    CUDA_TRY(cudaMemcpy(result, res.p, 5 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    return S3R_OK;
}

extern "C" uint64_t s3r_kernel_launches(const S3RRenderer *r) { return r ? r->launches : 0; }

extern "C" int s3r_get_timing(S3RRenderer *r, double *geometry_ms, double *raster_ms, uint64_t *chunks, int reset) {
    if (!r) { return fail(S3R_E_ARG, "renderer is null"); }
    CUDA_TRY(cudaSetDevice(r->device));
    for (int slot = 0; slot < S3RRenderer::RING; slot++) {  // drain the chunks still in the ring
        int rc = retire_timed_slot(r, slot);
        if (rc) { return rc; }
    }
    if (geometry_ms) { *geometry_ms = r->geometry_ms; }
    if (raster_ms) { *raster_ms = r->raster_ms; }
    if (chunks) { *chunks = r->timed_chunks; }
    if (reset) { r->geometry_ms = r->raster_ms = 0; r->timed_chunks = 0; r->kernel_acc.clear(); }
    return S3R_OK;
}

extern "C" int s3r_get_kernel_timing(S3RRenderer *r, uint32_t index, const char **name, double *ms, uint64_t *launches) {
    if (!r) { return fail(S3R_E_ARG, "renderer is null"); }
    CUDA_TRY(cudaSetDevice(r->device));
    for (int slot = 0; slot < S3RRenderer::RING; slot++) {
        int rc = retire_timed_slot(r, slot);
        if (rc) { return rc; }
    }
    if (index >= r->kernel_acc.size()) { return 1; }   // past the last kernel
    if (name) { *name = r->kernel_acc[index].name; }
    if (ms) { *ms = r->kernel_acc[index].ms; }
    if (launches) { *launches = r->kernel_acc[index].launches; }
    return S3R_OK;
}

extern "C" int s3r_set_option(S3RRenderer *r, const char *name, int64_t value) {
    if (!r || !name) { return fail(S3R_E_ARG, "null argument"); }
    if (!strcmp(name, "tma_store")) { r->opt_tma = value != 0; return S3R_OK; }
    if (!strcmp(name, "fused_small")) { r->opt_fused_small = value != 0; return S3R_OK; }
    if (!strcmp(name, "direct_small")) { r->opt_direct_small = value != 0; return S3R_OK; }
    if (!strcmp(name, "spans")) { r->opt_spans = value != 0; return S3R_OK; }
    if (!strcmp(name, "clusters")) {
        if (value < 0 || value > 2) { return fail(S3R_E_ARG, "clusters: 0 off, 1 on, 2 on for partitioned submissions"); }
        cudaStreamSynchronize(r->stream); r->opt_clusters = (int)value; return S3R_OK;
    }
    if (!strcmp(name, "cluster_cull")) { r->opt_cluster_cull = value != 0; return S3R_OK; }
    if (!strcmp(name, "tensor_store")) { r->opt_tmap = value != 0; return S3R_OK; }
    if (!strcmp(name, "flat_max")) {   // >= 16: the record-free direct walk handles boxes under 16 x 16 whatever this says
        if (value < 16 || value > 65536) { return fail(S3R_E_ARG, "flat_max out of range"); }
        r->opt_flat_max = (int)value; return S3R_OK;
    }
    if (!strcmp(name, "pack24")) { r->opt_pack24 = value != 0; return S3R_OK; }
    if (!strcmp(name, "host_bands")) { r->opt_host_bands = (int)std::max<int64_t>(1, value); return S3R_OK; }
    if (!strcmp(name, "copy_threads")) {
        cudaStreamSynchronize(r->stream);
        delete r->copier; r->copier = nullptr;
        r->opt_copy_threads = (int)value;
        return S3R_OK;
    }
    if (!strcmp(name, "timing")) { r->opt_timing = (int)std::max<int64_t>(0, std::min<int64_t>(value, 1 << 20)); r->timing_phase = 0; return S3R_OK; }
    if (!strcmp(name, "pin_host")) { r->opt_pin_host = value != 0; if (!value) { r->pins.clear(); } return S3R_OK; }
    if (!strcmp(name, "views_per_chunk")) {
        if (value < 1) { return fail(S3R_E_ARG, "views_per_chunk < 1"); }
        r->views_per_chunk = (uint32_t)value;
        return S3R_OK;
    }
    if (!strcmp(name, "setup_capacity")) {  // test hook: force the regrow path
        if (value < 1) { return fail(S3R_E_ARG, "setup_capacity < 1"); }
        FrameScratch &b = r->scratch;
        b.setup_cap = (uint32_t)value; b.tile_cap = 4; b.big_cap = 4; b.walk_cap = 8;
        return S3R_OK;
    }
    if (!strcmp(name, "rowtab_capacity")) {   // test hook: row-start table size in floats per view (0: empty, < 0: default)
        r->rowtab_limit = value; return S3R_OK;
    }
    return fail(S3R_E_ARG, std::string("unknown option ") + name);
}

// --------------------------------------------------------------------------------------------------
// the drop-in entry point — render-cpp/render.cpp:264-384
// --------------------------------------------------------------------------------------------------
namespace {
S3RRenderer *g_renderer = nullptr;
S3RCamera g_camera;
uint32_t g_depth_bytes = 0;   // depth_buffer.buffer_size, render.cpp:67-73

// ---- one process, several GPUs (env S3R_DEVICES="0,1,2,3" or "all") -----------------------------------------------
// The frame is split by interleaved tile rows (tile row a belongs to GPU a mod n: an even share of the screen whatever
// the scene looks like); every GPU holds the whole scene, skips the clusters that miss its rows, rasterises and shades
// its rows into a compact device buffer and copies them — over its OWN PCIe link — to their place in the caller's
// buffer.  One persistent host thread per GPU issues that GPU's launches and copies, so the n launch sequences run in
// parallel; updateAndRender stays synchronous (it returns when every thread has finished the frame).
// The caller's buffer is registered (cudaHostRegisterPortable) on first sight, as the reference's main loop keeps one
// double buffer for its lifetime (main.swift:117-118,156-165); a registration that went stale is detected by sentinels
// and the frame is then delivered through pinned staging (S3R_PIN_HOST=0 forces that path).
struct MultiJob { const float *matrix; float factor; uint32_t W, H; uint32_t *host_out; bool pinned; };

struct MultiGpu {
    struct Worker {
        S3RRenderer *r = nullptr;
        std::thread th;
        uint8_t *staging = nullptr;
        size_t staging_bytes = 0;
        int rc = 0;
        std::string error;
    };
    std::vector<Worker> w;
    std::mutex m;
    std::condition_variable cv_go, cv_done;
    std::atomic<uint64_t> generation{0};
    std::atomic<int> done{0};
    bool stop = false;
    MultiJob job{};
    int pin = 1, bands = 4;   // bands: raster / shading launches per GPU and frame, each followed by its rows' copy
    HostPins pins{cudaHostRegisterPortable};
    // S3R_MULTI_TRACE=1: where a frame's wall time goes (microseconds, summed; printed every 256 frames to stderr)
    int trace = 0;
    uint64_t traced = 0;
    std::chrono::steady_clock::time_point t_publish;
    double us_total = 0, us_pin = 0, us_tail = 0;   // main thread: whole call, registration + sentinels, last worker done -> return
    struct Trace {
        double wake = 0, launch = 0, copies = 0, finish = 0;
        std::chrono::steady_clock::time_point done;
        cudaEvent_t e0 = nullptr, eb[16] = {}, ee[16] = {};   // device timeline: frame start (render stream), every band's copy begin / end (copy stream)
        double begin_us[16] = {}, end_us[16] = {};
    };
    std::vector<Trace> tr;
};
static inline double us_since(std::chrono::steady_clock::time_point t0) {
    return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - t0).count();
}
MultiGpu *g_multi = nullptr;

int multi_worker_frame(MultiGpu *mg, int k) {
    MultiGpu::Worker &me = mg->w[(size_t)k];
    S3RRenderer *r = me.r;
    const MultiJob &j = mg->job;
    const uint32_t n = (uint32_t)mg->w.size(), tile_rows = (j.H + TILE_H - 1) / TILE_H;
    if (tile_rows <= (uint32_t)k) { return S3R_OK; }   // fewer tile rows than GPUs: nothing for this one
    const uint32_t owned = (tile_rows - (uint32_t)k + n - 1) / n;
    const size_t compact_px = (size_t)j.W * owned * TILE_H;
    CUDA_TRY(cudaSetDevice(r->device));
    CUDA_TRY(r->frame.ensure(compact_px));
    if (!j.pinned && me.staging_bytes < compact_px * 4) {
        if (me.staging) { cudaFreeHost(me.staging); me.staging = nullptr; me.staging_bytes = 0; }
        CUDA_TRY(cudaHostAlloc(reinterpret_cast<void **>(&me.staging), compact_px * 4, cudaHostAllocPortable));
        me.staging_bytes = compact_px * 4;
    }
    r->factor_override = j.factor;
    if (mg->trace) { mg->tr[(size_t)k].wake += us_since(mg->t_publish); }
    for (int attempt = 0; attempt < 8; attempt++) {
        const auto t_begin = std::chrono::steady_clock::now();
        // The GPU's tile rows are rendered in a few bands; band b's rows leave over PCIe (copy stream) while band b + 1 is
        // rasterised / shaded.  Owned tile row l = frame tile row l * n + k: TILE_H contiguous pixel rows, i.e. one "row" of a
        // 2-D copy whose destination pitch is n tile rows — one DMA descriptor per band, one more for a cut last tile row.
        const size_t tile_bytes = (size_t)TILE_H * j.W * 4;
        const uint32_t last_y = ((owned - 1u) * n + (uint32_t)k) * TILE_H, last_rows = std::min<uint32_t>(TILE_H, j.H - last_y);
        uint8_t *dst0 = j.pinned ? reinterpret_cast<uint8_t *>(j.host_out + (size_t)k * TILE_H * j.W) : me.staging;
        const size_t dpitch = j.pinned ? tile_bytes * n : tile_bytes;
        uint32_t done_tiles = 0;
        MultiGpu::Trace *tr = mg->trace ? &mg->tr[(size_t)k] : nullptr;
        int n_bands = 0;
        if (tr) {
            if (!tr->e0) { cudaEventCreate(&tr->e0); for (int b = 0; b < 16; b++) { cudaEventCreate(&tr->eb[b]); cudaEventCreate(&tr->ee[b]); } }
            CUDA_TRY(cudaEventRecord(tr->e0, r->stream));
        }
        const BandFn copy_band = [&](int b, uint32_t end_row) -> int {
            const uint32_t upto = std::min(owned, (end_row + TILE_H - 1u) / TILE_H);   // owned tile rows finished after band b
            CUDA_TRY(cudaStreamWaitEvent(r->copy_stream, r->ev_raster[b], 0));
            if (tr && b < 16) { CUDA_TRY(cudaEventRecord(tr->eb[b], r->copy_stream)); n_bands = b + 1; }
            const uint32_t full_end = (upto == owned && last_rows != (uint32_t)TILE_H) ? owned - 1u : upto;
            if (full_end > done_tiles) {
                CUDA_TRY(cudaMemcpy2DAsync(dst0 + dpitch * done_tiles, dpitch, reinterpret_cast<const uint8_t *>(r->frame.p) + tile_bytes * done_tiles,
                                           tile_bytes, tile_bytes, full_end - done_tiles, cudaMemcpyDeviceToHost, r->copy_stream));
            }
            if (upto == owned && full_end < owned && done_tiles < owned) {
                CUDA_TRY(cudaMemcpyAsync(dst0 + dpitch * full_end, reinterpret_cast<const uint8_t *>(r->frame.p) + tile_bytes * full_end,
                                         (size_t)last_rows * j.W * 4, cudaMemcpyDeviceToHost, r->copy_stream));
            }
            done_tiles = upto;
            if (tr && b < 16) { CUDA_TRY(cudaEventRecord(tr->ee[b], r->copy_stream)); }
            return S3R_OK;
        };
        int rc = render_chunk(r, j.matrix, 1, j.W, j.H, 0, j.H, n, (uint32_t)k, r->frame.p, r->stream, mg->bands, false, copy_band);
        if (rc) { return rc; }
        r->last_views = 1; r->last_W = j.W; r->last_H = j.H; r->last_stream = r->stream;
        const auto t_launched = std::chrono::steady_clock::now();
        CUDA_TRY(cudaStreamSynchronize(r->copy_stream));
        const auto t_copied = std::chrono::steady_clock::now();
        rc = finish_on(r, r->stream);   // waits for the launches and the copies; 1 = a capacity was regrown, render again
        if (mg->trace) {
            MultiGpu::Trace &t = mg->tr[(size_t)k];
            t.launch += std::chrono::duration<double, std::micro>(t_launched - t_begin).count();
            t.copies += std::chrono::duration<double, std::micro>(t_copied - t_launched).count();
            t.finish += us_since(t_copied);
            for (int b = 0; b < n_bands; b++) {
                float ms = 0;
                if (cudaEventElapsedTime(&ms, t.e0, t.eb[b]) == cudaSuccess) { t.begin_us[b] += ms * 1e3; }
                if (cudaEventElapsedTime(&ms, t.e0, t.ee[b]) == cudaSuccess) { t.end_us[b] += ms * 1e3; }
            }
        }
        if (rc < 0) { return rc; }
        if (rc == 0) {
            if (!j.pinned) {
                for (uint32_t l = 0; l < owned; l++) {
                    const uint32_t y = (l * n + (uint32_t)k) * TILE_H, rows = std::min<uint32_t>(TILE_H, j.H - y);
                    memcpy(j.host_out + (size_t)y * j.W, me.staging + (size_t)l * TILE_H * j.W * 4, (size_t)rows * j.W * 4);
                }
            }
            return S3R_OK;
        }
    }
    return fail(S3R_E_CUDA, "frame scratch still overflowing after 8 regrowths");
}

void multi_worker(MultiGpu *mg, int k) {
    uint64_t seen = 0;
    for (;;) {
        // a short spin first (frames follow each other within microseconds in a render loop), then sleep
        for (int spin = 0; spin < 4000 && mg->generation.load(std::memory_order_acquire) == seen; spin++) { __builtin_ia32_pause(); }
        if (mg->generation.load(std::memory_order_acquire) == seen) {
            std::unique_lock<std::mutex> g(mg->m);
            mg->cv_go.wait(g, [&] { return mg->generation.load(std::memory_order_acquire) != seen; });
        }
        seen = mg->generation.load(std::memory_order_acquire);
        if (mg->stop) { return; }
        MultiGpu::Worker &me = mg->w[(size_t)k];
        me.rc = multi_worker_frame(mg, k);
        if (me.rc) { me.error = g_error; }
        if (mg->trace) { mg->tr[(size_t)k].done = std::chrono::steady_clock::now(); }
        if (mg->done.fetch_add(1, std::memory_order_acq_rel) + 1 == (int)mg->w.size()) {
            std::lock_guard<std::mutex> g(mg->m);
            mg->cv_done.notify_one();
        }
    }
}

int multi_render(MultiGpu *mg, const float *matrix, float factor, uint32_t W, uint32_t H, uint32_t *host_out) {
    if (W == 0 || H == 0 || W > 65535 || H > 65535) { return fail(S3R_E_ARG, "bad frame geometry"); }
    const size_t px = (size_t)W * H;
    const auto t_call = std::chrono::steady_clock::now();
    for (int pass = 0; pass < 2; pass++) {
        cudaSetDevice(mg->w[0].r->device);
        const bool pinned = pass == 0 && mg->pin && mg->pins.pin(host_out, px * 4);
        if (pinned) { plant_sentinels(host_out, px); }
        mg->job = MultiJob{matrix, factor, W, H, host_out, pinned};
        if (mg->trace) { mg->us_pin += us_since(t_call); mg->t_publish = std::chrono::steady_clock::now(); }
        mg->done.store(0, std::memory_order_release);
        {
            std::lock_guard<std::mutex> g(mg->m);
            mg->generation.fetch_add(1, std::memory_order_acq_rel);
        }
        mg->cv_go.notify_all();
        for (int spin = 0; spin < 20000 && mg->done.load(std::memory_order_acquire) < (int)mg->w.size(); spin++) { __builtin_ia32_pause(); }
        if (mg->done.load(std::memory_order_acquire) < (int)mg->w.size()) {
            std::unique_lock<std::mutex> g(mg->m);
            mg->cv_done.wait(g, [&] { return mg->done.load(std::memory_order_acquire) >= (int)mg->w.size(); });
        }
        for (auto &wk : mg->w) { if (wk.rc) { return fail(wk.rc, wk.error); } }
        if (mg->trace) {
            auto last = mg->tr[0].done;
            for (auto &t : mg->tr) { last = std::max(last, t.done); }
            mg->us_tail += us_since(last);
        }
        if (!pinned || sentinels_gone(host_out, px)) {
            if (mg->trace) {
                mg->us_total += us_since(t_call);
                if (++mg->traced % 256 == 0) {
                    const double n = 256.0;
                    fprintf(stderr, "[s3r multi] per frame: call %.0f us, pin+sentinels %.0f, tail %.0f |", mg->us_total / n, mg->us_pin / n, mg->us_tail / n);
                    for (size_t i = 0; i < mg->tr.size(); i++) {
                        MultiGpu::Trace &t = mg->tr[i];
                        fprintf(stderr, " gpu%zu: wake %.0f launch %.0f copies %.0f finish %.0f, band copies on the device clock", i, t.wake / n, t.launch / n, t.copies / n, t.finish / n);
                        for (int b = 0; b < 16 && t.end_us[b] > 0; b++) { fprintf(stderr, " [%.0f-%.0f]", t.begin_us[b] / n, t.end_us[b] / n); t.begin_us[b] = t.end_us[b] = 0; }
                        fprintf(stderr, " |");
                        t.wake = t.launch = t.copies = t.finish = 0;
                    }
                    fprintf(stderr, "\n");
                    mg->us_total = mg->us_pin = mg->us_tail = 0;
                }
            }
            return S3R_OK;
        }
        // the DMA went to pages the CPU no longer sees (a registration outlived its allocation): drop every pin, go again through staging
        mg->pins.clear();
        mg->pin = 0;
    }
    return S3R_OK;
}

std::vector<int> drop_in_devices() {   // S3R_DEVICES: "all" or a comma-separated list; empty = single-GPU drop-in
    std::vector<int> out;
    const char *env = getenv("S3R_DEVICES");
    if (!env || !*env) { return out; }
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess) { count = 0; }
    if (!strcmp(env, "all")) { for (int d = 0; d < count; d++) { out.push_back(d); } return out; }
    for (const char *p = env; *p;) {
        char *e = nullptr;
        const long d = strtol(p, &e, 10);
        if (e == p) { break; }
        if (d >= 0 && d < count) { out.push_back((int)d); }
        p = *e == ',' ? e + 1 : e;
    }
    return out;
}

void drop_in_initialize() {  // render.cpp:160-176 (data.bin next to this shared object)
    Dl_info info;
    char path[PATH_MAX + 64];
    path[0] = 0;
    if (dladdr(reinterpret_cast<const void *>(&updateAndRender), &info) && info.dli_fname) {
        strncpy(path, info.dli_fname, PATH_MAX);
        path[PATH_MAX] = 0;
    }
    char *slash = strrchr(path, '/');
    if (!slash) { strcpy(path, "./"); slash = path + 1; }
    const char *candidates[3] = {"/data.bin", "/Resources/data.bin", "/../data-generator/data.bin"};
    bool found = false;
    for (const char *c : candidates) {
        strcpy(slash, c);
        FILE *fp = fopen(path, "rb");
        if (fp) { fclose(fp); found = true; break; }
    }
    if (!found) { exit(666); }  // render.cpp:173
    std::vector<int> devices = drop_in_devices();
    if (devices.size() <= 1) {
        int device = devices.empty() ? 0 : devices[0];
        if (devices.empty()) { if (const char *env = getenv("S3R_DEVICE")) { device = atoi(env); } }
        if (s3r_create(&g_renderer, device) != S3R_OK) {
            fprintf(stderr, "render.so: %s\n", s3r_last_error());
            exit(70);
        }
        if (const char *env = getenv("S3R_PIN_HOST")) { g_renderer->opt_pin_host = atoi(env) != 0; }
        if (s3r_load_scene_file(g_renderer, path) != S3R_OK) {
            fprintf(stderr, "render.so: %s: %s\n", path, s3r_last_error());
            exit(70);
        }
    } else {
        MultiGpu *mg = new MultiGpu();
        mg->w.resize(devices.size());
        if (const char *env = getenv("S3R_PIN_HOST")) { mg->pin = atoi(env) != 0; }
        if (const char *env = getenv("S3R_MULTI_BANDS")) { mg->bands = std::max(1, std::min(atoi(env), 16)); }
        if (const char *env = getenv("S3R_MULTI_TRACE")) { mg->trace = atoi(env); }
        mg->tr.resize(devices.size());
        std::vector<std::thread> loaders;
        std::vector<int> rcs(devices.size(), 0);
        std::vector<std::string> errs(devices.size());
        for (size_t k = 0; k < devices.size(); k++) {   // every GPU holds the whole scene: load them side by side
            loaders.emplace_back([&, k] {
                rcs[k] = s3r_create(&mg->w[k].r, devices[k]);
                if (rcs[k] == S3R_OK) { rcs[k] = s3r_load_scene_file(mg->w[k].r, path); }
                if (rcs[k] != S3R_OK) { errs[k] = s3r_last_error(); }
            });
        }
        for (auto &t : loaders) { t.join(); }
        for (size_t k = 0; k < devices.size(); k++) {
            if (rcs[k] != S3R_OK) { fprintf(stderr, "render.so: device %d: %s\n", devices[k], errs[k].c_str()); exit(70); }
        }
        for (size_t k = 0; k < devices.size(); k++) { mg->w[k].th = std::thread(multi_worker, mg, (int)k); }
        g_multi = mg;
        g_renderer = mg->w[0].r;
    }
    s3r_camera_reset(&g_camera);
}
}  // namespace

// Harness-only: puts the drop-in's camera back to the reference's initial state (render.cpp:51-65) so a
// benchmark can replay the same Input script; the loaded scene and device buffers are kept.
extern "C" void s3r_dropin_reset(void) {
    s3r_camera_reset(&g_camera);
}

// Harness-only: drops every registration of caller memory the drop-in holds (a harness that frees its frame buffers and
// lets the allocator recycle their addresses must not leave them registered: the next registration of that range fails,
// and a DMA through the stale one would land in pages nobody sees).  The next call registers again.
extern "C" void s3r_dropin_release_pins(void) {
    if (g_multi) {
        cudaSetDevice(g_multi->w[0].r->device);
        g_multi->pins.clear();
    } else if (g_renderer) {
        cudaSetDevice(g_renderer->device);
        g_renderer->pins.clear();
    }
}

// Harness-only: how many GPUs the drop-in renders on (0 before the first updateAndRender call).
extern "C" int s3r_dropin_devices(void) {
    return g_multi ? (int)g_multi->w.size() : (g_renderer ? 1 : 0);
}

extern "C" __attribute__((visibility("default"))) void updateAndRender(const PixelData *pixel_data, const Input *input) {
    if (!g_renderer) { drop_in_initialize(); }
    S3RInput in{input->up, input->down, input->left, input->right, input->mouse[0], input->mouse[1]};
    s3r_camera_update(&g_camera, &in);  // the first call forces the matrix rebuild (render.cpp:267-270)
    // render.cpp:275-280: factor is refreshed only when width * height * 4 changes (hazard H8)
    const uint32_t depth_bytes = pixel_data->width * pixel_data->height * (uint32_t)sizeof(float);
    if (g_depth_bytes != depth_bytes) {
        g_depth_bytes = depth_bytes;
        g_renderer->factor_override = s3r_factor(pixel_data->height);
    }
    // render.cpp:281-282 clears bufferSize bytes; we write width * height pixels (== bufferSize / 4, main.swift:163)
    const int rc = g_multi ? multi_render(g_multi, g_camera.matrix, g_renderer->factor_override, pixel_data->width, pixel_data->height, pixel_data->buffer)
                           : s3r_render_host(g_renderer, g_camera.matrix, 1, pixel_data->width, pixel_data->height, 0, pixel_data->height, pixel_data->buffer);
    if (rc != S3R_OK) {
        fprintf(stderr, "render.so: %s\n", s3r_last_error());
        exit(70);
    }
}

// --------------------------------------------------------------------------------------------------
// Frame sink (SURVEY.md 8(f) row 4): consumes device-resident frames — the memory layout the reference's shell
// hands to CoreImage as .BGRA8 (main.swift:124-128: bytes B, G, R, 0) — without a synchronous trip through the
// caller's host buffer.  Two containers: raw BGR0 frames, or YUV4MPEG2 4:2:0 (any player / encoder reads it), with
// the colour conversion done on the GPU so that 1.5 instead of 4 bytes per pixel cross PCIe.  Submission is
// asynchronous: conversion kernel and device->host copy on the caller's stream into a ring of pinned buffers, a
// writer thread waits for each copy's event and appends the frame to the file.
// --------------------------------------------------------------------------------------------------
#include <condition_variable>
#include <deque>
#include <mutex>

namespace {

// BT.601 limited range, the usual integer form; chroma from the rounded mean of the 2x2 block (edge blocks repeat
// their last column / row).  One thread per 2x2 block.
__global__ void __launch_bounds__(256) bgr0_to_i420(const uint32_t *frame, uint32_t W, uint32_t H, uint8_t *yp, uint8_t *up, uint8_t *vp) {
    const uint32_t cw = (W + 1u) / 2u, ch = (H + 1u) / 2u;
    const uint32_t bx = blockIdx.x * 16u + (threadIdx.x & 15u), by = blockIdx.y * 16u + (threadIdx.x >> 4);
    if (bx >= cw || by >= ch) { return; }
    uint32_t sr = 0, sg = 0, sb = 0;
#pragma unroll
    for (uint32_t k = 0; k < 4u; k++) {
        const uint32_t x = min(2u * bx + (k & 1u), W - 1u), y = min(2u * by + (k >> 1), H - 1u);
        const uint32_t p = frame[(size_t)y * W + x], r = (p >> 16) & 255u, g = (p >> 8) & 255u, b = p & 255u;
        sr += r; sg += g; sb += b;
        if (2u * bx + (k & 1u) < W && 2u * by + (k >> 1) < H) {
            yp[(size_t)y * W + x] = (uint8_t)(((66u * r + 129u * g + 25u * b + 128u) >> 8) + 16u);
        }
    }
    const int r = (int)((sr + 2u) >> 2), g = (int)((sg + 2u) >> 2), b = (int)((sb + 2u) >> 2);
    up[(size_t)by * cw + bx] = (uint8_t)(((-38 * r - 74 * g + 112 * b + 128) >> 8) + 128);
    vp[(size_t)by * cw + bx] = (uint8_t)(((112 * r - 94 * g - 18 * b + 128) >> 8) + 128);
}

}  // namespace

struct S3RSink {
    static const int RING = 4;
    int device = 0, format = 0;
    cudaStream_t default_stream = nullptr;   // the renderer's own stream (what s3r_render_device uses for stream = null)
    uint32_t W = 0, H = 0;
    size_t frame_bytes = 0;
    FILE *file = nullptr;
    uint8_t *dev_yuv = nullptr;          // format 1: conversion target (one frame; the copy that follows is stream-ordered)
    uint8_t *host[RING] = {};
    cudaEvent_t copied[RING] = {};
    bool busy[RING] = {};
    uint64_t submitted = 0, written = 0;
    bool closing = false, io_error = false;
    std::deque<int> jobs;
    std::mutex mu;
    std::condition_variable cv;
    std::thread writer;
};

static void sink_writer(S3RSink *k) {
    cudaSetDevice(k->device);
    while (true) {
        int slot;
        {
            std::unique_lock<std::mutex> lock(k->mu);
            k->cv.wait(lock, [&] { return !k->jobs.empty() || k->closing; });
            if (k->jobs.empty()) { return; }
            slot = k->jobs.front();
            k->jobs.pop_front();
        }
        const bool ok = cudaEventSynchronize(k->copied[slot]) == cudaSuccess &&
                        (k->format == 0 || fwrite("FRAME\n", 1, 6, k->file) == 6) &&
                        fwrite(k->host[slot], 1, k->frame_bytes, k->file) == k->frame_bytes;
        {
            std::lock_guard<std::mutex> lock(k->mu);
            if (ok) { k->written++; } else { k->io_error = true; }
            k->busy[slot] = false;
        }
        k->cv.notify_all();
    }
}

static void sink_free(S3RSink *k) {   // everything but the writer thread
    if (k->file) { fclose(k->file); }
    for (int i = 0; i < S3RSink::RING; i++) {
        if (k->host[i]) { cudaFreeHost(k->host[i]); }
        if (k->copied[i]) { cudaEventDestroy(k->copied[i]); }
    }
    if (k->dev_yuv) { cudaFree(k->dev_yuv); }
    delete k;
}

extern "C" int s3r_sink_open(S3RRenderer *r, const char *path, uint32_t width, uint32_t height, uint32_t fps_num,
                             uint32_t fps_den, int format, S3RSink **out) {
    if (!r || !path || !out) { return fail(S3R_E_ARG, "null argument"); }
    if (width == 0 || height == 0 || width > 65535 || height > 65535 || fps_num == 0 || fps_den == 0 || format < 0 || format > 1) {
        return fail(S3R_E_ARG, "bad sink geometry, rate or format");
    }
    CUDA_TRY(cudaSetDevice(r->device));
    S3RSink *k = new S3RSink();
    k->device = r->device; k->format = format; k->W = width; k->H = height; k->default_stream = r->stream;
    const size_t cw = (width + 1u) / 2u, ch = (height + 1u) / 2u;
    k->frame_bytes = format == 0 ? (size_t)width * height * 4u : (size_t)width * height + 2u * cw * ch;
    k->file = fopen(path, "wb");
    if (!k->file) { sink_free(k); return fail(S3R_E_IO, std::string("cannot create ") + path); }
    if (format == 1) {
        fprintf(k->file, "YUV4MPEG2 W%u H%u F%u:%u Ip A1:1 C420jpeg XCOLORRANGE=LIMITED\n", width, height, fps_num, fps_den);
        if (cudaMalloc(&k->dev_yuv, k->frame_bytes) != cudaSuccess) { sink_free(k); return fail(S3R_E_CUDA, "sink: cudaMalloc"); }
    }
    for (int i = 0; i < S3RSink::RING; i++) {
        if (cudaMallocHost(reinterpret_cast<void **>(&k->host[i]), k->frame_bytes) != cudaSuccess ||
            cudaEventCreateWithFlags(&k->copied[i], cudaEventDisableTiming) != cudaSuccess) {
            sink_free(k);
            return fail(S3R_E_CUDA, "sink: pinned ring allocation failed");
        }
    }
    k->writer = std::thread(sink_writer, k);
    *out = k;
    return S3R_OK;
}

extern "C" int s3r_sink_submit(S3RSink *k, const uint32_t *dev_frame, void *stream) {
    if (!k || !dev_frame) { return fail(S3R_E_ARG, "null argument"); }
    CUDA_TRY(cudaSetDevice(k->device));
    cudaStream_t s = stream ? static_cast<cudaStream_t>(stream) : k->default_stream;
    const int slot = (int)(k->submitted % S3RSink::RING);
    {
        std::unique_lock<std::mutex> lock(k->mu);   // back-pressure: at most RING frames between the GPU and the file
        k->cv.wait(lock, [&] { return !k->busy[slot]; });
        if (k->io_error) { return fail(S3R_E_IO, "sink: write failed"); }
        k->busy[slot] = true;
    }
    cudaError_t ce = cudaSuccess;
    if (k->format == 1) {
        const size_t cw = (k->W + 1u) / 2u, ch = (k->H + 1u) / 2u;
        uint8_t *yp = k->dev_yuv, *up = yp + (size_t)k->W * k->H, *vp = up + cw * ch;
        bgr0_to_i420<<<dim3((unsigned)((cw + 15u) / 16u), (unsigned)((ch + 15u) / 16u)), 256, 0, s>>>(dev_frame, k->W, k->H, yp, up, vp);
        ce = cudaGetLastError();
        if (ce == cudaSuccess) { ce = cudaMemcpyAsync(k->host[slot], k->dev_yuv, k->frame_bytes, cudaMemcpyDeviceToHost, s); }
    } else {
        ce = cudaMemcpyAsync(k->host[slot], dev_frame, k->frame_bytes, cudaMemcpyDeviceToHost, s);
    }
    if (ce == cudaSuccess) { ce = cudaEventRecord(k->copied[slot], s); }
    if (ce != cudaSuccess) {   // nothing was queued for the writer: give the ring slot back, or the next submit on it waits forever
        {
            std::lock_guard<std::mutex> lock(k->mu);
            k->busy[slot] = false;
        }
        k->cv.notify_all();
        return fail(S3R_E_CUDA, std::string("sink submit: ") + cudaGetErrorString(ce));
    }
    k->submitted++;
    {
        std::lock_guard<std::mutex> lock(k->mu);
        k->jobs.push_back(slot);
    }
    k->cv.notify_all();
    return S3R_OK;
}

extern "C" int s3r_sink_close(S3RSink *k, uint64_t *frames_written) {
    if (!k) { return fail(S3R_E_ARG, "sink is null"); }
    {
        std::lock_guard<std::mutex> lock(k->mu);
        k->closing = true;
    }
    k->cv.notify_all();
    if (k->writer.joinable()) { k->writer.join(); }   // drains the queue first
    cudaSetDevice(k->device);
    const bool bad = k->io_error || fflush(k->file) != 0;
    if (frames_written) { *frames_written = k->written; }
    sink_free(k);
    return bad ? fail(S3R_E_IO, "sink: write failed") : S3R_OK;
}
