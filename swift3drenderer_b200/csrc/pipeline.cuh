// pipeline.cuh — device-side data layout and kernel parameter block of the B200 renderer.
//
// HBM layout (all arrays 256-byte aligned cudaMalloc blocks):
//
//   scene (converted once from data.bin's AoS records; contents rewritten in place by the s3r_update_* calls, counts fixed)
//     pos_x/pos_y/pos_z   float[Vpad]        planar positions, streamed as float4 by the vertex stage
//     vi0/vi1/vi2         uint32[T]          planar vertex-index streams (corner 0/1/2 of triangle t)
//     ai0/ai1/ai2         uint32[T]          planar attribute-index streams
//     attr                uint4[2*A]         per attribute: {nx, ny, nz, kind} , {payload words 0..3}
//                                            (32-byte AoS on purpose: attributes are *gathered*)
//     texels              uint32[nTex<<18]   512x512 rip-map atlases, 0x00RRGGBB
//
//   per view (frame scratch, strided by view)
//     rv                  float4[Vpad]       raster-space vertices (x, y, z, -) from the vertex stage
//     vis / shade         64 B + 128 B per *recorded* surviving triangle (compacted): clipped, spawned or larger than
//                         16 x 16 pixels.  Small unclipped survivors never get a record (visibility-buffer path).
//     keys                u64[pixels]        general path: depth << 32 | ~order per pixel (atomicMax); zero = background
//     tile_count, entries (u32 survivor slots, tile_cap per tile, unordered), big_list, counters
//
// Screen tiles are TILE_W x TILE_H pixels, aligned to the full frame's origin (so a band-partitioned
// render bins and rasterises exactly the tiles the whole-frame render would).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace s3r {

#ifndef S3R_TILE_W
#define S3R_TILE_W 64
#define S3R_TILE_H 32
#endif
constexpr int TILE_W = S3R_TILE_W;
constexpr int TILE_H = S3R_TILE_H;
constexpr int RASTER_THREADS = 256;         // (TILE_W / SEG) * TILE_H
constexpr int SEG = 8;                      // pixels per thread in the visibility pass
constexpr int SEGS_PER_ROW = TILE_W / SEG;
static_assert(SEGS_PER_ROW * TILE_H == RASTER_THREADS, "one thread per 8-pixel segment");
constexpr int BATCH = 8;                    // triangles staged per visibility batch
#ifndef S3R_SORT_CAP
#define S3R_SORT_CAP 3840
#endif
#ifndef S3R_RASTER_CTAS
#define S3R_RASTER_CTAS 4
#endif
constexpr int SORT_CAP = S3R_SORT_CAP;      // survivors a small scene may have (in-kernel per-tile collection)
constexpr int RASTER_CTAS = S3R_RASTER_CTAS; // tile_raster CTAs per SM the launch bounds ask for
constexpr uint32_t BIG_TILES = 16;          // triangles over more tiles are binned cooperatively
constexpr uint32_t NO_TRI = 0xFFFFFFFFu;
constexpr int MAX_PEERS = 16;              // destinations of the fused frame assembly (ranks of one NVSwitch domain)
constexpr uint32_t RASTER_CHUNK = 64;       // bin-list entries one tile-kernel work item resolves (general path)
constexpr uint32_t SPAN_MAX = 8;            // small scenes: survivors whose tile-column checkpoints are walked once per frame (span_walk)
constexpr uint32_t SPAN_MIN = 128;          // ... those whose box is at least this wide or high

constexpr float kNear = 0.1f;                   // render-cpp/render.cpp:89
constexpr float kScale = 0x1.0a2c9ap-5f;        // near * tanf(fov / 2), render.cpp:92 (binary32 value of the reference build)
constexpr uint32_t kBackground = 0x001E1E1Eu;   // RGB(30, 30, 30), render.cpp:96

enum Counter : uint32_t {
    C_SETUPS = 0, C_ENTRIES = 1, C_BIG = 2, C_OVERFLOW = 3, C_NEAR = 4, C_CLIPPED = 5, C_SPAWNED = 6, C_CULLED = 7, C_WORK = 8,
    C_ITEMS = 11,    // (tile, chunk) items in the tile kernel's work queue (general path)
    C_QHEAD = 12,    // ... and how many of them have been taken
    C_DONE = 10,     // CTAs of post_setup that have finished (the last one closes the frame's geometry)
    C_DIRECT = 9,    // small unclipped survivors walked straight from the classify kernel (no setup record)
    C_ROWTAB = 15,   // general path: floats of row-start tables allocated so far (post_setup)
    C_FLATQ = 14,    // general path: rounds of the flat walk handed out so far (post_setup)
    C_SPANS = 13,    // small scenes: survivors with a checkpoint table this frame (<= SPAN_MAX)
    C_WALKQ = 18,    // cluster front: candidates queued for the direct-walk kernel
    C_WALKHEAD = 19, // ... and how many rounds of 256 the walk kernel's persistent CTAs have taken
    C_CLUSTERS = 20, // cluster front: clusters that survived the cluster-level rejection (cluster_cull)
    C_COUNT = 24
};

struct __align__(16) SetupVis {     // 64 bytes: everything the coverage/depth walk needs
    uint16_t xmin, xmax, ymin, ymax;
    uint32_t order;
    uint32_t kind;
    float wstart[3];
    float dx[3];
    float dy[3];
    float rvz[3];
};
static_assert(sizeof(SetupVis) == 64, "SetupVis must be 64 bytes");

struct __align__(16) SetupShade {   // 128 bytes: everything shading needs
    float cv[9];    // camera-space corners / z        (render.cpp:337)
    float n[9];     // camera-space normals / z        (render.cpp:338)
    float pay[9];   // colour: rgb/z per corner;  texture: (u/z, v/z) per corner in [0..5], dz in [6..7]
    float tpp[2];   // texture only                    (render.cpp:350-352)
    uint32_t kind;
    uint32_t texture;
    float area;     // diagnostic (dumped to tests)
};
static_assert(sizeof(SetupShade) == 128, "SetupShade must be 128 bytes");

struct WalkRecord;

struct Frame {
    // scene
    const float *pos_x, *pos_y, *pos_z;
    const uint32_t *vi0, *vi1, *vi2, *ai0, *ai1, *ai2;
    const uint4 *attr;
    const uint32_t *texels;
    uint32_t V, Vpad, T, A, n_tex;
    // spatial pre-partition of the triangle stream (cluster.hpp); cl_hdr == null: the unclustered front (vertex_stage +
    // triangle_classify) runs instead
    const uint4 *cl_hdr;          // 2 x uint4 per cluster, n_clusters + 1 (sentinel)
    const float *cl_px, *cl_py, *cl_pz;
    const uint32_t *cl_tri;
    uint4 *cluster_list;          // [views][list_cap] clusters that survived cluster_cull: {v_off, tri_off, t0, n_verts | n_tris << 16}; zeros = empty slot
    uint32_t list_cap;            // n_clusters + room for every CTA's partly used last chunk
    uint32_t n_clusters;
    struct WalkRecord *walk_q;    // [views][walk_cap] candidates of the direct walk (front kernel -> walk kernel)
    uint32_t walk_cap;
    int cluster_cull;             // 0: every cluster is processed per triangle (A/B and tests)
    // views
    const float *cams;  // n_views x 12
    float cam0[12];     // the matrix itself when the submission has one view (cam_inline): nothing is uploaded
    int cam_inline;
    uint32_t n_views;
    uint32_t W, H, y0, y1;
    float fw, fh, half_w, half_h, factor;
    float band_lo, band_hi;   // (float)y0, (float)y1: early band reject in the classify pass
    uint32_t tiles_x, tile_row0, tiles_y, n_tiles;   // tiles_y: tile rows this submission owns
    uint32_t row_stride, row_phase;                  // tile-row ownership: a % row_stride == row_phase (1, 0 = contiguous band)
    uint32_t rs_magic;                               // floor(2^32 / row_stride) + 1: a / row_stride == umulhi(a, rs_magic) for a * row_stride < 2^32
    uint32_t raster_row0, raster_rows;   // tile rows [raster_row0, raster_row0 + raster_rows) of the band go in one raster launch
    // per-view scratch
    float4 *rv;           // null on the cluster path: raster-space vertices live in shared memory only
    SetupVis *vis;
    SetupShade *shade;
    uint32_t *slot_of;    // [views][2T] order key -> survivor slot (written for recorded survivors only)
    uint4 *head;          // per survivor: {xmin | xmax << 16, ymin | ymax << 16, order, kind}
    uint32_t *worklist;   // [views][T] classify -> setup work items
    uint32_t setup_cap;
    uint32_t *counters;
    uint32_t *sticky;   // [8] across chunks: overflow bits (OR), max setups, max entries, max big, max walk-queue length
    uint32_t *tile_count;       // [views][tile_stride] entries binned per tile this frame
    uint32_t tile_stride;
    uint32_t *entries;          // per-tile lists of survivor slots (unordered)
    uint32_t tile_cap;          // capacity of every tile's list
    uint32_t *big_list;
    uint32_t big_cap;
    // general path: per-pixel depth keys (depth << 32 | ~order); the tile kernel's work queue.
    // Key layout (key_at in kernels.cu): the keys of 4 vertically adjacent pixels — output rows 4g .. 4g + 3 of one column —
    // share one 32-byte sector.  The L2 reduction path works per (instruction, sector), not per lane
    // (tools/probes/red_sector_probe.cu: 191 G reductions/s with one lane per sector, 381 G with two, 468 G with four),
    // and the walks' neighbouring lanes are neighbouring rows of one triangle at the same x.
    unsigned long long *keys;
    unsigned long long key_view_stride;   // keys per view: W * (output rows rounded up to 4)
    unsigned long long *pstate;   // [pixels][3] {slot << 32 | weight bits}: exact weights of the tile kernel's best candidate, each word tagged
    uint2 *raster_items;   // [views][items_cap] {tile, first entry of the chunk}
    uint32_t items_cap;
    // output
    // fused frame assembly (multi-GPU, general path): every owned pixel row is stored straight into the full-size
    // frames of all ranks (own HBM + NVLink peer memory) at its absolute position; `out` is not written then
    uint32_t *peer_out[MAX_PEERS];
    uint32_t n_peers;
    uint32_t *out;
    unsigned long long out_view_stride;  // output pixels per view
    unsigned long long pix_view_stride;  // pixels per view of the frame as rendered (pstate); equals out_view_stride unless ss_log2 > 0
    // supersampling: the frame above (W x H, rows [y0, y1)) is rendered with k x k samples per output pixel, k = 1 << ss_log2
    // (0, 1, 2), and every k x k block is box-resolved in the write-out: `out` holds (W >> ss_log2) x ((y1 - y0) >> ss_log2)
    // pixels per view.  W, H, y0 and y1 are multiples of k; row_stride == 1 and no peer frames when ss_log2 > 0.
    uint32_t ss_log2;
    int use_tma;
    uint32_t flat_max;  // recorded triangles under flat_max x flat_max pixels are walked flat (post_setup), larger ones by tiles
    int direct_small;   // 1 (general path): small unclipped survivors are walked by the classify kernel and shaded from the raw scene
    int direct_bin;     // 1: no bin arrays — every raster CTA collects its triangles from the setup list itself
    int out_packed24;   // 1: `out` is a byte buffer with 3 bytes per pixel (B, G, R), used for host transport
    // small scenes, whole-frame launches: exact weights of the largest survivors at the first walked pixel of every
    // (tile column, pixel row), written once per frame by span_walk and read by every tile's stage A
    float *coltab;          // [views][SPAN_MAX][tiles_x][3][span_h], null = every tile takes the exact jump itself
    uint32_t *span_slots;   // [views][SPAN_MAX] survivor slots that have a table (counters[C_SPANS] of them)
    uint32_t span_h;        // H rounded up to a multiple of 32
    // general path: row-start weights (render.cpp:378-379) of the tile-path triangles, walked once per frame by
    // post_setup; the tile kernel's stage A then needs only the jump along the row
    float *rowtab;          // [views][rowtab_cap]: per triangle a block [component][box row]
    uint32_t *rowbase;      // [views][setup_cap] block offset per survivor slot, NO_TRI = none (flat-walked, or the table was full)
    uint32_t rowtab_cap;
    // tile_raster write-out as ONE 3-D TMA tensor store per tile (box (64 x 32) >> ss_log2 x 1 of {x, output row, view}; rows
    // and columns outside the output are clipped by the hardware) instead of one bulk copy per row
    int use_tmap;
    CUtensorMap out_map;    // 64-byte aligned member of a __grid_constant__ parameter
    // visibility planes (s3r_render_device_visibility: row_stride == 1, ss_log2 == 0, no peer frames), laid out like `out`:
    // per pixel the scene index of the winning triangle (a triangle the near-plane clip appended reports its parent;
    // NO_TRI = background) and its interpolated 1/z (+0 = background).  Null = not requested.  Only the PLANES
    // instantiations of tile_raster and shade_tiles read these; with a plane set, out == null means visibility only:
    // nothing is shaded and no colour is written.
    uint32_t *tri_out;
    float *depth_out;
};

// Scene update (s3r_update_vertices): where new positions go and the cluster arrays the refit rewrites in place.
struct SceneUpdate {
    float *pos_x, *pos_y, *pos_z;
    uint4 *cl_hdr;                // n_clusters + 1 headers (2 x uint4 each); the refit rewrites {cx, cy, cz, radius, max_edge}
    float *cl_px, *cl_py, *cl_pz;
    const uint32_t *cl_tri;
    const uint32_t *cl_src;       // per cluster vertex: the original vertex index it copies
    uint32_t n_clusters;
};

// Launchers (kernels.cu).  Each returns the number of kernels it enqueued.  `marks` (optional): called after every kernel
// launch with the kernel's name — the host layer records a timing event there (option "timing").
struct LaunchMarks { void (*fn)(void *ctx, const char *kernel); void *ctx; };
int launch_geometry(const Frame &f, cudaStream_t s, const LaunchMarks *marks = nullptr);   // vertex stage, classify + direct walk, clip/setup, binning + flat walk
int launch_raster(const Frame &f, cudaStream_t s, const LaunchMarks *marks = nullptr);     // per-tile visibility + shading + write-out
int launch_geometry_small(const Frame &f, cudaStream_t s, const LaunchMarks *marks = nullptr);  // single-CTA-per-view fused geometry (+ span_walk when f.coltab is set)
void launch_vertex_stage(const Frame &f, cudaStream_t s);   // vertex stage alone into f.rv (raster-vertex dumps)
// positions xyz (count x 3 packed, device-readable) -> pos[first ..], then every cluster refit (plain launches)
int launch_scene_update(const SceneUpdate &u, const float *xyz, uint32_t first, uint32_t count, cudaStream_t s);
cudaError_t configure_kernels();
void launch_exact_math(uint32_t mode, unsigned long long lo, unsigned long long count, uint32_t seed, unsigned long long *result,
                       cudaStream_t st);
void launch_walk_jump(const float *s, const float *d, const uint32_t *n, float *out, uint32_t count, cudaStream_t st);

}  // namespace s3r
