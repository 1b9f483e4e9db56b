/*
 * include/s3r_b200.h — additional C-ABI entry points of the B200 renderer library.
 *
 * None of these exist in the reference (its only export is updateAndRender, include/render.h);
 * SURVEY.md section 8(b) allows a replacement to add entry points the Swift loop never calls as long as
 * updateAndRender's behaviour is unchanged.  They expose what the reference keeps in process
 * statics (render-cpp/render.cpp:51-113) as explicit objects, so that a harness can (a) load a
 * scene from an explicit path or from arrays, (b) step the camera on the host
 * (update_camera, render.cpp:134-156) and render explicit camera matrices, (c) keep frames
 * device-resident, (d) render many views per call (frame-parallel batches), and (e) render only a
 * screen-space band [y0, y1) of the frame (multi-GPU partition).
 *
 * Plain pointers and sizes only.  Every function returns 0 on success or a negative S3R_E_* code;
 * s3r_last_error() gives the text.  There is no CPU fallback: without a CUDA device every
 * rendering entry point fails.
 */
#ifndef S3R_B200_H
#define S3R_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define S3R_API __attribute__((visibility("default")))

#define S3R_OK 0
#define S3R_E_CUDA -1       /* CUDA runtime error (no device, launch failure, ...) */
#define S3R_E_IO -2         /* data.bin missing / unreadable */
#define S3R_E_SCENE -3      /* scene violates the format contract (w != 1, bad index, kind > 1, ...) */
#define S3R_E_ARG -4        /* invalid argument */
#define S3R_E_NOSCENE -5    /* no scene loaded */

typedef struct S3RRenderer S3RRenderer;

typedef struct {            /* same 24-byte layout as Input (render-cpp/render.hpp:15-21) */
    float up, down, left, right, mouse_x, mouse_y;
} S3RInput;

typedef struct {            /* the reference's `state` static, render-cpp/render.cpp:51-65 */
    float position[3];
    float axis_x[3], axis_y[3], axis_z[3];
    float matrix[12];       /* rows (axis, -axis . position), row-major 3x4 */
    float mouse[2];
    int32_t started;        /* 0 until the first update (which forces the matrix rebuild, :267-270) */
} S3RCamera;

typedef struct {            /* per-view pipeline counters of the last completed render */
    uint32_t triangles_in;
    uint32_t near_rejected;     /* max z <= near                        (render.cpp:306) */
    uint32_t clipped;           /* straddled the near plane             (render.cpp:308-310) */
    uint32_t spawned;           /* second triangle appended by clip()   (render.cpp:239-257) */
    uint32_t culled;            /* off-screen bbox or area < 10         (render.cpp:311-317) */
    uint32_t setups;            /* triangles handed to the rasteriser */
    uint32_t bin_entries;       /* (triangle, tile) pairs */
    uint32_t big_triangles;     /* binned cooperatively (more than S3R_BIG_TILES tiles) */
    uint32_t overflow;          /* bit0 setup capacity, bit1 bin capacity, bit2 big-list capacity (auto-regrown) */
    uint32_t reserved[7];
} S3RStats;

/* One surviving triangle as the rasteriser sees it; field-compatible with the oracle's dump. */
typedef struct {
    uint32_t order;             /* processing order key: index, or T + parent index for appended */
    uint32_t xmin, xmax, ymin, ymax;
    float area;
    float wstart[3], dx[3], dy[3], rvz[3];
    float cv[3][3], n[3][3];
    uint32_t kind, texture;
    float payload[3][3];
    float dz[2], tpp[2];
} S3RSetupDump;

/* ---- lifetime ---------------------------------------------------------------------------- */
S3R_API int s3r_create(S3RRenderer **out, int device);
S3R_API void s3r_destroy(S3RRenderer *r);
S3R_API const char *s3r_last_error(void);

/* ---- scene (data.bin: data-generator/main.swift:381-416, render-cpp/render.cpp:177-209) --- */
S3R_API int s3r_load_scene_file(S3RRenderer *r, const char *data_bin_path);
S3R_API int s3r_load_scene_arrays(S3RRenderer *r, const float *vertices_xyzw, uint64_t vertex_count,
                          const uint64_t *vertex_indices, const uint64_t *attribute_indices, uint64_t index_count,
                          const void *attributes_48b, uint64_t attribute_count, const uint32_t *texels,
                          uint64_t texel_count);
S3R_API int s3r_scene_counts(const S3RRenderer *r, uint64_t *vertices, uint64_t *indices, uint64_t *attributes,
                     uint64_t *texels);

/* ---- scene updates: new contents for the loaded scene, in place (animation) ---------------------
 * Counts, both index streams and the number of atlases are fixed at load: an update overwrites contents and never
 * reallocates the scene or the frame scratch (new geometry that needs more room takes the usual path: s3r_finish
 * returns 1, render again).
 *   s3r_update_vertices   positions of vertices [first, first + count): xyz holds count x 3 binary32, tightly packed
 *                         (w stays 1; non-finite values are accepted, as at load).  source_on_device = 0: host memory,
 *                         the call returns once the data has left the caller's buffer; 1: device memory of the renderer's
 *                         device, read by the enqueued work — keep it unchanged until that work has run.  Every cluster
 *                         of the load-time partition gets its private vertex copies gathered again and its bounds refit
 *                         by the load-time rule (membership and order stay).  Enqueues 2 kernels (1 for a scene without
 *                         triangles).
 *   s3r_update_attributes records [first, first + count): 48-byte records as in data.bin, from host memory only,
 *                         checked by the load rules (normal w == 0, kind <= 1, texture index < atlas count); a violation
 *                         returns S3R_E_SCENE.  A copy, no kernel.
 *   s3r_update_texels     atlases [first_atlas, first_atlas + atlases): atlases x 2^18 words, host or device memory
 *                         (source_on_device as above; host data has left the caller's buffer on return).  A copy.
 * Ordering: an update is enqueued on `stream` (a cudaStream_t, NULL = the renderer's own stream, the one s3r_render_host
 * uses).  Work enqueued on that stream before the update renders the old scene, work enqueued after it the new one;
 * across streams the caller orders, as for s3r_render_device.  s3r_dump_raster_vertices recomputes from the current
 * positions on the cluster path, so after an update it may describe the updated scene.
 * Errors (nothing is written): count = 0 is a no-op that enqueues nothing; a range past the scene, a null source with
 * count > 0, a flag other than 0 / 1 or a source that is not where the flag says (cudaPointerGetAttributes; managed
 * memory is neither) return S3R_E_ARG; no scene returns S3R_E_NOSCENE. */
S3R_API int s3r_update_vertices(S3RRenderer *r, uint64_t first, uint64_t count, const float *xyz,
                                int source_on_device, void *stream);
S3R_API int s3r_update_attributes(S3RRenderer *r, uint64_t first, uint64_t count, const void *records_48b, void *stream);
S3R_API int s3r_update_texels(S3RRenderer *r, uint32_t first_atlas, uint32_t atlases, const uint32_t *texels,
                              int source_on_device, void *stream);
/* Test hook: the device's cluster headers and cluster-private vertex copies as they are after all work enqueued so far,
 * laid out like s3r_debug_clusters' outputs (hdr_out: clusters + 1 records of 32 bytes, pos_out: three planes of v_cap
 * floats; each is filled when non-null and large enough).  counts_out = {clusters, cluster vertices, triangles}. */
S3R_API int s3r_dump_clusters(S3RRenderer *r, void *hdr_out, uint64_t hdr_cap, float *pos_out, uint64_t v_cap,
                              uint64_t counts_out[3]);

/* ---- camera on the host (update_camera, render-cpp/render.cpp:134-156) --------------------- */
S3R_API void s3r_camera_reset(S3RCamera *cam);
S3R_API void s3r_camera_update(S3RCamera *cam, const S3RInput *input);
S3R_API float s3r_factor(uint32_t height);   /* near * H / (2 * scale), render-cpp/render.cpp:279 */

/* ---- rendering ------------------------------------------------------------------------------
 * cameras: n_views x 12 floats (S3RCamera.matrix).  Rows [y0, y1) of each width x height frame are
 * produced (y0 = 0, y1 = height for a whole frame).  Output: n_views x (y1 - y0) x width uint32,
 * 0x00RRGGBB, tightly packed.
 *
 * s3r_render_device: dev_out is DEVICE memory; work is enqueued on `stream` (a cudaStream_t, NULL =
 *   the renderer's own stream) and NOT waited for.  Call s3r_finish before reading results; it
 *   returns 1 when an internal capacity overflowed (buffers have been regrown — render again).
 * s3r_render_host: host_out is HOST memory (pageable or pinned); synchronous, includes the
 *   device->host copy and any capacity retry.
 */
S3R_API int s3r_render_device(S3RRenderer *r, const float *cameras, uint32_t n_views, uint32_t width, uint32_t height,
                      uint32_t y0, uint32_t y1, uint32_t *dev_out, void *stream);
/* Supersampled anti-aliasing: k x k samples per output pixel, k = samples_per_axis in {1, 2, 4} (anything else, or
 * k * width or k * height over 65535, returns S3R_E_ARG).  width, height, y0, y1 and the output layout are in OUTPUT pixels,
 * exactly as for s3r_render_device / s3r_render_host; streams, view chunks, s3r_finish and capacity regrowth behave the same.
 * Definition: with F the frame s3r_render_device renders at k*width x k*height with the same camera (so s3r_factor(k*height),
 * half_w = k*width / 2, ... follow from that size), output pixel (x, y), channel c, is
 *     (sum over i, j < k of F[k*y + j][k*x + i].c  +  k*k / 2) >> log2(k*k)
 * — a box filter on the stored 8-bit values, rounding half up, no gamma conversion, top byte 0.  The band [y0, y1) renders
 * rows [k*y0, k*y1) of F.  Consequence: the k samples of an output pixel lie at offsets 0, 1/k, ..., (k-1)/k from its 1x
 * sample point, so the resolved image is shifted by (k-1)/(2k) pixel against the 1x frame (kept: a moved sample grid would
 * lose exact parity with the reference's frame).  The k x k samples are resolved on chip; only output pixels reach memory,
 * but visibility scratch is sized for F: at 3840 x 2160 with k = 4 the key plane is 1.06 GB and the tile kernel's weight
 * state 3.2 GB per view.  k = 1 is the plain call.  After a render with k > 1, s3r_get_stats, s3r_dump_setups and
 * s3r_dump_raster_vertices describe F.  Not available with peer frames set (S3R_E_ARG), nor for interleaved rows. */
S3R_API int s3r_render_device_ssaa(S3RRenderer *r, const float *cameras, uint32_t n_views, uint32_t width, uint32_t height,
                                   uint32_t y0, uint32_t y1, uint32_t samples_per_axis, uint32_t *dev_out, void *stream);
/* Visibility planes: which triangle each pixel shows and at what depth, for picking, depth compositing and deferred passes
 * driven by a triangle-ID buffer.  Everything works as in s3r_render_device (cameras, bands [y0, y1), view chunks, streams,
 * s3r_finish and its render-again contract, statistics and dumps).  Each non-null output is DEVICE memory with the colour
 * output's layout: n_views x (y1 - y0) x width, tightly packed.
 *   dev_triangle[p]: the scene triangle index t of the triangle that colours pixel p in the reference's frame; its corners
 *     are vertex_indices[3t .. 3t+2].  A triangle appended by the near-plane clip (render.cpp:239-257) reports the triangle
 *     it was cut from.  Background: 0xFFFFFFFF.
 *   dev_depth[p]: the reference's depth-buffer value at p (render.cpp:363-364), the binary32 interpolated 1/z
 *     (rvz0*w0 + rvz1*w1) + rvz2*w2 of that triangle; linear depth is 1 / dev_depth[p].  Background: +0.0f.
 *   dev_out: when non-null, the colour frame, bit-identical to s3r_render_device's.  When null, the call is a
 *     visibility-only render: nothing is shaded and no colour is written.
 * Any subset of the three outputs may be null, but not all three.  The planes cost two 4-byte stores per pixel and no
 * extra kernel launch.  S3R_E_ARG (nothing written): all three outputs null, peer frames set, or bad frame geometry as for
 * s3r_render_device.  Not available for host output, interleaved rows or supersampling. */
S3R_API int s3r_render_device_visibility(S3RRenderer *r, const float *cameras, uint32_t n_views, uint32_t width,
                                         uint32_t height, uint32_t y0, uint32_t y1, uint32_t *dev_out,
                                         uint32_t *dev_triangle, float *dev_depth, void *stream);
/* Interleaved partition for multi-GPU load balance: renders the tile rows a (s3r_tile_height() pixel rows
 * each, counted from the top of the frame) with a % row_stride == row_phase.  Output: those tile rows
 * compacted in order — ceil((ceil(H / th) - row_phase) / row_stride) * th rows of `width` uint32 per view
 * (rows beyond `height` in the last tile row are padding: untouched or background). */
S3R_API int s3r_render_device_rows(S3RRenderer *r, const float *cameras, uint32_t n_views, uint32_t width,
                                   uint32_t height, uint32_t row_stride, uint32_t row_phase, uint32_t *dev_out,
                                   void *stream);
S3R_API uint32_t s3r_tile_height(void);

/* ---- fused frame assembly over peer memory (multi-GPU screen partition) -----------------------
 * Replaces "render my rows, then all-gather" by "store my rows straight into every rank's frame":
 * the shading kernel writes each finished pixel row to its absolute position in up to 16 full-size
 * (n_views x height x width) destination frames — the rank's own and its NVLink peers'.  Frames are plain
 * device allocations shared through CUDA IPC:
 *   s3r_peer_frame_alloc   allocates `bytes` on the renderer's device, returns the pointer and a 64-byte
 *                          IPC handle to send to the other ranks (any transport);
 *   s3r_peer_frame_open    maps another process's allocation (peer access is enabled on demand);
 *   s3r_set_peer_frames    the destinations of the following s3r_render_device / _rows calls (n = 0
 *                          switches back to `dev_out`, which may be NULL while destinations are set).
 * The caller orders frames across ranks (a barrier / tiny all-reduce per frame, or a ring of frames).
 * General path only (scenes over 1920 triangles); other scenes return S3R_E_ARG while destinations are set. */
S3R_API int s3r_peer_frame_alloc(S3RRenderer *r, uint64_t bytes, void **dev_ptr, unsigned char ipc_handle_out[64]);
S3R_API int s3r_peer_frame_open(S3RRenderer *r, const unsigned char ipc_handle[64], void **dev_ptr);
S3R_API int s3r_peer_frame_release(S3RRenderer *r, void *dev_ptr);   /* frees (own) or unmaps (opened) */
S3R_API int s3r_set_peer_frames(S3RRenderer *r, void *const *dev_ptrs, uint32_t n);
S3R_API int s3r_copy_from_device(S3RRenderer *r, void *host_dst, const void *dev_src, uint64_t bytes);   /* test helper */
S3R_API int s3r_finish(S3RRenderer *r);
S3R_API int s3r_render_host(S3RRenderer *r, const float *cameras, uint32_t n_views, uint32_t width, uint32_t height,
                    uint32_t y0, uint32_t y1, uint32_t *host_out);
/* s3r_render_host with k x k supersampling: see s3r_render_device_ssaa. */
S3R_API int s3r_render_host_ssaa(S3RRenderer *r, const float *cameras, uint32_t n_views, uint32_t width, uint32_t height,
                                 uint32_t y0, uint32_t y1, uint32_t samples_per_axis, uint32_t *host_out);

/* ---- introspection (tests, bench) -------------------------------------------------------- */
/* statistics of view `view` (its index in the last call's batch, whatever views_per_chunk split it into) */
S3R_API int s3r_get_stats(S3RRenderer *r, uint32_t view, S3RStats *out);
/* raster-space vertices of the last render of `view` (V x 4 floats: x, y, z, unused), render.cpp:285-289.  This and
 * s3r_dump_setups keep only the views of the last chunk of a batch longer than views_per_chunk (S3R_E_ARG otherwise). */
S3R_API int s3r_dump_raster_vertices(S3RRenderer *r, uint32_t view, float *out_xyzw, uint64_t capacity_vertices);
/* surviving triangles of the last render of `view`, sorted by order key; *count receives the total */
S3R_API int s3r_dump_setups(S3RRenderer *r, uint32_t view, S3RSetupDump *out, uint64_t capacity, uint64_t *count);
S3R_API uint64_t s3r_kernel_launches(const S3RRenderer *r);   /* kernels launched by this renderer so far */
/* CUDA-event time accumulated per stage since the last reset (needs option "timing" = 1): the
 * geometry kernels (reset .. bin fill) and the tile rasteriser, measured on the launching stream;
 * *chunks = number of (multi-view) submissions covered. */
S3R_API int s3r_get_timing(S3RRenderer *r, double *geometry_ms, double *raster_ms, uint64_t *chunks, int reset);
/* Per-kernel CUDA-event time accumulated since the last reset (option "timing" = 1; reset through s3r_get_timing):
 * entry `index` = one kernel of the frame pipeline in launch order.  Returns 0 and fills *name (static string), *ms (sum
 * over the timed launches) and *launches; returns 1 when index is past the last kernel. */
S3R_API int s3r_get_kernel_timing(S3RRenderer *r, uint32_t index, const char **name, double *ms, uint64_t *launches);
S3R_API int s3r_set_option(S3RRenderer *r, const char *name, int64_t value);
/* options: "tma_store" (1 = cp.async.bulk tile write-out, default; 0 = plain stores),
 *          "pin_host" (1 = cudaHostRegister the caller's frame buffers; default 0 — only for callers that
 *                      keep the buffer mapped while they pass it; drop-in: env S3R_PIN_HOST=1),
 *          "views_per_chunk" (views per kernel launch set, 1..65535, default 256: a chunk's views are a grid dimension of
 *          its launches), "timing" (per-stage and per-kernel events, default 0
 *          = off; n > 1: on every n-th submission only),
 *          "fused_small" (1 = one fused geometry CTA per view for scenes of at most 1920 triangles, default),
 *          "direct_small" (general path: 1 = small unclipped survivors are walked by the classify kernel without a setup
 *          record, default; 0 = every survivor is recorded),
 *          "flat_max" (general path: recorded triangles whose box is under flat_max x flat_max pixels are walked flat, larger
 *          ones by tiles; 16 .. 65536, default 128),
 *          "tensor_store" (1 = tile_raster writes each tile with one TMA tensor store instead of 32 bulk row copies, default),
 *          "spans" (1 = small scenes, whole-frame launches: the row walks of the largest survivors are done once per
 *          frame by span_walk instead of by exact jumps in every tile, default),
 *          "pack24" (1 = 24-bit pixel transport over PCIe for host renders, default), "host_bands" (raster/
 *          copy pipeline depth of host renders, default 12), "copy_threads" (staging -> caller copy workers; default 0 =
 *          min(14, hardware threads - 2)),
 *          "setup_capacity" (test hook: shrink the survivor buffers to exercise regrowth),
 *          "rowtab_capacity" (test hook: cap the general path's row-start table at this many floats per view, 0 = empty —
 *          tile-path triangles that do not fit keep their exact jumps; < 0 = the default size),
 *          "clusters" (general path front: 1 = over the load-time clusters — batch / cluster rejection, per-warp vertex stage and
 *          front tests with raster-space vertices in shared memory only, direct walk from a candidate queue; 0 = vertex_stage +
 *          triangle_classify over the raw stream; 2 (default) = clusters for partitioned submissions — bands, interleaved rows —
 *          and the raw stream for whole frames),
 *          "cluster_cull" (1 = whole clusters are rejected by their bounds, default; 0 = every triangle is tested) */

/* Test hook: out[i] = the device build of walk_jump(start[i], delta[i], steps[i]) — the exact result of
 * steps[i] sequential binary32 additions (render-cpp/render.cpp:374-379).  Host arrays. */
S3R_API int s3r_debug_walk(S3RRenderer *r, const float *start, const float *delta, const uint32_t *steps,
                           float *out, uint32_t count);

/* Frame sink (SURVEY.md 8(f) row 4; replaces the reference shell's CoreImage -> Metal blit, main.swift:124-140, for
 * headless use): appends device-resident frames — 0x00RRGGBB words, i.e. bytes B, G, R, 0, the shell's .BGRA8 — to a
 * file without passing through a caller's host buffer.  format 0: raw BGR0 frames back to back; format 1: YUV4MPEG2
 * 4:2:0 (BT.601 limited range), converted on the GPU (1.5 bytes per pixel over PCIe).  s3r_sink_submit is asynchronous
 * and stream-ordered: enqueue it on the stream the frame was rendered on (null = the renderer's own stream, like
 * s3r_render_device); the frame may be overwritten by work enqueued after it.  At most four frames are in flight; s3r_sink_close drains them and reports how many reached the file. */
typedef struct S3RSink S3RSink;
S3R_API int s3r_sink_open(S3RRenderer *r, const char *path, uint32_t width, uint32_t height, uint32_t fps_num,
                          uint32_t fps_den, int format, S3RSink **out);
S3R_API int s3r_sink_submit(S3RSink *sink, const uint32_t *dev_frame, void *stream);
S3R_API int s3r_sink_close(S3RSink *sink, uint64_t *frames_written);

/* Test hook: compares the shading chain's hand-scheduled IEEE division / reciprocal square root (csrc/exact_math.cuh)
 * with the compiler's operators on the device.  mode 0: every binary32 bit pattern first .. first + count - 1 through
 * 1/sqrt; mode 1: `count` seeded pseudo-random operand sets through the divisions.  result[0] = mismatches,
 * result[1..4] = operands and values of the first one (bit patterns). */
S3R_API int s3r_debug_exact_math(S3RRenderer *r, uint32_t mode, uint64_t first, uint64_t count, uint32_t seed,
                                 uint64_t result[5]);

/* Test hook, callable without a GPU: the load-time spatial pre-partition of a triangle stream (csrc/cluster.hpp) — runs of
 * consecutive, spatially close triangles with a bounding sphere and their longest edge, in Morton order, which the general
 * path's front kernel rejects wholesale when they lie behind the near plane, off screen, outside the rows a GPU owns or
 * are too small to pass `area >= 10` (render-cpp/render.cpp:306-317).  counts_out = {clusters, cluster vertices, triangles};
 * hdr_out: (clusters + 1) x 32 bytes {cx, cy, cz, radius, max_edge, t0, v_off, tri_off}; pos_out: three planes of v_cap
 * floats; tri_out: one word per triangle (v0 | v1 << 8 | v2 << 16, cluster-local vertex numbers), room for index_count / 3. */
S3R_API int s3r_debug_clusters(const float *vertices_xyzw, uint64_t vertex_count, const uint64_t *vertex_indices,
                               uint64_t index_count, void *hdr_out, uint64_t hdr_cap, float *pos_out, uint64_t v_cap,
                               uint32_t *tri_out, uint64_t counts_out[3]);

/* Test hook, callable without a GPU: the tile-row band edges of a host render (s3r_render_host pipelines raster launches
 * with device-to-host copies band by band; the last band is tapered).  Returns the number of edges written (bands + 1),
 * edges_out needs room for 65. */
S3R_API int s3r_debug_band_edges(uint32_t tiles_y, int bands, int taper, uint32_t *edges_out, int capacity);

/* Harness-only: resets the camera owned by updateAndRender (include/render.h) to the reference's
 * initial state so that the same Input script can be replayed; scene and buffers stay loaded. */
S3R_API void s3r_dropin_reset(void);
/* Harness-only: the number of GPUs updateAndRender renders on (0 before its first call).  More than one when the
 * environment names several at the first call — S3R_DEVICES="0,1,2,3" or "all": the frame is then split by interleaved
 * tile rows, one host thread per GPU issues that GPU's launches, and every GPU copies its rows over its own PCIe link
 * straight into the caller's buffer (registered on first sight; S3R_PIN_HOST=0: through pinned staging).  The call stays
 * synchronous and its result bit-identical.  S3R_DEVICE=<k> selects the GPU of the single-GPU drop-in. */
S3R_API int s3r_dropin_devices(void);
/* Harness-only: unregisters every caller buffer the drop-in has registered with CUDA (call before freeing frame buffers
 * whose addresses the allocator may hand out again; the reference's main loop never frees its double buffer). */
S3R_API void s3r_dropin_release_pins(void);

#ifdef __cplusplus
}
#endif
#endif
