/*
 * camcal_b200.h -- C ABI of libcamcal_b200.so: the B200 (sm_100a) implementation of
 * the calibration-object evaluation path of yakir12/CameraCalibrations v0.7.3.
 *
 * The reference has no FFI of its own; its boundary is the Julia callable surface of
 * `Calibration` (src/meta.jl:82-103) and the bulk callers in
 * src/buildcalibrations.jl:28-67 and src/plot_calibration.jl:15-22,40.  Each entry
 * point below names the reference lines it replaces.  A Julia wrapper binds these
 * with `ccall` (see INTEGRATION.md and julia/CameraCalibrationsB200.jl); the Python
 * package cameracalibrations_b200 binds the same symbols with ctypes.
 *
 * Conventions
 *  - plain C types only; every function returns 0 (CC_OK) or a negative cc_status and
 *    never throws; cc_last_error_string() gives the text for the calling thread.
 *  - there is NO CPU fallback: without a CUDA device every compute entry point fails
 *    with CC_ERR_NO_DEVICE.
 *  - `*_f64` / `*_f32`, `rectify_*`, `reproj_*` take DEVICE pointers and are
 *    asynchronous on `stream` (a cudaStream_t passed as void*, NULL = default
 *    stream); `*_host` variants take HOST pointers, run a chunked
 *    H2D -> kernel -> D2H pipeline and return when the result is in host memory.
 *  - a cc_ctx belongs to one device and is not internally locked: use one context per
 *    host thread, or serialise the calls on it.  It owns the host pipeline's staging
 *    buffers, the cached rectification tile plans (the 8 most recent calibration /
 *    geometry sets) and the tile-scheduler counters; calls on different streams of the
 *    same context may overlap on the device.
 *  - rectification is out of place (src != dst).
 *  - point sets are SoA (one array per coordinate).  Pointers aligned to 16 bytes
 *    take the 128-bit vector path; unaligned pointers are accepted (scalar path).
 *  - frames are stored the way Julia stores `img[r, c]` (size (sz1, sz2)): pixel
 *    (r, c), 1-based, lives at  base + (c-1)*pitch + (r-1)  in PIXELS; the first
 *    RowCol component `r` is the contiguous axis (SURVEY.md F6).  Frame f of a batch
 *    starts frame_stride pixels after frame f-1.  u8c3 pixels are 3 interleaved
 *    bytes (RGB{N0f8}).
 *  - parameters are passed by value in host structs (cc_intr, cc_view); the library
 *    expands the rotation vector and the inverse maps once per call on the host,
 *    exactly what `Calibration(...)` / `img2obj` precompute (src/meta.jl:27-33,71-76).
 */
#ifndef CAMCAL_B200_H
#define CAMCAL_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CC_ABI_VERSION 1

typedef enum {
    CC_OK = 0,
    CC_ERR_INVALID_ARG = -1,  /* NULL pointer, non-positive size, bad flag          */
    CC_ERR_NO_DEVICE = -2,    /* no CUDA device / driver: there is no CPU fallback  */
    CC_ERR_CUDA = -3,         /* a CUDA runtime call failed (text in last error)    */
    CC_ERR_UNSUPPORTED = -4,  /* device is not sm_100                               */
    CC_ERR_NOMEM = -5
} cc_status;

/* Calibration.intrinsic (AffineMap diag + translation), Calibration.k and the
 * checker_size behind Calibration.scale -- src/meta.jl:17-25,
 * src/buildcalibrations.jl:1-6. */
typedef struct {
    double frow, fcol, crow, ccol, k, checker_size;
} cc_intr;

/* Calibration.extrinsics[i]: RotationVec + translation -- src/buildcalibrations.jl:3 */
typedef struct {
    double rvec[3], tvec[3];
} cc_view;

typedef struct cc_ctx cc_ctx; /* per-device scratch, staging buffers, streams */

/* coordinate arithmetic of the rectification map */
#define CC_COORD_F64 0u     /* reference precision: bit-exact index/weight selection  */
#define CC_COORD_F32 1u     /* fast path: map error bounded as for cc_rectify_map_f32  */
/* how source texels are fetched */
#define CC_GATHER_AUTO 0u   /* TMA-staged tiles when the frame layout allows, else direct */
#define CC_GATHER_DIRECT 16u
#define CC_GATHER_TMA 32u   /* fail with CC_ERR_INVALID_ARG if the layout cannot be staged */

int cc_abi_version(void);
const char *cc_last_error_string(void);
int cc_device_count(int *count);

int cc_ctx_create(int device, cc_ctx **out);
int cc_ctx_destroy(cc_ctx *ctx);
int cc_ctx_device(const cc_ctx *ctx, int *device);
int cc_ctx_synchronize(cc_ctx *ctx);
/* number of kernels this context has launched so far (bench.py's gpu_launches) */
int cc_ctx_launch_count(const cc_ctx *ctx, uint64_t *count);

/* pinned host memory for the *_host entry points (optional; pageable works, slower) */
int cc_host_alloc(void **ptr, size_t bytes);
int cc_host_free(void *ptr);
int cc_host_register(void *ptr, size_t bytes);
int cc_host_unregister(void *ptr);

/* ---- pixel -> world:  (c::Calibration)(i::RowCol, idx)  src/meta.jl:82, chain :31,
 *      inv_lens_distortion :50-57, get_inv_prespective_map :60-69, img2obj :71-76.
 *      z == NULL gives rectification(c, idx) = pop o image2real  (src/meta.jl:99-103).
 *      Bulk form of the broadcast c.(imgpoints, i), src/buildcalibrations.jl:46. */
int cc_img2world_f64(cc_ctx *ctx, const cc_intr *intr, const cc_view *view,
                     const double *row, const double *col, double *x, double *y,
                     double *z, size_t n, void *stream);
int cc_img2world_f32(cc_ctx *ctx, const cc_intr *intr, const cc_view *view,
                     const float *row, const float *col, float *x, float *y, float *z,
                     size_t n, void *stream);
int cc_img2world_f64_host(cc_ctx *ctx, const cc_intr *intr, const cc_view *view,
                          const double *row, const double *col, double *x, double *y,
                          double *z, size_t n);
int cc_img2world_f32_host(cc_ctx *ctx, const cc_intr *intr, const cc_view *view,
                          const float *row, const float *col, float *x, float *y,
                          float *z, size_t n);

/* ---- world -> pixel:  (c::Calibration)(xyz::XYZ, idx)  src/meta.jl:88, chain :29,
 *      lens_distortion :39-44.  z == NULL means z = 0 (points on the board plane).
 *      Bulk form of c.(objpoints, i), src/buildcalibrations.jl:29. */
int cc_world2img_f64(cc_ctx *ctx, const cc_intr *intr, const cc_view *view,
                     const double *x, const double *y, const double *z, double *row,
                     double *col, size_t n, void *stream);
int cc_world2img_f32(cc_ctx *ctx, const cc_intr *intr, const cc_view *view,
                     const float *x, const float *y, const float *z, float *row,
                     float *col, size_t n, void *stream);
int cc_world2img_f64_host(cc_ctx *ctx, const cc_intr *intr, const cc_view *view,
                          const double *x, const double *y, const double *z,
                          double *row, double *col, size_t n);
int cc_world2img_f32_host(cc_ctx *ctx, const cc_intr *intr, const cc_view *view,
                          const float *x, const float *y, const float *z, float *row,
                          float *col, size_t n);

/* ---- points of MANY views in one call: the broadcasts c.(pts_v, v) over the views of a calibration
 *      (src/buildcalibrations.jl:29,46; src/plot_calibration.jl:36-42).  Points
 *      [offsets[s], offsets[s+1]) use views[s].  offsets: HOST array of nviews + 1 entries,
 *      offsets[0] == 0, non-decreasing, n = offsets[nviews].  views: HOST array (a view may appear in
 *      several segments; empty segments are allowed).  Same arithmetic as the single-view entry
 *      points: every point's result is bit-identical to calling cc_img2world_* / cc_world2img_* with
 *      its own view.  z == NULL as there.  The device forms upload a per-segment table to the
 *      context (on `stream`) and make ONE launch whatever nviews is; the *_host forms upload it
 *      once and run the chunked pipeline.  n == 0: CC_OK, nothing launched. */
int cc_img2world_f64_views(cc_ctx *ctx, const cc_intr *intr, const cc_view *views, int nviews,
                           const size_t *offsets, const double *row, const double *col, double *x,
                           double *y, double *z, void *stream);
int cc_img2world_f32_views(cc_ctx *ctx, const cc_intr *intr, const cc_view *views, int nviews,
                           const size_t *offsets, const float *row, const float *col, float *x,
                           float *y, float *z, void *stream);
int cc_world2img_f64_views(cc_ctx *ctx, const cc_intr *intr, const cc_view *views, int nviews,
                           const size_t *offsets, const double *x, const double *y, const double *z,
                           double *row, double *col, void *stream);
int cc_world2img_f32_views(cc_ctx *ctx, const cc_intr *intr, const cc_view *views, int nviews,
                           const size_t *offsets, const float *x, const float *y, const float *z,
                           float *row, float *col, void *stream);
int cc_img2world_f64_views_host(cc_ctx *ctx, const cc_intr *intr, const cc_view *views, int nviews,
                                const size_t *offsets, const double *row, const double *col,
                                double *x, double *y, double *z);
int cc_img2world_f32_views_host(cc_ctx *ctx, const cc_intr *intr, const cc_view *views, int nviews,
                                const size_t *offsets, const float *row, const float *col, float *x,
                                float *y, float *z);
int cc_world2img_f64_views_host(cc_ctx *ctx, const cc_intr *intr, const cc_view *views, int nviews,
                                const size_t *offsets, const double *x, const double *y,
                                const double *z, double *row, double *col);
int cc_world2img_f32_views_host(cc_ctx *ctx, const cc_intr *intr, const cc_view *views, int nviews,
                                const size_t *offsets, const float *x, const float *y, const float *z,
                                float *row, float *col);

/* ---- interleaved points, the reference's own layout: Vector{RowCol} / Matrix{RowCol} (src/detect_fit.jl:19)
 *      and arrays of XYZ are (row, col) pairs and (x, y, z) triples in memory.
 *      rc: n x 2 interleaved (row, col).  img2world: out = n x out_dim interleaved, out_dim 3 gives
 *      (x, y, z) = c(::RowCol, i), out_dim 2 gives (x, y) = rectification(c, i) with z not computed.
 *      world2img: pts = n x in_dim interleaved, in_dim 3 is (x, y, z), in_dim 2 is (x, y) with z = 0.
 *      offsets == NULL: every point uses views[0] (nviews must be 1).  offsets != NULL: the segments of
 *      cc_*_views, and offsets[nviews] must equal n.  Every point's result is bit-identical to the SoA
 *      entry point with the same view.  16-byte aligned rc / out / pts take 128-bit accesses; any other
 *      base takes a scalar path with the same results.  Bad arguments (out_dim / in_dim not 2 or 3, a NULL
 *      point array with n > 0, offsets == NULL with nviews != 1, n != offsets[nviews], and what cc_*_views
 *      rejects) return CC_ERR_INVALID_ARG and write nothing.  n == 0: CC_OK, nothing launched.  The device
 *      forms make ONE launch on `stream`; the *_host forms run the chunked pipeline with one contiguous
 *      copy per direction and chunk. */
int cc_img2world_f64_aos(cc_ctx *ctx, const cc_intr *intr, const cc_view *views, int nviews,
                         const size_t *offsets, const double *rc, double *out, int out_dim,
                         size_t n, void *stream);
int cc_img2world_f32_aos(cc_ctx *ctx, const cc_intr *intr, const cc_view *views, int nviews,
                         const size_t *offsets, const float *rc, float *out, int out_dim,
                         size_t n, void *stream);
int cc_world2img_f64_aos(cc_ctx *ctx, const cc_intr *intr, const cc_view *views, int nviews,
                         const size_t *offsets, const double *pts, int in_dim, double *rc,
                         size_t n, void *stream);
int cc_world2img_f32_aos(cc_ctx *ctx, const cc_intr *intr, const cc_view *views, int nviews,
                         const size_t *offsets, const float *pts, int in_dim, float *rc,
                         size_t n, void *stream);
int cc_img2world_f64_aos_host(cc_ctx *ctx, const cc_intr *intr, const cc_view *views, int nviews,
                              const size_t *offsets, const double *rc, double *out, int out_dim,
                              size_t n);
int cc_img2world_f32_aos_host(cc_ctx *ctx, const cc_intr *intr, const cc_view *views, int nviews,
                              const size_t *offsets, const float *rc, float *out, int out_dim,
                              size_t n);
int cc_world2img_f64_aos_host(cc_ctx *ctx, const cc_intr *intr, const cc_view *views, int nviews,
                              const size_t *offsets, const double *pts, int in_dim, double *rc,
                              size_t n);
int cc_world2img_f32_aos_host(cc_ctx *ctx, const cc_intr *intr, const cc_view *views, int nviews,
                              const size_t *offsets, const float *pts, int in_dim, float *rc,
                              size_t n);

/* ---- full-frame rectification:  warp(img, tform, axs)  src/plot_calibration.jl:40
 *      with tform = real2image[i] o push(.,0) o inv(LinearMap(ratio*I)) (:17-18) and
 *      axs from get_axes (:1-6): output index (I1, I2) = axs_min + (a, b), same size
 *      as the input (cc_rectify_axes_* below: any output size).  Bilinear, OnGrid, out-of-range -> fill.  `ratio` is pixels per
 *      world unit (get_ratio, :8-13).  flags = CC_COORD_* | CC_GATHER_*.
 *      All `nframes` frames share the view: the map is computed once per tile and group of
 *      frames, so batches rectify faster per frame than single-frame calls.  The first call
 *      with a new (calibration, ratio, axs_min, frame geometry) builds the tile plan on the host
 *      and uploads it (one stream synchronisation); later calls with the same parameters are
 *      fully asynchronous. */
int cc_rectify_f32c1(cc_ctx *ctx, const cc_intr *intr, const cc_view *view, double ratio,
                     const int64_t axs_min[2], const float *src, float *dst, int sz1,
                     int sz2, size_t pitch, size_t frame_stride, int nframes, float fill,
                     unsigned flags, void *stream);
int cc_rectify_u8c3(cc_ctx *ctx, const cc_intr *intr, const cc_view *view, double ratio,
                    const int64_t axs_min[2], const uint8_t *src, uint8_t *dst, int sz1,
                    int sz2, size_t pitch, size_t frame_stride, int nframes,
                    const uint8_t fill[3], unsigned flags, void *stream);
int cc_rectify_f32c1_host(cc_ctx *ctx, const cc_intr *intr, const cc_view *view,
                          double ratio, const int64_t axs_min[2], const float *src,
                          float *dst, int sz1, int sz2, size_t pitch, size_t frame_stride,
                          int nframes, float fill, unsigned flags);
int cc_rectify_u8c3_host(cc_ctx *ctx, const cc_intr *intr, const cc_view *view,
                         double ratio, const int64_t axs_min[2], const uint8_t *src,
                         uint8_t *dst, int sz1, int sz2, size_t pitch,
                         size_t frame_stride, int nframes, const uint8_t fill[3],
                         unsigned flags);
/* Frames with DIFFERENT views in one call -- what the reference's plot does: every calibration
 * image is rectified with its own extrinsic, ratio and axes (src/plot_calibration.jl:36-42).
 * Frames [v * frames_per_view, (v+1) * frames_per_view) use views[v], ratios[v] and
 * axs_mins[2v], axs_mins[2v+1].  Device pointers, ordered on `stream`.  Groups of up to 64 views go
 * out as ONE launch each (view table in the kernel's parameter space, one staged box size for the
 * group, tile headers per view; the context caches the plans of the 4 most recent groups and of
 * the 64 most recent views); a layout the staged kernels cannot take (pitch not a multiple of
 * 16 bytes, footprints too large to stage) falls back to one launch per view.  Frames of one view
 * share the map; a call with one frame per view pays the map per frame. */
int cc_rectify_f32c1_views(cc_ctx *ctx, const cc_intr *intr, const cc_view *views, int nviews,
                           const double *ratios, const int64_t *axs_mins, const float *src,
                           float *dst, int sz1, int sz2, size_t pitch, size_t frame_stride,
                           int frames_per_view, float fill, unsigned flags, void *stream);
int cc_rectify_u8c3_views(cc_ctx *ctx, const cc_intr *intr, const cc_view *views, int nviews,
                          const double *ratios, const int64_t *axs_mins, const uint8_t *src,
                          uint8_t *dst, int sz1, int sz2, size_t pitch, size_t frame_stride,
                          int frames_per_view, const uint8_t fill[3], unsigned flags,
                          void *stream);
/* The same from HOST memory (pinned or pageable): arguments as cc_rectify_*_views, any number
 * of views; returns when dst holds the result.  The frames stream through the chunk pipeline of
 * cc_rectify_*_host (4 slot streams, ~32 MB chunks, CAMCAL_CHUNK_MB / CAMCAL_CHUNK_RAMP); a chunk
 * may start or end inside a view and span two 64-view groups, and makes one staged launch per
 * group it touches.  Each group's plan is obtained once per call; a missing one is built on host
 * threads while the previous group streams.  A group the staged kernels cannot take (1080p u8c3
 * lines of 3240 bytes, CC_GATHER_DIRECT, footprints too large to stage) runs one launch per view
 * on the chunk's stream.  Every frame is bit-identical to cc_rectify_*_views; host padding
 * between lines and frames is never written. */
int cc_rectify_views_f32c1_host(cc_ctx *ctx, const cc_intr *intr, const cc_view *views, int nviews,
                                const double *ratios, const int64_t *axs_mins, const float *src,
                                float *dst, int sz1, int sz2, size_t pitch, size_t frame_stride,
                                int frames_per_view, float fill, unsigned flags);
int cc_rectify_views_u8c3_host(cc_ctx *ctx, const cc_intr *intr, const cc_view *views, int nviews,
                               const double *ratios, const int64_t *axs_mins, const uint8_t *src,
                               uint8_t *dst, int sz1, int sz2, size_t pitch, size_t frame_stride,
                               int frames_per_view, const uint8_t fill[3], unsigned flags);
/* Rectification into output axes of any size: warp(img, tform, axs) with axs any two index ranges
 * (downscale, crop, upscale), one view or many.
 *  - Output layout: pixel (a+1, b+1) of output frame f, 0 <= a < out_sz1, 0 <= b < out_sz2, is
 *    stored at dst + f*out_frame_stride + b*out_pitch + a (u8c3: times 3 bytes).
 *  - It holds warp(img_f, tform_v, (axs_mins[2v] .+ (0:out_sz1-1), axs_mins[2v+1] .+ (0:out_sz2-1)))
 *    at that index: the world point ((axs_min[0]+a)/ratio, (axs_min[1]+b)/ratio, 0), the scale
 *    convention of cc_rectify_*.
 *  - Source frames: sz1 x sz2 pixels, lines `pitch` and frames `frame_stride` pixels apart, as for
 *    cc_rectify_*.
 *  - Views: frames [v*frames_per_view, (v+1)*frames_per_view) of src and of dst use views[v],
 *    ratios[v] and axs_mins[2v .. 2v+1]; all views share the output extent.
 *  - nviews == 1 takes the path of cc_rectify_f32c1 / _u8c3 (the _host forms: of their _host forms);
 *    nviews > 1 the path of cc_rectify_*_views / cc_rectify_views_*_host: groups of up to 64 views per
 *    staged launch, one launch per view where a group cannot be staged.  flags as for cc_rectify_*.
 *  - When the output extent, pitch and frame stride equal the source's, the output is byte-identical
 *    to that entry point's and the call makes the same number of launches.
 *  - CC_COORD_F64: a pixel's value does not depend on the output window that contains it (a crop of a
 *    larger call equals that call's window bit for bit).  CC_COORD_F32: the kernels sample the map
 *    cc_rectify_map_f32 returns for the same (ratio, axs_min, out_sz1, out_sz2), with its accuracy.
 *  - CC_ERR_INVALID_ARG, nothing written and nothing enqueued: out_sz1 or out_sz2 outside (0, 2^22),
 *    out_pitch < out_sz1, overlapping output frames (more than one frame), out_pitch*out_sz2 >= 2^30,
 *    and every rule of cc_rectify_* on the source, src != dst included.
 *  - The _host forms take host memory and return when dst holds the result; host padding between
 *    output lines and frames is never written. */
int cc_rectify_axes_f32c1(cc_ctx *ctx, const cc_intr *intr, const cc_view *views, int nviews,
                          const double *ratios, const int64_t *axs_mins, int out_sz1, int out_sz2,
                          const float *src, int sz1, int sz2, size_t pitch, size_t frame_stride,
                          float *dst, size_t out_pitch, size_t out_frame_stride,
                          int frames_per_view, float fill, unsigned flags, void *stream);
int cc_rectify_axes_u8c3(cc_ctx *ctx, const cc_intr *intr, const cc_view *views, int nviews,
                         const double *ratios, const int64_t *axs_mins, int out_sz1, int out_sz2,
                         const uint8_t *src, int sz1, int sz2, size_t pitch, size_t frame_stride,
                         uint8_t *dst, size_t out_pitch, size_t out_frame_stride,
                         int frames_per_view, const uint8_t fill[3], unsigned flags, void *stream);
int cc_rectify_axes_f32c1_host(cc_ctx *ctx, const cc_intr *intr, const cc_view *views, int nviews,
                               const double *ratios, const int64_t *axs_mins, int out_sz1,
                               int out_sz2, const float *src, int sz1, int sz2, size_t pitch,
                               size_t frame_stride, float *dst, size_t out_pitch,
                               size_t out_frame_stride, int frames_per_view, float fill,
                               unsigned flags);
int cc_rectify_axes_u8c3_host(cc_ctx *ctx, const cc_intr *intr, const cc_view *views, int nviews,
                              const double *ratios, const int64_t *axs_mins, int out_sz1,
                              int out_sz2, const uint8_t *src, int sz1, int sz2, size_t pitch,
                              size_t frame_stride, uint8_t *dst, size_t out_pitch,
                              size_t out_frame_stride, int frames_per_view,
                              const uint8_t fill[3], unsigned flags);
/* the map alone (source row/col sampled by each output pixel), FP64, frame layout */
int cc_rectify_map_f64(cc_ctx *ctx, const cc_intr *intr, const cc_view *view, double ratio,
                       const int64_t axs_min[2], double *map_row, double *map_col, int sz1,
                       int sz2, size_t pitch, void *stream);

/* the map the CC_COORD_F32 fast path samples (same arithmetic as its kernels), FP32: within 1e-3 px
 * of the exact map wherever the FP64 map is inside the frame, the point is in front of the camera
 * (P3 > 0) and the lens is monotone there (1 + 3k r^2 > 0); elsewhere within the conditioning bound of
 * oracle/map_ref.py: |err| <= s u sum_z |d(row, col)/dz| |z| over the roundings z of the kernel's
 * sequence, u = 2^-24, s = 1.0625 (past the fold of the lens: about 2e-2 px at in-frame pixels of a
 * 4K camera with k = -0.12) */
int cc_rectify_map_f32(cc_ctx *ctx, const cc_intr *intr, const cc_view *view, double ratio,
                       const int64_t axs_min[2], float *map_row, float *map_col, int sz1,
                       int sz2, size_t pitch, void *stream);

/* ---- image-file ingest on the device (SURVEY 8f: the step upstream of rectification) ----------
 * The reference reads every calibration image with FileIO.load and converts it to RGB before warp
 * (src/plot_calibration.jl:37; also src/detect_fit.jl:6,64).  cc_jpeg_decode_u8c3 takes the
 * COMPRESSED bytes (host pointers) of n baseline JPEG streams and leaves the decoded frames in
 * device memory in the u8c3 layout above -- element (r, c) of frame i at
 * dst[((i * frame_stride) + c * pitch + r) * 3], i.e. the memory of the Julia array RGB.(load(file)) --
 * ready for cc_rectify_u8c3 / cc_rectify_u8c3_views on the same stream.  Decoding is nvJPEG (CUDA
 * toolkit library, resolved at run time: without libnvjpeg.so.12 -> CC_ERR_UNSUPPORTED); the
 * raster -> frame transposition is a kernel of this library.  Grey JPEGs decode to R = G = B.
 * sz1 = image rows (height), sz2 = image columns (width); every stream must have that size.
 * cc_jpeg_info parses the header only: rows, columns, components (nvJPEG still needs a CUDA device). */
int cc_jpeg_info(const uint8_t *jpeg, size_t length, int *sz1, int *sz2, int *channels);
int cc_jpeg_decode_u8c3(cc_ctx *ctx, const uint8_t *const *jpegs, const size_t *lengths, int n,
                        uint8_t *dst, int sz1, int sz2, size_t pitch, size_t frame_stride,
                        void *stream);

/* get_ratio / get_axes (src/plot_calibration.jl:1-13): tiny host-side helpers so a
 * binding needs nothing else to drive cc_rectify_*.  corners: (a, b) at [a + n1*b]. */
int cc_get_ratio(const double *rows, const double *cols, int n1, int n2,
                 double checker_size, double *ratio);
int cc_get_axes(double ratio, double checker_size, int n1, int n2, int sz1, int sz2,
                int64_t axs_min[2]);

/* ---- reprojection residual + Jacobian + normal-equation blocks.
 *      Residual: _reprojection, src/buildcalibrations.jl:28-31.  Jacobian / J'J: the
 *      arithmetic OpenCV.calibrateCamera reduces for the flags of src/detect_fit.jl:40
 *      (ZERO_TANGENT + FIX_K2 + FIX_K3 + FIX_ASPECT_RATIO); free parameters per view
 *      e = (rvec, tvec), shared i = (f, crow, ccol, k) with frow = aspect*f, fcol = f.
 *        views    device, nviews cc_view
 *        obj      device, ncorners x 3 (x,y,z interleaved; shared by all views)
 *        img      device, nviews x ncorners x 2 (row,col interleaved)
 *        per_view device, nviews x 66: [JtJ_ee 6x6 | JtJ_ei 6x4 | Jtr_e 6]
 *        shared   device, 21: [JtJ_ii 4x4 | Jtr_i 4 | sum r^2]  (this device's views;
 *                 all-reduce it across ranks with NCCL -- the host layer does that)
 *      The reduction order is fixed: results are bit-reproducible run to run. */
#define CC_PER_VIEW 66
#define CC_SHARED 21
int cc_reproj_jtj_f64(cc_ctx *ctx, const cc_intr *intr, double aspect, const cc_view *views,
                      int nviews, const double *obj, const double *img, int ncorners,
                      double *per_view, double *shared, void *stream);
int cc_reproj_jtj_f64_host(cc_ctx *ctx, const cc_intr *intr, double aspect,
                           const cc_view *views, int nviews, const double *obj,
                           const double *img, int ncorners, double *per_view,
                           double *shared);

/* ---- calculate_errors, src/buildcalibrations.jl:37-67, fused on the device.
 *        n1 x n2 corners per view (a fastest); inv_rows/inv_cols: nviews x
 *        inverse_samples pre-drawn pixels in [1, sz] (the reference draws rand());
 *        sums (device, 4): raw sums {reprojection, projection, distance, inverse}
 *        before the RMS normalisation (all-reduce, then normalise on the host). */
int cc_calculate_errors_f64(cc_ctx *ctx, const cc_intr *intr, const cc_view *views,
                            int nviews, const double *obj, const double *img, int n1, int n2,
                            const double *inv_rows, const double *inv_cols,
                            int inverse_samples, double *sums, void *stream);
/* the same with HOST arrays (copies in, the four sums back; one synchronisation) */
int cc_calculate_errors_f64_host(cc_ctx *ctx, const cc_intr *intr, const cc_view *views,
                                 int nviews, const double *obj, const double *img, int n1,
                                 int n2, const double *inv_rows, const double *inv_cols,
                                 int inverse_samples, double *sums);

/* ---- one Levenberg-Marquardt step on those blocks (the solve OpenCV.calibrateCamera runs
 *      inside the reference's fit, src/detect_fit.jl:47; flags :40; CRITERIA
 *      src/CameraCalibrations.jl:16).  Arrowhead system, Schur complement on the 4 shared
 *      parameters; Marquardt damping  diag *= (1 + lambda).
 *      phase 1  cc_lm_schur_f64 : per view  Y = A'^-1 B (6x4), z = A'^-1 g (6)  -> yz (device,
 *               nviews x 30); schur (device, CC_LM_SCHUR = 21): [S 4x4 | s 4 | #views whose
 *               6x6 block was not positive definite], summed over THIS device's views in a fixed
 *               order.  All-reduce schur across ranks when views are sharded (host layer).
 *      phase 2  cc_lm_update_f64: (C' - S) di = -(gi - s);  de = -(z + Y di);
 *               views_out = views_in + de;  delta (device, CC_LM_DELTA = 8):
 *               [di 4 | sum |de|^2 | sum |rvec,tvec|^2 | 1.0 if the 4x4 solve succeeded | 0].
 *               free_mask: bit j set = shared parameter j (f, crow, ccol, k) is free
 *               (CALIB_FIX_K1 clears bit 3).  `shared` is the all-reduced block of cc_reproj_jtj. */
#define CC_LM_YZ 30
#define CC_LM_SCHUR 21
#define CC_LM_DELTA 8
int cc_lm_schur_f64(cc_ctx *ctx, const double *per_view, int nviews, double lambda, double *yz,
                    double *schur, void *stream);
int cc_lm_update_f64(cc_ctx *ctx, const double *shared, const double *schur, double lambda,
                     unsigned free_mask, const double *yz, const cc_view *views_in, int nviews,
                     cc_view *views_out, double *delta, void *stream);
/* The whole fit on one device with HOST arrays: the call that replaces
 * OpenCV.calibrateCamera(objectPoints, imagePoints, ..., flags, CRITERIA) of
 * src/detect_fit.jl:47.  intr/views: starting values in, fitted values out (frow = aspect*fcol is
 * kept, CALIB_FIX_ASPECT_RATIO); lambda schedule of CvLevMarq (1e-3, /10 accepted, *10 rejected);
 * stops after max_iter steps or when |step| < eps * |parameters| (CRITERIA: 30, 1e-3).
 * rms = sqrt(sum |residual|^2 / (nviews * ncorners)), what calibrateCamera returns. */
int cc_lm_fit_f64_host(cc_ctx *ctx, cc_intr *intr, double aspect, unsigned free_mask,
                       cc_view *views, int nviews, const double *obj, const double *img,
                       int ncorners, int max_iter, double eps, double *rms, int *iterations);
/* The same fit on DEVICE arrays, asynchronous on `stream` until the fitted intrinsics are handed
 * back (one wait at the end), with THIS RANK'S views when the context has a communicator
 * (cc_comm_init_rank): views/img hold the rank's shard, obj is replicated, intr goes in equal and
 * comes out equal on every rank.  The loop state (damping, accept/reject, stopping rule) lives in
 * device memory: an iteration costs two NCCL all-reduces (21 and 23 doubles) and NO host
 * synchronisation.  nviews may be 0 on a rank.  rms counts the points of all ranks. */
int cc_lm_fit_f64(cc_ctx *ctx, cc_intr *intr, double aspect, unsigned free_mask, cc_view *views,
                  int nviews, const double *obj, const double *img, int ncorners, int max_iter,
                  double eps, double *rms, int *iterations, void *stream);

/* Starting values for cc_lm_fit_f64 from the detections alone, as calibrateCamera derives them
 * inside the reference's fit (src/detect_fit.jl:34-36,47): principal point at the image centre,
 * focal length from the homographies (cvInitIntrinsicParams2D, FIX_ASPECT_RATIO when aspect > 0),
 * one pose per view from its homography; k = 0.  Device arrays (this rank's views); `views` is
 * written, `intr` (host) gets frow, fcol, crow, ccol, k -- checker_size is left as passed in.
 * obj must lie in the plane z = 0 (a checkerboard).  One stream wait (5 doubles come back). */
int cc_lm_initial_guess_f64(cc_ctx *ctx, const double *obj, const double *img, int nviews,
                            int ncorners, int sz1, int sz2, double aspect, cc_intr *intr,
                            cc_view *views, void *stream);

/* ---- multi-GPU: one process per GPU, one context per process, NCCL over NVLink for the small
 *      shared blocks only (the reduction over views of src/buildcalibrations.jl:28-31,60-65 and
 *      of the fit).  Frames, points and per-view blocks never cross GPUs.
 *      Bootstrap: rank 0 calls cc_comm_unique_id and hands the 128 bytes to the other ranks by
 *      any means (MPI, a file, torch.distributed); every rank then calls cc_comm_init_rank.
 *      NCCL is resolved at run time: without libnccl.so.2 these return CC_ERR_UNSUPPORTED and
 *      everything else still works.  A context without a communicator is a world of one, for
 *      which cc_allreduce_shared is a no-op. */
#define CC_COMM_ID_BYTES 128
int cc_comm_unique_id(void *id128);
int cc_comm_init_rank(cc_ctx *ctx, int nranks, int rank, const void *id128);
int cc_comm_destroy(cc_ctx *ctx);
int cc_comm_size(const cc_ctx *ctx, int *nranks, int *rank);
int cc_comm_nccl_version(int *version);
/* in-place sum of `count` doubles (device) over the ranks, asynchronous on `stream`:
 * cc_reproj_jtj_f64's `shared`, cc_calculate_errors_f64's `sums`, cc_lm_schur_f64's `schur` */
int cc_allreduce_shared(cc_ctx *ctx, double *buf, size_t count, void *stream);
/* One process, several GPUs (a single Julia session driving the whole box): ndev contexts, one per
 * device of devs[], joined in ONE communicator (ncclCommInitAll) -- the multi-device context of
 * SURVEY 8b.  cc_allreduce_shared_group sums bufs[i] (device memory of ctxs[i]) over the group in
 * place with one grouped NCCL call, each on streams[i] (streams == NULL: the default streams).
 * Entry points that wait on a collective internally (cc_lm_fit_f64) need one host thread per
 * context; all other calls are asynchronous and may be issued device after device from one thread. */
int cc_ctx_create_group(int ndev, const int *devs, cc_ctx **ctxs);
int cc_ctx_destroy_group(int ndev, cc_ctx **ctxs);
int cc_allreduce_shared_group(cc_ctx *const *ctxs, int ndev, double *const *bufs, size_t count,
                              void *const *streams);
/* number of all-reduces this context has issued so far */
int cc_ctx_collective_count(const cc_ctx *ctx, uint64_t *count);

#ifdef __cplusplus
}
#endif
#endif
