// abi.cu -- the extern "C" surface of libcamcal_b200.so (include/camcal_b200.h):
// argument checking, per-device context, and the host pipelines behind the *_host entry points.
// No compute lives here and nothing here can fall back to the CPU.
#include <algorithm>
#include <vector>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cmath>
#include <new>
#include <optional>

#include "lm_state.cuh"

namespace cc {

static thread_local char g_err[512] = "";

int set_error(int status, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return status;
}

int cuda_fail(cudaError_t e, const char* what) {
    const int st = (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver) ? CC_ERR_NO_DEVICE
                   : (e == cudaErrorMemoryAllocation ? CC_ERR_NOMEM : CC_ERR_CUDA);
    return set_error(st, "%s: %s (%s)", what, cudaGetErrorString(e), cudaGetErrorName(e));
}

// launchers implemented in the kernel translation units (the fit's: lm_state.cuh)
template <typename T>
int point_table_upload(cc_ctx*, bool, const ChainD*, int, const size_t*, cudaStream_t, PointTable*);
int point_table_release(cc_ctx*, cudaStream_t);
template <typename T>
int launch_points(cc_ctx*, const PointSrc&, const PointIO<T>&, size_t, cudaStream_t);
template <typename PX>
int launch_rectify(cc_ctx*, const RectCall<PX>&, int, int, const PX*, PX*, cudaStream_t);
template <typename PX>
int launch_rectify_group(cc_ctx*, const RectCall<PX>&, int, int, const PX*, PX*, cudaStream_t, bool*);
int rectify_views_per_launch();
struct RectViewsHost;
template <typename PX>
int rect_vh_begin(cc_ctx*, const RectCall<PX>&, RectViewsHost**);
int rect_vh_prepare(RectViewsHost*, int);
template <typename PX>
int rect_vh_launch(RectViewsHost*, const RectCall<PX>&, int, int, int, const PX*, PX*, cudaStream_t, bool*);
void rect_vh_retire(RectViewsHost*, int);
int rect_vh_end(RectViewsHost*);
template <typename T>
int launch_rectify_map(cc_ctx*, const ChainD&, double, const int64_t[2], T*, T*, int, int, size_t, cudaStream_t);

static int check_params(const cc_ctx* ctx, const cc_intr* intr, const cc_view* view) {
    CC_REQUIRE(ctx != nullptr, "ctx is NULL");
    CC_REQUIRE(intr != nullptr, "intr is NULL");
    CC_REQUIRE(view != nullptr, "view is NULL");
    CC_REQUIRE(intr->frow != 0.0 && intr->fcol != 0.0, "focal lengths must be non-zero");
    CC_REQUIRE(intr->checker_size != 0.0, "checker_size must be non-zero");
    return CC_OK;
}

// Every entry point runs on the context's device and leaves the CALLER's current device as it
// found it (one process may drive several GPUs: a call on cuda:1 must not redirect the host's
// later allocations).  `if ((rc = enter(ctx))) return rc;` declares the guard in the enclosing scope.
struct DeviceGuard {
    int prev = -1;
    int set(cc_ctx* ctx) {
        CC_REQUIRE(ctx != nullptr, "ctx is NULL");
        int cur = -1;
        CC_CUDA(cudaGetDevice(&cur));
        if (cur != ctx->device) {
            CC_CUDA(cudaSetDevice(ctx->device));
            prev = cur;
        }
        return CC_OK;
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};
#define enter(ctx) _cc_guard.set(ctx)
#define CC_GUARD DeviceGuard _cc_guard

// ---- host pipeline ---------------------------------------------------------------
static int ensure_stream(cc_ctx* ctx, int k) {
    if (!ctx->pipe_stream[k]) CC_CUDA(cudaStreamCreateWithFlags(&ctx->pipe_stream[k], cudaStreamNonBlocking));
    return CC_OK;
}
static int ensure_slot(cc_ctx* ctx, int k, size_t in_bytes, size_t out_bytes) {
    if (!ctx->pipe_stream[k]) CC_CUDA(cudaStreamCreateWithFlags(&ctx->pipe_stream[k], cudaStreamNonBlocking));
    if (ctx->pipe_in_bytes[k] < in_bytes) {
        if (ctx->pipe_in[k]) CC_CUDA(cudaFree(ctx->pipe_in[k]));
        ctx->pipe_in[k] = nullptr; ctx->pipe_in_bytes[k] = 0;
        CC_CUDA(cudaMalloc(&ctx->pipe_in[k], in_bytes));
        ctx->pipe_in_bytes[k] = in_bytes;
    }
    if (ctx->pipe_out_bytes[k] < out_bytes) {
        if (ctx->pipe_out[k]) CC_CUDA(cudaFree(ctx->pipe_out[k]));
        ctx->pipe_out[k] = nullptr; ctx->pipe_out_bytes[k] = 0;
        CC_CUDA(cudaMalloc(&ctx->pipe_out[k], out_bytes));
        ctx->pipe_out_bytes[k] = out_bytes;
    }
    return CC_OK;
}

static int drain(cc_ctx* ctx) {
    for (int k = 0; k < cc_ctx::NSLOT; ++k)
        if (ctx->pipe_stream[k]) CC_CUDA(cudaStreamSynchronize(ctx->pipe_stream[k]));
    return CC_OK;
}

static size_t round_up(size_t v, size_t m) { return (v + m - 1) / m * m; }

constexpr size_t kPointChunk = (size_t)1 << 22;   // points per pipeline stage

// ---- point-map pipelines ----------------------------------------------------------
// Every point-map entry point fills a PointIO and calls points_device or points_host.  offsets == NULL: views[0]
// maps all `count` points (nviews must be 1).  Otherwise points [offsets[s], offsets[s+1]) use views[s], and
// offsets[nviews] must equal count; the SoA `_views` calls pass no count, so their offsets are required and give it.
template <typename T> static PointIO<T> soa_img2world(const T* row, const T* col, T* x, T* y, T* z) {
    return {false, false, 2, z ? 3 : 2, {row, col}, {x, y, z}};
}
template <typename T> static PointIO<T> soa_world2img(const T* x, const T* y, const T* z, T* row, T* col) {
    return {true, false, z ? 3 : 2, 2, {x, y, z}, {row, col}};
}
template <typename T> static PointIO<T> aos_img2world(const T* rc, T* out, int out_dim) {
    return {false, true, 2, out_dim, {rc}, {out}};
}
template <typename T> static PointIO<T> aos_world2img(const T* pts, int in_dim, T* rc) {
    return {true, true, in_dim, 2, {pts}, {rc}};
}

// Checks everything before anything is written or enqueued.  *n: the call's points.  *single: the view whose chain
// maps every point, passed by value with no table (the SINGLE kernel), or -1 (TABLE).
template <typename T>
static int check_points(const cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews,
                        const size_t* offsets, std::optional<size_t> count, const PointIO<T>& io, size_t* n,
                        int* single) {
    CC_REQUIRE(io.in_dim >= 2 && io.in_dim <= 3 && io.out_dim >= 2 && io.out_dim <= 3,
               "out_dim / in_dim must be 2 or 3");
    if (count && offsets == nullptr) {
        CC_REQUIRE(nviews == 1, "offsets == NULL needs nviews == 1");
    } else {
        CC_REQUIRE(ctx != nullptr, "ctx is NULL");
        CC_REQUIRE(nviews >= 1, "nviews must be at least 1");
        CC_REQUIRE(views != nullptr && offsets != nullptr, "views / offsets is NULL");
        CC_REQUIRE(offsets[0] == 0, "offsets[0] must be 0");
        for (int s = 0; s < nviews; ++s) CC_REQUIRE(offsets[s + 1] >= offsets[s], "offsets must not decrease");
    }
    const int rc = check_params(ctx, intr, views);
    if (rc) return rc;
    *n = count ? *count : offsets[nviews];
    CC_REQUIRE(offsets == nullptr || offsets[nviews] == *n, "offsets[nviews] must equal n");
    bool arrays = true;
    for (int d = 0; d < io.in_arrays(); ++d) arrays = arrays && io.in[d];
    for (int d = 0; d < io.out_arrays(); ++d) arrays = arrays && io.out[d];
    CC_REQUIRE(*n == 0 || arrays, "NULL point array");
    // An AoS call whose points all lie in one segment takes that view's SINGLE kernel.  The SoA `_views` calls
    // keep the table even then: at one segment it is faster than SINGLE for some maps and slower for others
    // (DESIGN.md §4.1).
    *single = offsets == nullptr ? 0 : -1;
    for (int s = 0; io.aos && offsets && s < nviews && *single < 0; ++s)
        if (offsets[s + 1] - offsets[s] == *n) *single = s;
    return CC_OK;
}

// SINGLE: views[single]'s chain in *ch.  TABLE: the chains of all segments, uploaded on st.  The chains are built
// on the host, one per segment, exactly as for one view: every point's result is bit-identical to a single-view
// call with its own view.
template <typename T>
static int point_src(cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews, const size_t* offsets,
                     int single, bool to_img, cudaStream_t st, ChainD* ch, PointSrc* src) {
    *src = PointSrc{nullptr, {}, 0, 0, nviews};
    if (single >= 0) {
        build_chain(intr, views + single, ch);
        src->chain = ch;
        return CC_OK;
    }
    std::vector<ChainD> chs((size_t)nviews);
    for (int s = 0; s < nviews; ++s) build_chain(intr, views + s, &chs[s]);
    return point_table_upload<T>(ctx, to_img, chs.data(), nviews, offsets, st, &src->tb);
}

// Device form: at most one table upload and ONE launch on the caller's stream, whatever nviews is.
template <typename T>
static int points_device(cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews, const size_t* offsets,
                         std::optional<size_t> count, const PointIO<T>& io, void* stream) {
    size_t n = 0;
    int single = -1, rc = check_points(ctx, intr, views, nviews, offsets, count, io, &n, &single);
    if (rc) return rc;
    CC_GUARD;
    if ((rc = enter(ctx)) || n == 0) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    ChainD ch;
    PointSrc src;
    if ((rc = point_src<T>(ctx, intr, views, nviews, offsets, single, io.to_img, st, &ch, &src))) return rc;
    rc = launch_points<T>(ctx, src, io, n, st);
    const int rr = src.chain ? (int)CC_OK : point_table_release(ctx, st);
    return rc ? rc : rr;
}

// Moves points [off, off + m) of a host call through slot k: up, one launch, down.  A side of `dim` coordinates
// takes dim arrays of m points at stride cap in the slot (SoA), or one range of dim * m elements (AoS).  cap is a
// multiple of 64, so every chunk takes the vector path.
template <typename T>
static int stage_chunk(cc_ctx* ctx, int k, const PointSrc& src, const PointIO<T>& io, size_t off, size_t m,
                       size_t cap) {
    cudaStream_t st = ctx->pipe_stream[k];
    const size_t ein = io.aos ? io.in_dim : 1, eout = io.aos ? io.out_dim : 1;   // elements per point and array
    PointIO<T> dev = io;
    for (int d = 0; d < io.in_arrays(); ++d) {
        T* slot = static_cast<T*>(ctx->pipe_in[k]) + d * cap;
        dev.in[d] = slot;
        CC_CUDA(cudaMemcpyAsync(slot, io.in[d] + ein * off, ein * m * sizeof(T), cudaMemcpyHostToDevice, st));
    }
    for (int d = 0; d < io.out_arrays(); ++d) dev.out[d] = static_cast<T*>(ctx->pipe_out[k]) + d * cap;
    const int rc = launch_points<T>(ctx, src, dev, m, st);
    if (rc) return rc;
    for (int d = 0; d < io.out_arrays(); ++d)
        CC_CUDA(cudaMemcpyAsync(io.out[d] + eout * off, dev.out[d], eout * m * sizeof(T), cudaMemcpyDeviceToHost, st));
    return CC_OK;
}

// Host form: chunks of kPointChunk points go round-robin through the NSLOT slots, with one drain at the end.  A
// table goes up once on slot 0's stream and every other slot's stream waits for it; each chunk's launch gets the
// segments it covers and its first point's index in the call.
template <typename T>
static int points_host(cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews, const size_t* offsets,
                       std::optional<size_t> count, const PointIO<T>& io) {
    size_t n = 0;
    int single = -1, rc = check_points(ctx, intr, views, nviews, offsets, count, io, &n, &single);
    if (rc) return rc;
    CC_GUARD;
    if ((rc = enter(ctx)) || n == 0) return rc;
    const size_t cap = n < kPointChunk ? round_up(n, 64) : kPointChunk;
    const size_t nchunks = (n + cap - 1) / cap;
    ChainD ch;
    PointSrc src;
    if ((rc = ensure_stream(ctx, 0))) return rc;
    if ((rc = point_src<T>(ctx, intr, views, nviews, offsets, single, io.to_img, ctx->pipe_stream[0], &ch, &src)))
        return rc;
    if (!src.chain) {
        if ((rc = point_table_release(ctx, ctx->pipe_stream[0]))) return rc;
        for (int k = 1; k < cc_ctx::NSLOT && (size_t)k < nchunks; ++k) {
            if ((rc = ensure_stream(ctx, k))) return rc;
            CC_CUDA(cudaStreamWaitEvent(ctx->pipe_stream[k], ctx->pt_event, 0));
        }
    }
    size_t off = 0;
    for (int it = 0; rc == CC_OK && off < n; ++it, off += cap) {
        const int k = it % cc_ctx::NSLOT;
        const size_t m = (n - off) < cap ? (n - off) : cap;
        if (!src.chain) {
            src.base = off;
            src.seg_lo = (int)(std::upper_bound(offsets, offsets + nviews + 1, off) - offsets) - 1;
            src.seg_hi = (int)(std::upper_bound(offsets, offsets + nviews + 1, off + m - 1) - offsets);
        }
        if ((rc = ensure_slot(ctx, k, io.in_dim * cap * sizeof(T), io.out_dim * cap * sizeof(T)))) break;
        rc = stage_chunk<T>(ctx, k, src, io, off, m, cap);
    }
    const int rd = drain(ctx);                     // the table's readers are done before the call returns
    return rc ? rc : rd;
}

// Frames per chunk of the frame pipelines: a few whole frames, ~32 MB per chunk (measured on B200 / PCIe Gen5:
// 8 MB chunks 9.7, 16 MB 10.7, 32 MB 11.0, 64 MB 10.8 Gpix/s end to end on 64 x 1080p fp32 frames), at most
// max_per.  The first chunk's upload and the last chunk's download overlap with nothing: the batch starts with
// chunks of 1, 2, 4 ... frames and ends with ... 4, 2, 1 (CAMCAL_CHUNK_RAMP=0: uniform chunks), so the exposed
// head and tail are one frame each instead of one 32 MB chunk each.  *per_out: the body's chunk.
static std::vector<int> chunk_schedule(int nframes, size_t frame_bytes, int max_per, int* per_out) {
    size_t chunk_mb = 32;
    if (const char* e = getenv("CAMCAL_CHUNK_MB")) chunk_mb = (size_t)std::max(1, atoi(e));   // tuning knob
    int per = (int)((chunk_mb << 20) / frame_bytes);
    if (per < 1) per = 1;
    if (per > max_per) per = max_per;
    if (per > nframes) per = nframes;
    bool ramp = true;
    if (const char* e = getenv("CAMCAL_CHUNK_RAMP")) ramp = atoi(e) != 0;   // tuning knob
    int ramp_frames = 0, ramp_steps = 0;                     // frames / chunks of one ramp: 1 + 2 + ... (< per)
    for (int c = 1; ramp && c < per; c *= 2) { ramp_frames += c; ++ramp_steps; }
    if (2 * ramp_frames + per > nframes) ramp_frames = ramp_steps = 0;
    std::vector<int> sizes;
    for (int f0 = 0, it = 0, m = 0; f0 < nframes; f0 += m, ++it) {
        const int left = nframes - f0;
        if (it < ramp_steps) m = 1 << it;                                    // head: 1, 2, 4 ...
        else if (left > ramp_frames) m = std::min(per, left - ramp_frames);  // body
        else { m = 1; while (2 * m - 1 < left) m *= 2; }                     // tail: left = 2m - 1 -> m, ... 2, 1
        sizes.push_back(m);
    }
    *per_out = per;
    return sizes;
}

// ---- rectification ---------------------------------------------------------------
// Every rectification entry point calls rectify_device or rectify_host with its views and its frame layout: a
// single-view call is one view whose frames per view are the call's nframes; `many` marks the `_views` calls.

// Every rule of a rectification call, checked before anything is written, enqueued or the device is touched.  The
// map entry points pass fr.fpv = 0: no frames.
static int check_rect(const cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews, const double* ratios,
                      const int64_t* axs_mins, const RectFrames& fr, const void* src, const void* dst, bool fill_ok) {
    CC_REQUIRE(ctx != nullptr, "ctx is NULL");
    CC_REQUIRE(intr != nullptr, "intr is NULL");
    CC_REQUIRE(nviews >= 0 && fr.fpv >= 0, "bad counts: nviews and frame counts must not be negative");
    const long long nframes = (long long)nviews * fr.fpv;
    CC_REQUIRE(nframes <= 65535, "at most 65535 frames per call");
    if (nviews > 0) {
        CC_REQUIRE(views != nullptr, "view is NULL");
        CC_REQUIRE(ratios != nullptr, "ratios is NULL");
        CC_REQUIRE(axs_mins != nullptr, "axs_min is NULL");
        CC_REQUIRE(fr.sz1 > 0 && fr.sz2 > 0, "frame size must be positive");
        CC_REQUIRE(fr.sz1 < (1 << 22) && fr.sz2 < (1 << 22), "frame extent must be < 2^22");
        CC_REQUIRE(fr.pitch >= (size_t)fr.sz1, "pitch smaller than sz1");
        CC_REQUIRE(nframes <= 1 || fr.frame_stride >= fr.pitch * (size_t)(fr.sz2 - 1) + fr.sz1, "frames overlap");
        CC_REQUIRE(fr.pitch * (size_t)fr.sz2 < (size_t)1 << 30, "frame too large (pitch*sz2 must be < 2^30)");
    }
    const int64_t lim = (int64_t)1 << 30;
    for (int v = 0; v < nviews; ++v) {
        const int rc = check_params(ctx, intr, views + v);
        if (rc) return rc;
        CC_REQUIRE(ratios[v] > 0.0 && ratios[v] == ratios[v], "ratio must be positive");
        const int64_t* axs = axs_mins + 2 * v;
        CC_REQUIRE(axs[0] > -lim && axs[0] < lim && axs[1] > -lim && axs[1] < lim, "axs_min out of range");
    }
    CC_REQUIRE(nframes == 0 || (src && dst), "NULL frame pointer");
    CC_REQUIRE(nframes == 0 || src != dst, "rectification is not in place: src == dst");
    CC_REQUIRE(fill_ok, "fill is NULL");
    return CC_OK;
}

// the fill of a call as the kernels take it; false: a NULL u8c3 fill
static bool make_fill(float f, float* out) {
    *out = f;
    return true;
}
static bool make_fill(const uint8_t* f, uchar3* out) {
    if (f) *out = make_uchar3(f[0], f[1], f[2]);
    return f != nullptr;
}

// Device form.  A single-view call is one launch on the caller's stream.  A `_views` call launches groups of up to 64
// views in one staged launch each (CAMCAL_VIEWS_SINGLE=0, a tuning knob, turns that off); the views of a group that
// cannot be staged get one launch each.
template <typename PX, typename FILL>
static int rectify_device(cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews, const double* ratios,
                          const int64_t* axs_mins, const PX* src, PX* dst, const RectFrames& fr, FILL fill,
                          unsigned flags, void* stream, bool many) {
    RectCall<PX> c{fr, {nullptr, ratios, axs_mins, nviews}, {}, flags};
    int rc = check_rect(ctx, intr, views, nviews, ratios, axs_mins, fr, src, dst, make_fill(fill, &c.fill));
    if (rc) return rc;
    CC_GUARD;
    if ((rc = enter(ctx)) || nviews == 0 || fr.fpv == 0) return rc;
    std::vector<ChainD> chs((size_t)nviews);
    for (int v = 0; v < nviews; ++v) build_chain(intr, views + v, &chs[v]);
    c.views.chs = chs.data();
    cudaStream_t stream_ = (cudaStream_t)stream;
    if (!many) return launch_rectify(ctx, c, 0, fr.fpv, src, dst, stream_);
    const size_t view_elems = (size_t)fr.fpv * fr.frame_stride * RectPx<PX>::channels;
    std::vector<char> done((size_t)nviews, 0);
    bool single = true;
    if (const char* e = getenv("CAMCAL_VIEWS_SINGLE")) single = atoi(e) != 0;
    int ndone = 0;
    const int per = rectify_views_per_launch();
    for (int v0 = 0; single && v0 < nviews; v0 += per) {
        const int nv = std::min(per, nviews - v0);
        bool ok = false;
        if ((rc = launch_rectify_group(ctx, c, v0, nv, src + v0 * view_elems, dst + v0 * view_elems, stream_, &ok)))
            return rc;
        if (ok) { for (int v = v0; v < v0 + nv; ++v) done[v] = 1; ndone += nv; }
    }
    if (ndone == nviews) return CC_OK;
    // One launch per view.  On a single stream the launches serialise: every persistent kernel ramps up
    // and drains alone (a 1080p frame is ~15 us of launch + tail for ~5 us of work).  The views are
    // therefore spread round-robin over the context's side streams, forked from and joined to `stream`
    // with events, so consecutive views overlap.
    const int lanes = std::min<int>(cc_ctx::NSLOT, nviews);
    cudaEvent_t fork = nullptr, join[cc_ctx::NSLOT] = {};
    if (lanes > 1) {
        CC_CUDA(cudaEventCreateWithFlags(&fork, cudaEventDisableTiming));
        CC_CUDA(cudaEventRecord(fork, stream_));
        for (int k = 0; k < lanes; ++k) {
            if ((rc = ensure_stream(ctx, k))) return rc;
            CC_CUDA(cudaStreamWaitEvent(ctx->pipe_stream[k], fork, 0));
        }
    }
    for (int v = 0; v < nviews; ++v) {
        if (done[v]) continue;
        cudaStream_t st = lanes > 1 ? ctx->pipe_stream[v % lanes] : stream_;
        if ((rc = launch_rectify(ctx, c, v, fr.fpv, src + v * view_elems, dst + v * view_elems, st))) break;
    }
    if (lanes > 1) {                                  // join even after an error: nothing stays forked
        for (int k = 0; k < lanes; ++k) {
            if (cudaEventCreateWithFlags(&join[k], cudaEventDisableTiming) == cudaSuccess) {
                cudaEventRecord(join[k], ctx->pipe_stream[k]);
                cudaStreamWaitEvent(stream_, join[k], 0);
                cudaEventDestroy(join[k]);            // released once the wait has consumed it
            }
        }
        cudaEventDestroy(fork);
    }
    return rc;
}

// m frames from `from` to `to` (kind: which way): one side is a slot, frames pitch * sz2 apart, the other the caller's
// host frames, frame_stride apart.  One copy when the host frames are dense, else one 2-D copy per frame.
static int copy_frames(const RectFrames& fr, size_t pxb, int m, const void* from, void* to, cudaMemcpyKind kind,
                       cudaStream_t st) {
    const size_t line = fr.pitch * pxb, slot_frame = line * fr.sz2, host_frame = fr.frame_stride * pxb;
    const bool up = kind == cudaMemcpyHostToDevice, dense = host_frame == slot_frame && fr.pitch == (size_t)fr.sz1;
    const size_t from_frame = up ? host_frame : slot_frame, to_frame = up ? slot_frame : host_frame;
    for (int f = 0; f < (dense ? 1 : m); ++f) {
        const uint8_t* s = static_cast<const uint8_t*>(from) + (size_t)f * from_frame;
        uint8_t* d = static_cast<uint8_t*>(to) + (size_t)f * to_frame;
        const cudaError_t e = dense ? cudaMemcpyAsync(d, s, (size_t)m * slot_frame, kind, st)
                                    : cudaMemcpy2DAsync(d, line, s, line, (size_t)fr.sz1 * pxb, fr.sz2, kind, st);
        if (e != cudaSuccess) return cuda_fail(e, "copy");
    }
    return CC_OK;
}

// Host form: the chunk pipeline over the frame axis of the whole call.  Chunks of whole frames (chunk_schedule) go
// round-robin through the NSLOT slots: up, launches, down.  A single-view call launches the single-view kernels over
// each chunk.  The chunks of a `_views` call ignore view boundaries and span at most two 64-view groups (a chunk holds
// at most 64 views' frames).  Such a chunk makes one staged launch per group it touches, over the window of that
// group's frames it holds (rectify.cu: RectViewsHost); a group without a staged plan runs the window's views through
// the single-view kernels on the chunk's own slot stream.  The next group's plan is built on host threads while the
// device streams the current one: before waiting for it, the uploads of the next NSLOT chunks are enqueued.  Every
// call drains the slot streams before it returns, after an error too, so no copy into `dst` is left in flight.
template <typename PX, typename FILL>
static int rectify_host(cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews, const double* ratios,
                        const int64_t* axs_mins, const PX* src, PX* dst, const RectFrames& fr, FILL fill,
                        unsigned flags, bool many) {
    RectCall<PX> c{fr, {nullptr, ratios, axs_mins, nviews}, {}, flags};
    int rc = check_rect(ctx, intr, views, nviews, ratios, axs_mins, fr, src, dst, make_fill(fill, &c.fill));
    if (rc) return rc;
    CC_GUARD;
    if ((rc = enter(ctx)) || nviews == 0 || fr.fpv == 0) return rc;
    std::vector<ChainD> chs((size_t)nviews);
    for (int v = 0; v < nviews; ++v) build_chain(intr, views + v, &chs[v]);
    c.views.chs = chs.data();
    const size_t pxb = RectPx<PX>::bytes, frame_bytes = fr.pitch * (size_t)fr.sz2 * pxb;
    c.fr.frame_stride = fr.pitch * (size_t)fr.sz2;           // device frames are stored pitch*sz2
    const int nframes = nviews * fr.fpv, gframes = many ? rectify_views_per_launch() * fr.fpv : nframes;
    int per = 0;
    const std::vector<int> chunks = chunk_schedule(nframes, frame_bytes, gframes, &per);
    const int nchunks = (int)chunks.size();
    std::vector<int> first((size_t)nchunks + 1, 0);
    for (int i = 0; i < nchunks; ++i) first[i + 1] = first[i] + chunks[i];
    const uint8_t* hsrc = reinterpret_cast<const uint8_t*>(src);
    uint8_t* hdst = reinterpret_cast<uint8_t*>(dst);
    // frame f of a chunk in slot buffer p
    auto at = [&](void* p, int f) { return reinterpret_cast<PX*>(static_cast<uint8_t*>(p) + (size_t)f * frame_bytes); };
    RectViewsHost* vh = nullptr;
    if (many && (rc = rect_vh_begin(ctx, c, &vh))) return rc;
    std::vector<char> uploaded((size_t)nchunks, 0), prepared((size_t)((nframes + gframes - 1) / gframes), 0);
    // chunk i's frames to its slot (the slot's previous chunk, i - NSLOT, is enqueued in full by then); +64 bytes:
    // vector gathers may touch the aligned word holding the last texel
    auto upload = [&](int i) -> int {
        if (i >= nchunks || uploaded[i]) return CC_OK;
        const int k = i % cc_ctx::NSLOT;
        int r = ensure_slot(ctx, k, per * frame_bytes + 64, per * frame_bytes + 64);
        if (!r) r = copy_frames(fr, pxb, chunks[i], hsrc + (size_t)first[i] * fr.frame_stride * pxb, ctx->pipe_in[k],
                                cudaMemcpyHostToDevice, ctx->pipe_stream[k]);
        uploaded[i] = r == CC_OK;
        return r;
    };
    int retired = 0;                                        // groups whose chunks are all enqueued
    for (int i = 0; rc == CC_OK && i < nchunks; ++i) {
        const int f0 = first[i], m = chunks[i], g_lo = f0 / gframes, g_hi = (f0 + m - 1) / gframes;
        for (int gi = g_lo; vh && rc == CC_OK && gi <= g_hi; ++gi) {
            if (prepared[gi]) continue;
            for (int j = 0; rc == CC_OK && j < cc_ctx::NSLOT; ++j) rc = upload(i + j);
            if (rc == CC_OK) rc = rect_vh_prepare(vh, gi);
            prepared[gi] = 1;
        }
        if (rc == CC_OK) rc = upload(i);
        if (rc) break;
        const int k = i % cc_ctx::NSLOT;
        cudaStream_t st = ctx->pipe_stream[k];
        if (!vh) rc = launch_rectify(ctx, c, 0, m, at(ctx->pipe_in[k], 0), at(ctx->pipe_out[k], 0), st);
        for (int gi = g_lo; vh && rc == CC_OK && gi <= g_hi; ++gi) {
            const int a = std::max(f0, gi * gframes), b = std::min(f0 + m, (gi + 1) * gframes);
            bool ok = false;
            rc = rect_vh_launch(vh, c, gi, a - gi * gframes, b - a, at(ctx->pipe_in[k], a - f0),
                                at(ctx->pipe_out[k], a - f0), st, &ok);
            for (int v = a / fr.fpv; rc == CC_OK && !ok && v <= (b - 1) / fr.fpv; ++v) {
                const int fa = std::max(a, v * fr.fpv), fb = std::min(b, (v + 1) * fr.fpv);
                rc = launch_rectify(ctx, c, v, fb - fa, at(ctx->pipe_in[k], fa - f0), at(ctx->pipe_out[k], fa - f0), st);
            }
        }
        if (rc) break;
        rc = copy_frames(fr, pxb, m, ctx->pipe_out[k], hdst + (size_t)f0 * fr.frame_stride * pxb, cudaMemcpyDeviceToHost,
                         st);
        for (; vh && (retired < g_hi || (retired == g_hi && f0 + m == std::min(nframes, (g_hi + 1) * gframes))); ++retired)
            rect_vh_retire(vh, retired);
    }
    const int re = rect_vh_end(vh);                         // every plan fenced, uploads complete
    const int rd = drain(ctx);
    return rc ? rc : re ? re : rd;
}

// the map alone: FP64 (the exact coordinates) or FP32 (the fast ones)
template <typename T>
static int rectify_map(cc_ctx* ctx, const cc_intr* intr, const cc_view* view, double ratio, const int64_t* axs_min,
                       T* map_row, T* map_col, int sz1, int sz2, size_t pitch, void* stream) {
    int rc = check_rect(ctx, intr, view, 1, &ratio, axs_min, {sz1, sz2, pitch, pitch * (size_t)sz2, 0}, nullptr,
                        nullptr, true);
    if (rc) return rc;
    CC_REQUIRE(map_row && map_col, "NULL map pointer");
    CC_GUARD;
    if ((rc = enter(ctx))) return rc;
    ChainD ch;
    build_chain(intr, view, &ch);
    return launch_rectify_map<T>(ctx, ch, ratio, axs_min, map_row, map_col, sz1, sz2, pitch, (cudaStream_t)stream);
}

// ---- fit: residual / J'J, calculate_errors, Levenberg-Marquardt ------------------
// Each check runs every rule of its entry points before the device is touched, anything is uploaded or launched.
// A pointer is required only when the call reads it.  img is read as 16-byte (row, col) pairs: the device forms
// check its alignment; a staged host call is aligned by construction.
static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

static int check_reproj_jtj(const cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews,
                            const double* obj, const double* img, int ncorners, const double* per_view,
                            const double* shared, bool host) {
    CC_REQUIRE(ctx && intr, "NULL argument");
    CC_REQUIRE(nviews >= 0 && ncorners > 0, "bad sizes");
    CC_REQUIRE(shared != nullptr, "shared is NULL");
    CC_REQUIRE(nviews == 0 || (views && obj && img && per_view), host ? "NULL host pointer" : "NULL device pointer");
    CC_REQUIRE(intr->checker_size != 0.0, "checker_size must be non-zero");
    CC_REQUIRE(host || aligned16(img), "img must be 16-byte aligned");
    return CC_OK;
}

static int check_calculate_errors(const cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews,
                                  const double* obj, const double* img, int n1, int n2, const double* inv_rows,
                                  const double* inv_cols, int inverse_samples, const double* sums, bool host) {
    CC_REQUIRE(ctx && intr && sums, "NULL argument");
    CC_REQUIRE(nviews >= 0 && n1 >= 1 && n2 >= 1 && inverse_samples >= 0, "bad sizes");
    CC_REQUIRE(nviews == 0 || (views && obj && img), host ? "NULL host pointer" : "NULL device pointer");
    CC_REQUIRE(inverse_samples == 0 || nviews == 0 || (inv_rows && inv_cols), "NULL sample pointer");
    CC_REQUIRE(intr->checker_size != 0.0 && intr->frow != 0.0 && intr->fcol != 0.0, "bad intrinsics");
    CC_REQUIRE(host || aligned16(img), "img must be 16-byte aligned");
    CC_REQUIRE(calc_errors_smem(n1, n2) <= kCalcErrorsSmemMax, "too many corners per view for the fused kernel");
    return CC_OK;
}

// The host form fits at least one view; the device form may hold no views on a rank of a sharded fit.
static int check_lm_fit(const cc_ctx* ctx, const cc_intr* intr, double aspect, unsigned free_mask,
                        const cc_view* views, int nviews, const double* obj, const double* img, int ncorners,
                        int max_iter, double eps, bool host) {
    CC_REQUIRE(ctx && intr && obj, "NULL argument");
    CC_REQUIRE(nviews >= (host ? 1 : 0) && ncorners > 0, "bad sizes");
    CC_REQUIRE(nviews == 0 || (views && img), "NULL view / image-point array");
    CC_REQUIRE(free_mask != 0u && free_mask < 16u, "free_mask selects among the 4 shared parameters");
    CC_REQUIRE(max_iter >= 0 && eps >= 0.0, "bad stopping rule");
    CC_REQUIRE(aspect > 0.0 && intr->fcol != 0.0 && intr->checker_size != 0.0, "bad starting intrinsics");
    CC_REQUIRE(host || aligned16(img), "img must be 16-byte aligned");
    return CC_OK;
}

static int check_lm_schur(const cc_ctx* ctx, const double* per_view, int nviews, double lambda, const double* yz,
                          const double* schur) {
    CC_REQUIRE(ctx && schur, "NULL argument");
    CC_REQUIRE(nviews >= 0, "bad sizes");
    CC_REQUIRE(nviews == 0 || (per_view && yz), "NULL device pointer");
    CC_REQUIRE(lambda >= 0.0 && lambda == lambda, "lambda must be non-negative");
    return CC_OK;
}

static int check_lm_update(const cc_ctx* ctx, const double* shared, const double* schur, double lambda,
                           unsigned free_mask, const double* yz, const cc_view* views_in, int nviews,
                           const cc_view* views_out, const double* delta) {
    CC_REQUIRE(ctx && shared && schur && delta, "NULL argument");
    CC_REQUIRE(nviews >= 0, "bad sizes");
    CC_REQUIRE(nviews == 0 || (yz && views_in && views_out), "NULL device pointer");
    CC_REQUIRE(lambda >= 0.0 && lambda == lambda, "lambda must be non-negative");
    CC_REQUIRE(free_mask != 0u && free_mask < 16u, "free_mask selects among the 4 shared parameters");
    return CC_OK;
}

static int check_initial_guess(const cc_ctx* ctx, const double* obj, const double* img, int nviews, int ncorners,
                               int sz1, int sz2, const cc_intr* intr, const cc_view* views) {
    CC_REQUIRE(ctx && intr && obj, "NULL argument");
    CC_REQUIRE(nviews >= 0 && ncorners >= 4 && sz1 > 0 && sz2 > 0, "bad sizes (a homography needs >= 4 corners)");
    CC_REQUIRE(nviews == 0 || (views && img), "NULL view / image-point array");
    return CC_OK;
}

// One host array of a staged call: `up` (if not NULL) is uploaded before the body runs, `down` (if not NULL)
// receives the array after it.  A span may be both.
struct HostSpan {
    const void* up;
    void* down;
    size_t bytes;
};

// The host form of a fit entry point: the spans go to slot 0 at 256-byte offsets, up on the slot's stream; body runs
// the device form's launcher on the slot's device copies (d[i] for span i) and that stream; then the downloads, and
// one synchronisation.  The caller has checked the arguments and entered the context's device.
template <size_t N, typename Body>
static int stage_host(cc_ctx* ctx, const HostSpan (&spans)[N], Body body) {
    size_t off[N + 1] = {0};
    for (size_t i = 0; i < N; ++i) off[i + 1] = off[i] + round_up(spans[i].bytes, 256);
    int rc = ensure_slot(ctx, 0, off[N], 0);
    if (rc) return rc;
    cudaStream_t st = ctx->pipe_stream[0];
    void* d[N];
    for (size_t i = 0; i < N; ++i) {
        d[i] = static_cast<uint8_t*>(ctx->pipe_in[0]) + off[i];
        if (spans[i].up && spans[i].bytes)
            CC_CUDA(cudaMemcpyAsync(d[i], spans[i].up, spans[i].bytes, cudaMemcpyHostToDevice, st));
    }
    if ((rc = body(d, st))) return rc;
    for (size_t i = 0; i < N; ++i)
        if (spans[i].down && spans[i].bytes)
            CC_CUDA(cudaMemcpyAsync(spans[i].down, d[i], spans[i].bytes, cudaMemcpyDeviceToHost, st));
    CC_CUDA(cudaStreamSynchronize(st));
    return CC_OK;
}

}  // namespace cc

using namespace cc;

extern "C" {

int cc_abi_version(void) { return CC_ABI_VERSION; }

const char* cc_last_error_string(void) { return g_err; }

int cc_device_count(int* count) {
    CC_REQUIRE(count != nullptr, "count is NULL");
    *count = 0;
    CC_CUDA(cudaGetDeviceCount(count));
    return CC_OK;
}

int cc_ctx_create(int device, cc_ctx** out) {
    CC_REQUIRE(out != nullptr, "out is NULL");
    *out = nullptr;
    int n = 0;
    CC_CUDA(cudaGetDeviceCount(&n));
    if (n == 0) return set_error(CC_ERR_NO_DEVICE, "no CUDA device (libcamcal_b200 has no CPU fallback)");
    CC_REQUIRE(device >= 0 && device < n, "device index out of range");
    CC_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    CC_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return set_error(CC_ERR_UNSUPPORTED, "device %d is sm_%d%d; libcamcal_b200 carries sm_100a code only",
                         device, prop.major, prop.minor);
    cc_ctx* ctx = new (std::nothrow) cc_ctx();
    if (!ctx) return set_error(CC_ERR_NOMEM, "out of host memory");
    memset(ctx, 0, sizeof(*ctx));
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    ctx->cc_major = prop.major;
    ctx->cc_minor = prop.minor;
    *out = ctx;
    return CC_OK;
}

int cc_ctx_destroy(cc_ctx* ctx) {
    if (!ctx) return CC_OK;
    cudaSetDevice(ctx->device);
    for (int k = 0; k < cc_ctx::NSLOT; ++k) {
        if (ctx->pipe_stream[k]) { cudaStreamSynchronize(ctx->pipe_stream[k]); cudaStreamDestroy(ctx->pipe_stream[k]); }
        if (ctx->pipe_in[k]) cudaFree(ctx->pipe_in[k]);
        if (ctx->pipe_out[k]) cudaFree(ctx->pipe_out[k]);
    }
    if (ctx->jtj_scratch) cudaFree(ctx->jtj_scratch);
    if (ctx->scratch_event) cudaEventDestroy(ctx->scratch_event);
    lm_free_workspace(ctx);
    comm_free(ctx);
    rectify_free_plans(ctx);
    rectify_free_sched(ctx);
    ingest_free(ctx);
    point_table_free(ctx);
    delete ctx;
    return CC_OK;
}

int cc_ctx_device(const cc_ctx* ctx, int* device) {
    CC_REQUIRE(ctx && device, "NULL argument");
    *device = ctx->device;
    return CC_OK;
}

int cc_ctx_synchronize(cc_ctx* ctx) {
    CC_GUARD;
    int rc = enter(ctx);
    if (rc) return rc;
    CC_CUDA(cudaDeviceSynchronize());
    return CC_OK;
}

int cc_ctx_launch_count(const cc_ctx* ctx, uint64_t* count) {
    CC_REQUIRE(ctx && count, "NULL argument");
    *count = ctx->launches;
    return CC_OK;
}

int cc_host_alloc(void** ptr, size_t bytes) {
    CC_REQUIRE(ptr != nullptr, "ptr is NULL");
    CC_CUDA(cudaHostAlloc(ptr, bytes ? bytes : 1, cudaHostAllocPortable));
    return CC_OK;
}
int cc_host_free(void* ptr) {
    if (ptr) CC_CUDA(cudaFreeHost(ptr));
    return CC_OK;
}
int cc_host_register(void* ptr, size_t bytes) {
    CC_REQUIRE(ptr != nullptr && bytes > 0, "bad host range");
    CC_CUDA(cudaHostRegister(ptr, bytes, cudaHostRegisterPortable));
    return CC_OK;
}
int cc_host_unregister(void* ptr) {
    CC_REQUIRE(ptr != nullptr, "ptr is NULL");
    CC_CUDA(cudaHostUnregister(ptr));
    return CC_OK;
}

// ---- point maps ------------------------------------------------------------------
int cc_img2world_f64(cc_ctx* ctx, const cc_intr* intr, const cc_view* view, const double* row,
                     const double* col, double* x, double* y, double* z, size_t n, void* stream) {
    return points_device(ctx, intr, view, 1, nullptr, n, soa_img2world(row, col, x, y, z), stream);
}
int cc_img2world_f32(cc_ctx* ctx, const cc_intr* intr, const cc_view* view, const float* row,
                     const float* col, float* x, float* y, float* z, size_t n, void* stream) {
    return points_device(ctx, intr, view, 1, nullptr, n, soa_img2world(row, col, x, y, z), stream);
}
int cc_world2img_f64(cc_ctx* ctx, const cc_intr* intr, const cc_view* view, const double* x,
                     const double* y, const double* z, double* row, double* col, size_t n,
                     void* stream) {
    return points_device(ctx, intr, view, 1, nullptr, n, soa_world2img(x, y, z, row, col), stream);
}
int cc_world2img_f32(cc_ctx* ctx, const cc_intr* intr, const cc_view* view, const float* x,
                     const float* y, const float* z, float* row, float* col, size_t n,
                     void* stream) {
    return points_device(ctx, intr, view, 1, nullptr, n, soa_world2img(x, y, z, row, col), stream);
}

int cc_img2world_f64_host(cc_ctx* ctx, const cc_intr* intr, const cc_view* view, const double* row,
                          const double* col, double* x, double* y, double* z, size_t n) {
    return points_host(ctx, intr, view, 1, nullptr, n, soa_img2world(row, col, x, y, z));
}
int cc_img2world_f32_host(cc_ctx* ctx, const cc_intr* intr, const cc_view* view, const float* row,
                          const float* col, float* x, float* y, float* z, size_t n) {
    return points_host(ctx, intr, view, 1, nullptr, n, soa_img2world(row, col, x, y, z));
}
int cc_world2img_f64_host(cc_ctx* ctx, const cc_intr* intr, const cc_view* view, const double* x,
                          const double* y, const double* z, double* row, double* col, size_t n) {
    return points_host(ctx, intr, view, 1, nullptr, n, soa_world2img(x, y, z, row, col));
}
int cc_world2img_f32_host(cc_ctx* ctx, const cc_intr* intr, const cc_view* view, const float* x,
                          const float* y, const float* z, float* row, float* col, size_t n) {
    return points_host(ctx, intr, view, 1, nullptr, n, soa_world2img(x, y, z, row, col));
}

int cc_img2world_f64_views(cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews, const size_t* offsets,
                           const double* row, const double* col, double* x, double* y, double* z, void* stream) {
    return points_device(ctx, intr, views, nviews, offsets, std::nullopt, soa_img2world(row, col, x, y, z), stream);
}
int cc_img2world_f32_views(cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews, const size_t* offsets,
                           const float* row, const float* col, float* x, float* y, float* z, void* stream) {
    return points_device(ctx, intr, views, nviews, offsets, std::nullopt, soa_img2world(row, col, x, y, z), stream);
}
int cc_world2img_f64_views(cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews, const size_t* offsets,
                           const double* x, const double* y, const double* z, double* row, double* col, void* stream) {
    return points_device(ctx, intr, views, nviews, offsets, std::nullopt, soa_world2img(x, y, z, row, col), stream);
}
int cc_world2img_f32_views(cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews, const size_t* offsets,
                           const float* x, const float* y, const float* z, float* row, float* col, void* stream) {
    return points_device(ctx, intr, views, nviews, offsets, std::nullopt, soa_world2img(x, y, z, row, col), stream);
}
int cc_img2world_f64_views_host(cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews,
                                const size_t* offsets, const double* row, const double* col, double* x, double* y,
                                double* z) {
    return points_host(ctx, intr, views, nviews, offsets, std::nullopt, soa_img2world(row, col, x, y, z));
}
int cc_img2world_f32_views_host(cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews,
                                const size_t* offsets, const float* row, const float* col, float* x, float* y,
                                float* z) {
    return points_host(ctx, intr, views, nviews, offsets, std::nullopt, soa_img2world(row, col, x, y, z));
}
int cc_world2img_f64_views_host(cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews,
                                const size_t* offsets, const double* x, const double* y, const double* z,
                                double* row, double* col) {
    return points_host(ctx, intr, views, nviews, offsets, std::nullopt, soa_world2img(x, y, z, row, col));
}
int cc_world2img_f32_views_host(cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews,
                                const size_t* offsets, const float* x, const float* y, const float* z,
                                float* row, float* col) {
    return points_host(ctx, intr, views, nviews, offsets, std::nullopt, soa_world2img(x, y, z, row, col));
}

int cc_img2world_f64_aos(cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews, const size_t* offsets,
                         const double* rc, double* out, int out_dim, size_t n, void* stream) {
    return points_device(ctx, intr, views, nviews, offsets, n, aos_img2world(rc, out, out_dim), stream);
}
int cc_img2world_f32_aos(cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews, const size_t* offsets,
                         const float* rc, float* out, int out_dim, size_t n, void* stream) {
    return points_device(ctx, intr, views, nviews, offsets, n, aos_img2world(rc, out, out_dim), stream);
}
int cc_world2img_f64_aos(cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews, const size_t* offsets,
                         const double* pts, int in_dim, double* rc, size_t n, void* stream) {
    return points_device(ctx, intr, views, nviews, offsets, n, aos_world2img(pts, in_dim, rc), stream);
}
int cc_world2img_f32_aos(cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews, const size_t* offsets,
                         const float* pts, int in_dim, float* rc, size_t n, void* stream) {
    return points_device(ctx, intr, views, nviews, offsets, n, aos_world2img(pts, in_dim, rc), stream);
}
int cc_img2world_f64_aos_host(cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews,
                              const size_t* offsets, const double* rc, double* out, int out_dim, size_t n) {
    return points_host(ctx, intr, views, nviews, offsets, n, aos_img2world(rc, out, out_dim));
}
int cc_img2world_f32_aos_host(cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews,
                              const size_t* offsets, const float* rc, float* out, int out_dim, size_t n) {
    return points_host(ctx, intr, views, nviews, offsets, n, aos_img2world(rc, out, out_dim));
}
int cc_world2img_f64_aos_host(cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews,
                              const size_t* offsets, const double* pts, int in_dim, double* rc, size_t n) {
    return points_host(ctx, intr, views, nviews, offsets, n, aos_world2img(pts, in_dim, rc));
}
int cc_world2img_f32_aos_host(cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews,
                              const size_t* offsets, const float* pts, int in_dim, float* rc, size_t n) {
    return points_host(ctx, intr, views, nviews, offsets, n, aos_world2img(pts, in_dim, rc));
}

// ---- rectification ---------------------------------------------------------------
int cc_rectify_f32c1(cc_ctx* ctx, const cc_intr* intr, const cc_view* view, double ratio,
                     const int64_t axs_min[2], const float* src, float* dst, int sz1, int sz2,
                     size_t pitch, size_t frame_stride, int nframes, float fill, unsigned flags,
                     void* stream) {
    return rectify_device(ctx, intr, view, 1, &ratio, axs_min, src, dst, {sz1, sz2, pitch, frame_stride, nframes}, fill,
                          flags, stream, false);
}

int cc_rectify_u8c3(cc_ctx* ctx, const cc_intr* intr, const cc_view* view, double ratio,
                    const int64_t axs_min[2], const uint8_t* src, uint8_t* dst, int sz1, int sz2,
                    size_t pitch, size_t frame_stride, int nframes, const uint8_t fill[3],
                    unsigned flags, void* stream) {
    return rectify_device(ctx, intr, view, 1, &ratio, axs_min, src, dst, {sz1, sz2, pitch, frame_stride, nframes}, fill,
                          flags, stream, false);
}

int cc_rectify_f32c1_views(cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews, const double* ratios,
                           const int64_t* axs_mins, const float* src, float* dst, int sz1, int sz2, size_t pitch,
                           size_t frame_stride, int frames_per_view, float fill, unsigned flags, void* stream) {
    return rectify_device(ctx, intr, views, nviews, ratios, axs_mins, src, dst,
                          {sz1, sz2, pitch, frame_stride, frames_per_view}, fill, flags, stream, true);
}

int cc_rectify_u8c3_views(cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews, const double* ratios,
                          const int64_t* axs_mins, const uint8_t* src, uint8_t* dst, int sz1, int sz2, size_t pitch,
                          size_t frame_stride, int frames_per_view, const uint8_t fill[3], unsigned flags,
                          void* stream) {
    return rectify_device(ctx, intr, views, nviews, ratios, axs_mins, src, dst,
                          {sz1, sz2, pitch, frame_stride, frames_per_view}, fill, flags, stream, true);
}

int cc_rectify_f32c1_host(cc_ctx* ctx, const cc_intr* intr, const cc_view* view, double ratio,
                          const int64_t axs_min[2], const float* src, float* dst, int sz1, int sz2,
                          size_t pitch, size_t frame_stride, int nframes, float fill,
                          unsigned flags) {
    return rectify_host(ctx, intr, view, 1, &ratio, axs_min, src, dst, {sz1, sz2, pitch, frame_stride, nframes}, fill,
                        flags, false);
}

int cc_rectify_u8c3_host(cc_ctx* ctx, const cc_intr* intr, const cc_view* view, double ratio,
                         const int64_t axs_min[2], const uint8_t* src, uint8_t* dst, int sz1,
                         int sz2, size_t pitch, size_t frame_stride, int nframes,
                         const uint8_t fill[3], unsigned flags) {
    return rectify_host(ctx, intr, view, 1, &ratio, axs_min, src, dst, {sz1, sz2, pitch, frame_stride, nframes}, fill,
                        flags, false);
}

// many views from host memory
int cc_rectify_views_f32c1_host(cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews,
                                const double* ratios, const int64_t* axs_mins, const float* src, float* dst,
                                int sz1, int sz2, size_t pitch, size_t frame_stride, int frames_per_view,
                                float fill, unsigned flags) {
    return rectify_host(ctx, intr, views, nviews, ratios, axs_mins, src, dst,
                        {sz1, sz2, pitch, frame_stride, frames_per_view}, fill, flags, true);
}

int cc_rectify_views_u8c3_host(cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews,
                               const double* ratios, const int64_t* axs_mins, const uint8_t* src, uint8_t* dst,
                               int sz1, int sz2, size_t pitch, size_t frame_stride, int frames_per_view,
                               const uint8_t fill[3], unsigned flags) {
    return rectify_host(ctx, intr, views, nviews, ratios, axs_mins, src, dst,
                        {sz1, sz2, pitch, frame_stride, frames_per_view}, fill, flags, true);
}

int cc_rectify_map_f64(cc_ctx* ctx, const cc_intr* intr, const cc_view* view, double ratio,
                       const int64_t axs_min[2], double* map_row, double* map_col, int sz1, int sz2,
                       size_t pitch, void* stream) {
    return rectify_map(ctx, intr, view, ratio, axs_min, map_row, map_col, sz1, sz2, pitch, stream);
}

int cc_rectify_map_f32(cc_ctx* ctx, const cc_intr* intr, const cc_view* view, double ratio,
                       const int64_t axs_min[2], float* map_row, float* map_col, int sz1, int sz2,
                       size_t pitch, void* stream) {
    return rectify_map(ctx, intr, view, ratio, axs_min, map_row, map_col, sz1, sz2, pitch, stream);
}

int cc_jpeg_info(const uint8_t* jpeg, size_t length, int* sz1, int* sz2, int* channels) {
    CC_REQUIRE(jpeg && length > 0, "NULL / empty JPEG stream");
    return jpeg_info(jpeg, length, sz1, sz2, channels);
}

int cc_jpeg_decode_u8c3(cc_ctx* ctx, const uint8_t* const* jpegs, const size_t* lengths, int n, uint8_t* dst,
                        int sz1, int sz2, size_t pitch, size_t frame_stride, void* stream) {
    CC_REQUIRE(ctx != nullptr, "NULL context");
    CC_REQUIRE(n >= 0, "negative image count");
    if (n == 0) return CC_OK;
    CC_REQUIRE(jpegs && lengths && dst, "NULL argument");
    CC_REQUIRE(sz1 > 0 && sz2 > 0 && pitch >= (size_t)sz1, "bad frame size / pitch");
    CC_REQUIRE(n <= 1 || frame_stride >= pitch * (size_t)(sz2 - 1) + sz1, "frames overlap");
    for (int i = 0; i < n; ++i) CC_REQUIRE(jpegs[i] && lengths[i] > 0, "NULL / empty JPEG stream");
    int rc;
    CC_GUARD;
    if ((rc = enter(ctx))) return rc;
    return jpeg_decode_u8c3(ctx, jpegs, lengths, n, dst, sz1, sz2, pitch, frame_stride, (cudaStream_t)stream);
}

// get_ratio, src/plot_calibration.jl:8-13
int cc_get_ratio(const double* rows, const double* cols, int n1, int n2, double checker_size,
                 double* ratio) {
    CC_REQUIRE(rows && cols && ratio, "NULL argument");
    CC_REQUIRE(n1 >= 2 && n2 >= 2, "need at least 2x2 corners");
    CC_REQUIRE(checker_size != 0.0, "checker_size must be non-zero");
    double s1 = 0.0, s2 = 0.0;
    for (int b = 0; b < n2; ++b)
        for (int a = 0; a + 1 < n1; ++a) {
            const double dr = rows[a + 1 + n1 * b] - rows[a + n1 * b];
            const double dc = cols[a + 1 + n1 * b] - cols[a + n1 * b];
            s1 += std::sqrt(dr * dr + dc * dc);
        }
    for (int b = 0; b + 1 < n2; ++b)
        for (int a = 0; a < n1; ++a) {
            const double dr = rows[a + n1 * (b + 1)] - rows[a + n1 * b];
            const double dc = cols[a + n1 * (b + 1)] - cols[a + n1 * b];
            s2 += std::sqrt(dr * dr + dc * dc);
        }
    const double l = (s1 / (double)((n1 - 1) * n2) + s2 / (double)(n1 * (n2 - 1))) / 2.0;
    *ratio = l / checker_size;
    return CC_OK;
}

// get_axes, src/plot_calibration.jl:1-6 (round(Int, .) = round-half-even = rint)
int cc_get_axes(double ratio, double checker_size, int n1, int n2, int sz1, int sz2,
                int64_t axs_min[2]) {
    CC_REQUIRE(axs_min != nullptr, "axs_min is NULL");
    const double w1 = std::rint(ratio * checker_size * (double)(n1 - 1));
    const double w2 = std::rint(ratio * checker_size * (double)(n2 - 1));
    axs_min[0] = (int64_t)std::rint((w1 - (double)sz1) / 2.0);
    axs_min[1] = (int64_t)std::rint((w2 - (double)sz2) / 2.0);
    return CC_OK;
}

// ---- residual / Jacobian, calculate_errors ---------------------------------------
int cc_reproj_jtj_f64(cc_ctx* ctx, const cc_intr* intr, double aspect, const cc_view* views,
                      int nviews, const double* obj, const double* img, int ncorners,
                      double* per_view, double* shared, void* stream) {
    int rc = check_reproj_jtj(ctx, intr, views, nviews, obj, img, ncorners, per_view, shared, false);
    CC_GUARD;
    if (rc || (rc = enter(ctx))) return rc;
    return launch_reproj_jtj(ctx, intr, aspect, views, nviews, obj, img, ncorners, per_view, shared,
                             (cudaStream_t)stream);
}

int cc_reproj_jtj_f64_host(cc_ctx* ctx, const cc_intr* intr, double aspect, const cc_view* views,
                           int nviews, const double* obj, const double* img, int ncorners,
                           double* per_view, double* shared) {
    int rc = check_reproj_jtj(ctx, intr, views, nviews, obj, img, ncorners, per_view, shared, true);
    CC_GUARD;
    if (rc || (rc = enter(ctx))) return rc;
    const size_t nv = (size_t)nviews, nc = nviews > 0 ? (size_t)ncorners : 0;
    const HostSpan spans[] = {{views, nullptr, nv * sizeof(cc_view)},
                              {obj, nullptr, nc * 3 * sizeof(double)},
                              {img, nullptr, nv * nc * 2 * sizeof(double)},
                              {nullptr, per_view, nv * CC_PER_VIEW * sizeof(double)},
                              {nullptr, shared, CC_SHARED * sizeof(double)}};
    return stage_host(ctx, spans, [&](void* const* d, cudaStream_t st) {
        return launch_reproj_jtj(ctx, intr, aspect, (const cc_view*)d[0], nviews, (const double*)d[1],
                                 (const double*)d[2], ncorners, (double*)d[3], (double*)d[4], st);
    });
}

int cc_calculate_errors_f64(cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews,
                            const double* obj, const double* img, int n1, int n2,
                            const double* inv_rows, const double* inv_cols, int inverse_samples,
                            double* sums, void* stream) {
    int rc = check_calculate_errors(ctx, intr, views, nviews, obj, img, n1, n2, inv_rows, inv_cols,
                                    inverse_samples, sums, false);
    CC_GUARD;
    if (rc || (rc = enter(ctx))) return rc;
    return launch_calc_errors(ctx, intr, views, nviews, obj, img, n1, n2, inv_rows, inv_cols,
                              inverse_samples, sums, (cudaStream_t)stream);
}

// host arrays in, the four raw sums out: what calculate_errors (src/buildcalibrations.jl:37-67) needs from a
// caller that holds the detections on the host, like the reference does
int cc_calculate_errors_f64_host(cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews,
                                 const double* obj, const double* img, int n1, int n2, const double* inv_rows,
                                 const double* inv_cols, int inverse_samples, double* sums) {
    int rc = check_calculate_errors(ctx, intr, views, nviews, obj, img, n1, n2, inv_rows, inv_cols,
                                    inverse_samples, sums, true);
    CC_GUARD;
    if (rc || (rc = enter(ctx))) return rc;
    const size_t nv = (size_t)nviews, nc = nviews > 0 ? (size_t)n1 * n2 : 0, ns = nv * inverse_samples;
    const HostSpan spans[] = {{views, nullptr, nv * sizeof(cc_view)},
                              {obj, nullptr, nc * 3 * sizeof(double)},
                              {img, nullptr, nv * nc * 2 * sizeof(double)},
                              {inv_rows, nullptr, ns * sizeof(double)},
                              {inv_cols, nullptr, ns * sizeof(double)},
                              {nullptr, sums, 4 * sizeof(double)}};
    return stage_host(ctx, spans, [&](void* const* d, cudaStream_t st) {
        return launch_calc_errors(ctx, intr, (const cc_view*)d[0], nviews, (const double*)d[1], (const double*)d[2],
                                  n1, n2, (const double*)d[3], (const double*)d[4], inverse_samples, (double*)d[5], st);
    });
}

// ---- Levenberg-Marquardt -----------------------------------------------------------
int cc_lm_schur_f64(cc_ctx* ctx, const double* per_view, int nviews, double lambda, double* yz,
                    double* schur, void* stream) {
    int rc = check_lm_schur(ctx, per_view, nviews, lambda, yz, schur);
    CC_GUARD;
    if (rc || (rc = enter(ctx))) return rc;
    return launch_lm_schur(ctx, per_view, nviews, lambda, yz, schur, (cudaStream_t)stream);
}

int cc_lm_update_f64(cc_ctx* ctx, const double* shared, const double* schur, double lambda,
                     unsigned free_mask, const double* yz, const cc_view* views_in, int nviews,
                     cc_view* views_out, double* delta, void* stream) {
    int rc = check_lm_update(ctx, shared, schur, lambda, free_mask, yz, views_in, nviews, views_out, delta);
    CC_GUARD;
    if (rc || (rc = enter(ctx))) return rc;
    return launch_lm_update(ctx, shared, schur, lambda, free_mask, yz, views_in, nviews, views_out, delta,
                            (cudaStream_t)stream);
}

int cc_lm_fit_f64_host(cc_ctx* ctx, cc_intr* intr, double aspect, unsigned free_mask, cc_view* views,
                       int nviews, const double* obj, const double* img, int ncorners, int max_iter,
                       double eps, double* rms, int* iterations) {
    int rc = check_lm_fit(ctx, intr, aspect, free_mask, views, nviews, obj, img, ncorners, max_iter, eps, true);
    CC_GUARD;
    if (rc || (rc = enter(ctx))) return rc;
    const size_t nv = (size_t)nviews, nc = (size_t)ncorners;
    const HostSpan spans[] = {{views, views, nv * sizeof(cc_view)},
                              {obj, nullptr, nc * 3 * sizeof(double)},
                              {img, nullptr, nv * nc * 2 * sizeof(double)}};
    return stage_host(ctx, spans, [&](void* const* d, cudaStream_t st) {
        return lm_fit_device(ctx, intr, aspect, free_mask, (cc_view*)d[0], nviews, (const double*)d[1],
                             (const double*)d[2], ncorners, max_iter, eps, rms, iterations, st);
    });
}

int cc_lm_fit_f64(cc_ctx* ctx, cc_intr* intr, double aspect, unsigned free_mask, cc_view* views, int nviews,
                  const double* obj, const double* img, int ncorners, int max_iter, double eps, double* rms,
                  int* iterations, void* stream) {
    int rc = check_lm_fit(ctx, intr, aspect, free_mask, views, nviews, obj, img, ncorners, max_iter, eps, false);
    CC_GUARD;
    if (rc || (rc = enter(ctx))) return rc;
    return lm_fit_device(ctx, intr, aspect, free_mask, views, nviews, obj, img, ncorners, max_iter, eps, rms,
                         iterations, (cudaStream_t)stream);
}

int cc_lm_initial_guess_f64(cc_ctx* ctx, const double* obj, const double* img, int nviews, int ncorners, int sz1,
                            int sz2, double aspect, cc_intr* intr, cc_view* views, void* stream) {
    int rc = check_initial_guess(ctx, obj, img, nviews, ncorners, sz1, sz2, intr, views);
    CC_GUARD;
    if (rc || (rc = enter(ctx))) return rc;
    return launch_initial_guess(ctx, obj, img, nviews, ncorners, sz1, sz2, aspect, intr, views, (cudaStream_t)stream);
}

int cc_ctx_collective_count(const cc_ctx* ctx, uint64_t* count) {
    CC_REQUIRE(ctx && count, "NULL argument");
    *count = ctx->collectives;
    return CC_OK;
}

}  // extern "C"
