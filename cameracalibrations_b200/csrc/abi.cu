// abi.cu -- the extern "C" surface of libcamcal_b200.so (include/camcal_b200.h):
// argument checking, per-device context, and the chunked host pipeline behind the
// *_host entry points.  No compute lives here and nothing here can fall back to the CPU.
#include <algorithm>
#include <vector>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cmath>
#include <new>
#include <optional>

#include "common.cuh"

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

// launchers implemented in the kernel translation units
template <typename T>
int point_table_upload(cc_ctx*, bool, const ChainD*, int, const size_t*, cudaStream_t, PointTable*);
int point_table_release(cc_ctx*, cudaStream_t);
template <typename T>
int launch_points(cc_ctx*, const PointSrc&, const PointIO<T>&, size_t, cudaStream_t);
int check_rect_args(const int64_t axs_min[2], int sz1, int sz2, size_t pitch, size_t frame_stride,
                    int nframes, double ratio);
int launch_rectify_f32c1(cc_ctx*, const ChainD&, double, const int64_t[2], const float*, float*, int,
                         int, size_t, size_t, int, float, unsigned, cudaStream_t);
int launch_rectify_u8c3(cc_ctx*, const ChainD&, double, const int64_t[2], const uint8_t*, uint8_t*,
                        int, int, size_t, size_t, int, const uint8_t[3], unsigned, cudaStream_t);
int launch_rectify_f32c1_views(cc_ctx*, const ChainD*, const double*, const int64_t*, int, const float*, float*, int, int,
                               size_t, size_t, int, float, unsigned, cudaStream_t, bool*);
int launch_rectify_u8c3_views(cc_ctx*, const ChainD*, const double*, const int64_t*, int, const uint8_t*, uint8_t*, int,
                              int, size_t, size_t, int, const uint8_t[3], unsigned, cudaStream_t, bool*);
int rectify_views_per_launch();
struct RectViewsHost;
int rect_vh_begin(cc_ctx*, const ChainD*, const double*, const int64_t*, int, int, int, size_t, int, int, bool,
                  RectViewsHost**);
int rect_vh_prepare(RectViewsHost*, int);
int rect_vh_launch_f32c1(RectViewsHost*, int, int, int, const float*, float*, float, unsigned, cudaStream_t, bool*);
int rect_vh_launch_u8c3(RectViewsHost*, int, int, int, const uint8_t*, uint8_t*, const uint8_t[3], unsigned, cudaStream_t,
                        bool*);
void rect_vh_retire(RectViewsHost*, int);
int rect_vh_end(RectViewsHost*);
int launch_rectify_map(cc_ctx*, const ChainD&, double, const int64_t[2], double*, double*, int, int,
                       size_t, cudaStream_t);
int launch_rectify_map_f32(cc_ctx*, const ChainD&, double, const int64_t[2], float*, float*, int, int,
                           size_t, cudaStream_t);
int launch_reproj_jtj(cc_ctx*, const cc_intr*, double, const cc_view*, int, const double*,
                      const double*, int, double*, double*, cudaStream_t);
int launch_calc_errors(cc_ctx*, const cc_intr*, const cc_view*, int, const double*, const double*,
                       int, int, const double*, const double*, int, double*, cudaStream_t);
int launch_lm_schur(cc_ctx*, const double*, int, double, double*, double*, cudaStream_t);
int lm_fit_host(cc_ctx*, cc_intr*, double, unsigned, cc_view*, int, const double*, const double*, int, int, double,
                double*, int*);
int launch_lm_update(cc_ctx*, const double*, const double*, double, unsigned, const double*, const cc_view*,
                     int, cc_view*, double*, cudaStream_t);
int lm_fit_device(cc_ctx*, cc_intr*, double, unsigned, cc_view*, int, const double*, const double*, int, int, double,
                  double*, int*, cudaStream_t);
int launch_initial_guess(cc_ctx*, const double*, const double*, int, int, int, int, double, cc_intr*, cc_view*,
                         cudaStream_t);

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

static int cuda_check(cudaError_t e, const char* what) { return e == cudaSuccess ? (int)CC_OK : cuda_fail(e, what); }

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

// frames: chunk = a few whole frames (~32 MB per stage)
template <typename PX, typename LAUNCH>
static int rectify_host(cc_ctx* ctx, const PX* src, PX* dst, int sz1, int sz2, size_t pitch,
                        size_t frame_stride, int nframes, size_t px_bytes, LAUNCH launch) {
    int rc;
    CC_GUARD;
    if ((rc = enter(ctx))) return rc;
    const size_t frame_elems = pitch * (size_t)sz2;          // device frames are stored pitch*sz2
    const size_t frame_bytes = frame_elems * px_bytes;
    int per = 0;
    const std::vector<int> chunks = chunk_schedule(nframes, frame_bytes, nframes, &per);
    const bool dense = frame_stride == frame_elems && pitch == (size_t)sz1;
    for (int f0 = 0, it = 0, m = 0; f0 < nframes; f0 += m, ++it) {
        const int k = it % cc_ctx::NSLOT;
        m = chunks[it];
        // +64 bytes: vector gathers may touch the aligned word holding the last texel
        if ((rc = ensure_slot(ctx, k, per * frame_bytes + 64, per * frame_bytes + 64))) return rc;
        cudaStream_t st = ctx->pipe_stream[k];
        uint8_t* din = static_cast<uint8_t*>(ctx->pipe_in[k]);
        uint8_t* dout = static_cast<uint8_t*>(ctx->pipe_out[k]);
        const uint8_t* hs = reinterpret_cast<const uint8_t*>(src) + (size_t)f0 * frame_stride * px_bytes;
        uint8_t* hd = reinterpret_cast<uint8_t*>(dst) + (size_t)f0 * frame_stride * px_bytes;
        if (dense) {
            CC_CUDA(cudaMemcpyAsync(din, hs, (size_t)m * frame_bytes, cudaMemcpyHostToDevice, st));
        } else {
            for (int f = 0; f < m; ++f)
                CC_CUDA(cudaMemcpy2DAsync(din + (size_t)f * frame_bytes, pitch * px_bytes,
                                          hs + (size_t)f * frame_stride * px_bytes, pitch * px_bytes,
                                          (size_t)sz1 * px_bytes, sz2, cudaMemcpyHostToDevice, st));
        }
        if ((rc = launch(reinterpret_cast<const PX*>(din), reinterpret_cast<PX*>(dout), frame_elems, m, st)))
            return rc;
        if (dense) {
            CC_CUDA(cudaMemcpyAsync(hd, dout, (size_t)m * frame_bytes, cudaMemcpyDeviceToHost, st));
        } else {
            for (int f = 0; f < m; ++f)
                CC_CUDA(cudaMemcpy2DAsync(hd + (size_t)f * frame_stride * px_bytes, pitch * px_bytes,
                                          dout + (size_t)f * frame_bytes, pitch * px_bytes,
                                          (size_t)sz1 * px_bytes, sz2, cudaMemcpyDeviceToHost, st));
        }
    }
    return drain(ctx);
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
    int rc = check_params(ctx, intr, view);
    if (rc) return rc;
    if ((rc = check_rect_args(axs_min, sz1, sz2, pitch, frame_stride, nframes, ratio))) return rc;
    CC_REQUIRE(nframes == 0 || (src && dst), "NULL frame pointer");
    CC_REQUIRE(nframes == 0 || (const void*)src != (const void*)dst, "rectification is not in place: src == dst");
    CC_GUARD;
    if ((rc = enter(ctx))) return rc;
    ChainD ch;
    build_chain(intr, view, &ch);
    return launch_rectify_f32c1(ctx, ch, ratio, axs_min, src, dst, sz1, sz2, pitch, frame_stride,
                                nframes, fill, flags, (cudaStream_t)stream);
}

int cc_rectify_u8c3(cc_ctx* ctx, const cc_intr* intr, const cc_view* view, double ratio,
                    const int64_t axs_min[2], const uint8_t* src, uint8_t* dst, int sz1, int sz2,
                    size_t pitch, size_t frame_stride, int nframes, const uint8_t fill[3],
                    unsigned flags, void* stream) {
    int rc = check_params(ctx, intr, view);
    if (rc) return rc;
    if ((rc = check_rect_args(axs_min, sz1, sz2, pitch, frame_stride, nframes, ratio))) return rc;
    CC_REQUIRE(nframes == 0 || (src && dst), "NULL frame pointer");
    CC_REQUIRE(nframes == 0 || (const void*)src != (const void*)dst, "rectification is not in place: src == dst");
    CC_REQUIRE(fill != nullptr, "fill is NULL");
    CC_GUARD;
    if ((rc = enter(ctx))) return rc;
    ChainD ch;
    build_chain(intr, view, &ch);
    return launch_rectify_u8c3(ctx, ch, ratio, axs_min, src, dst, sz1, sz2, pitch, frame_stride,
                               nframes, fill, flags, (cudaStream_t)stream);
}

}  // extern "C"

// the argument rules of the many-view rectification calls (device and host forms alike)
static int check_rect_views(cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews, const double* ratios,
                            const int64_t* axs_mins, const void* src, const void* dst, int sz1, int sz2, size_t pitch,
                            size_t frame_stride, int frames_per_view) {
    CC_REQUIRE(ctx && intr && (nviews == 0 || (views && ratios && axs_mins)), "NULL argument");
    CC_REQUIRE(nviews >= 0 && frames_per_view >= 0, "bad counts");
    CC_REQUIRE((long long)nviews * frames_per_view <= 65535, "at most 65535 frames per call");
    int rc = CC_OK;
    for (int v = 0; v < nviews; ++v) {
        if ((rc = check_params(ctx, intr, views + v))) return rc;
        if ((rc = check_rect_args(axs_mins + 2 * v, sz1, sz2, pitch, frame_stride, frames_per_view, ratios[v]))) return rc;
    }
    CC_REQUIRE(nviews * frames_per_view == 0 || (src && dst), "NULL frame pointer");
    CC_REQUIRE(nviews * frames_per_view == 0 || src != dst, "rectification is not in place: src == dst");
    CC_REQUIRE(nviews * frames_per_view <= 1 || frame_stride >= pitch * (size_t)(sz2 - 1) + sz1, "frames overlap");
    return CC_OK;
}

// Frames with DIFFERENT views in one call: the reference's plot loop rectifies every calibration
// image with its own extrinsic (src/plot_calibration.jl:36-42).  frames [v * frames_per_view,
// (v + 1) * frames_per_view) use views[v], ratios[v], axs_mins[2v .. 2v+1].  Every view is one
// launch with its own cached tile plan.
template <typename P, typename F, typename G>
static int rectify_views(cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews, const double* ratios,
                         const int64_t* axs_mins, const P* src, P* dst, int sz1, int sz2, size_t pitch,
                         size_t frame_stride, int frames_per_view, int channels, cudaStream_t stream, F launch,
                         G launch_group) {
    int rc = check_rect_views(ctx, intr, views, nviews, ratios, axs_mins, src, dst, sz1, sz2, pitch, frame_stride,
                              frames_per_view);
    if (rc) return rc;
    CC_GUARD;
    if ((rc = enter(ctx))) return rc;
    if (nviews == 0 || frames_per_view == 0) return CC_OK;
    // Groups of up to 64 views in ONE launch each (rectify.cu: launch_rectify_*_views) when the layout can be
    // staged; CAMCAL_VIEWS_SINGLE=0 (tuning knob) or a group that cannot be staged: one launch per view, below.
    std::vector<ChainD> chs((size_t)nviews);
    for (int v = 0; v < nviews; ++v) build_chain(intr, views + v, &chs[v]);
    std::vector<char> done((size_t)nviews, 0);
    bool single = true;
    if (const char* e = getenv("CAMCAL_VIEWS_SINGLE")) single = atoi(e) != 0;
    int ndone = 0;
    const int per = rectify_views_per_launch();
    for (int v0 = 0; single && v0 < nviews; v0 += per) {
        const int nv = std::min(per, nviews - v0);
        const size_t off = (size_t)v0 * frames_per_view * frame_stride * channels;
        bool ok = false;
        if ((rc = launch_group(chs.data() + v0, ratios + v0, axs_mins + 2 * v0, nv, src + off, dst + off, stream, &ok))) return rc;
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
        CC_CUDA(cudaEventRecord(fork, stream));
        for (int k = 0; k < lanes; ++k) {
            if ((rc = ensure_stream(ctx, k))) return rc;
            CC_CUDA(cudaStreamWaitEvent(ctx->pipe_stream[k], fork, 0));
        }
    }
    for (int v = 0; v < nviews; ++v) {
        if (done[v]) continue;
        const size_t off = (size_t)v * frames_per_view * frame_stride * channels;
        cudaStream_t st = lanes > 1 ? ctx->pipe_stream[v % lanes] : stream;
        if ((rc = launch(chs[v], ratios[v], axs_mins + 2 * v, src + off, dst + off, st))) break;
    }
    if (lanes > 1) {                                  // join even after an error: nothing stays forked
        for (int k = 0; k < lanes; ++k) {
            if (cudaEventCreateWithFlags(&join[k], cudaEventDisableTiming) == cudaSuccess) {
                cudaEventRecord(join[k], ctx->pipe_stream[k]);
                cudaStreamWaitEvent(stream, join[k], 0);
                cudaEventDestroy(join[k]);            // released once the wait has consumed it
            }
        }
        cudaEventDestroy(fork);
    }
    return rc;
}


// Frames of many views from host memory in one call (cc_rectify_views_*_host): the chunk pipeline of rectify_host
// over the frame axis of the whole call.  Chunks ignore view boundaries and span at most two 64-view groups (a
// chunk holds at most 64 views' frames).  A chunk makes one staged launch per group it touches, over the window of
// that group's frames it holds (rectify.cu: RectViewsHost); a group without a staged plan runs the window's views
// through the single-view kernels on the chunk's own slot stream.  The next group's plan is built on host threads
// while the device streams the current one: before waiting for it, the uploads of the next NSLOT chunks are
// enqueued.  LAUNCH_GROUP(vh, g, w0, wn, src, dst, st, ok) / LAUNCH_ONE(v, src, dst, nframes, st).
template <typename PX, typename LAUNCH_GROUP, typename LAUNCH_ONE>
static int rectify_views_host(cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews, const double* ratios,
                              const int64_t* axs_mins, const PX* src, PX* dst, int sz1, int sz2, size_t pitch,
                              size_t frame_stride, int fpv, int pxb, unsigned flags, std::vector<ChainD>* chs,
                              LAUNCH_GROUP launch_group, LAUNCH_ONE launch_one) {
    int rc = check_rect_views(ctx, intr, views, nviews, ratios, axs_mins, src, dst, sz1, sz2, pitch, frame_stride, fpv);
    if (rc) return rc;
    CC_GUARD;
    if ((rc = enter(ctx))) return rc;
    if (nviews == 0 || fpv == 0) return CC_OK;
    chs->resize((size_t)nviews);
    for (int v = 0; v < nviews; ++v) build_chain(intr, views + v, &(*chs)[v]);
    const int nframes = nviews * fpv, gframes = rectify_views_per_launch() * fpv;
    const size_t frame_elems = pitch * (size_t)sz2;          // device frames are stored pitch*sz2
    const size_t frame_bytes = frame_elems * pxb;
    int per = 0;
    const std::vector<int> chunks = chunk_schedule(nframes, frame_bytes, gframes, &per);
    const int nchunks = (int)chunks.size();
    std::vector<int> first((size_t)nchunks + 1, 0);
    for (int c = 0; c < nchunks; ++c) first[c + 1] = first[c] + chunks[c];
    const bool dense = frame_stride == frame_elems && pitch == (size_t)sz1;
    const uint8_t* hsrc = reinterpret_cast<const uint8_t*>(src);
    uint8_t* hdst = reinterpret_cast<uint8_t*>(dst);
    RectViewsHost* vh = nullptr;
    if ((rc = rect_vh_begin(ctx, chs->data(), ratios, axs_mins, nviews, sz1, sz2, pitch, fpv, pxb,
                            !(flags & CC_GATHER_DIRECT), &vh)))
        return rc;
    std::vector<char> uploaded((size_t)nchunks, 0), prepared((size_t)((nframes + gframes - 1) / gframes), 0);
    // chunk c's frames to its slot (the slot's previous chunk, c - NSLOT, is enqueued in full by then)
    auto upload = [&](int c) -> int {
        if (c >= nchunks || uploaded[c]) return CC_OK;
        const int k = c % cc_ctx::NSLOT, m = chunks[c];
        int r = ensure_slot(ctx, k, per * frame_bytes + 64, per * frame_bytes + 64);   // +64: see rectify_host
        if (r) return r;
        uint8_t* din = static_cast<uint8_t*>(ctx->pipe_in[k]);
        const uint8_t* hs = hsrc + (size_t)first[c] * frame_stride * pxb;
        if (dense) {
            CC_CUDA(cudaMemcpyAsync(din, hs, (size_t)m * frame_bytes, cudaMemcpyHostToDevice, ctx->pipe_stream[k]));
        } else {
            for (int f = 0; f < m; ++f)
                CC_CUDA(cudaMemcpy2DAsync(din + (size_t)f * frame_bytes, pitch * pxb, hs + (size_t)f * frame_stride * pxb,
                                          pitch * pxb, (size_t)sz1 * pxb, sz2, cudaMemcpyHostToDevice, ctx->pipe_stream[k]));
        }
        uploaded[c] = 1;
        return CC_OK;
    };
    int retired = 0;                                        // groups whose chunks are all enqueued
    for (int c = 0; rc == CC_OK && c < nchunks; ++c) {
        const int f0 = first[c], m = chunks[c], g_lo = f0 / gframes, g_hi = (f0 + m - 1) / gframes;
        for (int gi = g_lo; rc == CC_OK && gi <= g_hi; ++gi) {
            if (prepared[gi]) continue;
            for (int j = 0; rc == CC_OK && j < cc_ctx::NSLOT; ++j) rc = upload(c + j);
            if (rc == CC_OK) rc = rect_vh_prepare(vh, gi);
            prepared[gi] = 1;
        }
        if (rc == CC_OK) rc = upload(c);
        if (rc) break;
        const int k = c % cc_ctx::NSLOT;
        cudaStream_t st = ctx->pipe_stream[k];
        uint8_t* din = static_cast<uint8_t*>(ctx->pipe_in[k]);
        uint8_t* dout = static_cast<uint8_t*>(ctx->pipe_out[k]);
        for (int gi = g_lo; rc == CC_OK && gi <= g_hi; ++gi) {
            const int a = std::max(f0, gi * gframes), b = std::min(f0 + m, (gi + 1) * gframes);
            const size_t off = (size_t)(a - f0) * frame_bytes;
            bool ok = false;
            rc = launch_group(vh, gi, a - gi * gframes, b - a, reinterpret_cast<const PX*>(din + off),
                              reinterpret_cast<PX*>(dout + off), st, &ok);
            for (int v = a / fpv; rc == CC_OK && !ok && v <= (b - 1) / fpv; ++v) {
                const int fa = std::max(a, v * fpv), fb = std::min(b, (v + 1) * fpv);
                const size_t o = (size_t)(fa - f0) * frame_bytes;
                rc = launch_one(v, reinterpret_cast<const PX*>(din + o), reinterpret_cast<PX*>(dout + o), fb - fa, st);
            }
        }
        if (rc) break;
        uint8_t* hd = hdst + (size_t)f0 * frame_stride * pxb;
        if (dense) {
            rc = cuda_check(cudaMemcpyAsync(hd, dout, (size_t)m * frame_bytes, cudaMemcpyDeviceToHost, st), "copy");
        } else {
            for (int f = 0; rc == CC_OK && f < m; ++f)
                rc = cuda_check(cudaMemcpy2DAsync(hd + (size_t)f * frame_stride * pxb, pitch * pxb, dout + (size_t)f * frame_bytes,
                                                  pitch * pxb, (size_t)sz1 * pxb, sz2, cudaMemcpyDeviceToHost, st), "copy");
        }
        for (; retired < g_hi || (retired == g_hi && f0 + m == std::min(nframes, (g_hi + 1) * gframes)); ++retired)
            rect_vh_retire(vh, retired);
    }
    const int re = rect_vh_end(vh);                         // every plan fenced, uploads complete
    const int rd = drain(ctx);
    return rc ? rc : re ? re : rd;
}

extern "C" {

int cc_rectify_f32c1_views(cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews, const double* ratios,
                           const int64_t* axs_mins, const float* src, float* dst, int sz1, int sz2, size_t pitch,
                           size_t frame_stride, int frames_per_view, float fill, unsigned flags, void* stream) {
    return rectify_views(ctx, intr, views, nviews, ratios, axs_mins, src, dst, sz1, sz2, pitch, frame_stride,
                         frames_per_view, 1, (cudaStream_t)stream,
                         [&](const ChainD& ch, double ratio, const int64_t* axs, const float* s, float* d, cudaStream_t st) {
                             return launch_rectify_f32c1(ctx, ch, ratio, axs, s, d, sz1, sz2, pitch, frame_stride,
                                                         frames_per_view, fill, flags, st);
                         },
                         [&](const ChainD* chs, const double* rs, const int64_t* axs, int nv, const float* s, float* d,
                             cudaStream_t st, bool* ok) {
                             *ok = false;
                             if (flags & CC_GATHER_DIRECT) return (int)CC_OK;
                             return launch_rectify_f32c1_views(ctx, chs, rs, axs, nv, s, d, sz1, sz2, pitch, frame_stride,
                                                               frames_per_view, fill, flags, st, ok);
                         });
}

int cc_rectify_u8c3_views(cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews, const double* ratios,
                          const int64_t* axs_mins, const uint8_t* src, uint8_t* dst, int sz1, int sz2, size_t pitch,
                          size_t frame_stride, int frames_per_view, const uint8_t fill[3], unsigned flags,
                          void* stream) {
    CC_REQUIRE(fill != nullptr, "fill is NULL");
    return rectify_views(ctx, intr, views, nviews, ratios, axs_mins, src, dst, sz1, sz2, pitch, frame_stride,
                         frames_per_view, 3, (cudaStream_t)stream,
                         [&](const ChainD& ch, double ratio, const int64_t* axs, const uint8_t* s, uint8_t* d, cudaStream_t st) {
                             return launch_rectify_u8c3(ctx, ch, ratio, axs, s, d, sz1, sz2, pitch, frame_stride,
                                                        frames_per_view, fill, flags, st);
                         },
                         [&](const ChainD* chs, const double* rs, const int64_t* axs, int nv, const uint8_t* s, uint8_t* d,
                             cudaStream_t st, bool* ok) {
                             *ok = false;
                             if (flags & CC_GATHER_DIRECT) return (int)CC_OK;
                             return launch_rectify_u8c3_views(ctx, chs, rs, axs, nv, s, d, sz1, sz2, pitch, frame_stride,
                                                              frames_per_view, fill, flags, st, ok);
                         });
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

int cc_rectify_f32c1_host(cc_ctx* ctx, const cc_intr* intr, const cc_view* view, double ratio,
                          const int64_t axs_min[2], const float* src, float* dst, int sz1, int sz2,
                          size_t pitch, size_t frame_stride, int nframes, float fill,
                          unsigned flags) {
    int rc = check_params(ctx, intr, view);
    if (rc) return rc;
    if ((rc = check_rect_args(axs_min, sz1, sz2, pitch, frame_stride, nframes, ratio))) return rc;
    CC_REQUIRE(nframes == 0 || (src && dst), "NULL frame pointer");
    CC_REQUIRE(nframes == 0 || (const void*)src != (const void*)dst, "rectification is not in place: src == dst");
    ChainD ch;
    build_chain(intr, view, &ch);
    return rectify_host<float>(
        ctx, src, dst, sz1, sz2, pitch, frame_stride, nframes, sizeof(float),
        [&](const float* s, float* d, size_t fs, int m, cudaStream_t st) {
            return launch_rectify_f32c1(ctx, ch, ratio, axs_min, s, d, sz1, sz2, pitch, fs, m, fill,
                                        flags, st);
        });
}

int cc_rectify_u8c3_host(cc_ctx* ctx, const cc_intr* intr, const cc_view* view, double ratio,
                         const int64_t axs_min[2], const uint8_t* src, uint8_t* dst, int sz1,
                         int sz2, size_t pitch, size_t frame_stride, int nframes,
                         const uint8_t fill[3], unsigned flags) {
    int rc = check_params(ctx, intr, view);
    if (rc) return rc;
    if ((rc = check_rect_args(axs_min, sz1, sz2, pitch, frame_stride, nframes, ratio))) return rc;
    CC_REQUIRE(nframes == 0 || (src && dst), "NULL frame pointer");
    CC_REQUIRE(nframes == 0 || (const void*)src != (const void*)dst, "rectification is not in place: src == dst");
    CC_REQUIRE(fill != nullptr, "fill is NULL");
    ChainD ch;
    build_chain(intr, view, &ch);
    return rectify_host<uint8_t>(
        ctx, src, dst, sz1, sz2, pitch, frame_stride, nframes, 3,
        [&](const uint8_t* s, uint8_t* d, size_t fs, int m, cudaStream_t st) {
            return launch_rectify_u8c3(ctx, ch, ratio, axs_min, s, d, sz1, sz2, pitch, fs, m, fill,
                                       flags, st);
        });
}

// ---- many views from host memory ----------------------------------------------------
int cc_rectify_views_f32c1_host(cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews,
                                const double* ratios, const int64_t* axs_mins, const float* src, float* dst,
                                int sz1, int sz2, size_t pitch, size_t frame_stride, int frames_per_view,
                                float fill, unsigned flags) {
    std::vector<ChainD> chs;
    return rectify_views_host(ctx, intr, views, nviews, ratios, axs_mins, src, dst, sz1, sz2, pitch, frame_stride,
                              frames_per_view, (int)sizeof(float), flags, &chs,
                              [&](RectViewsHost* vh, int gi, int w0, int wn, const float* s, float* d, cudaStream_t st, bool* ok) {
                                  return rect_vh_launch_f32c1(vh, gi, w0, wn, s, d, fill, flags, st, ok);
                              },
                              [&](int v, const float* s, float* d, int m, cudaStream_t st) {
                                  return launch_rectify_f32c1(ctx, chs[v], ratios[v], axs_mins + 2 * v, s, d, sz1, sz2,
                                                              pitch, pitch * (size_t)sz2, m, fill, flags, st);
                              });
}

int cc_rectify_views_u8c3_host(cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews,
                               const double* ratios, const int64_t* axs_mins, const uint8_t* src, uint8_t* dst,
                               int sz1, int sz2, size_t pitch, size_t frame_stride, int frames_per_view,
                               const uint8_t fill[3], unsigned flags) {
    CC_REQUIRE(fill != nullptr, "fill is NULL");
    std::vector<ChainD> chs;
    return rectify_views_host(ctx, intr, views, nviews, ratios, axs_mins, src, dst, sz1, sz2, pitch, frame_stride,
                              frames_per_view, 3, flags, &chs,
                              [&](RectViewsHost* vh, int gi, int w0, int wn, const uint8_t* s, uint8_t* d, cudaStream_t st, bool* ok) {
                                  return rect_vh_launch_u8c3(vh, gi, w0, wn, s, d, fill, flags, st, ok);
                              },
                              [&](int v, const uint8_t* s, uint8_t* d, int m, cudaStream_t st) {
                                  return launch_rectify_u8c3(ctx, chs[v], ratios[v], axs_mins + 2 * v, s, d, sz1, sz2,
                                                             pitch, pitch * (size_t)sz2, m, fill, flags, st);
                              });
}

int cc_rectify_map_f64(cc_ctx* ctx, const cc_intr* intr, const cc_view* view, double ratio,
                       const int64_t axs_min[2], double* map_row, double* map_col, int sz1, int sz2,
                       size_t pitch, void* stream) {
    int rc = check_params(ctx, intr, view);
    if (rc) return rc;
    if ((rc = check_rect_args(axs_min, sz1, sz2, pitch, pitch * (size_t)sz2, 1, ratio))) return rc;
    CC_REQUIRE(map_row && map_col, "NULL map pointer");
    CC_GUARD;
    if ((rc = enter(ctx))) return rc;
    ChainD ch;
    build_chain(intr, view, &ch);
    return launch_rectify_map(ctx, ch, ratio, axs_min, map_row, map_col, sz1, sz2, pitch,
                              (cudaStream_t)stream);
}

int cc_rectify_map_f32(cc_ctx* ctx, const cc_intr* intr, const cc_view* view, double ratio,
                       const int64_t axs_min[2], float* map_row, float* map_col, int sz1, int sz2,
                       size_t pitch, void* stream) {
    int rc = check_params(ctx, intr, view);
    if (rc) return rc;
    if ((rc = check_rect_args(axs_min, sz1, sz2, pitch, pitch * (size_t)sz2, 1, ratio))) return rc;
    CC_REQUIRE(map_row && map_col, "NULL map pointer");
    CC_GUARD;
    if ((rc = enter(ctx))) return rc;
    ChainD ch;
    build_chain(intr, view, &ch);
    return launch_rectify_map_f32(ctx, ch, ratio, axs_min, map_row, map_col, sz1, sz2, pitch,
                                  (cudaStream_t)stream);
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

// ---- residual / Jacobian ---------------------------------------------------------
int cc_reproj_jtj_f64(cc_ctx* ctx, const cc_intr* intr, double aspect, const cc_view* views,
                      int nviews, const double* obj, const double* img, int ncorners,
                      double* per_view, double* shared, void* stream) {
    CC_REQUIRE(ctx && intr, "NULL argument");
    CC_REQUIRE(nviews >= 0 && ncorners > 0, "bad sizes");
    CC_REQUIRE(shared != nullptr, "shared is NULL");
    CC_REQUIRE(nviews == 0 || (views && obj && img && per_view), "NULL device pointer");
    CC_REQUIRE(intr->checker_size != 0.0, "checker_size must be non-zero");
    CC_GUARD;
    int rc = enter(ctx);
    if (rc) return rc;
    return launch_reproj_jtj(ctx, intr, aspect, views, nviews, obj, img, ncorners, per_view, shared,
                             (cudaStream_t)stream);
}

int cc_reproj_jtj_f64_host(cc_ctx* ctx, const cc_intr* intr, double aspect, const cc_view* views,
                           int nviews, const double* obj, const double* img, int ncorners,
                           double* per_view, double* shared) {
    CC_REQUIRE(ctx && intr, "NULL argument");
    CC_REQUIRE(nviews >= 0 && ncorners > 0, "bad sizes");
    CC_REQUIRE(shared != nullptr, "shared is NULL");
    CC_REQUIRE(nviews == 0 || (views && obj && img && per_view), "NULL host pointer");
    CC_REQUIRE(intr->checker_size != 0.0, "checker_size must be non-zero");
    CC_GUARD;
    int rc = enter(ctx);
    if (rc) return rc;
    const size_t nv = (size_t)(nviews > 0 ? nviews : 1);
    const size_t b_views = round_up(nv * sizeof(cc_view), 256);
    const size_t b_obj = round_up((size_t)ncorners * 3 * sizeof(double), 256);
    const size_t b_img = round_up(nv * ncorners * 2 * sizeof(double), 256);
    const size_t b_pv = round_up(nv * CC_PER_VIEW * sizeof(double), 256);
    if ((rc = ensure_slot(ctx, 0, b_views + b_obj + b_img, b_pv + 256))) return rc;
    cudaStream_t st = ctx->pipe_stream[0];
    uint8_t* din = static_cast<uint8_t*>(ctx->pipe_in[0]);
    uint8_t* dout = static_cast<uint8_t*>(ctx->pipe_out[0]);
    cc_view* d_views = reinterpret_cast<cc_view*>(din);
    double* d_obj = reinterpret_cast<double*>(din + b_views);
    double* d_img = reinterpret_cast<double*>(din + b_views + b_obj);
    double* d_pv = reinterpret_cast<double*>(dout);
    double* d_sh = reinterpret_cast<double*>(dout + b_pv);
    if (nviews > 0) {
        CC_CUDA(cudaMemcpyAsync(d_views, views, (size_t)nviews * sizeof(cc_view), cudaMemcpyHostToDevice, st));
        CC_CUDA(cudaMemcpyAsync(d_obj, obj, (size_t)ncorners * 3 * sizeof(double), cudaMemcpyHostToDevice, st));
        CC_CUDA(cudaMemcpyAsync(d_img, img, (size_t)nviews * ncorners * 2 * sizeof(double), cudaMemcpyHostToDevice, st));
    }
    if ((rc = launch_reproj_jtj(ctx, intr, aspect, d_views, nviews, d_obj, d_img, ncorners, d_pv, d_sh, st)))
        return rc;
    if (nviews > 0)
        CC_CUDA(cudaMemcpyAsync(per_view, d_pv, (size_t)nviews * CC_PER_VIEW * sizeof(double), cudaMemcpyDeviceToHost, st));
    CC_CUDA(cudaMemcpyAsync(shared, d_sh, CC_SHARED * sizeof(double), cudaMemcpyDeviceToHost, st));
    CC_CUDA(cudaStreamSynchronize(st));
    return CC_OK;
}

int cc_calculate_errors_f64(cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews,
                            const double* obj, const double* img, int n1, int n2,
                            const double* inv_rows, const double* inv_cols, int inverse_samples,
                            double* sums, void* stream) {
    CC_REQUIRE(ctx && intr && sums, "NULL argument");
    CC_REQUIRE(nviews >= 0 && n1 >= 1 && n2 >= 1 && inverse_samples >= 0, "bad sizes");
    CC_REQUIRE(nviews == 0 || (views && obj && img), "NULL device pointer");
    CC_REQUIRE(inverse_samples == 0 || (inv_rows && inv_cols), "NULL sample pointer");
    CC_REQUIRE(intr->checker_size != 0.0 && intr->frow != 0.0 && intr->fcol != 0.0, "bad intrinsics");
    CC_GUARD;
    int rc = enter(ctx);
    if (rc) return rc;
    return launch_calc_errors(ctx, intr, views, nviews, obj, img, n1, n2, inv_rows, inv_cols,
                              inverse_samples, sums, (cudaStream_t)stream);
}

// host arrays in, the four raw sums out: what calculate_errors (src/buildcalibrations.jl:37-67) needs from a
// caller that holds the detections on the host, like the reference does
int cc_calculate_errors_f64_host(cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews,
                                 const double* obj, const double* img, int n1, int n2, const double* inv_rows,
                                 const double* inv_cols, int inverse_samples, double* sums) {
    CC_REQUIRE(ctx && intr && sums, "NULL argument");
    CC_REQUIRE(nviews >= 0 && n1 >= 1 && n2 >= 1 && inverse_samples >= 0, "bad sizes");
    CC_REQUIRE(nviews == 0 || (views && obj && img), "NULL host pointer");
    CC_REQUIRE(inverse_samples == 0 || nviews == 0 || (inv_rows && inv_cols), "NULL sample pointer");
    CC_REQUIRE(intr->checker_size != 0.0 && intr->frow != 0.0 && intr->fcol != 0.0, "bad intrinsics");
    CC_GUARD;
    int rc = enter(ctx);
    if (rc) return rc;
    const size_t nv = (size_t)(nviews > 0 ? nviews : 1), nc = (size_t)n1 * n2;
    const size_t b_views = round_up(nv * sizeof(cc_view), 256);
    const size_t b_obj = round_up(nc * 3 * sizeof(double), 256);
    const size_t b_img = round_up(nv * nc * 2 * sizeof(double), 256);
    const size_t b_inv = round_up(nv * (size_t)std::max(inverse_samples, 1) * sizeof(double), 256);
    if ((rc = ensure_slot(ctx, 0, b_views + b_obj + b_img + 2 * b_inv, 256))) return rc;
    cudaStream_t st = ctx->pipe_stream[0];
    uint8_t* din = static_cast<uint8_t*>(ctx->pipe_in[0]);
    cc_view* d_views = reinterpret_cast<cc_view*>(din);
    double* d_obj = reinterpret_cast<double*>(din + b_views);
    double* d_img = reinterpret_cast<double*>(din + b_views + b_obj);
    double* d_ir = reinterpret_cast<double*>(din + b_views + b_obj + b_img);
    double* d_ic = reinterpret_cast<double*>(din + b_views + b_obj + b_img + b_inv);
    double* d_sums = static_cast<double*>(ctx->pipe_out[0]);
    if (nviews > 0) {
        CC_CUDA(cudaMemcpyAsync(d_views, views, (size_t)nviews * sizeof(cc_view), cudaMemcpyHostToDevice, st));
        CC_CUDA(cudaMemcpyAsync(d_obj, obj, nc * 3 * sizeof(double), cudaMemcpyHostToDevice, st));
        CC_CUDA(cudaMemcpyAsync(d_img, img, (size_t)nviews * nc * 2 * sizeof(double), cudaMemcpyHostToDevice, st));
        if (inverse_samples > 0) {
            CC_CUDA(cudaMemcpyAsync(d_ir, inv_rows, (size_t)nviews * inverse_samples * sizeof(double), cudaMemcpyHostToDevice, st));
            CC_CUDA(cudaMemcpyAsync(d_ic, inv_cols, (size_t)nviews * inverse_samples * sizeof(double), cudaMemcpyHostToDevice, st));
        }
    }
    if ((rc = launch_calc_errors(ctx, intr, d_views, nviews, d_obj, d_img, n1, n2, d_ir, d_ic, inverse_samples, d_sums, st)))
        return rc;
    CC_CUDA(cudaMemcpyAsync(sums, d_sums, 4 * sizeof(double), cudaMemcpyDeviceToHost, st));
    CC_CUDA(cudaStreamSynchronize(st));
    return CC_OK;
}

// ---- Levenberg-Marquardt step -----------------------------------------------------
int cc_lm_schur_f64(cc_ctx* ctx, const double* per_view, int nviews, double lambda, double* yz,
                    double* schur, void* stream) {
    CC_REQUIRE(ctx && schur, "NULL argument");
    CC_REQUIRE(nviews >= 0, "bad sizes");
    CC_REQUIRE(nviews == 0 || (per_view && yz), "NULL device pointer");
    CC_REQUIRE(lambda >= 0.0 && lambda == lambda, "lambda must be non-negative");
    CC_GUARD;
    int rc = enter(ctx);
    if (rc) return rc;
    return launch_lm_schur(ctx, per_view, nviews, lambda, yz, schur, (cudaStream_t)stream);
}

int cc_lm_update_f64(cc_ctx* ctx, const double* shared, const double* schur, double lambda,
                     unsigned free_mask, const double* yz, const cc_view* views_in, int nviews,
                     cc_view* views_out, double* delta, void* stream) {
    CC_REQUIRE(ctx && shared && schur && delta, "NULL argument");
    CC_REQUIRE(nviews >= 0, "bad sizes");
    CC_REQUIRE(nviews == 0 || (yz && views_in && views_out), "NULL device pointer");
    CC_REQUIRE(lambda >= 0.0 && lambda == lambda, "lambda must be non-negative");
    CC_REQUIRE(free_mask != 0u && free_mask < 16u, "free_mask selects among the 4 shared parameters");
    CC_GUARD;
    int rc = enter(ctx);
    if (rc) return rc;
    return launch_lm_update(ctx, shared, schur, lambda, free_mask, yz, views_in, nviews, views_out, delta,
                            (cudaStream_t)stream);
}

int cc_lm_fit_f64_host(cc_ctx* ctx, cc_intr* intr, double aspect, unsigned free_mask, cc_view* views,
                       int nviews, const double* obj, const double* img, int ncorners, int max_iter,
                       double eps, double* rms, int* iterations) {
    CC_REQUIRE(ctx && intr && views && obj && img, "NULL argument");
    CC_REQUIRE(nviews > 0 && ncorners > 0, "bad sizes");
    CC_REQUIRE(free_mask != 0u && free_mask < 16u, "free_mask selects among the 4 shared parameters");
    CC_REQUIRE(max_iter >= 0 && eps >= 0.0, "bad stopping rule");
    CC_REQUIRE(aspect > 0.0 && intr->fcol != 0.0 && intr->checker_size != 0.0, "bad starting intrinsics");
    CC_GUARD;
    int rc = enter(ctx);
    if (rc) return rc;
    return lm_fit_host(ctx, intr, aspect, free_mask, views, nviews, obj, img, ncorners, max_iter, eps, rms,
                       iterations);
}

int cc_lm_fit_f64(cc_ctx* ctx, cc_intr* intr, double aspect, unsigned free_mask, cc_view* views, int nviews,
                  const double* obj, const double* img, int ncorners, int max_iter, double eps, double* rms,
                  int* iterations, void* stream) {
    CC_REQUIRE(ctx && intr && obj, "NULL argument");
    CC_REQUIRE(nviews >= 0 && ncorners > 0, "bad sizes");
    CC_REQUIRE(nviews == 0 || (views && img), "NULL view / image-point array");
    CC_REQUIRE(free_mask != 0u && free_mask < 16u, "free_mask selects among the 4 shared parameters");
    CC_REQUIRE(max_iter >= 0 && eps >= 0.0, "bad stopping rule");
    CC_REQUIRE(aspect > 0.0 && intr->fcol != 0.0 && intr->checker_size != 0.0, "bad starting intrinsics");
    CC_GUARD;
    int rc = enter(ctx);
    if (rc) return rc;
    return lm_fit_device(ctx, intr, aspect, free_mask, views, nviews, obj, img, ncorners, max_iter, eps, rms,
                         iterations, (cudaStream_t)stream);
}

int cc_lm_initial_guess_f64(cc_ctx* ctx, const double* obj, const double* img, int nviews, int ncorners, int sz1,
                            int sz2, double aspect, cc_intr* intr, cc_view* views, void* stream) {
    CC_REQUIRE(ctx && intr && obj, "NULL argument");
    CC_REQUIRE(nviews >= 0 && ncorners >= 4 && sz1 > 0 && sz2 > 0, "bad sizes (a homography needs >= 4 corners)");
    CC_REQUIRE(nviews == 0 || (views && img), "NULL view / image-point array");
    CC_GUARD;
    int rc = enter(ctx);
    if (rc) return rc;
    return launch_initial_guess(ctx, obj, img, nviews, ncorners, sz1, sz2, aspect, intr, views, (cudaStream_t)stream);
}

int cc_ctx_collective_count(const cc_ctx* ctx, uint64_t* count) {
    CC_REQUIRE(ctx && count, "NULL argument");
    *count = ctx->collectives;
    return CC_OK;
}

}  // extern "C"
