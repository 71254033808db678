// common.cuh -- shared declarations of libcamcal_b200 (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>

#include "../../include/camcal_b200.h"

struct cc_ctx;
namespace cc {

// What `Calibration(...)` / `img2obj` derive once per view (src/meta.jl:27-33, 71-76),
// expanded on the host and passed to kernels by value.  Row-major 3x3.
template <typename T>
struct Chain {
    T R[9], t[3], Rinv[9], tinv[3];
    T a_row, b_row, a_col, b_col;   // inv(intrinsic): u = a*rc + b
    T frow, fcol, crow, ccol, k;
    T inv_cs, cs_back;              // scale and inv(scale)
};
using ChainD = Chain<double>;
using ChainF = Chain<float>;

// The rest of a chain from its R and t and the intrinsics: inv(extrinsic), inv(intrinsic), scale and its inverse.
// Fused only where the source says fma(), so the host build (-ffp-contract=off) and the device build (-fmad=false)
// give the same bits.
__host__ __device__ inline void complete_chain(const cc_intr& in, ChainD& ch) {
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) ch.Rinv[3 * i + j] = ch.R[3 * j + i];
    for (int i = 0; i < 3; ++i) {
        const double* m = ch.Rinv + 3 * i;
        ch.tinv[i] = fma(m[2], -ch.t[2], fma(m[1], -ch.t[1], m[0] * -ch.t[0]));
    }
    ch.frow = in.frow; ch.fcol = in.fcol;
    ch.crow = in.crow; ch.ccol = in.ccol;
    ch.k = in.k;
    ch.a_row = 1.0 / in.frow;
    ch.a_col = 1.0 / in.fcol;
    ch.b_row = ch.a_row * (-in.crow);
    ch.b_col = ch.a_col * (-in.ccol);
    ch.inv_cs = 1.0 / in.checker_size;
    ch.cs_back = 1.0 / ch.inv_cs;
}

// host: rotation vector -> matrix and derived maps (chain_host.cu)
void rodrigues_host(const double r[3], double R[9]);
void build_chain(const cc_intr* in, const cc_view* vw, ChainD* out);
void narrow_chain(const ChainD& d, ChainF* f);
void rectify_free_plans(struct ::cc_ctx* ctx);
void rectify_free_sched(struct ::cc_ctx* ctx);
void ingest_free(struct ::cc_ctx* ctx);
int jpeg_info(const uint8_t* data, size_t length, int* sz1, int* sz2, int* channels);
int jpeg_decode_u8c3(struct ::cc_ctx* ctx, const uint8_t* const* jpegs, const size_t* lengths, int n, uint8_t* dst,
                     int sz1, int sz2, size_t pitch, size_t frame_stride, cudaStream_t st);
void comm_free(struct ::cc_ctx* ctx);
void lm_free_workspace(struct ::cc_ctx* ctx);
void point_table_free(struct ::cc_ctx* ctx);
// the device chain table of the multi-view point maps (pointmap.cu): rows, then segment offsets
struct PointTable {
    const void* rows;
    const size_t* off;
};
// The arrays of a point map.  SoA: one array per coordinate.  AoS: in[0] / out[0] hold packed points of in_dim /
// out_dim coordinates.  img2world out_dim 2: z is not computed; world2img in_dim 2: z = 0.  Unused entries are NULL.
template <typename T> struct PointIO {
    bool to_img;           // world -> pixel
    bool aos;
    int in_dim, out_dim;   // 2 or 3
    const T* in[3];
    T* out[3];
    int in_arrays() const { return aos ? 1 : in_dim; }
    int out_arrays() const { return aos ? 1 : out_dim; }
};
// The views of one launch.  SINGLE (chain != NULL): every point uses *chain, passed by value.  TABLE: the launch's
// points are points base + [0, n) of the call, in segments [seg_lo, seg_hi) of the uploaded table tb.
struct PointSrc {
    const ChainD* chain;
    PointTable tb;
    size_t base;
    int seg_lo, seg_hi;
};
// The pixel of a rectified frame: PX elements (channels) and bytes per pixel, and the fill as the kernels take it
// (f32c1: one float; u8c3: three bytes)
template <typename PX> struct RectPx;
template <> struct RectPx<float> { static constexpr int channels = 1, bytes = 4; using Fill = float; };
template <> struct RectPx<uint8_t> { static constexpr int channels = 3, bytes = 3; using Fill = uchar3; };
// A rectification call.  Source frames are sz1 x sz2 pixels, lines `pitch` pixels and frames `frame_stride` pixels
// apart; output frames out_sz1 x out_sz2, lines out_pitch and frames out_frame_stride apart (the cc_rectify_* entry
// points other than cc_rectify_axes_*: the source's own geometry, rect_frames).  View v (chs[v], ratios[v],
// axs_mins[2v .. 2v+1]) rectifies frames [v * fpv, (v + 1) * fpv); a single-view call is one view with all the frames.
struct RectFrames {
    int sz1, sz2;
    size_t pitch, frame_stride;
    int fpv;
    int out_sz1, out_sz2;
    size_t out_pitch, out_frame_stride;
};
// a call whose output has the source's geometry
inline RectFrames rect_frames(int sz1, int sz2, size_t pitch, size_t frame_stride, int fpv) {
    return {sz1, sz2, pitch, frame_stride, fpv, sz1, sz2, pitch, frame_stride};
}
struct RectViews {
    const ChainD* chs;
    const double* ratios;
    const int64_t* axs_mins;
    int n;
};
template <typename PX> struct RectCall {
    RectFrames fr;
    RectViews views;
    typename RectPx<PX>::Fill fill;
    unsigned flags;
};

// error plumbing (abi.cu)
int set_error(int status, const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);

}  // namespace cc

struct cc_ctx {
    int device;
    int sm_count;
    int cc_major, cc_minor;
    unsigned long long launches;
    // reprojection scratch: [21][nviews] component-major partials
    double* jtj_scratch;
    size_t jtj_scratch_elems;
    // the scratch is shared by reproj_jtj / calc_errors / lm_*: calls on DIFFERENT streams are ordered
    // through an event recorded on the previous user's stream (lm_state.cuh: ScratchHold)
    cudaStream_t scratch_stream;
    cudaEvent_t scratch_event;
    int scratch_used;
    // host pipeline: NSLOT streams with device staging buffers
    static const int NSLOT = 4;
    cudaStream_t pipe_stream[NSLOT];
    void* pipe_in[NSLOT];
    void* pipe_out[NSLOT];
    size_t pipe_in_bytes[NSLOT];
    size_t pipe_out_bytes[NSLOT];
    // TMA descriptor encode entry point (driver API, resolved at ctx creation)
    void* encode_tiled;
    // rectification footprints of single views (rectify.cu: RectPlan, host memory only), most recent NPLAN
    // parameter sets
    static const int NPLAN = 64;
    void* rect_plans[NPLAN];
    int rect_plan_next;
    // the device tables every staged rectification launch reads (rectify.cu: GroupPlan): plans of one view in
    // the first NPLAN slots, plans of more views in the last NGROUP, each part evicting round-robin
    // (group_plan_next[0] / [1]).  Tables go up on rect_upload; an evicted plan's buffers are overwritten after
    // its readers, or the plan is retired (plans_retired) and freed once they have finished.
    // cc_rectify_views_*_host joins its slot streams on rect_join (rect_join_event: one per slot).
    static const int NGROUP = 4;
    void* group_plans[NPLAN + NGROUP];
    int group_plan_next[2];
    cudaStream_t rect_upload, rect_join;
    cudaEvent_t rect_join_event[NSLOT];
    void* plans_retired;
    // ticket counters of the persistent rectification kernels (rectify.cu: RectSched)
    static const int NSCHED = 16;
    void* sched_pool;
    cudaEvent_t sched_event[NSCHED];
    cudaStream_t sched_stream[NSCHED];
    unsigned char sched_used[NSCHED];
    unsigned sched_next;
    // NCCL communicator of this context (comm.cu); NULL / 1 rank: a world of one
    void* nccl_comm;
    int comm_nranks, comm_rank;
    unsigned long long collectives;       // all-reduces issued so far
    // workspace of the device-resident LM loop (lm.cu: LmWorkspace), grown on demand
    void* lm_ws;
    // nvJPEG handle / state / raster scratch of the image ingest (ingest.cu: Ingest), created on first use
    void* ingest;
    // chain table of the multi-view point maps (pointmap.cu: point_table_upload), grown on demand; a call
    // on a stream other than the previous user's waits for pt_event, recorded after that user's kernels
    void* pt_table;
    size_t pt_table_bytes;
    cudaEvent_t pt_event;
    cudaStream_t pt_stream;
    int pt_used;
    // pinned staging of the table upload; pt_stage_event: the last upload out of it has completed
    void* pt_stage;
    size_t pt_stage_bytes;
    cudaEvent_t pt_stage_event;
};

#define CC_CUDA(call)                                                     \
    do {                                                                  \
        cudaError_t _e = (call);                                          \
        if (_e != cudaSuccess) return cc::cuda_fail(_e, #call);           \
    } while (0)

#define CC_REQUIRE(cond, msg)                                             \
    do {                                                                  \
        if (!(cond)) return cc::set_error(CC_ERR_INVALID_ARG, "%s", msg); \
    } while (0)

// ---- device helpers -------------------------------------------------------
namespace cc {

// streaming 128-bit accesses: inputs are read once, outputs written once
__device__ __forceinline__ double2 ldg_stream(const double2* p) {
    double2 v;
    asm volatile("ld.global.nc.L1::no_allocate.v2.f64 {%0,%1}, [%2];"
                 : "=d"(v.x), "=d"(v.y) : "l"(p));
    return v;
}
__device__ __forceinline__ float4 ldg_stream(const float4* p) {
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}
__device__ __forceinline__ void stg_stream(double2* p, double2 v) {
    asm volatile("st.global.cs.v2.f64 [%0], {%1,%2};" :: "l"(p), "d"(v.x), "d"(v.y) : "memory");
}
__device__ __forceinline__ void stg_stream(float4* p, float4 v) {
    asm volatile("st.global.cs.v4.f32 [%0], {%1,%2,%3,%4};"
                 :: "l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void stg_stream(uint4* p, uint4 v) {
    asm volatile("st.global.cs.v4.u32 [%0], {%1,%2,%3,%4};"
                 :: "l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// 2^-23-accurate reciprocal seed on the SFU (MUFU.RCP64H)
__device__ __forceinline__ double rcp_approx(double a) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(a));
    return r;
}

}  // namespace cc
