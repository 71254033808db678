// pointmap.cu -- batched pixel<->world maps over SoA point sets and interleaved (AoS) points.
//
// Replaces the Julia broadcasts c.(imgpoints, i) / c.(objpoints, i)
// (src/buildcalibrations.jl:29,46) over the callables of src/meta.jl:82,88.
//
// HBM-bound streaming kernels: every array is read or written exactly once with
// 128-bit accesses (double2 / float4), L1 no-allocate loads and evict-first stores;
// a persistent grid of (SM count x resident CTAs) strides over the vectors with two
// independent vectors in flight per thread.  Algorithmic bytes per point:
// img2world 40 B (f64) / 20 B (f32), 32 / 16 B without z; world2img 40 / 20 B
// (32 / 16 B when z == NULL).
#include <cstring>
#include <type_traits>

#include "chain_device.cuh"

namespace cc {

template <typename T> struct Vec;
template <> struct Vec<double> { using type = double2; static constexpr int N = 2; };
template <> struct Vec<float>  { using type = float4;  static constexpr int N = 4; };

template <typename T> __device__ __forceinline__ T& lane(typename Vec<T>::type& v, int i);
template <> __device__ __forceinline__ double& lane<double>(double2& v, int i) { return i == 0 ? v.x : v.y; }
template <> __device__ __forceinline__ float& lane<float>(float4& v, int i) {
    return i == 0 ? v.x : (i == 1 ? v.y : (i == 2 ? v.z : v.w));
}

constexpr int kThreads = 256;
constexpr int kUnroll = 2;

// ---- view sources -------------------------------------------------------------------------------
// SINGLE: one chain for every point, passed by value (constant bank) -- the source is a Chain<T>.
// TABLE:  per-segment chains in a device table plus segment offsets -- the source is a ViewTable<Row>.
//         Points [off[s], off[s+1]) use segment s; a launch covers points base + [0, n).
//
// The table stores only the fields of Chain<T> its direction reads (18 values instead of 35).
template <typename T> struct RowW2I { T R[9], t[3], k, frow, fcol, crow, ccol, inv_cs; };
template <typename T> struct RowI2W { T a_row, b_row, a_col, b_col, k, Rinv[9], tinv[3], cs_back; };

template <typename T> __host__ __device__ __forceinline__ void pack(const Chain<T>& c, RowW2I<T>& r) {
    for (int i = 0; i < 9; ++i) r.R[i] = c.R[i];
    for (int i = 0; i < 3; ++i) r.t[i] = c.t[i];
    r.k = c.k; r.frow = c.frow; r.fcol = c.fcol; r.crow = c.crow; r.ccol = c.ccol; r.inv_cs = c.inv_cs;
}
template <typename T> __host__ __device__ __forceinline__ void pack(const Chain<T>& c, RowI2W<T>& r) {
    r.a_row = c.a_row; r.b_row = c.b_row; r.a_col = c.a_col; r.b_col = c.b_col; r.k = c.k;
    for (int i = 0; i < 9; ++i) r.Rinv[i] = c.Rinv[i];
    for (int i = 0; i < 3; ++i) r.tinv[i] = c.tinv[i];
    r.cs_back = c.cs_back;
}
// the fields world2img / img2world do not read are left unset
template <typename T> __device__ __forceinline__ void unpack(const RowW2I<T>& r, Chain<T>& c) {
#pragma unroll
    for (int i = 0; i < 9; ++i) c.R[i] = r.R[i];
#pragma unroll
    for (int i = 0; i < 3; ++i) c.t[i] = r.t[i];
    c.k = r.k; c.frow = r.frow; c.fcol = r.fcol; c.crow = r.crow; c.ccol = r.ccol; c.inv_cs = r.inv_cs;
}
template <typename T> __device__ __forceinline__ void unpack(const RowI2W<T>& r, Chain<T>& c) {
    c.a_row = r.a_row; c.b_row = r.b_row; c.a_col = r.a_col; c.b_col = r.b_col; c.k = r.k;
#pragma unroll
    for (int i = 0; i < 9; ++i) c.Rinv[i] = r.Rinv[i];
#pragma unroll
    for (int i = 0; i < 3; ++i) c.tinv[i] = r.tinv[i];
    c.cs_back = r.cs_back;
}

template <typename Row> struct ViewTable {
    const Row* rows;       // one per segment
    const size_t* off;     // segment offsets, nseg + 1 entries
    size_t base;           // index of this launch's point 0 among the call's points
    int seg_lo, seg_hi;    // the launch's points lie in segments [seg_lo, seg_hi)
};

template <typename S> struct IsTable : std::false_type {};
template <typename Row> struct IsTable<ViewTable<Row>> : std::true_type {};

// ---- layouts ---------------------------------------------------------------------------------------
// SoA: one array per coordinate.  AoS: one array of packed points, D coordinates each ((row, col) pairs,
// (x, y, z) or (x, y) points).  A group of N consecutive points (N = Vec<T>::N) is D 16-byte vectors in
// either layout: vector g of each coordinate array (SoA), or vectors D*g .. D*g + D-1 of the packed array
// (AoS).  Coordinate d of the group's point e is lane e of vector d (SoA), or scalar k = D*e + d of the
// group: lane k % N of vector k / N (AoS).  The indices are compile-time constants after unrolling, so the
// AoS permutation is register moves only.
template <typename T, int D, bool AOS>
__device__ __forceinline__ T& coord(typename Vec<T>::type* g, int d, int e) {
    constexpr int N = Vec<T>::N;
    if constexpr (AOS) return lane<T>(g[(D * e + d) / N], (D * e + d) % N);
    else return lane<T>(g[d], e);
}

// ---- per-point loops ------------------------------------------------------------------------------
// Points [p0, p1) (p0 a multiple of N): groups of N points through 16-byte vectors when vec_ok, thread
// `tid` of `nthreads` taking groups tid, tid + nthreads, ... two at a time, then the scalar tail; scalar
// throughout when !vec_ok.  chain(p) gives the chain of point p, asked for in increasing p within a thread.
// AOS: `row` holds the (row, col) pairs and `x` the (x, y[, z]) points; col, y and z are not used.
template <typename T, bool HAS_Z, bool AOS, typename CH>
__device__ __forceinline__ void img2world_range(CH&& chain, const T* __restrict__ row,
                                                 const T* __restrict__ col, T* __restrict__ x,
                                                 T* __restrict__ y, T* __restrict__ z, size_t p0,
                                                 size_t p1, size_t tid, size_t nthreads, bool vec_ok) {
    using V = typename Vec<T>::type;
    constexpr int N = Vec<T>::N;
    constexpr int DO = HAS_Z ? 3 : 2;
    size_t done = p0;
    if (vec_ok) {
        const size_t nvec = p1 / N;
        const V* rv = reinterpret_cast<const V*>(row);
        const V* cv = reinterpret_cast<const V*>(col);
        V* xv = reinterpret_cast<V*>(x);
        V* yv = reinterpret_cast<V*>(y);
        V* zv = reinterpret_cast<V*>(z);
        for (size_t i = p0 / N + tid; i < nvec; i += nthreads * kUnroll) {
            V in[kUnroll][2];
#pragma unroll
            for (int u = 0; u < kUnroll; ++u) {
                const size_t j = i + u * nthreads;
                if (j < nvec) {
                    if constexpr (AOS) { in[u][0] = ldg_stream(rv + 2 * j); in[u][1] = ldg_stream(rv + 2 * j + 1); }
                    else { in[u][0] = ldg_stream(rv + j); in[u][1] = ldg_stream(cv + j); }
                }
            }
#pragma unroll
            for (int u = 0; u < kUnroll; ++u) {
                const size_t j = i + u * nthreads;
                if (j < nvec) {
                    V o[3];            // o[2]: z lanes that are computed but not stored when !HAS_Z
#pragma unroll
                    for (int e = 0; e < N; ++e)
                        img2world(chain(j * N + e), coord<T, 2, AOS>(in[u], 0, e), coord<T, 2, AOS>(in[u], 1, e),
                                  coord<T, DO, AOS>(o, 0, e), coord<T, DO, AOS>(o, 1, e),
                                  HAS_Z ? coord<T, DO, AOS>(o, 2, e) : lane<T>(o[2], e));
                    if constexpr (AOS) {
#pragma unroll
                        for (int d = 0; d < DO; ++d) stg_stream(xv + DO * j + d, o[d]);
                    } else {
                        stg_stream(xv + j, o[0]);
                        stg_stream(yv + j, o[1]);
                        if (HAS_Z) stg_stream(zv + j, o[2]);
                    }
                }
            }
        }
        done = nvec * N;
    }
    for (size_t i = done + tid; i < p1; i += nthreads) {   // tail / unaligned pointers
        T ox, oy, oz;
        if constexpr (AOS) {
            img2world(chain(i), row[2 * i], row[2 * i + 1], ox, oy, oz);
            x[DO * i] = ox; x[DO * i + 1] = oy;
            if (HAS_Z) x[DO * i + 2] = oz;
        } else {
            img2world(chain(i), row[i], col[i], ox, oy, oz);
            x[i] = ox; y[i] = oy;
            if (HAS_Z) z[i] = oz;
        }
    }
}

// AOS: `x` holds the (x, y[, z]) points and `row` the (row, col) pairs; y, z and col are not used.
template <typename T, bool HAS_Z, bool AOS, typename CH>
__device__ __forceinline__ void world2img_range(CH&& chain, const T* __restrict__ x,
                                                const T* __restrict__ y, const T* __restrict__ z,
                                                T* __restrict__ row, T* __restrict__ col, size_t p0,
                                                size_t p1, size_t tid, size_t nthreads, bool vec_ok) {
    using V = typename Vec<T>::type;
    constexpr int N = Vec<T>::N;
    constexpr int DI = HAS_Z ? 3 : 2;
    size_t done = p0;
    if (vec_ok) {
        const size_t nvec = p1 / N;
        const V* xv = reinterpret_cast<const V*>(x);
        const V* yv = reinterpret_cast<const V*>(y);
        const V* zv = reinterpret_cast<const V*>(z);
        V* rv = reinterpret_cast<V*>(row);
        V* cv = reinterpret_cast<V*>(col);
        for (size_t i = p0 / N + tid; i < nvec; i += nthreads * kUnroll) {
            V in[kUnroll][3];
#pragma unroll
            for (int u = 0; u < kUnroll; ++u) {
                const size_t j = i + u * nthreads;
                if (j < nvec) {
                    if constexpr (AOS) {
#pragma unroll
                        for (int d = 0; d < DI; ++d) in[u][d] = ldg_stream(xv + DI * j + d);
                    } else {
                        in[u][0] = ldg_stream(xv + j);
                        in[u][1] = ldg_stream(yv + j);
                        if (HAS_Z) in[u][2] = ldg_stream(zv + j);
                    }
                }
            }
#pragma unroll
            for (int u = 0; u < kUnroll; ++u) {
                const size_t j = i + u * nthreads;
                if (j < nvec) {
                    V o[2];
#pragma unroll
                    for (int e = 0; e < N; ++e)
                        world2img(chain(j * N + e), coord<T, DI, AOS>(in[u], 0, e), coord<T, DI, AOS>(in[u], 1, e),
                                  HAS_Z ? coord<T, DI, AOS>(in[u], 2, e) : T(0), coord<T, 2, AOS>(o, 0, e),
                                  coord<T, 2, AOS>(o, 1, e));
                    if constexpr (AOS) {
                        stg_stream(rv + 2 * j, o[0]);
                        stg_stream(rv + 2 * j + 1, o[1]);
                    } else {
                        stg_stream(rv + j, o[0]);
                        stg_stream(cv + j, o[1]);
                    }
                }
            }
        }
        done = nvec * N;
    }
    for (size_t i = done + tid; i < p1; i += nthreads) {
        T orow, ocol;
        if constexpr (AOS) {
            world2img(chain(i), x[DI * i], x[DI * i + 1], HAS_Z ? x[DI * i + 2] : T(0), orow, ocol);
            row[2 * i] = orow; row[2 * i + 1] = ocol;
        } else {
            world2img(chain(i), x[i], y[i], HAS_Z ? z[i] : T(0), orow, ocol);
            row[i] = orow; col[i] = ocol;
        }
    }
}

// ---- TABLE: tiles of segments ---------------------------------------------------------------------
// Every CTA of the persistent grid takes a contiguous run of kTile-point tiles (kTile is a multiple
// of both vector widths, so a tile's vectors stay 16-byte aligned whatever the segment boundaries).
// Warp 0 finds the tile's first segment; a tile inside one segment (the common case for large
// segments) runs the single-view loop on that chain, staged in shared memory; a tile that crosses
// segment boundaries walks a per-thread segment cursor over the offsets and reads each point's chain
// from the table (L1-resident).  The offsets are never expanded into a per-point index.
constexpr size_t kTile = 4096;

// First segment s in [lo, hi) with off[s + 1] > p; one exists.  The whole warp calls it.  The first
// round looks at the 32 segments from lo on (the next tile usually starts in one of them); later
// rounds split what is left 32 ways.
__device__ __forceinline__ int find_segment(const size_t* __restrict__ off, int lo, int hi, size_t p) {
    const int lane = threadIdx.x & 31;
    for (bool near = true;; near = false) {
        const int step = (near || hi - lo <= 32) ? 1 : (hi - lo + 31) / 32;
        const int c = lo + lane * step;
        const bool after = c >= hi || __ldg(off + c + 1) > p;       // monotone over the lanes
        const unsigned b = __ballot_sync(0xffffffffu, after);
        if (b == 0) { lo += 31 * step + 1; continue; }
        const int L = __ffs(b) - 1;
        if (step == 1) return lo + L;
        if (L == 0) return lo;
        const int nlo = lo + (L - 1) * step + 1;
        hi = min(hi, lo + L * step + 1);
        lo = nlo;
    }
}

template <typename T, typename Row, typename BODY>
__device__ __forceinline__ void for_each_tile(const ViewTable<Row>& tb, size_t n, BODY&& body) {
    __shared__ Chain<T> s_chain[2];        // double-buffered: one barrier per tile
    __shared__ int s_seg[2];
    __shared__ int s_inside[2];
    const size_t ntiles = (n + kTile - 1) / kTile;
    const size_t per = ntiles / gridDim.x, extra = ntiles % gridDim.x;
    const size_t t0 = blockIdx.x * per + min((size_t)blockIdx.x, extra);
    const size_t t1 = t0 + per + (blockIdx.x < extra ? 1 : 0);
    int lo = tb.seg_lo;
    for (size_t t = t0; t < t1; ++t) {
        const int b = (int)(t & 1);
        const size_t p0 = t * kTile, p1 = min(n, p0 + kTile);
        if (threadIdx.x < 32) {
            lo = find_segment(tb.off, lo, tb.seg_hi, tb.base + p0);
            if (threadIdx.x == 0) {
                const int inside = __ldg(tb.off + lo + 1) >= tb.base + p1;
                s_seg[b] = lo;
                s_inside[b] = inside;
                if (inside) unpack(tb.rows[lo], s_chain[b]);
            }
        }
        __syncthreads();
        if (s_inside[b]) {
            body(p0, p1, [&](size_t) -> const Chain<T>& { return s_chain[b]; });
        } else {
            int s = s_seg[b];
            body(p0, p1, [&](size_t p) {
                while (__ldg(tb.off + s + 1) <= tb.base + p) ++s;
                Chain<T> c;
                unpack(tb.rows[s], c);
                return c;
            });
        }
    }
}

// Resident CTAs per SM asked of ptxas: none for SINGLE (its code is what it always was).  For TABLE, 3 where
// that measured faster on a B200 (1000 W): FP64 pixel->world and FP32 world->pixel (0.72 -> 0.85x and
// 0.95 -> 1.05x of the single-view rate at 1 segment); it made FP64 world->pixel slower (1.00 -> 0.90x) and
// left FP32 pixel->world unchanged, so those two keep the compiler's choice.
template <typename SRC, bool ASK> constexpr int kTableMinBlocks = IsTable<SRC>::value && ASK ? 3 : 0;

template <typename T, bool HAS_Z, typename SRC = Chain<T>>
__global__ void __launch_bounds__(kThreads, kTableMinBlocks<SRC, std::is_same<T, double>::value>)
img2world_kernel(const SRC src, const T* __restrict__ row, const T* __restrict__ col,
                 T* __restrict__ x, T* __restrict__ y, T* __restrict__ z, size_t n, bool vec_ok) {
    if constexpr (IsTable<SRC>::value) {
        for_each_tile<T>(src, n, [&](size_t p0, size_t p1, auto&& chain) {
            img2world_range<T, HAS_Z, false>(chain, row, col, x, y, z, p0, p1, threadIdx.x, kThreads, vec_ok);
        });
    } else {
        const size_t tid = (size_t)blockIdx.x * kThreads + threadIdx.x;
        const size_t nthreads = (size_t)gridDim.x * kThreads;
        img2world_range<T, HAS_Z, false>([&](size_t) -> const Chain<T>& { return src; }, row, col, x, y, z,
                                         0, n, tid, nthreads, vec_ok);
    }
}

template <typename T, bool HAS_Z, typename SRC = Chain<T>>
__global__ void __launch_bounds__(kThreads, kTableMinBlocks<SRC, std::is_same<T, float>::value>)
world2img_kernel(const SRC src, const T* __restrict__ x, const T* __restrict__ y,
                 const T* __restrict__ z, T* __restrict__ row, T* __restrict__ col, size_t n,
                 bool vec_ok) {
    if constexpr (IsTable<SRC>::value) {
        for_each_tile<T>(src, n, [&](size_t p0, size_t p1, auto&& chain) {
            world2img_range<T, HAS_Z, false>(chain, x, y, z, row, col, p0, p1, threadIdx.x, kThreads, vec_ok);
        });
    } else {
        const size_t tid = (size_t)blockIdx.x * kThreads + threadIdx.x;
        const size_t nthreads = (size_t)gridDim.x * kThreads;
        world2img_range<T, HAS_Z, false>([&](size_t) -> const Chain<T>& { return src; }, x, y, z, row, col,
                                         0, n, tid, nthreads, vec_ok);
    }
}

// AoS kernels: rc = n (row, col) pairs; xyz = n points of 3 (HAS_Z) or 2 coordinates.  Their bodies repeat
// the SoA kernels' instead of sharing a device function: with one, the SoA kernels' code changed.
template <typename T, bool HAS_Z, typename SRC = Chain<T>>
__global__ void __launch_bounds__(kThreads, kTableMinBlocks<SRC, std::is_same<T, double>::value>)
img2world_aos_kernel(const SRC src, const T* __restrict__ rc, T* __restrict__ xyz, size_t n, bool vec_ok) {
    if constexpr (IsTable<SRC>::value) {
        for_each_tile<T>(src, n, [&](size_t p0, size_t p1, auto&& chain) {
            img2world_range<T, HAS_Z, true>(chain, rc, nullptr, xyz, nullptr, nullptr, p0, p1, threadIdx.x, kThreads,
                                            vec_ok);
        });
    } else {
        const size_t tid = (size_t)blockIdx.x * kThreads + threadIdx.x;
        const size_t nthreads = (size_t)gridDim.x * kThreads;
        img2world_range<T, HAS_Z, true>([&](size_t) -> const Chain<T>& { return src; }, rc, nullptr, xyz, nullptr,
                                        nullptr, 0, n, tid, nthreads, vec_ok);
    }
}

template <typename T, bool HAS_Z, typename SRC = Chain<T>>
__global__ void __launch_bounds__(kThreads, kTableMinBlocks<SRC, std::is_same<T, float>::value>)
world2img_aos_kernel(const SRC src, const T* __restrict__ xyz, T* __restrict__ rc, size_t n, bool vec_ok) {
    if constexpr (IsTable<SRC>::value) {
        for_each_tile<T>(src, n, [&](size_t p0, size_t p1, auto&& chain) {
            world2img_range<T, HAS_Z, true>(chain, xyz, nullptr, nullptr, rc, nullptr, p0, p1, threadIdx.x, kThreads,
                                            vec_ok);
        });
    } else {
        const size_t tid = (size_t)blockIdx.x * kThreads + threadIdx.x;
        const size_t nthreads = (size_t)gridDim.x * kThreads;
        world2img_range<T, HAS_Z, true>([&](size_t) -> const Chain<T>& { return src; }, xyz, nullptr, nullptr, rc,
                                        nullptr, 0, n, tid, nthreads, vec_ok);
    }
}

static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

template <typename K>
static int grid_for(cc_ctx* ctx, K kernel, size_t work_items) {
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kThreads, 0) != cudaSuccess ||
        per_sm < 1)
        per_sm = 1;
    size_t want = (work_items + (size_t)kThreads * kUnroll - 1) / ((size_t)kThreads * kUnroll);
    size_t cap = (size_t)ctx->sm_count * per_sm;
    if (want < 1) want = 1;
    return (int)(want < cap ? want : cap);
}

template <typename T> static Chain<T> pick_chain(const ChainD& d);
template <> Chain<double> pick_chain<double>(const ChainD& d) { return d; }
template <> Chain<float> pick_chain<float>(const ChainD& d) { ChainF f; narrow_chain(d, &f); return f; }

// ---- multi-view calls: the device chain table ----------------------------------------------------
// One table per context: the rows of the call's segments, then its nseg + 1 offsets.  It is
// uploaded on the caller's stream from pinned staging, grows on demand and is freed with the
// context.  Calls on different streams of one context may overlap: a call on a stream other than
// the previous user's waits for the event that user recorded after its last kernel, so the table is
// never overwritten under a kernel still reading it.  The staging buffer is rewritten only after
// the previous upload out of it has completed.
template <typename T>
int point_table_upload(cc_ctx* ctx, bool to_img, const ChainD* chains, int nseg, const size_t* offsets,
                       cudaStream_t st, PointTable* out) {
    const size_t row_bytes = to_img ? sizeof(RowW2I<T>) : sizeof(RowI2W<T>);
    const size_t rows_bytes = ((size_t)nseg * row_bytes + 15) / 16 * 16;
    const size_t bytes = rows_bytes + ((size_t)nseg + 1) * sizeof(size_t);
    if (ctx->pt_stage_event) CC_CUDA(cudaEventSynchronize(ctx->pt_stage_event));
    else CC_CUDA(cudaEventCreateWithFlags(&ctx->pt_stage_event, cudaEventDisableTiming));
    if (ctx->pt_stage_bytes < bytes) {
        if (ctx->pt_stage) CC_CUDA(cudaFreeHost(ctx->pt_stage));
        ctx->pt_stage = nullptr; ctx->pt_stage_bytes = 0;
        CC_CUDA(cudaHostAlloc(&ctx->pt_stage, bytes, cudaHostAllocPortable));
        ctx->pt_stage_bytes = bytes;
    }
    uint8_t* h = static_cast<uint8_t*>(ctx->pt_stage);
    for (int s = 0; s < nseg; ++s) {
        const Chain<T> c = pick_chain<T>(chains[s]);
        if (to_img) pack(c, reinterpret_cast<RowW2I<T>*>(h)[s]);
        else pack(c, reinterpret_cast<RowI2W<T>*>(h)[s]);
    }
    memcpy(h + rows_bytes, offsets, ((size_t)nseg + 1) * sizeof(size_t));
    if (ctx->pt_used && ctx->pt_stream != st) CC_CUDA(cudaStreamWaitEvent(st, ctx->pt_event, 0));
    if (ctx->pt_table_bytes < bytes) {
        if (ctx->pt_table) {
            if (ctx->pt_used) CC_CUDA(cudaEventSynchronize(ctx->pt_event));
            CC_CUDA(cudaFree(ctx->pt_table));
        }
        ctx->pt_table = nullptr; ctx->pt_table_bytes = 0;
        CC_CUDA(cudaMalloc(&ctx->pt_table, bytes));
        ctx->pt_table_bytes = bytes;
    }
    uint8_t* d = static_cast<uint8_t*>(ctx->pt_table);
    CC_CUDA(cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, st));
    CC_CUDA(cudaEventRecord(ctx->pt_stage_event, st));
    out->rows = d;
    out->off = reinterpret_cast<const size_t*>(d + rows_bytes);
    return CC_OK;
}

// after the call's last kernel that reads the table, on that kernel's stream
int point_table_release(cc_ctx* ctx, cudaStream_t st) {
    if (!ctx->pt_event) CC_CUDA(cudaEventCreateWithFlags(&ctx->pt_event, cudaEventDisableTiming));
    CC_CUDA(cudaEventRecord(ctx->pt_event, st));
    ctx->pt_stream = st;
    ctx->pt_used = 1;
    return CC_OK;
}

void point_table_free(cc_ctx* ctx) {
    if (ctx->pt_event) cudaEventSynchronize(ctx->pt_event);
    if (ctx->pt_stage_event) cudaEventSynchronize(ctx->pt_stage_event);
    if (ctx->pt_table) cudaFree(ctx->pt_table);
    if (ctx->pt_stage) cudaFreeHost(ctx->pt_stage);
    if (ctx->pt_event) cudaEventDestroy(ctx->pt_event);
    if (ctx->pt_stage_event) cudaEventDestroy(ctx->pt_stage_event);
}

template <typename K>
static int grid_tiles(cc_ctx* ctx, K kernel, size_t n) {
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kThreads, 0) != cudaSuccess ||
        per_sm < 1)
        per_sm = 1;
    const size_t tiles = (n + kTile - 1) / kTile;
    const size_t cap = (size_t)ctx->sm_count * per_sm;
    return (int)(tiles < cap ? tiles : cap);
}

// ---- the launcher ------------------------------------------------------------------------------
// The kernel of one direction, layout, z and view source: SINGLE on a grid-stride grid over the vectors (the points
// when !vec), TABLE on one CTA per tile up to the resident limit.
template <typename T, bool TO_IMG, bool AOS, bool HAS_Z, typename SRC>
static void launch_kernel(cc_ctx* ctx, const SRC& src, const PointIO<T>& io, size_t n, bool vec, cudaStream_t st) {
    auto go = [&](auto k, auto... arrays) {
        const int grid = IsTable<SRC>::value ? grid_tiles(ctx, k, n) : grid_for(ctx, k, vec ? n / Vec<T>::N + 1 : n);
        k<<<grid, kThreads, 0, st>>>(src, arrays..., n, vec);
    };
    if constexpr (AOS && TO_IMG) go(world2img_aos_kernel<T, HAS_Z, SRC>, io.in[0], io.out[0]);
    else if constexpr (AOS) go(img2world_aos_kernel<T, HAS_Z, SRC>, io.in[0], io.out[0]);
    else if constexpr (TO_IMG) go(world2img_kernel<T, HAS_Z, SRC>, io.in[0], io.in[1], io.in[2], io.out[0], io.out[1]);
    else go(img2world_kernel<T, HAS_Z, SRC>, io.in[0], io.in[1], io.out[0], io.out[1], io.out[2]);
}

// f(std::true_type) or f(std::false_type): a run-time flag as a template argument
template <typename F> static void with_bool(bool b, F&& f) {
    if (b) f(std::true_type{});
    else f(std::false_type{});
}

// One launch over points [0, n) of io on st; none when n == 0.  The vector path needs every array the kernel
// dereferences 16-byte aligned.
template <typename T>
int launch_points(cc_ctx* ctx, const PointSrc& src, const PointIO<T>& io, size_t n, cudaStream_t st) {
    if (n == 0) return CC_OK;
    bool vec = true;
    for (int d = 0; d < io.in_arrays(); ++d) vec = vec && aligned16(io.in[d]);
    for (int d = 0; d < io.out_arrays(); ++d) vec = vec && aligned16(io.out[d]);
    const bool has_z = (io.to_img ? io.in_dim : io.out_dim) == 3;
    with_bool(io.to_img, [&](auto to_img) { with_bool(io.aos, [&](auto aos) { with_bool(has_z, [&](auto z) {
        constexpr bool TO_IMG = decltype(to_img)::value, AOS = decltype(aos)::value, HAS_Z = decltype(z)::value;
        using Row = std::conditional_t<TO_IMG, RowW2I<T>, RowI2W<T>>;
        if (src.chain)
            launch_kernel<T, TO_IMG, AOS, HAS_Z>(ctx, pick_chain<T>(*src.chain), io, n, vec, st);
        else
            launch_kernel<T, TO_IMG, AOS, HAS_Z>(
                ctx, ViewTable<Row>{static_cast<const Row*>(src.tb.rows), src.tb.off, src.base, src.seg_lo, src.seg_hi},
                io, n, vec, st);
    }); }); });
    ctx->launches++;
    CC_CUDA(cudaGetLastError());
    return CC_OK;
}

template int point_table_upload<double>(cc_ctx*, bool, const ChainD*, int, const size_t*, cudaStream_t, PointTable*);
template int point_table_upload<float>(cc_ctx*, bool, const ChainD*, int, const size_t*, cudaStream_t, PointTable*);
template int launch_points<double>(cc_ctx*, const PointSrc&, const PointIO<double>&, size_t, cudaStream_t);
template int launch_points<float>(cc_ctx*, const PointSrc&, const PointIO<float>&, size_t, cudaStream_t);

}  // namespace cc

