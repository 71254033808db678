// rectify.cu -- full-frame rectification (backward warp + bilinear gather): host side.
//
// Replaces warp(img, tform, axs) of src/plot_calibration.jl:40 (tform/axs from
// image_transformations :15-22 and get_axes :1-6) for batches of frames that share one
// view.  The map is never stored in memory: algorithmic traffic is one read and one write of
// every pixel (8 B/px fp32 gray, 6 B/px u8 RGB).
//
// Decomposition.  The first RowCol axis is contiguous in memory.  A tile is 32 consecutive
// first-axis pixels (lane = pixel, so every store instruction writes one full 128-byte line
// and consecutive lanes sample consecutive source texels) x 32 second-axis lines, 8 lines per
// consumer warp.  A work unit is one tile of a GROUP of consecutive frames: the tile's map
// (tap offsets, weights, pixel classes) is built once per unit and reused for every frame of
// the group (rectify_f32c1.cuh, rectify_u8c3.cuh).
//
// This file: the tile plan (per-tile source box, floor constants, valid ranges; built on the
// host once per calibration/geometry, cached in the context, uploaded once), the tensor map of
// the source frames, the persistent grid and its ticket counter (rectify_ring.cuh), and the
// choice between the TMA-staged kernels and the direct ones (pointers/pitches TMA cannot
// address, footprints too large to stage).
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <thread>
#include <vector>

#include "rectify_device.cuh"
#include "tma.cuh"

namespace cc {

constexpr int kT = 32;                 // strip width along the first axis = lanes of a warp
constexpr int kWarps = 4;              // consumer warps per CTA
constexpr int kTLf = 32;               // f32c1: lines per tile (a warp owns kTLf / kWarps of them)
constexpr int kTLu = 32;               // u8c3: lines per tile
constexpr int kTLmax = 32;             // most lines of a tile (sizes the per-stage q2 slots)
// most frames one unit rectifies with one map (measured, profiles/r1_rectify.md: the costlier the
// map, the larger the group; the cheaper, the finer the units for the tail of the ticket queue)
constexpr int kFGf32Exact = 12, kFGf32Fast = 4, kFGu8Exact = 16, kFGu8Fast = 16;
constexpr int kMaxStages = 8;
// dynamic shared memory one CTA may spend on its ring (4 resident CTAs of 48 KB + static slots fit in 227 KB)
constexpr int kRingBytes = 48 * 1024;
// f32c1 staged line pitch granularity in bytes (dense boxes; u8c3 lines take the bank-disjoint pitch of box_dims)
constexpr int kPitchAlignF32 = 16;
// __launch_bounds__ min CTAs/SM of the staged kernels (fast / exact coordinates)
constexpr int kMinBlocks = 1, kMinBlocksExact = 4;
constexpr int kMinBlocksU8 = 1, kMinBlocksU8Exact = 3;
constexpr int kConsumerThreads = 32 * kWarps;

struct TileCfg {
    int box1, box2;        // staged box, in pixels (box1 along the contiguous axis)
    int pitch_b;           // bytes between consecutive lines of a staged box (see plan_boxes)
    int stages;
    int ntiles2;           // tiles along the second axis
    int box_bytes;         // bytes one TMA load delivers = stage stride (multiple of 128)
    // persistent f32c1 kernels: work units (strip x, tile y, frame z), x fastest
    int strips;            // tiles along the first axis
    uint32_t units;        // strips * ntiles2 * frame groups
    int fg;                // frames per group: the tile's map is built once per group and reused
    uint32_t reserved;     // unused: keeps the offsets of the fields below, and with them the kernels' SASS
    // *_views_kernel only (frames with different views in ONE launch): units are (strip x, tile y, group) with
    // group = view * gpv + frame group of the view; the tile headers / q2 terms of view v start at v * tiles / v * sz2
    int fpv;               // frames per view
    int gpv;               // frame groups per view
    int tiles;             // strips * ntiles2
    // *_views_kernel frame window: the launch covers frames [w0, w0 + g.nframes) of the group (the tensor map and
    // dst start at frame w0).  Units cover the frame groups g0, g0 + 1 ... that meet the window; frame groups
    // stay inside a view, and those at the window's edges are cut to it.  w0 = g0 = 0: the whole group.
    int w0;
    uint32_t g0;
};

// Frames with different views in one launch (cc_rectify_*_views): what the single-view kernels take as
// launch parameters, per view, in the kernel's parameter space (constant bank: a warp-uniform index).
constexpr int kMaxViews = 64;
struct ViewParams { RectExact pe; RectFast pf; RectGeom g; };
struct ViewTable { ViewParams v[kMaxViews]; };

// f32c1: per-tile header precomputed on the host (RectPlan), read straight from global memory
struct __align__(16) TileHdr {
    double Mk1, Mk2;       // exact: 2^52 - K   (K = global 1-based index of local tap 0)
    float mk1, mk2;        // fast:  1.5*2^23 - K
    uint32_t R1, R2;       // number of valid local first-tap indices per axis (0: nothing staged)
    int x0, y0;            // box origin: TMA coordinates (x0: f32 texels / u8 BYTES of the line, multiple of 16 bytes; y0: lines; may be negative)
    uint32_t base_off;     // byte offset of local tap (0, 0) inside the stage (pixels are 4 or 3 bytes)
    uint32_t view;         // *_views_kernel: index of the unit's view, written by the producer (0 in the plan tables)
};
static_assert(sizeof(TileHdr) == 48, "TileHdr is read as three 16-byte words");

// per-stage slot of the persistent f32c1 kernels, published by the producer warp
struct SmemRing {
    uint64_t full[kMaxStages];
    uint64_t empty[kMaxStages];
    int4 pos[kMaxStages];            // (strip x, tile y, frame z, -); z < 0: no more work
    TileHdr hdr[kMaxStages];
    double q2[kMaxStages][kTLmax];   // exact path: second-axis world term of the lines of each staged tile
};

// global ticket counter of one launch (self-resetting: the last producer zeroes it)
struct RectSched { uint32_t next, done; };

}  // namespace cc
#include "rectify_ring.cuh"
#include "rectify_f32c1.cuh"
#include "rectify_u8c3.cuh"
namespace cc {

// --------------------------------------------------------------------------------------
// the map alone (FP64): the source coordinate each output pixel samples
// --------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kConsumerThreads)
rectify_map_kernel(const RectExact p, const RectGeom g, double* __restrict__ map_row,
                   double* __restrict__ map_col) {
    const int lane_id = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int a = blockIdx.x * kT + lane_id;
    if (a >= g.sz1) return;
    const RowTermD rt = rect_row_term(p, g.axs0 + a);
#pragma unroll
    for (int e = 0; e < kT / kWarps; ++e) {
        const int b = blockIdx.y * kT + warp * (kT / kWarps) + e;
        if (b < g.sz2) {
            double row, col;
            rect_coord(p, rt, rect_q2(p, g.axs1 + b), row, col);
            map_row[(long long)b * g.pitch + a] = row;
            map_col[(long long)b * g.pitch + a] = col;
        }
    }
}

// the FP32 fast path's map: the same arithmetic as the fast staged kernels (rect_row_term /
// rect_coord on RectFast), written out as floats
__global__ void __launch_bounds__(kConsumerThreads)
rectify_map_f32_kernel(const RectFast p, const RectGeom g, float* __restrict__ map_row,
                       float* __restrict__ map_col) {
    const int lane_id = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int a = blockIdx.x * kT + lane_id;
    if (a >= g.sz1) return;
    const RowTermF rt = rect_row_term(p, g.axs0 + a);
#pragma unroll
    for (int e = 0; e < kT / kWarps; ++e) {
        const int b = blockIdx.y * kT + warp * (kT / kWarps) + e;
        if (b < g.sz2) {
            float row, col;
            rect_coord(p, rt, (float)(g.axs1 + b) - p.c2, row, col);
            map_row[(long long)b * g.pitch + a] = row;
            map_col[(long long)b * g.pitch + a] = col;
        }
    }
}

// --------------------------------------------------------------------------------------
// host side
// --------------------------------------------------------------------------------------
static RectGeom make_geom(const int64_t axs_min[2], int sz1, int sz2, size_t pitch,
                          size_t frame_stride, int nframes) {
    RectGeom g;
    memset(&g, 0, sizeof(g));
    g.axs0 = (int)axs_min[0]; g.axs1 = (int)axs_min[1];
    g.sz1 = sz1; g.sz2 = sz2; g.pitch = (long long)pitch; g.frame_stride = (long long)frame_stride;
    g.nframes = nframes;
    return g;
}

static RectExact make_exact(const ChainD& ch, double ratio) {
    RectExact p;
    for (int i = 0; i < 3; ++i) { p.R0[i] = ch.R[3 * i]; p.R1[i] = ch.R[3 * i + 1]; p.t[i] = ch.t[i]; }
    p.inv_ratio = 1.0 / ratio;     // inv(LinearMap(ratio*I)), src/plot_calibration.jl:16-17
    p.inv_cs = ch.inv_cs; p.k = ch.k;
    p.frow = ch.frow; p.fcol = ch.fcol; p.crow = ch.crow; p.ccol = ch.ccol;
    return p;
}

// fast path: fold scale, 1/ratio and the rotation columns in double, shift the origin to
// the centre of the output so the FP32 products stay small
static RectFast make_fast(const ChainD& ch, double ratio, const RectGeom& g) {
    RectFast p;
    const double sc = (1.0 / ratio) * ch.inv_cs;
    const double c1r = std::nearbyint((double)g.axs0 + 0.5 * (g.sz1 - 1));
    const double c2r = std::nearbyint((double)g.axs1 + 0.5 * (g.sz2 - 1));
    for (int i = 0; i < 3; ++i) {
        const double A = ch.R[3 * i] * sc, C = ch.R[3 * i + 1] * sc;
        p.A[i] = (float)A; p.Cc[i] = (float)C;
        p.T[i] = (float)(ch.t[i] + A * c1r + C * c2r);
    }
    p.c1 = (float)c1r; p.c2 = (float)c2r;
    p.k = (float)ch.k; p.frow = (float)ch.frow; p.fcol = (float)ch.fcol;
    p.crow = (float)ch.crow; p.ccol = (float)ch.ccol;
    return p;
}

// host evaluation of the map (double) for the box-size estimate only
static void host_coord(const ChainD& ch, double inv_ratio, long long I1, long long I2, double* row,
                       double* col) {
    const double q1 = ((double)I1 * inv_ratio) * ch.inv_cs, q2 = ((double)I2 * inv_ratio) * ch.inv_cs;
    const double P1 = ch.R[1] * q2 + (ch.R[0] * q1 + ch.t[0]);
    const double P2 = ch.R[4] * q2 + (ch.R[3] * q1 + ch.t[1]);
    const double P3 = ch.R[7] * q2 + (ch.R[6] * q1 + ch.t[2]);
    const double u = P1 / P3, v = P2 / P3;
    const double radial = 1.0 + ch.k * (u * u + v * v);
    *row = ch.frow * radial * u + ch.crow;
    *col = ch.fcol * radial * v + ch.ccol;
}

// Tile plan.  For every output tile: the bounding box of its source footprint (32 samples on the
// tile perimeter, evaluated in double) and everything the kernels derive from it.  A plan
// depends on the calibration, ratio/axes, frame size and tile shape only -- not on the pixels --
// so it is built once on the host, uploaded once and reused by every later call with the same
// parameters (a video stream): the kernels' producer warp then only issues TMA loads.
struct PlanKey { ChainD ch; double ratio; RectGeom g; int tw, tl, pxb; };

struct RectPlan {
    PlanKey key;
    int n1, n2;                    // tiles along the first / second axis
    int need1, need2;              // largest footprint (pixels), incl. taps and slack
    int box1, box2, box_bytes;     // staged box (pixels) and its size; box_bytes == 0: not stageable
    int pitch_b;                   // bytes per staged line
    int tilt;                      // sign of d(source line)/d(first output index): which way a warp's taps change lines
    std::vector<int> origin;       // per tile: floor(min row), floor(min col) of the perimeter samples
    std::vector<unsigned char> p3_ok;
    std::vector<TileHdr> hdr;      // tile headers
    std::vector<double> q2;        // exact path: second-axis world term of every output line
    TileHdr* d_hdr;
    double* d_q2;
    int per_sm[2];                 // resident CTAs per SM of the staged kernel, [exact], cached (0: not queried yet)
    size_t per_sm_smem[2];
};

static void plan_free(RectPlan* p) {
    if (!p) return;
    if (p->d_hdr) cudaFree(p->d_hdr);
    if (p->d_q2) cudaFree(p->d_q2);
    delete p;
}

static void multi_free(void* mp);
static void multi_free_retired(cc_ctx* ctx);

void rectify_free_plans(cc_ctx* ctx) {
    for (int i = 0; i < cc_ctx::NPLAN; ++i) {
        plan_free(static_cast<RectPlan*>(ctx->rect_plans[i]));
        ctx->rect_plans[i] = nullptr;
    }
    for (int i = 0; i < cc_ctx::NMULTI; ++i) {
        multi_free(ctx->multi_plans[i]);
        ctx->multi_plans[i] = nullptr;
    }
    multi_free_retired(ctx);
    if (ctx->rect_upload) { cudaStreamSynchronize(ctx->rect_upload); cudaStreamDestroy(ctx->rect_upload); ctx->rect_upload = nullptr; }
    if (ctx->rect_join) { cudaStreamSynchronize(ctx->rect_join); cudaStreamDestroy(ctx->rect_join); ctx->rect_join = nullptr; }
    for (int k = 0; k < cc_ctx::NSLOT; ++k)
        if (ctx->rect_join_event[k]) { cudaEventDestroy(ctx->rect_join_event[k]); ctx->rect_join_event[k] = nullptr; }
}

static void plan_footprints(RectPlan* p, bool threads) {
    const ChainD& ch = p->key.ch;
    const RectGeom& g = p->key.g;
    const int tw = p->key.tw, tl = p->key.tl;
    const double inv_ratio = 1.0 / p->key.ratio;
    p->n1 = (g.sz1 + tw - 1) / tw;
    p->n2 = (g.sz2 + tl - 1) / tl;
    p->origin.assign((size_t)p->n1 * p->n2 * 2, -4);
    p->p3_ok.assign((size_t)p->n1 * p->n2, 1);
    // strips [s0, s1) of the plan; partial maxima / tilt votes of the range go to out[3]
    auto strips = [&](int s0, int s1, long long* out) {
    int m1 = 0, m2 = 0;
    long long tilt = 0;
    for (int t1 = s0; t1 < s1; ++t1) {
        const int a_lo = t1 * tw, a_hi = std::min(a_lo + tw - 1, g.sz1 - 1);
        for (int t2 = 0; t2 < p->n2; ++t2) {
            const int b_lo = t2 * tl, b_hi = std::min(b_lo + tl - 1, g.sz2 - 1);
            double rmin = 0, rmax = 0, cmin = 0, cmax = 0;
            bool finite = true;
            double c_first = 0, c_last = 0;         // source line at the two ends of the tile's first output line
            for (int j = 0; j < 32; ++j) {          // 8 samples on each of the four edges
                const int k = j & 7;
                const bool far = (j & 8) != 0;
                int ca, cb;
                if (j < 16) { ca = far ? a_hi : a_lo; cb = b_lo + ((b_hi - b_lo) * k) / 7; }
                else        { cb = far ? b_hi : b_lo; ca = a_lo + ((a_hi - a_lo) * k) / 7; }
                double r, c;
                host_coord(ch, inv_ratio, g.axs0 + ca, g.axs1 + cb, &r, &c);
                finite = finite && std::isfinite(r) && std::isfinite(c);
                if (j == 0) { rmin = rmax = r; cmin = cmax = c; }
                if (j == 16) c_first = c;
                if (j == 23) c_last = c;
                rmin = std::min(rmin, r); rmax = std::max(rmax, r);
                cmin = std::min(cmin, c); cmax = std::max(cmax, c);
            }
            // P3 is monotone in each output index: the four corners bound it over the tile.  The
            // branch-free reciprocal of the exact kernels needs a sane exponent and one sign.
            double p3min = 0, p3max = 0;
            for (int j = 0; j < 4; ++j) {
                const long long I1 = g.axs0 + ((j & 1) ? a_hi : a_lo), I2 = g.axs1 + ((j & 2) ? b_hi : b_lo);
                const double q1 = ((double)I1 * inv_ratio) * ch.inv_cs, q2 = ((double)I2 * inv_ratio) * ch.inv_cs;
                const double P3 = std::fma(ch.R[7], q2, std::fma(ch.R[6], q1, ch.t[2]));
                if (j == 0) p3min = p3max = P3;
                p3min = std::min(p3min, P3); p3max = std::max(p3max, P3);
            }
            const bool p3_ok = std::isfinite(p3min) && std::isfinite(p3max) &&
                               ((p3min > 1e-270 && p3max < 1e270) || (p3max < -1e-270 && p3min > -1e270));
            const size_t t = (size_t)t1 * p->n2 + t2;
            p->p3_ok[t] = p3_ok ? 1 : 0;
            if (!finite) continue;                  // origin stays at (-4, -4): the range tests fail
            tilt += (c_last > c_first) - (c_last < c_first);
            // clamp so that far-away footprints still give a legal (fully out-of-frame) box
            const double rc = std::min(std::max(rmin, -4.0), (double)g.sz1 + 4.0);
            const double cc_ = std::min(std::max(cmin, -4.0), (double)g.sz2 + 4.0);
            p->origin[2 * t] = (int)std::floor(rc);
            p->origin[2 * t + 1] = (int)std::floor(cc_);
            // tiles entirely outside the frame never gather
            if (rmax < 1.0 || cmax < 1.0 || rmin > g.sz1 || cmin > g.sz2) continue;
            m1 = std::max(m1, (int)(std::floor(rmax) - std::floor(rmin)));
            m2 = std::max(m2, (int)(std::floor(cmax) - std::floor(cmin)));
        }
    }
    out[0] = m1; out[1] = m2; out[2] = tilt;
    };
    // large plans (a 4K frame has 8160 tiles x 36 coordinate evaluations) are split over host threads; every
    // tile writes its own slots of origin / p3_ok, the partials are combined in strip order
    const long long tiles = (long long)p->n1 * p->n2;
    const int nt = !threads ? 1 : (int)std::max(1ll, std::min<long long>({tiles / 512, 16ll, (long long)std::max(1u, std::thread::hardware_concurrency()), (long long)p->n1}));
    std::vector<long long> part((size_t)nt * 3, 0);
    if (nt == 1) {
        strips(0, p->n1, part.data());
    } else {
        std::vector<std::thread> th;
        for (int t = 0; t < nt; ++t) {
            const int s0 = (int)((long long)p->n1 * t / nt), s1 = (int)((long long)p->n1 * (t + 1) / nt);
            bool spawned = false;
            if (t + 1 < nt) {
                try { th.emplace_back(strips, s0, s1, part.data() + 3 * t); spawned = true; }
                catch (...) {}                  // no thread to be had: this range runs here (nothing throws across the C ABI)
            }
            if (!spawned) strips(s0, s1, part.data() + 3 * t);
        }
        for (auto& x : th) x.join();
    }
    int m1 = 0, m2 = 0;
    long long tilt = 0;
    for (int t = 0; t < nt; ++t) { m1 = std::max(m1, (int)part[3 * t]); m2 = std::max(m2, (int)part[3 * t + 1]); tilt += part[3 * t + 2]; }
    // taps floor-1 .. floor; 2 texels of slack below (origin) and 1 above
    p->need1 = m1 + 2 + 3;
    p->need2 = m2 + 2 + 3;
    p->tilt = tilt >= 0 ? 1 : -1;
}

// box size from the footprint; tile headers
//
// f32c1 (4-byte pixels): the box origin along the first axis is a texel index rounded down to 4
// texels (16 bytes, what TMA can address); dense lines (pitch = box width).
//
// u8c3 (3-byte pixels): the TMA tensor is the line of BYTES, so the origin is a byte offset rounded
// down to 16 bytes -- at most 15 bytes (5 texels) of slack instead of the 15 texels a texel-granular
// origin needs -- and the tile header carries the byte offset of local tap 0.  Line pitch: the lanes
// of a warp read consecutive 3-byte texels (32 lanes span ~24-26 words); on a rotated map the upper
// part of the warp samples the neighbouring source line, `pitch` bytes away.  Both parts hit disjoint
// banks iff the pitch in words is +4 (mod 32) in the direction the source line changes: with a
// multiple of 128 bytes the two lanes at the change share a bank (ncu, round 2: 1.2 wavefronts per
// LDS), with anything else whole groups of lanes collide (1.7 wavefronts with 192-byte lines).
static int floor_to(int v, int m) { return v >= 0 ? (v / m) * m : -(((-v) + m - 1) / m) * m; }

// staged box of a footprint of need1 x need2 texels (tilt: RectPlan.tilt); box_bytes == 0: not worth staging
struct BoxDims { int box1, box2, pitch_b, box_bytes; };

static BoxDims box_dims(int need1, int need2, int tilt, int pxb) {
    BoxDims d;
    if (pxb == 4) {
        const int unit = 4;
        d.box1 = (need1 + unit - 1 + unit - 1) / unit * unit;          // + unit - 1: the origin is rounded down
        d.pitch_b = (d.box1 * pxb + kPitchAlignF32 - 1) / kPitchAlignF32 * kPitchAlignF32;
        d.box1 = d.pitch_b / pxb;                                      // usable pixels per line
    } else {
        const int need_b = need1 * 3 + 15;                             // + 15: the byte origin is rounded down
        int pitch = (need_b + 15) / 16 * 16;
        const int want = tilt >= 0 ? 4 : 28;                           // pitch in words, mod 32
        const int dense = pitch;
        while ((pitch / 4) % 32 != want) pitch += 16;
        // a TMA box line holds at most 256 elements (bytes here): a footprint whose bank-disjoint pitch does
        // not fit keeps the dense pitch (some bank conflicts) rather than losing the staged path altogether
        if (pitch > 256 && dense <= 256) pitch = dense;
        d.pitch_b = pitch;
        d.box1 = pitch / 3;
    }
    d.box2 = need2;
    while (((size_t)d.pitch_b * d.box2) % 128) ++d.box2;              // every stage base stays 128-byte aligned
    const int box1_elems = (pxb == 4) ? d.pitch_b / 4 : d.pitch_b;
    d.box_bytes = d.pitch_b * d.box2;
    if (box1_elems > 256 || d.box2 > 256 || d.box_bytes > 40 * 1024) d.box_bytes = 0;   // not worth staging
    return d;
}

// tile headers of a plan's footprints for a staged box of the given size (the plan's own, or the common box of
// a group of views: any box at least as large as the plan's footprint gives the same pixels)
static void fill_headers(const RectPlan* p, const BoxDims& d, TileHdr* hdr) {
    const RectGeom& g = p->key.g;
    const int pxb = p->key.pxb;
    const size_t ntiles = (size_t)p->n1 * p->n2;
    for (size_t t = 0; t < ntiles; ++t) {
        TileHdr& h = hdr[t];
        memset(&h, 0, sizeof(h));
        const int y0 = p->origin[2 * t + 1] - 2;
        // first tap g1 (0-based texel index): inside the box (both taps) and inside the frame
        int g_lo, g_hi;
        if (pxb == 4) {
            const int x0 = floor_to(p->origin[2 * t] - 2, 4);
            h.x0 = x0;
            g_lo = std::max(0, x0);
            g_hi = std::min(x0 + d.box1 - 2, g.sz1 - 2);
            h.base_off = (uint32_t)(g_lo - x0) * 4u;
        } else {
            const int xb0 = floor_to((p->origin[2 * t] - 2) * 3, 16);
            h.x0 = xb0;
            g_lo = std::max(0, xb0 >= 0 ? (xb0 + 2) / 3 : 0);                       // 3 g1 >= xb0
            g_hi = std::min((xb0 + d.pitch_b - 6) >= 0 ? (xb0 + d.pitch_b - 6) / 3 : -1, g.sz1 - 2);   // 3 g1 + 6 <= xb0 + pitch
            h.base_off = (uint32_t)(3 * g_lo - xb0);
        }
        const int lo2 = std::max(0, -y0), hi2 = std::min(d.box2 - 2, g.sz2 - 2 - y0);
        h.y0 = y0;
        h.R1 = p->p3_ok[t] ? (uint32_t)std::max(0, g_hi - g_lo + 1) : 0u;
        h.R2 = (uint32_t)std::max(0, hi2 - lo2 + 1);
        const int k1 = 1 + g_lo, k2 = 1 + y0 + lo2;       // global 1-based index of local tap 0
        h.Mk1 = 4503599627370496.0 - (double)k1;
        h.Mk2 = 4503599627370496.0 - (double)k2;
        h.mk1 = 12582912.0f - (float)k1;
        h.mk2 = 12582912.0f - (float)k2;
        h.base_off += (uint32_t)lo2 * (uint32_t)d.pitch_b;
    }
}

static void plan_boxes(RectPlan* p) {
    const RectGeom& g = p->key.g;
    const BoxDims d = box_dims(p->need1, p->need2, p->tilt, p->key.pxb);
    p->box1 = d.box1; p->box2 = d.box2; p->pitch_b = d.pitch_b; p->box_bytes = d.box_bytes;
    // the second-axis world terms do not depend on the box (the views call needs them for unstageable plans too)
    p->q2.resize((size_t)g.sz2);
    const double inv_ratio = 1.0 / p->key.ratio;
    for (int b = 0; b < g.sz2; ++b)       // rect_q2() of rectify_device.cuh, same two products
        p->q2[b] = ((double)((long long)g.axs1 + b) * inv_ratio) * p->key.ch.inv_cs;
    if (!p->box_bytes) return;
    p->hdr.resize((size_t)p->n1 * p->n2);
    fill_headers(p, d, p->hdr.data());
}

// tile headers and q2 terms of a plan to the device (once); false: out of device memory
static bool plan_upload(RectPlan* p, cudaStream_t st) {
    if (p->d_hdr || p->hdr.empty()) return true;
    const size_t hb = p->hdr.size() * sizeof(TileHdr), qb = p->q2.size() * sizeof(double);
    if (cudaMalloc(&p->d_hdr, hb) != cudaSuccess || cudaMalloc(&p->d_q2, qb) != cudaSuccess ||
        cudaMemcpyAsync(p->d_hdr, p->hdr.data(), hb, cudaMemcpyHostToDevice, st) != cudaSuccess ||
        cudaMemcpyAsync(p->d_q2, p->q2.data(), qb, cudaMemcpyHostToDevice, st) != cudaSuccess) {
        cudaGetLastError();
        if (p->d_hdr) cudaFree(p->d_hdr);
        if (p->d_q2) cudaFree(p->d_q2);
        p->d_hdr = nullptr; p->d_q2 = nullptr;
        return false;
    }
    // later calls may come on other streams: make the tables visible to all of them
    cudaStreamSynchronize(st);
    return true;
}

static RectPlan* plan_find(cc_ctx* ctx, const PlanKey& key) {
    for (int i = 0; i < cc_ctx::NPLAN; ++i) {
        RectPlan* p = static_cast<RectPlan*>(ctx->rect_plans[i]);
        if (p && memcmp(&p->key, &key, sizeof(key)) == 0) return p;
    }
    return nullptr;
}

// footprints, box and headers of one parameter set: host arithmetic only (safe to run on several threads;
// threads: split a large plan over host threads itself -- off when the caller already runs one plan per thread)
static RectPlan* plan_build(const PlanKey& key, bool threads) {
    RectPlan* p = new (std::nothrow) RectPlan();
    if (!p) return nullptr;
    p->key = key; p->d_hdr = nullptr; p->d_q2 = nullptr;
    p->per_sm[0] = p->per_sm[1] = 0; p->per_sm_smem[0] = p->per_sm_smem[1] = 0;
    plan_footprints(p, threads);
    plan_boxes(p);
    return p;
}

static void plan_insert(cc_ctx* ctx, RectPlan* p) {
    const int slot = ctx->rect_plan_next++ % cc_ctx::NPLAN;
    if (ctx->rect_plans[slot]) {
        cudaDeviceSynchronize();       // an evicted plan may still be read by a running kernel
        plan_free(static_cast<RectPlan*>(ctx->rect_plans[slot]));
    }
    ctx->rect_plans[slot] = p;
}

static PlanKey plan_key(const ChainD& ch, double ratio, const RectGeom& g, int tw, int tl, int pxb) {
    PlanKey key;
    memset(&key, 0, sizeof(key));
    key.ch = ch; key.ratio = ratio; key.g = g; key.g.nframes = 0; key.g.frame_stride = 0;
    key.tw = tw; key.tl = tl; key.pxb = pxb;
    return key;
}

// find or build the plan of this (calibration, geometry, tile shape); its tables go to the device on first use
static RectPlan* plan_get(cc_ctx* ctx, const ChainD& ch, double ratio, const RectGeom& g, int tw, int tl,
                          int pxb, cudaStream_t st) {
    const PlanKey key = plan_key(ch, ratio, g, tw, tl, pxb);
    if (RectPlan* p = plan_find(ctx, key)) return plan_upload(p, st) ? p : nullptr;
    RectPlan* p = plan_build(key, true);
    if (!p) return nullptr;
    if (!plan_upload(p, st)) {
        plan_free(p);
        return nullptr;
    }
    plan_insert(ctx, p);
    return p;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);

static EncodeTiledFn encoder(cc_ctx* ctx) {
    if (!ctx->encode_tiled) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            ctx->encode_tiled = fn;
    }
    return reinterpret_cast<EncodeTiledFn>(ctx->encode_tiled);
}

// ring stages of a staged box: measured (profiles/r1_rectify.md), occupancy beats ring depth; small boxes afford more
// stages.  The ring hides the TMA round trip: per SM, (stages - 1) x resident CTAs x the USEFUL bytes of a box must
// cover bandwidth x latency (~30 KB of reads at the HBM roofline, profiles/r2_rectify.md)
static int ring_stages(int box_bytes) {
    int stages = std::min(kMaxStages, std::max(2, kRingBytes / box_bytes));
    while (stages > 2 && stages * box_bytes > 56 * 1024) --stages;
    return stages;
}

// TMA can address the frames: 16-byte aligned base, lines and (more than one frame) frames
static bool tma_aligned(const void* src, int pxb, size_t pitch, size_t frame_stride, int nframes) {
    return !((reinterpret_cast<uintptr_t>(src) & 15u) || ((pitch * pxb) & 15u) || (nframes > 1 && ((frame_stride * pxb) & 15u)));
}

// the tensor map of `nframes` frames at src (pxb bytes per pixel) in boxes d, and the box and ring of *cfg; false: the
// map cannot be encoded
static bool stage_box(cc_ctx* ctx, const void* src, int pxb, int sz1, int sz2, size_t pitch, size_t frame_stride,
                      int nframes, const BoxDims& d, CUtensorMap* tmap, TileCfg* cfg) {
    EncodeTiledFn enc = encoder(ctx);
    if (!enc) return false;
    const size_t pitch_b = pitch * pxb;
    cuuint64_t dims[3] = {(cuuint64_t)sz1 * (pxb == 4 ? 1 : 3), (cuuint64_t)sz2, (cuuint64_t)std::max(nframes, 1)};
    cuuint64_t strides[2] = {(cuuint64_t)pitch_b, (cuuint64_t)(nframes > 1 ? frame_stride * pxb : pitch_b * sz2)};
    cuuint32_t box[3] = {(cuuint32_t)(pxb == 4 ? d.pitch_b / 4 : d.pitch_b), (cuuint32_t)d.box2, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    memset(tmap, 0, sizeof(*tmap));
    if (enc(tmap, pxb == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<void*>(src),
            dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
        return false;
    cfg->box1 = d.box1; cfg->box2 = d.box2; cfg->pitch_b = d.pitch_b; cfg->box_bytes = d.box_bytes;
    cfg->stages = ring_stages(d.box_bytes);
    return true;
}

// Decide whether the TMA-staged variant applies and build its tensor map + tile config.
static bool plan_tma(cc_ctx* ctx, const ChainD& ch, double ratio, const RectGeom& g, const void* src, int pxb, int tl,
                     cudaStream_t st, CUtensorMap* tmap, TileCfg* cfg, RectPlan** plan_out) {
    if (!tma_aligned(src, pxb, g.pitch, g.frame_stride, g.nframes) || !encoder(ctx)) return false;
    RectPlan* plan = plan_get(ctx, ch, ratio, g, kT, tl, pxb, st);
    if (!plan || !plan->box_bytes) return false;
    const BoxDims d = {plan->box1, plan->box2, plan->pitch_b, plan->box_bytes};
    if (!stage_box(ctx, src, pxb, g.sz1, g.sz2, g.pitch, g.frame_stride, g.nframes, d, tmap, cfg)) return false;
    *plan_out = plan;
    return true;
}

// cudaFuncAttributeMaxDynamicSharedMemorySize belongs to the KERNEL (per device), not to a plan:
// the library remembers the largest value it has set per staged kernel and device and only ever
// raises it (a smaller plan must not lower the limit under a cached larger one, whichever context
// of the process made either call).
static std::mutex g_smem_mu;
static size_t g_smem_attr[64][12];
template <typename K>
static int set_smem(cc_ctx* ctx, int kslot, K kernel, size_t bytes) {
    if (bytes <= 32 * 1024) return CC_OK;     // static smem (barriers + headers) counts against the 48 KB default too
    std::lock_guard<std::mutex> lk(g_smem_mu);
    size_t& cur = g_smem_attr[ctx->device & 63][kslot];
    if (bytes > cur) {
        CC_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
        cur = bytes;
    }
    return CC_OK;
}

// Ticket counters: a small ring of self-resetting counters per context.  Launches on different
// streams may overlap, so consecutive launches take different counters, and a counter is only
// handed out again after the launch that used it last has finished (event wait on the new stream).
static int sched_acquire(cc_ctx* ctx, cudaStream_t st, RectSched** out) {
    if (!ctx->sched_pool) {
        CC_CUDA(cudaMalloc(&ctx->sched_pool, cc_ctx::NSCHED * sizeof(RectSched)));
        CC_CUDA(cudaMemset(ctx->sched_pool, 0, cc_ctx::NSCHED * sizeof(RectSched)));
        for (int i = 0; i < cc_ctx::NSCHED; ++i)
            CC_CUDA(cudaEventCreateWithFlags(&ctx->sched_event[i], cudaEventDisableTiming));
    }
    const int slot = ctx->sched_next % cc_ctx::NSCHED;
    if (ctx->sched_used[slot] && ctx->sched_stream[slot] != st)
        CC_CUDA(cudaStreamWaitEvent(st, ctx->sched_event[slot], 0));
    *out = static_cast<RectSched*>(ctx->sched_pool) + slot;
    return CC_OK;
}

static void sched_release(cc_ctx* ctx, cudaStream_t st) {
    const int slot = ctx->sched_next++ % cc_ctx::NSCHED;
    cudaEventRecord(ctx->sched_event[slot], st);
    ctx->sched_used[slot] = 1;
    ctx->sched_stream[slot] = st;
}

void rectify_free_sched(cc_ctx* ctx) {
    if (!ctx->sched_pool) return;
    for (int i = 0; i < cc_ctx::NSCHED; ++i) cudaEventDestroy(ctx->sched_event[i]);
    cudaFree(ctx->sched_pool);
    ctx->sched_pool = nullptr;
}

// persistent grid of a staged kernel: every CTA slot of the device (tickets do the balancing)
template <typename K, typename PL>
static int persistent_grid(cc_ctx* ctx, int kslot, K kernel, size_t smem, const TileCfg& cfg, PL* plan, bool exact,
                           uint32_t* gsz) {
    // the occupancy query and the shared-memory attribute cost microseconds per call: once per plan
    int rc = set_smem(ctx, kslot, kernel, smem);
    if (rc) return rc;
    int per_sm = plan->per_sm_smem[exact] == smem ? plan->per_sm[exact] : 0;
    if (per_sm == 0) {
        CC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kConsumerThreads + 32, smem));
        plan->per_sm[exact] = per_sm;
        plan->per_sm_smem[exact] = smem;
    }
    *gsz = std::min<uint32_t>(cfg.units, (uint32_t)ctx->sm_count * (uint32_t)std::max(per_sm, 1));
    if (getenv("CAMCAL_DEBUG"))
        fprintf(stderr, "[camcal] staged: box %dx%d pitch %d (%d B) stages %d units %u (fg %d) grid %u (%d/SM) smem %zu\n",
                cfg.box1, cfg.box2, cfg.pitch_b, cfg.box_bytes, cfg.stages, cfg.units, cfg.fg, *gsz, per_sm, smem);
    return CC_OK;
}

// Frames per group.  The map of a tile (indices, weights) depends on the calibration only, so a
// unit rectifies the same tile of `fg` consecutive frames and computes the map once.  Larger
// groups amortise better; smaller ones leave more units for the tail of the ticket queue: keep
// at least ~8 units per resident CTA slot.
static int unit_cfg(cc_ctx* ctx, TileCfg* cfg, int sz1, int sz2, int nframes, int tw, int tl, int fg_max) {
    cfg->strips = (sz1 + tw - 1) / tw;
    cfg->ntiles2 = (sz2 + tl - 1) / tl;
    const long long tiles = (long long)cfg->strips * cfg->ntiles2;
    const long long want = (long long)ctx->sm_count * 6 * 8;
    int fg = std::min(fg_max, nframes);
    while (fg > 1 && tiles * ((nframes + fg - 1) / fg) < want) fg = (fg + 1) / 2;
    if (const char* e = getenv("CAMCAL_FG")) fg = std::max(1, std::min(nframes, atoi(e)));   // tuning knob
    cfg->fg = fg;
    const long long groups = (nframes + fg - 1) / fg;
    CC_REQUIRE(tiles * groups < (1ll << 31), "too many tiles in one call: split the batch");
    cfg->units = (uint32_t)(tiles * groups);
    return CC_OK;
}

// grid of the direct (unstaged) kernels: ~64 CTAs per SM worth of work, at least 32 lines per CTA
static dim3 direct_grid(cc_ctx* ctx, int sz1, int sz2, int nframes, int* lines) {
    const int strips = (sz1 + kT - 1) / kT;
    const long long per_line_ctas = (long long)strips * nframes;
    const long long segs = std::max<long long>(1, ((long long)ctx->sm_count * 64 + per_line_ctas - 1) / per_line_ctas);
    *lines = (int)std::max<long long>(32, (sz2 + segs - 1) / segs);
    return dim3(strips, (sz2 + *lines - 1) / *lines, nframes);
}

// --------------------------------------------------------------------------------------
// The pixel formats: every fact the launchers below need that differs between fp32 gray and 8-bit RGB.  staged /
// views / direct: the kernel of each family; *_slot: its g_smem_attr slot (exact; + 1: fast); ring: the ring of a
// staged launch (nf: frames per stage), returns its dynamic shared memory; launch: the one <<<>>> of every kernel of
// the format, with the format's arguments after `dst`.
// --------------------------------------------------------------------------------------
template <typename PX> struct RectFmt;

template <> struct RectFmt<float> {
    static constexpr int pxb = RectPx<float>::bytes, tl = kTLf, fg_exact = kFGf32Exact, fg_fast = kFGf32Fast, views_slot = 6;
    static auto staged(bool e, int nf) {
        return nf == 2 ? (e ? rectify_f32c1_kernel<true> : rectify_f32c1_kernel<false>)
                       : (e ? rectify_f32c1_single_kernel<true> : rectify_f32c1_single_kernel<false>);
    }
    static int staged_slot(int nf) { return nf == 2 ? 0 : 4; }
    static auto views(bool e) { return e ? rectify_f32c1_views_kernel<true> : rectify_f32c1_views_kernel<false>; }
    static auto direct(bool e) { return e ? rectify_f32c1_direct_kernel<true> : rectify_f32c1_direct_kernel<false>; }
    // two frames per ring stage when the ring holds at least four boxes (large boxes keep one) and the units have at
    // least two frames (single frames, e.g. the per-view launches of cc_rectify_*_views, keep one); the views kernel
    // holds one frame per stage
    static size_t ring(TileCfg& cfg, bool views, int* nf) {
        *nf = (!views && cfg.stages >= 4 && cfg.fg >= 2) ? 2 : 1;
        cfg.stages /= *nf;
        return (size_t)cfg.stages * *nf * cfg.box_bytes;
    }
    static bool dst_ok(const float*, const RectFrames&, int) { return true; }
    template <typename K, typename... A>
    static void launch(K k, dim3 grid, int threads, size_t smem, cudaStream_t st, const RectCall<float>& c, const A&... a) {
        k<<<grid, threads, smem, st>>>(a..., c.fill);
    }
};

template <> struct RectFmt<uint8_t> {
    static constexpr int pxb = RectPx<uint8_t>::bytes, tl = kTLu, fg_exact = kFGu8Exact, fg_fast = kFGu8Fast, views_slot = 8;
    static auto staged(bool e, int) { return e ? rectify_u8c3_kernel<true> : rectify_u8c3_kernel<false>; }
    static int staged_slot(int) { return 2; }
    static auto views(bool e) { return e ? rectify_u8c3_views_kernel<true> : rectify_u8c3_views_kernel<false>; }
    static auto direct(bool e) { return e ? rectify_u8c3_direct_kernel<true> : rectify_u8c3_direct_kernel<false>; }
    // one frame per stage; + 16: the word-granular gather may read the aligned words that hold the last tap bytes
    static size_t ring(TileCfg& cfg, bool, int* nf) {
        *nf = 1;
        return (size_t)cfg.stages * cfg.box_bytes + 16;
    }
    // the staged kernel writes whole 32-bit words: 4-byte aligned output lines
    static bool dst_ok(const uint8_t* dst, const RectFrames& fr, int nframes) {
        return (reinterpret_cast<uintptr_t>(dst) & 3u) == 0 && ((fr.pitch * 3) & 3u) == 0 &&
               (nframes <= 1 || ((fr.frame_stride * 3) & 3u) == 0);
    }
    // frame_bytes: the bytes of one frame that belong to the caller (the last line is only sz1 pixels long)
    template <typename K, typename... A>
    static void launch(K k, dim3 grid, int threads, size_t smem, cudaStream_t st, const RectCall<uint8_t>& c,
                       const A&... a) {
        const unsigned frame_bytes = (unsigned)((c.fr.pitch * (size_t)(c.fr.sz2 - 1) + (size_t)c.fr.sz1) * 3);
        k<<<grid, threads, smem, st>>>(a..., c.fill, frame_bytes);
    }
};

// One launch of the single-view kernels: frames [0, nframes) of view v at src / dst (the call's layout), on st.
template <typename PX>
int launch_rectify(cc_ctx* ctx, const RectCall<PX>& c, int v, int nframes, const PX* src, PX* dst, cudaStream_t st) {
    using F = RectFmt<PX>;
    if (nframes == 0) return CC_OK;
    const ChainD& ch = c.views.chs[v];
    const double ratio = c.views.ratios[v];
    const RectGeom g = make_geom(c.views.axs_mins + 2 * v, c.fr.sz1, c.fr.sz2, c.fr.pitch, c.fr.frame_stride, nframes);
    const RectExact pe = make_exact(ch, ratio);
    const RectFast pf = make_fast(ch, ratio, g);
    const bool exact = !(c.flags & CC_COORD_F32);
    CUtensorMap tmap;
    TileCfg cfg;
    memset(&cfg, 0, sizeof(cfg));
    RectPlan* plan = nullptr;
    const bool tma = !(c.flags & CC_GATHER_DIRECT) && F::dst_ok(dst, c.fr, nframes) &&
                     plan_tma(ctx, ch, ratio, g, src, F::pxb, F::tl, st, &tmap, &cfg, &plan);
    if ((c.flags & CC_GATHER_TMA) && !tma)
        return set_error(CC_ERR_INVALID_ARG, "TMA gather not available for this layout / footprint");
    int rc = CC_OK;
    if (tma) {
        if ((rc = unit_cfg(ctx, &cfg, c.fr.sz1, c.fr.sz2, nframes, kT, F::tl, exact ? F::fg_exact : F::fg_fast))) return rc;
        int nf = 1;
        const size_t smem = F::ring(cfg, false, &nf);
        const auto k = F::staged(exact, nf);
        uint32_t gsz = 0;
        if ((rc = persistent_grid(ctx, F::staged_slot(nf) + !exact, k, smem, cfg, plan, exact, &gsz))) return rc;
        RectSched* sched = nullptr;
        if ((rc = sched_acquire(ctx, st, &sched))) return rc;
        F::launch(k, gsz, kConsumerThreads + 32, smem, st, c, tmap, pe, pf, g, cfg, plan->d_hdr, plan->d_q2, sched, src, dst);
        sched_release(ctx, st);
    } else {
        int lines = 0;
        const dim3 grid = direct_grid(ctx, c.fr.sz1, c.fr.sz2, nframes, &lines);
        F::launch(F::direct(exact), grid, kConsumerThreads, 0, st, c, pe, pf, g, lines, src, dst);
    }
    ctx->launches++;
    CC_CUDA(cudaGetLastError());
    return CC_OK;
}

// --------------------------------------------------------------------------------------
// Frames with different views in ONE launch (cc_rectify_*_views; the reference's plot loop,
// src/plot_calibration.jl:36-42).  The views of a group share the frame layout, so they share the tensor map
// and -- with the largest footprint of the group as the common staged box -- the ring; what differs per view
// (coordinate parameters, axes, tile headers, q2 terms) is indexed by the unit's view.  One launch per view
// (round 2's first version) spent more time in 64 ramp-ups, tails and host launches than in the work.
// --------------------------------------------------------------------------------------
struct MultiPlan {
    std::vector<PlanKey> keys;     // the views of the group, in order
    BoxDims d;                     // the common staged box
    int n1, n2;
    TileHdr* d_hdr;                // [view][tile]
    double* d_q2;                  // [view][sz2]
    size_t hdr_cap, q2_cap;        // bytes allocated at d_hdr / d_q2
    int per_sm[2];
    size_t per_sm_smem[2];
    std::vector<TileHdr> h_hdr;    // the tables on the host, until their upload has completed
    std::vector<double> h_q2;
    // The host form (cc_rectify_views_*_host) uploads on its own stream: `ready` follows the upload, and the slot
    // streams wait for it.  `fence` follows the last launches that read the tables, on `fence_stream` (a device
    // call on another stream waits for it first, so it covers every reader): the host form reuses or frees the
    // buffers of an evicted plan after it, without synchronising the device.
    cudaEvent_t ready;
    cudaEvent_t fence;
    cudaStream_t fence_stream;
    bool fenced;
    MultiPlan* next_retired;       // cc_ctx::multi_retired: evicted, freed once its fence has passed
};

static void multi_free(void* p) {
    MultiPlan* mp = static_cast<MultiPlan*>(p);
    if (!mp) return;
    if (mp->d_hdr) cudaFree(mp->d_hdr);
    if (mp->d_q2) cudaFree(mp->d_q2);
    if (mp->ready) cudaEventDestroy(mp->ready);
    if (mp->fence) cudaEventDestroy(mp->fence);
    delete mp;
}

// plans retired by the host form: their readers are fenced, so this waits for those only
static void multi_free_retired(cc_ctx* ctx) {
    MultiPlan* mp = static_cast<MultiPlan*>(ctx->multi_retired);
    ctx->multi_retired = nullptr;
    while (mp) {
        MultiPlan* next = mp->next_retired;
        if (mp->fenced) cudaEventSynchronize(mp->fence);
        multi_free(mp);
        mp = next;
    }
}

static MultiPlan* multi_find(cc_ctx* ctx, const std::vector<PlanKey>& keys) {
    for (int i = 0; i < cc_ctx::NMULTI; ++i) {
        MultiPlan* mp = static_cast<MultiPlan*>(ctx->multi_plans[i]);
        if (mp && mp->keys.size() == keys.size() && memcmp(mp->keys.data(), keys.data(), keys.size() * sizeof(PlanKey)) == 0)
            return mp;
    }
    return nullptr;
}

// the views [missing] of a group on up to 16 host threads (the plot loop is a one-shot call: 64 cold views cost
// 64 x ~0.5 ms of host arithmetic on one thread); then every duplicate of an earlier view gets that view's plan
static void plans_build(const std::vector<PlanKey>& keys, std::vector<RectPlan*>& pl, const std::vector<int>& missing) {
    if (!missing.empty()) {
        const int nt = (int)std::min<size_t>(missing.size(), std::min(16u, std::max(1u, std::thread::hardware_concurrency())));
        std::vector<std::thread> th;
        auto work = [&](int t) { for (size_t i = (size_t)t; i < missing.size(); i += (size_t)nt) pl[missing[i]] = plan_build(keys[missing[i]], nt == 1); };
        for (int t = 1; t < nt; ++t) {
            try { th.emplace_back(work, t); }
            catch (...) { work(t); }            // no thread to be had: this share runs here
        }
        work(0);
        for (auto& x : th) x.join();
    }
    for (size_t v = 0; v < pl.size(); ++v)
        if (!pl[v])                                        // a duplicate of an earlier view (or out of memory)
            for (size_t w = 0; w < v && !pl[v]; ++w)
                if (memcmp(&keys[w], &keys[v], sizeof(PlanKey)) == 0) pl[v] = pl[w];
}

// views of a group without a plan, each distinct view once
static std::vector<int> plans_missing(const std::vector<PlanKey>& keys, const std::vector<RectPlan*>& pl) {
    std::vector<int> missing;
    for (size_t v = 0; v < keys.size(); ++v) {
        bool dup = false;                                  // the same view twice: build it once
        for (size_t w = 0; w < v && !pl[v] && !dup; ++w) dup = memcmp(&keys[w], &keys[v], sizeof(PlanKey)) == 0;
        if (!pl[v] && !dup) missing.push_back((int)v);
    }
    return missing;
}

// the common box and the host tables of a group from its views' footprints (host arithmetic only);
// nullptr: a view has no plan (out of memory) or the group cannot be staged
static MultiPlan* multi_assemble(const std::vector<PlanKey>& keys, const std::vector<RectPlan*>& pl, int pxb) {
    const int nviews = (int)keys.size();
    int need1 = 0, need2 = 0;
    long long tilt = 0;
    for (int v = 0; v < nviews; ++v) {
        if (!pl[v]) return nullptr;
        need1 = std::max(need1, pl[v]->need1); need2 = std::max(need2, pl[v]->need2);
        tilt += pl[v]->tilt;
    }
    MultiPlan* mp = new (std::nothrow) MultiPlan();
    if (!mp) return nullptr;
    mp->keys = keys;
    mp->d = box_dims(need1, need2, tilt >= 0 ? 1 : -1, pxb);
    mp->n1 = pl[0]->n1; mp->n2 = pl[0]->n2;
    if (getenv("CAMCAL_DEBUG"))
        fprintf(stderr, "[camcal] views: common footprint %d x %d -> box %d x %d pitch %d (%d B)\n", need1, need2, mp->d.box1,
                mp->d.box2, mp->d.pitch_b, mp->d.box_bytes);
    if (!mp->d.box_bytes) { delete mp; return nullptr; }
    const size_t ntiles = (size_t)mp->n1 * mp->n2, sz2 = (size_t)keys[0].g.sz2;
    mp->h_hdr.resize(ntiles * nviews);
    mp->h_q2.resize(sz2 * nviews);
    for (int v = 0; v < nviews; ++v) {
        fill_headers(pl[v], mp->d, mp->h_hdr.data() + (size_t)v * ntiles);
        memcpy(mp->h_q2.data() + (size_t)v * sz2, pl[v]->q2.data(), sz2 * sizeof(double));
    }
    return mp;
}

// find or build the plan of a group of views; nullptr: not stageable (or out of memory) -- the caller falls
// back to one launch per view
static MultiPlan* multi_get(cc_ctx* ctx, const ChainD* chs, const double* ratios, const RectGeom* gs, int nviews,
                            int tw, int tl, int pxb, cudaStream_t st) {
    std::vector<PlanKey> keys((size_t)nviews);
    for (int v = 0; v < nviews; ++v) keys[v] = plan_key(chs[v], ratios[v], gs[v], tw, tl, pxb);
    if (MultiPlan* mp = multi_find(ctx, keys)) return mp;
    // footprints per view: the cached RectPlans, the missing ones built on host threads and cached without their
    // device tables (the group uploads its own).  Assembled before inserting: inserting may evict an earlier plan.
    std::vector<RectPlan*> pl((size_t)nviews, nullptr);
    for (int v = 0; v < nviews; ++v) pl[v] = plan_find(ctx, keys[v]);
    const std::vector<int> missing = plans_missing(keys, pl);
    plans_build(keys, pl, missing);
    MultiPlan* mp = multi_assemble(keys, pl, pxb);
    for (int v : missing) if (pl[v]) plan_insert(ctx, pl[v]);
    if (!mp) return nullptr;
    const size_t hb = mp->h_hdr.size() * sizeof(TileHdr), qb = mp->h_q2.size() * sizeof(double);
    if (cudaMalloc(&mp->d_hdr, hb) != cudaSuccess || cudaMalloc(&mp->d_q2, qb) != cudaSuccess ||
        cudaMemcpyAsync(mp->d_hdr, mp->h_hdr.data(), hb, cudaMemcpyHostToDevice, st) != cudaSuccess ||
        cudaMemcpyAsync(mp->d_q2, mp->h_q2.data(), qb, cudaMemcpyHostToDevice, st) != cudaSuccess) {
        cudaGetLastError();
        multi_free(mp);
        return nullptr;
    }
    mp->hdr_cap = hb; mp->q2_cap = qb;
    cudaStreamSynchronize(st);         // the host vectors go away; later calls may come on other streams
    std::vector<TileHdr>().swap(mp->h_hdr);
    std::vector<double>().swap(mp->h_q2);
    const int slot = ctx->multi_plan_next++ % cc_ctx::NMULTI;
    if (ctx->multi_plans[slot]) {
        cudaDeviceSynchronize();       // an evicted plan may still be read by a running kernel
        multi_free(ctx->multi_plans[slot]);
    }
    ctx->multi_plans[slot] = mp;
    return mp;
}

// a launch on `st` reads mp's tables: readers on another stream come first (the fence then covers them all)
static void multi_read_begin(MultiPlan* mp, cudaStream_t st) {
    if (mp->ready) cudaStreamWaitEvent(st, mp->ready, 0);
    if (mp->fenced && mp->fence_stream != st) cudaStreamWaitEvent(st, mp->fence, 0);
}
static void multi_read_end(MultiPlan* mp, cudaStream_t st) {
    if (!mp->fence && cudaEventCreateWithFlags(&mp->fence, cudaEventDisableTiming) != cudaSuccess) { mp->fence = nullptr; return; }
    cudaEventRecord(mp->fence, st);
    mp->fenced = true;
    mp->fence_stream = st;
}

struct ViewsLaunch {
    CUtensorMap tmap;
    TileCfg cfg;
    ViewTable vt;
    RectGeom g;
    MultiPlan* mp;
};

// frame groups of fg frames (inside views of fpv frames) that meet frames [w0, w0 + wn) of a group; *g0: the first
static long long window_groups(int fpv, int fg, int w0, int wn, uint32_t* g0) {
    const int gpv = (fpv + fg - 1) / fg;
    const int v_lo = w0 / fpv, v_hi = (w0 + wn - 1) / fpv;
    const long long lo = (long long)v_lo * gpv + (w0 - v_lo * fpv) / fg;
    const long long hi = (long long)v_hi * gpv + (w0 + wn - 1 - v_hi * fpv) / fg;
    *g0 = (uint32_t)lo;
    return hi - lo + 1;
}

// tensor map, unit configuration and view table of one launch of a group's plan (views [v0, v0 + nv) of the call)
// over frames [w0, w0 + wn) of the group; src: the window's first frame.  *ok = false: the launch does not apply
template <typename PX>
static int views_window(cc_ctx* ctx, MultiPlan* mp, const RectCall<PX>& c, int v0, int nv, const PX* src, int w0,
                        int wn, ViewsLaunch* L, bool* ok) {
    using F = RectFmt<PX>;
    const RectFrames& fr = c.fr;
    *ok = false;
    TileCfg& cfg = L->cfg;
    memset(&cfg, 0, sizeof(cfg));
    if (!stage_box(ctx, src, F::pxb, fr.sz1, fr.sz2, fr.pitch, fr.frame_stride, wn, mp->d, &L->tmap, &cfg)) return CC_OK;
    cfg.strips = (fr.sz1 + kT - 1) / kT;
    cfg.ntiles2 = (fr.sz2 + F::tl - 1) / F::tl;
    cfg.tiles = cfg.strips * cfg.ntiles2;
    // frames per group: as unit_cfg (keep ~8 units per resident CTA slot), within a view
    const long long want = (long long)ctx->sm_count * 6 * 8;
    int fg = std::min(!(c.flags & CC_COORD_F32) ? F::fg_exact : F::fg_fast, fr.fpv);
    uint32_t g0 = 0;
    while (fg > 1 && (long long)cfg.tiles * window_groups(fr.fpv, fg, w0, wn, &g0) < want) fg = (fg + 1) / 2;
    const long long units = (long long)cfg.tiles * window_groups(fr.fpv, fg, w0, wn, &g0);
    cfg.fg = fg;
    cfg.fpv = fr.fpv;
    cfg.gpv = (fr.fpv + fg - 1) / fg;
    cfg.w0 = w0;
    cfg.g0 = g0;
    CC_REQUIRE(units < (1ll << 31), "too many tiles in one call: split the batch");
    cfg.units = (uint32_t)units;
    for (int v = 0; v < nv; ++v) {
        const RectGeom gv = make_geom(c.views.axs_mins + 2 * (v0 + v), fr.sz1, fr.sz2, fr.pitch, fr.frame_stride, wn);
        L->vt.v[v].pe = make_exact(c.views.chs[v0 + v], c.views.ratios[v0 + v]);
        L->vt.v[v].pf = make_fast(c.views.chs[v0 + v], c.views.ratios[v0 + v], gv);
        L->vt.v[v].g = gv;
    }
    for (int v = nv; v < kMaxViews; ++v) L->vt.v[v] = L->vt.v[0];
    L->g = L->vt.v[0].g;
    L->mp = mp;
    *ok = true;
    return CC_OK;
}

// the staged views kernel on a prepared launch
template <typename PX>
static int views_run(cc_ctx* ctx, ViewsLaunch* L, const RectCall<PX>& c, const PX* src, PX* dst, cudaStream_t st) {
    using F = RectFmt<PX>;
    const bool exact = !(c.flags & CC_COORD_F32);
    int nf = 1;
    const size_t smem = F::ring(L->cfg, true, &nf);
    const auto k = F::views(exact);
    uint32_t gsz = 0;
    int rc = persistent_grid(ctx, F::views_slot + !exact, k, smem, L->cfg, L->mp, exact, &gsz);
    RectSched* sched = nullptr;
    if (!rc) rc = sched_acquire(ctx, st, &sched);
    if (rc) return rc;
    multi_read_begin(L->mp, st);
    F::launch(k, gsz, kConsumerThreads + 32, smem, st, c, L->tmap, L->vt, L->g, L->cfg, L->mp->d_hdr, L->mp->d_q2, sched,
              src, dst);
    multi_read_end(L->mp, st);
    sched_release(ctx, st);
    ctx->launches++;
    CC_CUDA(cudaGetLastError());
    return CC_OK;
}

// Views [v0, v0 + nv) of a device call in one staged launch; src / dst: the group's first frame.  *ok = false: the
// group cannot be staged (the caller runs one launch per view).
template <typename PX>
int launch_rectify_group(cc_ctx* ctx, const RectCall<PX>& c, int v0, int nv, const PX* src, PX* dst, cudaStream_t st,
                         bool* ok) {
    using F = RectFmt<PX>;
    const RectFrames& fr = c.fr;
    const int nframes = nv * fr.fpv;
    *ok = false;
    if ((c.flags & CC_GATHER_DIRECT) || !F::dst_ok(dst, fr, nframes) || nv < 1 || nv > kMaxViews || fr.fpv < 1 ||
        !tma_aligned(src, F::pxb, fr.pitch, fr.frame_stride, nframes) || !encoder(ctx))
        return CC_OK;
    std::vector<RectGeom> gs((size_t)nv);
    for (int v = 0; v < nv; ++v)
        gs[v] = make_geom(c.views.axs_mins + 2 * (v0 + v), fr.sz1, fr.sz2, fr.pitch, fr.frame_stride, nframes);
    MultiPlan* mp = multi_get(ctx, c.views.chs + v0, c.views.ratios + v0, gs.data(), nv, kT, F::tl, F::pxb, st);
    if (!mp) {
        if (getenv("CAMCAL_DEBUG")) fprintf(stderr, "[camcal] views: group of %d not stageable (pxb %d)\n", nv, F::pxb);
        return CC_OK;
    }
    ViewsLaunch L;                     // 15 KB: the view table goes to the kernel by value
    int rc = views_window(ctx, mp, c, v0, nv, src, 0, nframes, &L, ok);
    if (rc || !*ok) return rc;
    return views_run(ctx, &L, c, src, dst, st);
}

// --------------------------------------------------------------------------------------
// Frames of many views from host memory (cc_rectify_views_*_host): the chunk pipeline of abi.cu moves the
// frames; this session owns the group plans of the call.  Each group of up to 64 views gets its plan once per
// call.  A missing plan is built on host threads while the device streams the previous group's chunks, goes up
// on the context's upload stream, and the slot streams wait for its `ready` event.  Nothing here synchronises
// the device: an evicted plan's buffers are reused (or retired) after its fence.
// --------------------------------------------------------------------------------------
struct RectViewsHost {
    cc_ctx* ctx;
    RectViews views;
    RectFrames fr;                         // the layout of the slot buffers: frames pitch * sz2 apart
    int ngroups, pxb, tl;
    bool stage;                            // the layout can be staged at all
    std::vector<MultiPlan*> mp;            // per group: its plan (nullptr: per-view launches)
    std::vector<char> state;               // per group: 0 nothing yet, 1 being built, 2 ready
    std::vector<char> used;                // per group: a launch read its plan since the last fence
    // the group being built off this thread: keys, copies of the cached footprints, result
    int job_group;
    std::thread job;
    std::vector<PlanKey> job_keys;
    std::vector<RectPlan> job_found;
    MultiPlan* job_out;
    std::vector<MultiPlan*> installed;     // plans this call uploaded (their host tables go at the end)
    std::vector<std::vector<TileHdr>> held_hdr;   // host tables of plans evicted during the call (uploads in flight)
    std::vector<std::vector<double>> held_q2;
};

static std::vector<PlanKey> group_keys(const RectViewsHost* h, int gi) {
    const int v0 = gi * kMaxViews, nv = std::min(kMaxViews, h->views.n - v0);
    std::vector<PlanKey> keys((size_t)nv);
    for (int v = 0; v < nv; ++v) {
        const RectGeom g = make_geom(h->views.axs_mins + 2 * (v0 + v), h->fr.sz1, h->fr.sz2, h->fr.pitch, 0, 0);
        keys[v] = plan_key(h->views.chs[v0 + v], h->views.ratios[v0 + v], g, kT, h->tl, h->pxb);
    }
    return keys;
}

// the host half of group gi's plan (footprints, box, tables) on its own thread; a cached group plan is taken as is
static void vh_start(RectViewsHost* h, int gi) {
    if (gi >= h->ngroups || h->state[gi] || !h->stage) return;
    std::vector<PlanKey> keys = group_keys(h, gi);
    if (MultiPlan* mp = multi_find(h->ctx, keys)) { h->mp[gi] = mp; h->state[gi] = 2; return; }
    // copies of the cached footprints: the context's plan cache may change while the job runs
    h->job_found.clear();
    h->job_found.reserve(keys.size());
    std::vector<int> found_at(keys.size(), -1);
    for (size_t v = 0; v < keys.size(); ++v)
        if (RectPlan* p = plan_find(h->ctx, keys[v])) { found_at[v] = (int)h->job_found.size(); h->job_found.push_back(*p); }
    h->job_keys.swap(keys);
    h->job_out = nullptr;
    h->job_group = gi;
    h->state[gi] = 1;
    auto work = [h, found_at]() {
        const std::vector<PlanKey>& keys = h->job_keys;
        std::vector<RectPlan*> pl(keys.size(), nullptr);
        for (size_t v = 0; v < keys.size(); ++v) if (found_at[v] >= 0) pl[v] = &h->job_found[found_at[v]];
        const std::vector<int> missing = plans_missing(keys, pl);
        plans_build(keys, pl, missing);
        h->job_out = multi_assemble(keys, pl, h->pxb);
        for (int v : missing) plan_free(pl[v]);        // the footprints live on in the group plan only
    };
    try { h->job = std::thread(work); }
    catch (...) { work(); }                             // no thread to be had: built here
}

// wait for the job of group gi; the tables go up on the upload stream into a free or evicted slot (never the
// plan of group gi - 1, whose chunks may still be enqueued)
static int vh_install(RectViewsHost* h, int gi) {
    cc_ctx* ctx = h->ctx;
    if (h->job.joinable()) h->job.join();
    h->job_found.clear();
    MultiPlan* mp = h->job_out;
    h->job_out = nullptr;
    h->state[gi] = 2;
    if (!mp) {
        if (getenv("CAMCAL_DEBUG")) fprintf(stderr, "[camcal] views: group of %zu not stageable (pxb %d)\n", h->job_keys.size(), h->pxb);
        return CC_OK;
    }
    const MultiPlan* keep = gi > 0 ? h->mp[gi - 1] : nullptr;
    int slot = -1;
    for (int i = 0; i < cc_ctx::NMULTI && slot < 0; ++i) {
        const int s = (ctx->multi_plan_next + i) % cc_ctx::NMULTI;
        if (!ctx->multi_plans[s] || ctx->multi_plans[s] != keep) slot = s;
    }
    ctx->multi_plan_next = slot + 1;
    const size_t hb = mp->h_hdr.size() * sizeof(TileHdr), qb = mp->h_q2.size() * sizeof(double);
    if (MultiPlan* old = static_cast<MultiPlan*>(ctx->multi_plans[slot])) {
        ctx->multi_plans[slot] = nullptr;
        h->installed.erase(std::remove(h->installed.begin(), h->installed.end(), old), h->installed.end());
        h->held_hdr.emplace_back(); h->held_hdr.back().swap(old->h_hdr);
        h->held_q2.emplace_back(); h->held_q2.back().swap(old->h_q2);
        if (old->fenced) CC_CUDA(cudaStreamWaitEvent(ctx->rect_upload, old->fence, 0));
        if (old->hdr_cap >= hb && old->q2_cap >= qb) {  // same frame size: the upload overwrites it after its readers
            mp->d_hdr = old->d_hdr; mp->d_q2 = old->d_q2; mp->hdr_cap = old->hdr_cap; mp->q2_cap = old->q2_cap;
            old->d_hdr = nullptr; old->d_q2 = nullptr;
            multi_free(old);
        } else {                                        // freed at the start of the next host call
            old->next_retired = static_cast<MultiPlan*>(ctx->multi_retired);
            ctx->multi_retired = old;
        }
    }
    if (!mp->d_hdr) {                                   // room for a full group: later groups of this size reuse it
        const size_t hcap = std::max(hb, (size_t)mp->n1 * mp->n2 * kMaxViews * sizeof(TileHdr));
        const size_t qcap = std::max(qb, (size_t)h->fr.sz2 * kMaxViews * sizeof(double));
        if (cudaMalloc(&mp->d_hdr, hcap) != cudaSuccess || cudaMalloc(&mp->d_q2, qcap) != cudaSuccess) {
            cudaGetLastError();
            multi_free(mp);
            return set_error(CC_ERR_CUDA, "out of device memory for the tile plans of a group of views");
        }
        mp->hdr_cap = hcap; mp->q2_cap = qcap;
    }
    if (cudaEventCreateWithFlags(&mp->ready, cudaEventDisableTiming) != cudaSuccess) {
        mp->ready = nullptr;
        multi_free(mp);
        cudaGetLastError();
        return set_error(CC_ERR_CUDA, "cannot create the upload event of a group plan");
    }
    ctx->multi_plans[slot] = mp;
    h->installed.push_back(mp);
    h->mp[gi] = mp;
    CC_CUDA(cudaMemcpyAsync(mp->d_hdr, mp->h_hdr.data(), hb, cudaMemcpyHostToDevice, ctx->rect_upload));
    CC_CUDA(cudaMemcpyAsync(mp->d_q2, mp->h_q2.data(), qb, cudaMemcpyHostToDevice, ctx->rect_upload));
    CC_CUDA(cudaEventRecord(mp->ready, ctx->rect_upload));
    return CC_OK;
}

// dc: the call in the layout of the slot buffers (frames pitch * sz2 apart)
template <typename PX>
int rect_vh_begin(cc_ctx* ctx, const RectCall<PX>& dc, RectViewsHost** out) {
    using F = RectFmt<PX>;
    *out = nullptr;
    multi_free_retired(ctx);
    if (!ctx->rect_upload) CC_CUDA(cudaStreamCreateWithFlags(&ctx->rect_upload, cudaStreamNonBlocking));
    if (!ctx->rect_join) CC_CUDA(cudaStreamCreateWithFlags(&ctx->rect_join, cudaStreamNonBlocking));
    for (int k = 0; k < cc_ctx::NSLOT; ++k)
        if (!ctx->rect_join_event[k]) CC_CUDA(cudaEventCreateWithFlags(&ctx->rect_join_event[k], cudaEventDisableTiming));
    RectViewsHost* h = new (std::nothrow) RectViewsHost();
    if (!h) return set_error(CC_ERR_NOMEM, "out of host memory");
    h->ctx = ctx; h->views = dc.views; h->fr = dc.fr;
    h->ngroups = (dc.views.n + kMaxViews - 1) / kMaxViews;
    h->pxb = F::pxb; h->tl = F::tl;
    // staged iff the device frames (pitch * sz2 elements, buffers 256-byte aligned) can be TMA-addressed
    h->stage = !(dc.flags & CC_GATHER_DIRECT) && ((dc.fr.pitch * F::pxb) & 15u) == 0 && encoder(ctx) != nullptr;
    h->mp.assign((size_t)h->ngroups, nullptr);
    h->state.assign((size_t)h->ngroups, 0);
    h->used.assign((size_t)h->ngroups, 0);
    h->job_group = -1;
    h->job_out = nullptr;
    *out = h;
    vh_start(h, 0);
    return CC_OK;
}

int rect_vh_prepare(RectViewsHost* h, int gi) {
    int rc = CC_OK;
    if (h->stage && h->state[gi] != 2) {
        if (h->state[gi] == 0) vh_start(h, gi);
        if (h->state[gi] == 1 && (rc = vh_install(h, gi))) return rc;
    }
    vh_start(h, gi + 1);                               // the next group's plan is built while this one streams
    return CC_OK;
}

// frames [w0, w0 + wn) of group gi, src / dst: the window's first frame in a slot, on st; *ok = false: the group has
// no plan (the caller runs its single-view launches)
template <typename PX>
int rect_vh_launch(RectViewsHost* h, const RectCall<PX>& dc, int gi, int w0, int wn, const PX* src, PX* dst,
                   cudaStream_t st, bool* ok) {
    *ok = false;
    if (!h->mp[gi]) return CC_OK;
    const int v0 = gi * kMaxViews, nv = std::min(kMaxViews, h->views.n - v0);
    ViewsLaunch L;
    int rc = views_window(h->ctx, h->mp[gi], dc, v0, nv, src, w0, wn, &L, ok);
    if (rc || !*ok) return rc;
    h->used[gi] = 1;
    return views_run(h->ctx, &L, dc, src, dst, st);
}

// no chunk of this call reads group gi's plan after the ones enqueued so far: its fence joins the slot streams
void rect_vh_retire(RectViewsHost* h, int gi) {
    cc_ctx* ctx = h->ctx;
    MultiPlan* mp = gi < h->ngroups ? h->mp[gi] : nullptr;
    if (!mp || !h->used[gi]) return;
    h->used[gi] = 0;
    for (int k = 0; k < cc_ctx::NSLOT; ++k) {
        if (!ctx->pipe_stream[k]) continue;
        cudaEventRecord(ctx->rect_join_event[k], ctx->pipe_stream[k]);
        cudaStreamWaitEvent(ctx->rect_join, ctx->rect_join_event[k], 0);
    }
    multi_read_end(mp, ctx->rect_join);
}

// after the last chunk (or an error): every plan fenced, the uploads complete, the host tables released
int rect_vh_end(RectViewsHost* h) {
    if (!h) return CC_OK;
    cc_ctx* ctx = h->ctx;
    if (h->job.joinable()) h->job.join();
    if (h->job_out) multi_free(h->job_out);
    for (int gi = 0; gi < h->ngroups; ++gi) rect_vh_retire(h, gi);
    const cudaError_t e = cudaStreamSynchronize(ctx->rect_upload);
    for (MultiPlan* mp : h->installed) {
        std::vector<TileHdr>().swap(mp->h_hdr);
        std::vector<double>().swap(mp->h_q2);
        if (mp->ready) { cudaEventDestroy(mp->ready); mp->ready = nullptr; }
    }
    delete h;
    return e == cudaSuccess ? CC_OK : cuda_fail(e, "plan upload");
}

int rectify_views_per_launch() { return kMaxViews; }

// the map alone of one view: FP64 with the exact kernels' arithmetic, FP32 with the fast ones'
template <typename T>
int launch_rectify_map(cc_ctx* ctx, const ChainD& chd, double ratio, const int64_t axs_min[2], T* map_row, T* map_col,
                       int sz1, int sz2, size_t pitch, cudaStream_t st) {
    const RectGeom g = make_geom(axs_min, sz1, sz2, pitch, pitch * (size_t)sz2, 1);
    const dim3 grid((sz1 + kT - 1) / kT, (sz2 + kT - 1) / kT);
    if constexpr (std::is_same_v<T, double>)
        rectify_map_kernel<<<grid, kConsumerThreads, 0, st>>>(make_exact(chd, ratio), g, map_row, map_col);
    else
        rectify_map_f32_kernel<<<grid, kConsumerThreads, 0, st>>>(make_fast(chd, ratio, g), g, map_row, map_col);
    ctx->launches++;
    CC_CUDA(cudaGetLastError());
    return CC_OK;
}

template int launch_rectify<float>(cc_ctx*, const RectCall<float>&, int, int, const float*, float*, cudaStream_t);
template int launch_rectify<uint8_t>(cc_ctx*, const RectCall<uint8_t>&, int, int, const uint8_t*, uint8_t*, cudaStream_t);
template int launch_rectify_group<float>(cc_ctx*, const RectCall<float>&, int, int, const float*, float*, cudaStream_t,
                                         bool*);
template int launch_rectify_group<uint8_t>(cc_ctx*, const RectCall<uint8_t>&, int, int, const uint8_t*, uint8_t*,
                                           cudaStream_t, bool*);
template int rect_vh_begin<float>(cc_ctx*, const RectCall<float>&, RectViewsHost**);
template int rect_vh_begin<uint8_t>(cc_ctx*, const RectCall<uint8_t>&, RectViewsHost**);
template int rect_vh_launch<float>(RectViewsHost*, const RectCall<float>&, int, int, int, const float*, float*,
                                   cudaStream_t, bool*);
template int rect_vh_launch<uint8_t>(RectViewsHost*, const RectCall<uint8_t>&, int, int, int, const uint8_t*, uint8_t*,
                                     cudaStream_t, bool*);
template int launch_rectify_map<double>(cc_ctx*, const ChainD&, double, const int64_t[2], double*, double*, int, int,
                                        size_t, cudaStream_t);
template int launch_rectify_map<float>(cc_ctx*, const ChainD&, double, const int64_t[2], float*, float*, int, int,
                                       size_t, cudaStream_t);

}  // namespace cc
