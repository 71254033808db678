// rectify_u8c3.cuh -- 8-bit RGB (RGB{N0f8}, 3 interleaved bytes) rectification kernels
// (included by rectify.cu).  Same skeleton as rectify_f32c1.cuh: persistent CTAs, ticket
// scheduler, host-built tile plan, one TMA box per tile, raw-bit addressing.
//
// Per pixel the two taps of one source line are 6 contiguous bytes at byte offset 3*i: they are
// fetched as three aligned 32-bit words and funnelled with PRMT.  Bytes become floats without a
// conversion instruction (an isolated byte IS the denormal float b * 2^-149; a packed FMUL2 by
// 2^100 makes it normal and exact), the blend runs on PAIRS of lines in FFMA2/FADD2 in that scaled
// domain, and the final FFMA2 by 2^49 onto a rounding magic undoes the scale.
//
// Exact variant (FP64 coordinates): indices and weights come from the FP64 chain, bit for bit
// like the oracle.  The blend of 8-bit taps is then done in FP32 with a CERTIFIED rounding:
//   |v32 - v64| <= 5.3e-5 LSB  (three roundings at ulp(255)/2 = 7.6e-6 each, accumulated:
//   3.8e-5, plus the weights' FP32 representation error 2 * 255 * 2^-25 = 1.5e-5),
// so whenever v32 is farther than 6.5e-5 from a rounding boundary, rint(v32) == rint(v64).
// The pixels that are closer (1.3e-4 of the values; exact .5 ties included) are re-blended in
// FP64 with the oracle's operation order.  The output is therefore bit-identical to the FP64
// blend while ~99.9 % of the pixels never touch the FP64 pipe after the coordinate chain.
//
// Stores: the 32 pixels of a warp's line are 96 contiguous bytes; two shuffles and one PRMT per
// line turn the per-lane 0x00BBGGRR into 24 aligned words (full 32-byte sectors).
#pragma once

namespace cc {

struct Taps6 { uint32_t lo, hi; };   // bytes [o, o+4) and [o+4, o+8) of a byte stream

// PRMT with a selector register whose nibbles are all < 8 (sel6): __byte_perm() would first mask
// the selector with 0x7777 (one LOP3 per pixel and frame in the hot loop)
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
    return d;
}

template <typename LD>
__device__ __forceinline__ Taps6 load6(const uint32_t* words, unsigned o, unsigned sel, LD ld) {
    const uint32_t* w = words + (o >> 2);
    const uint32_t w0 = ld(w), w1 = ld(w + 1), w2 = ld(w + 2);
    Taps6 t;
    t.lo = prmt(w0, w1, sel);
    t.hi = prmt(w1, w2, sel);
    return t;
}
__device__ __forceinline__ unsigned sel6(unsigned o) { return 0x3210u + 0x1111u * (o & 3u); }

// Shared-memory loads as ordinary C++ loads (not volatile asm): the compiler is free to hoist the
// loads of the next pixels above the arithmetic and the stores of the current ones; the "memory"
// clobber of the mbarrier wait/arrive keeps them inside one stage's lifetime.
__device__ __forceinline__ uint32_t lds_u32(uint32_t addr) {
    return *reinterpret_cast<const uint32_t*>(__cvta_shared_to_generic(addr));
}
template <int OFF>
__device__ __forceinline__ uint32_t lds_u32_off(uint32_t addr) {
    return *reinterpret_cast<const uint32_t*>(__cvta_shared_to_generic(addr + OFF));
}
// six bytes out of the three words at word-aligned shared address wa
__device__ __forceinline__ Taps6 lds6w(uint32_t wa, unsigned sel) {
    const uint32_t w0 = lds_u32(wa), w1 = lds_u32_off<4>(wa), w2 = lds_u32_off<8>(wa);
    Taps6 t;
    t.lo = prmt(w0, w1, sel);
    t.hi = prmt(w1, w2, sel);
    return t;
}
// byte k of w as a float without a conversion instruction: 0x4B000000 | b  ==  2^23 + b
__device__ __forceinline__ float byte_f(uint32_t w, int k) {
    return __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7440u + (unsigned)k)) - 8388608.0f;
}
__device__ __forceinline__ double byte_d(uint32_t w, int k) { return (double)((w >> (8 * k)) & 0xffu); }

// t0 = source line i2, t1 = line i2+1;  t.lo = [a00.r a00.g a00.b a10.r], t.hi = [a10.g a10.b . .]
template <bool EXACT>
__device__ __forceinline__ uint32_t blend_rgb(const Taps6& t0, const Taps6& t1, double d1d, double d2d,
                                              float d1f, float d2f) {
    uint32_t r, g, b;
    if (EXACT) {
        r = (uint32_t)(int)rint(bilerp(byte_d(t0.lo, 0), byte_d(t0.lo, 3), byte_d(t1.lo, 0), byte_d(t1.lo, 3), d1d, d2d));
        g = (uint32_t)(int)rint(bilerp(byte_d(t0.lo, 1), byte_d(t0.hi, 0), byte_d(t1.lo, 1), byte_d(t1.hi, 0), d1d, d2d));
        b = (uint32_t)(int)rint(bilerp(byte_d(t0.lo, 2), byte_d(t0.hi, 1), byte_d(t1.lo, 2), byte_d(t1.hi, 1), d1d, d2d));
    } else {
        // round-to-nearest by magic add; weights in [0,1] keep the result inside [0,255]
        const float m = 12582912.0f;
        const float fr = bilerp_fast(byte_f(t0.lo, 0), byte_f(t0.lo, 3), byte_f(t1.lo, 0), byte_f(t1.lo, 3), d1f, d2f) + m;
        const float fg = bilerp_fast(byte_f(t0.lo, 1), byte_f(t0.hi, 0), byte_f(t1.lo, 1), byte_f(t1.hi, 0), d1f, d2f) + m;
        const float fb = bilerp_fast(byte_f(t0.lo, 2), byte_f(t0.hi, 1), byte_f(t1.lo, 2), byte_f(t1.hi, 1), d1f, d2f) + m;
        r = __float_as_uint(fr); g = __float_as_uint(fg); b = __float_as_uint(fb);
    }
    // low bytes of r, g, b -> 0x00BBGGRR
    return __byte_perm(__byte_perm(r, g, 0x0040), b, 0x0410);
}

constexpr float kTwo49 = 562949953421312.0f;           // 2^49
// distance of a blended value from the integer it rounds to, against the certification bound
constexpr float kCertThr = 0.5f - 6.5e-5f;

__device__ __forceinline__ void store_rgb(uint8_t* q, uint32_t rgb) {
    q[0] = (uint8_t)rgb; q[1] = (uint8_t)(rgb >> 8); q[2] = (uint8_t)(rgb >> 16);
}

// generic per-pixel path with every check and direct global taps
template <bool EXACT>
__device__ __forceinline__ uint32_t sample_direct_u8(const RectExact& pe, const RectFast& pf,
                                                     const RowTermD& rtd, const RowTermF& rtf,
                                                     const RectGeom& g, const uint8_t* __restrict__ sframe,
                                                     unsigned pitch3, unsigned frame_bytes, int b,
                                                     uint32_t fill) {
    int g1, g2;
    double d1d = 0, d2d = 0;
    float d1f = 0, d2f = 0;
    if (EXACT) {
        double row, col;
        rect_coord(pe, rtd, rect_q2(pe, g.axs1 + b), row, col);
        if (!(lin_ok(row, g.sz1) & lin_ok(col, g.sz2))) return fill;
        lin_floor(row, g1, d1d);
        lin_floor(col, g2, d2d);
        lin_fix_edge(g.sz1, g1, d1d);
        lin_fix_edge(g.sz2, g2, d2d);
        g1 -= 1; g2 -= 1;
    } else {
        float row, col;
        int t1, t2;
        rect_coord(pf, rtf, (float)(g.axs1 + b) - pf.c2, row, col);
        lin_floor_fast(row, t1, d1f);
        lin_floor_fast(col, t2, d2f);
        g1 = t1 - (kMagicBits + 1); g2 = t2 - (kMagicBits + 1);
        if (!(((unsigned)g1 <= (unsigned)(g.sz1 - 2)) & ((unsigned)g2 <= (unsigned)(g.sz2 - 2)))) return fill;
    }
    const unsigned off = (unsigned)g2 * pitch3 + (unsigned)g1 * 3u;
    Taps6 t0, t1;
    // word-granular gather from a 4-byte aligned base; the byte path for the last few taps of
    // the frame so nothing outside the caller's buffer is touched
    if (off + pitch3 + 12u <= frame_bytes) {
        const unsigned mis = (unsigned)(reinterpret_cast<uintptr_t>(sframe) & 3u);
        const uint32_t* gwords = reinterpret_cast<const uint32_t*>(sframe - mis);
        auto ld = [](const uint32_t* p) { return __ldg(p); };
        t0 = load6(gwords, off + mis, sel6(off + mis), ld);
        t1 = load6(gwords, off + pitch3 + mis, sel6(off + pitch3 + mis), ld);
    } else {
        const uint8_t* q = sframe + off;
        t0.lo = q[0] | (q[1] << 8) | (q[2] << 16) | ((uint32_t)q[3] << 24);
        t0.hi = q[4] | (q[5] << 8);
        q += pitch3;
        t1.lo = q[0] | (q[1] << 8) | (q[2] << 16) | ((uint32_t)q[3] << 24);
        t1.hi = q[4] | (q[5] << 8);
    }
    return blend_rgb<EXACT>(t0, t1, d1d, d2d, d1f, d2f);
}

// ---- direct kernel: no staging -------------------------------------------------------------
template <bool EXACT>
__global__ void __launch_bounds__(kConsumerThreads)
rectify_u8c3_direct_kernel(const __grid_constant__ RectExact pe, const __grid_constant__ RectFast pf,
                           const __grid_constant__ RectGeom g, const int lines_per_cta,
                           const uint8_t* __restrict__ src, uint8_t* __restrict__ dst, uchar3 fill3,
                           unsigned frame_bytes) {
    const int lane_id = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int a = blockIdx.x * kT + lane_id;
    if (a >= g.sz1) return;
    const int frame = blockIdx.z;
    const uint8_t* sframe = src + (long long)frame * g.frame_stride * 3;
    const unsigned pitch3 = (unsigned)g.pitch * 3u;
    const uint32_t fill = fill3.x | (fill3.y << 8) | (fill3.z << 16);
    RowTermD rtd;
    RowTermF rtf;
    if (EXACT) rtd = rect_row_term(pe, g.axs0 + a); else rtf = rect_row_term(pf, g.axs0 + a);
    const int b_begin = blockIdx.y * lines_per_cta;
    const int b_end = min(b_begin + lines_per_cta, g.sz2);
    uint8_t* o = dst + ((long long)frame * g.frame_stride + (long long)(b_begin + warp) * g.pitch + a) * 3;
    for (int b = b_begin + warp; b < b_end; b += kWarps, o += (long long)kWarps * pitch3)
        store_rgb(o, sample_direct_u8<EXACT>(pe, pf, rtd, rtf, g, sframe, pitch3, frame_bytes, b, fill));
}

// ---- staged kernel (persistent; scheduling and producer: rectify_ring.cuh) ------------------
// Same unit structure as rectify_f32c1_kernel: the map of a tile is built once per group of frames
// and kept in registers (8 pixels per lane); every frame then only gathers, blends and stores.
//
// Per pixel the map is the byte offset of tap (0,0) inside a stage and the FOUR bilinear weights
//   w00 = (1-d1)(1-d2), w10 = d1(1-d2), w01 = (1-d1)d2, w11 = d1 d2          (a_xy: x = first axis)
// as FP32 numbers scaled by 2^100, for pairs of lines (FFMA2 lanes).  A tap byte's bit pattern is
// the denormal float b * 2^-149, so one FMUL2 and three FFMA2 per channel and pair of pixels give
// v * 2^-49 with no unpacking arithmetic at all, and the FFMA2 by 2^49 onto 2^23 leaves rint(v) in
// the low byte (v >= 0: weights and taps are non-negative).
//
// Exact variant: weights are the FP64 products rounded to FP32.  Error of the FP32 blend against
// the FP64 blend of the oracle:
//   four roundings of partial sums < 256 (half an ulp = 7.63e-6 each)            3.05e-5
//   representation of the weights (relative 2^-24, sum of w_i b_i <= 255)        1.52e-5
// so |v32 - v64| <= 4.6e-5 LSB, and whenever v32 is farther than 6.5e-5 from a rounding boundary
// rint(v32) == rint(v64).  Every lane keeps max |v32 - rint(v32)| per pixel; once per frame the
// warp votes, and the pixels that are closer (1.3e-4 of the values; exact .5 ties included) are
// re-blended in FP64 in the oracle's operation order and patched with byte stores.  The output is
// bit-identical to the FP64 blend.
//
// Tap bytes (exact variant): source line i2 is three aligned words + PRMT (ALU pipe), line i2+1 six
// LDS.U8 (the load unit isolates the bytes).
//
// One frame per ring stage: two (as in rectify_f32c1.cuh) cost registers here and were measured
// slower (profiles/r2_rectify.md).
//
// Stores: the 32 pixels of a warp's line are 96 contiguous bytes = 24 words.  Lane L (L % 4 != 3)
// builds word L - L/4 from its own packed pixel and lane L+1's (one shuffle, one PRMT).
constexpr float kMagic23 = 8388608.0f;                 // 2^23: rint(v) in the low mantissa byte, low 24 bits of the pattern zero

template <int OFF>
__device__ __forceinline__ uint32_t lds_u8_off(uint32_t addr) {
    return *reinterpret_cast<const uint8_t*>(__cvta_shared_to_generic(addr + OFF));
}

// predicated streaming store (no branch around it)
__device__ __forceinline__ void stcs_if(bool p, uint32_t* q, uint32_t v) {
    asm volatile("{ .reg .pred p; setp.ne.u32 p, %0, 0; @p st.global.cs.u32 [%1], %2; }" :: "r"((uint32_t)p), "l"(q), "r"(v));
}

// the 12 tap bytes of one pixel as denormal-float bit patterns: [c] a00, [3+c] a10, [6+c] a01, [9+c] a11
struct TapF { uint32_t m[12]; };

// A0: shared address of tap (0,0) of source line i2 rounded down to a word, `sel` funnelling its bytes;
// A1b: byte address of tap (0,0) of line i2+1
__device__ __forceinline__ TapF load_taps(uint32_t A0, unsigned sel, uint32_t A1b) {
    TapF t;
    const Taps6 r0 = lds6w(A0, sel);
    t.m[0] = __byte_perm(r0.lo, 0u, 0x4440); t.m[1] = __byte_perm(r0.lo, 0u, 0x4441); t.m[2] = __byte_perm(r0.lo, 0u, 0x4442);
    t.m[3] = __byte_perm(r0.lo, 0u, 0x4443); t.m[4] = __byte_perm(r0.hi, 0u, 0x4440); t.m[5] = __byte_perm(r0.hi, 0u, 0x4441);
    t.m[6] = lds_u8_off<0>(A1b); t.m[7] = lds_u8_off<1>(A1b); t.m[8] = lds_u8_off<2>(A1b);
    t.m[9] = lds_u8_off<3>(A1b); t.m[10] = lds_u8_off<4>(A1b); t.m[11] = lds_u8_off<5>(A1b);
    return t;
}
__device__ __forceinline__ float2 tap2(const TapF& p, const TapF& q, int k) {
    return make_float2(__uint_as_float(p.m[k]), __uint_as_float(q.m[k]));
}

// one channel of two pixels: scaled blend, rounding, and the distance from the rounded value
__device__ __forceinline__ float2 blend_ch2(const TapF& p, const TapF& q, int c, float2 w00, float2 w10,
                                            float2 w01, float2 w11, float2& dist) {
    float2 acc = mul2(w00, tap2(p, q, c));
    acc = fma2(w10, tap2(p, q, 3 + c), acc);
    acc = fma2(w01, tap2(p, q, 6 + c), acc);
    acc = fma2(w11, tap2(p, q, 9 + c), acc);
    const float2 f = fma2(acc, bc2(kTwo49), bc2(kMagic23));
    dist = fma2(acc, bc2(-kTwo49), add2(f, bc2(-kMagic23)));       // rint(v) - v, exact
    return f;
}
__device__ __forceinline__ uint32_t pack_rgb(float fr, float fg, float fb) {
    // patterns are 0x4B000000 + value: the multiples of 2^8 and 2^16 of 0x4B000000 vanish mod 2^32
    return __float_as_uint(fr) + (__float_as_uint(fg) << 8) + (__float_as_uint(fb) << 16);
}
__device__ __forceinline__ float max_abs3(float a, float b, float c) { return fmaxf(fmaxf(fabsf(a), fabsf(b)), fabsf(c)); }

// two pixels (lines e, e+1 of a lane): packed 0x..BBGGRR each, and max |v - rint(v)| per pixel
__device__ __forceinline__ void blend_px2(const TapF& p, const TapF& q, float2 w00, float2 w10, float2 w01,
                                          float2 w11, uint32_t& rgb_p, uint32_t& rgb_q, float2& dmax) {
    float2 dr, dg, db;
    const float2 fr = blend_ch2(p, q, 0, w00, w10, w01, w11, dr);
    const float2 fg = blend_ch2(p, q, 1, w00, w10, w01, w11, dg);
    const float2 fb = blend_ch2(p, q, 2, w00, w10, w01, w11, db);
    rgb_p = pack_rgb(fr.x, fg.x, fb.x);
    rgb_q = pack_rgb(fr.y, fg.y, fb.y);
    dmax = make_float2(max_abs3(dr.x, dg.x, db.x), max_abs3(dr.y, dg.y, db.y));
}

// ---- FP32-coordinate (fast) variant: integer blend on the raw tap bytes -----------------------
// IDP.2A multiplies two bytes of one register by two 16-bit halves of another and accumulates in
// 32 bits.  The two source lines of a pixel have the same byte phase (the staged pitch is a multiple
// of 4), so after the funnel PRMTs the bytes of a00 / a01 sit at the same position of two registers:
// three PRMTs interleave them into VERTICAL pairs
//   X0 = (R0 R0' G0 G0')   X1 = (B0 B0' R1 R1')   X2 = (G1 G1' B1 B1')      (' = line i2 + 1)
// and with W0 = (w00, w01), W1 = (w10, w11) as 16-bit fixed-point weights (sum 2^16) every channel
// is two IDP.2A -- no byte is ever isolated.  Per pixel: 6 LDS + 7 PRMT + 6 IDP.2A + 2 PRMT (pack)
// = 21 instructions against 28.5 of the FP32 formulation (9 loads, 8 PRMT, 7.5 FFMA2/FMUL2, 4 pack).
// Weight quantisation: 4 * 255 * 2^-17 = 0.008 LSB (the fast variant's contract is +-1 LSB).

__device__ __forceinline__ uint32_t blend_px_idp(const Taps6& u, const Taps6& v, uint32_t W0, uint32_t W1) {
    const uint32_t X0 = __byte_perm(u.lo, v.lo, 0x5140), X1 = __byte_perm(u.lo, v.lo, 0x7362);
    const uint32_t X2 = __byte_perm(u.hi, v.hi, 0x5140);
    const uint32_t r = __dp2a_hi(W1, X1, __dp2a_lo(W0, X0, 0x8000u));      // + 0.5: the byte is bits 16..23
    const uint32_t g = __dp2a_lo(W1, X2, __dp2a_hi(W0, X0, 0x8000u));
    const uint32_t b = __dp2a_hi(W1, X2, __dp2a_lo(W0, X1, 0x8000u));
    return __byte_perm(__byte_perm(r, g, 0x6262), b, 0x7610);              // 0x00BBGGRR
}
// (1-d1)(1-d2), d1(1-d2), (1-d1)d2, d1 d2 as 16-bit fixed point; the three products are rounded,
// w00 takes the rest so that the sum is 2^16 (clamped: 0 <= w00 <= 65535)
__device__ __forceinline__ void idp_weights(float d1, float d2, uint32_t& W0, uint32_t& W1) {
    const float m = 12582912.0f, e2 = 1.0f - d2;
    const uint32_t w10 = __float_as_uint(fmaf(d1 * e2, 65536.0f, m)) & 0x1ffffu;
    const uint32_t w01 = __float_as_uint(fmaf((1.0f - d1) * d2, 65536.0f, m)) & 0x1ffffu;
    const uint32_t w11 = __float_as_uint(fmaf(d1 * d2, 65536.0f, m)) & 0x1ffffu;
    const int w00 = 65536 - (int)(w10 + w01 + w11);
    W0 = (uint32_t)min(max(w00, 0), 65535) | (min(w01, 65535u) << 16);
    W1 = min(w10, 65535u) | (min(w11, 65535u) << 16);
}

// FP64 blend of one pixel in the oracle's operation order (taps re-read from the stage)
__device__ __noinline__ uint32_t reblend_exact_u8(const RectExact* pe, const RectGeom* g, int a, int b,
                                                  uint32_t A0, uint32_t A1) {
    const RowTermD rtd = rect_row_term(*pe, g->axs0 + a);
    double row, col, d1, d2;
    int i1, i2;
    rect_coord(*pe, rtd, rect_q2(*pe, g->axs1 + b), row, col);
    lin_floor(row, i1, d1);
    lin_floor(col, i2, d2);
    uint32_t t[12];
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        asm volatile("ld.shared.u8 %0, [%1];" : "=r"(t[k]) : "r"(A0 + k));
        asm volatile("ld.shared.u8 %0, [%1];" : "=r"(t[6 + k]) : "r"(A1 + k));
    }
    uint32_t out = 0;
#pragma unroll
    for (int c = 0; c < 3; ++c)
        out |= (uint32_t)(int)rint(bilerp((double)t[c], (double)t[3 + c], (double)t[6 + c], (double)t[9 + c], d1, d2)) << (8 * c);
    return out;
}

// the kernel body (the __global__ wrappers are below).  VIEWS: frames with different views in one launch
// (cc_rectify_u8c3_views) -- coordinate parameters and axes of the unit's view come from the view table in the
// kernel's parameter space (vt; index = TileHdr.view)
template <bool EXACT, bool VIEWS>
__device__ __forceinline__ void rectify_u8c3_body(const CUtensorMap& tmap, const RectExact& pe0, const RectFast& pf0,
                                                  const RectGeom& g, const TileCfg& cfg, const TileHdr* __restrict__ plan,
                                                  const double* __restrict__ q2tab, RectSched* __restrict__ sched,
                                                  const uint8_t* __restrict__ src, uint8_t* __restrict__ dst, uchar3 fill3,
                                                  unsigned frame_bytes, const ViewTable* vt) {
    constexpr int TL = kTLu;                      // lines per tile
    constexpr int LPW = TL / kWarps;              // lines per warp per tile = pixels per lane
    constexpr int NP = LPW / 2;                   // pairs of lines
    constexpr bool IDP = !EXACT;                  // fast variant: integer blend on vertical byte pairs
    static_assert(LPW % 2 == 0 && LPW <= 16, "pairs of lines; masks are 16 bits");
    extern __shared__ __align__(128) uint8_t stage_mem[];
    __shared__ SmemRing ring;
    const int lane_id = threadIdx.x & 31;
    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);   // warp-uniform for the compiler
    ring_init(&ring, cfg.stages);

    if (warp == kWarps) {                              // ---- producer warp
        producer_loop<EXACT, TL, 1, 1, VIEWS>(&tmap, g, cfg, plan, q2tab, sched, &ring, stage_mem, lane_id);
        return;
    }

    // ---- consumer warps
    const unsigned pitch3 = (unsigned)g.pitch * 3u;
    const uint32_t box_pitch_b = (uint32_t)cfg.pitch_b;       // bytes per box line (multiple of 128)
    const uint32_t stage0 = smem_u32(stage_mem);
    const uint32_t fill = fill3.x | (fill3.y << 8) | (fill3.z << 16);
    // store: lane L (L % 4 != 3) writes word L - L/4 of the line = own pixel's tail + next pixel's head
    const int lq = lane_id & 3;
    const unsigned wsel = lq == 0 ? 0x4210u : (lq == 1 ? 0x5421u : 0x6542u);
    const int widx = lane_id - (lane_id >> 2);

    // the map of the current unit
    uint32_t rel[LPW];                                 // tap (0,0) offset inside a stage, rounded down to a word
    uint32_t selv[LPW];                                // PRMT selector that funnels the 6 tap bytes out of 3 words
    uint32_t relb[LPW];                                // the unrounded byte offset
    float2 w00[NP], w10[NP], w01[NP], w11[NP];         // weights * 2^100, pairs of lines
    uint32_t m_staged = 0, m_fill = 0, m_skip = 0;
    bool all_staged = false;
    int a = 0, b0 = 0;
    long long off0 = 0;

    int s = 0;
    uint32_t phase = 0;
    int4 pos = make_int4(0, 0, 0, 0);
    int frames_left = 0, frame_z = 0;
    [[maybe_unused]] uint32_t view = 0;
    for (;;) {
        mbar_wait(&ring.full[s], phase);
        // the slot is read on a unit's first frame only; frame index and frames left are carried in
        // warp-uniform registers (declared uniform through a shuffle) -- no LDS + two dependent branches
        // in front of every frame
        if (frames_left == 0) {
            pos = ring.pos[s];
            if (pos.z < 0) break;
            frame_z = __shfl_sync(0xffffffffu, pos.z, 0);
            frames_left = __shfl_sync(0xffffffffu, pos.w, 0);
        } else {
            pos.w = 0;
        }
        if (VIEWS && pos.w) view = __shfl_sync(0xffffffffu, ring.hdr[s].view, 0);
        const RectExact& pe = VIEWS ? vt->v[view].pe : pe0;
        const RectFast& pf = VIEWS ? vt->v[view].pf : pf0;
        const RectGeom& gv = VIEWS ? vt->v[view].g : g;     // axs0 / axs1 of the view (everything else is the launch's)
        if (pos.w) {                                   // ---- first frame of a unit: build the map
            const TileHdr* h = &ring.hdr[s];
            const int a_w = pos.x * kT;
            a = a_w + lane_id;
            b0 = pos.y * TL + warp * LPW;
            off0 = ((long long)b0 * g.pitch + a_w) * 3;        // the warp's first output byte of line b0
            const int a_c = min(a, g.sz1 - 1);         // out-of-frame lanes shadow the last pixel
            const uint32_t R1 = h->R1, R2 = h->R2;
            const uint32_t rel0 = h->base_off;
            m_staged = m_fill = m_skip = 0;
            if ((!EXACT && !VIEWS) || a_w + kT > g.sz1 || b0 + LPW > g.sz2) {   // partial tile (warp-uniform test; measured: pays only in the exact kernel and with a map per frame)
#pragma unroll
                for (int e = 0; e < LPW; ++e)
                    if (a >= g.sz1 || b0 + e >= g.sz2) m_skip |= 1u << e;
            }
            if (EXACT) {
                const RowTermD rtd = rect_row_term(pe, gv.axs0 + a_c);
                const double Mk1 = h->Mk1, Mk2 = h->Mk2;
                const double* q2p = &ring.q2[s][warp * LPW];
                const double up = 1.2676506002282294e30;      // 2^100
#pragma unroll
                for (int e = 0; e < LPW; ++e) {
                    double row, col, d1, d2;
                    rect_coord_nobranch(pe, rtd, q2p[e], row, col);
                    uint32_t t1, t2, h1, h2;
                    floor_index<kFloorFrnd>(row, Mk1, t1, h1, d1);
                    floor_index<kFloorDaddRm>(col, Mk2, t2, h2, d2);
                    const bool st = (((h1 ^ 0x43300000u) | (h2 ^ 0x43300000u)) == 0u) & (t1 < R1) & (t2 < R2);
                    rel[e] = rel0 + t2 * box_pitch_b + t1 * 3u;
                    relb[e] = rel[e];
                    selv[e] = sel6(rel[e]); rel[e] &= ~3u;   // stages are 128-byte aligned: (address & 3) == (rel & 3)
                    const double e1 = 1.0 - d1, e2 = 1.0 - d2;
                    const float v00 = (float)((e1 * e2) * up), v10 = (float)((d1 * e2) * up);
                    const float v01 = (float)((e1 * d2) * up), v11 = (float)((d1 * d2) * up);
                    if (e & 1) { w00[e / 2].y = v00; w10[e / 2].y = v10; w01[e / 2].y = v01; w11[e / 2].y = v11; }
                    else       { w00[e / 2].x = v00; w10[e / 2].x = v10; w01[e / 2].x = v01; w11[e / 2].x = v11; }
                    if (st) m_staged |= 1u << e;
                    else if (!(lin_ok(row, g.sz1) & lin_ok(col, g.sz2))) m_fill |= 1u << e;   // rare: border tiles
                }
            } else {
                const RowTermF rtf = rect_row_term(pf, gv.axs0 + a_c);
                const float mk1 = h->mk1, mk2 = h->mk2;
                float2 ip;
                ip.x = (float)(gv.axs1 + b0) - pf.c2;
                ip.y = ip.x + 1.0f;
#pragma unroll
                for (int hh = 0; hh < NP; ++hh) {
                    float2 row, col, d1, d2;
                    rect_coord2(pf, rtf, ip, row, col);
                    ip = add2(ip, bc2(2.0f));
                    uint32_t t1[2], t2[2];
                    floor_bits_fast2(row, mk1, t1[0], t1[1], d1);
                    floor_bits_fast2(col, mk2, t2[0], t2[1], d2);
                    uint32_t a0, a1, c0, c1;           // W0 / W1 of the two pixels live in w00 / w10 (bit patterns)
                    idp_weights(d1.x, d2.x, a0, a1);
                    idp_weights(d1.y, d2.y, c0, c1);
                    w00[hh] = make_float2(__uint_as_float(a0), __uint_as_float(c0));
                    w10[hh] = make_float2(__uint_as_float(a1), __uint_as_float(c1));
                    const float rr[2] = {row.x, row.y}, cc_[2] = {col.x, col.y};
#pragma unroll
                    for (int j = 0; j < 2; ++j) {
                        const int e = 2 * hh + j;
                        const uint32_t l1 = t1[j] - (uint32_t)kMagicBits, l2 = t2[j] - (uint32_t)kMagicBits;
                        const bool st = (l1 < R1) & (l2 < R2);
                        rel[e] = rel0 + l2 * box_pitch_b + l1 * 3u;
                        relb[e] = rel[e];
                        selv[e] = sel6(rel[e]); rel[e] &= ~3u;
                        if (st) m_staged |= 1u << e;
                        if (!VIEWS) {
                            // (unconditional: four FSETPs cost less than a divergent branch here; measured)
                            const bool inframe = (rr[j] >= 1.0f) & (rr[j] < (float)g.sz1) & (cc_[j] >= 1.0f) & (cc_[j] < (float)g.sz2);
                            if (!inframe) m_fill |= 1u << e;
                        }
                    }
                }
                // VIEWS: the map is built per frame, so the fill class (nine instructions per pixel) is worked out
                // for the warps that need it only -- border tiles, 4 % -- from the same coordinates once more
                if (VIEWS && !__all_sync(0xffffffffu, m_staged == (1u << LPW) - 1u)) {
                    ip.x = (float)(gv.axs1 + b0) - pf.c2;
                    ip.y = ip.x + 1.0f;
#pragma unroll
                    for (int hh = 0; hh < LPW / 2; ++hh) {
                        float2 row, col;
                        rect_coord2(pf, rtf, ip, row, col);
                        ip = add2(ip, bc2(2.0f));
                        if (!((row.x >= 1.0f) & (row.x < (float)g.sz1) & (col.x >= 1.0f) & (col.x < (float)g.sz2))) m_fill |= 1u << (2 * hh);
                        if (!((row.y >= 1.0f) & (row.y < (float)g.sz1) & (col.y >= 1.0f) & (col.y < (float)g.sz2))) m_fill |= 1u << (2 * hh + 1);
                    }
                }
            }
            if (R1 == 0u || R2 == 0u) { m_staged = 0; m_fill = 0; }   // tile the plan marked unusable
            constexpr uint32_t kAll = (1u << LPW) - 1u;
            all_staged = __all_sync(0xffffffffu, (m_staged == kAll) & (m_skip == 0u));
        }

        // ---- every frame of the unit: gather, blend, store
        const uint8_t* sframe = src + (long long)frame_z * g.frame_stride * 3;
        // (a running output pointer, as in the f32c1 kernel, costs this one registers: ptxas goes from
        // 96 to 104 and the fast variant from 4 to 3 CTAs per SM -- measured 0.204 vs 0.194 ms on c3)
        uint8_t* oline = dst + (long long)frame_z * g.frame_stride * 3 + off0;
        const uint32_t sbase = stage0 + (uint32_t)s * (uint32_t)cfg.box_bytes;
        const uint32_t sbase1 = sbase + box_pitch_b;
        if (all_staged) {
            uint32_t* ow = reinterpret_cast<uint32_t*>(oline) + widx;
            [[maybe_unused]] float2 dm[NP];
#pragma unroll
            for (int hh = 0; hh < NP; ++hh) {
                const int e = 2 * hh;
#ifdef CAMCAL_CHECK_BOUNDS      // the chk build (Makefile): every tap byte of both lines inside the stage
                for (int j = 0; j < 2; ++j) {
                    const uint32_t o = sbase + rel[e + j];
                    if (o < sbase || o + box_pitch_b + 12u > sbase + (uint32_t)cfg.box_bytes + 4u || (o & 3u)) __trap();
                }
#endif
                uint32_t rgb_p, rgb_q;
                if (IDP) {
                    const Taps6 pu = lds6w(sbase + rel[e], selv[e]), pv = lds6w(sbase1 + rel[e], selv[e]);
                    const Taps6 qu = lds6w(sbase + rel[e + 1], selv[e + 1]), qv = lds6w(sbase1 + rel[e + 1], selv[e + 1]);
                    rgb_p = blend_px_idp(pu, pv, __float_as_uint(w00[hh].x), __float_as_uint(w10[hh].x));
                    rgb_q = blend_px_idp(qu, qv, __float_as_uint(w00[hh].y), __float_as_uint(w10[hh].y));
                } else {
                    const TapF tp = load_taps(sbase + rel[e], selv[e], sbase1 + relb[e]);
                    const TapF tq = load_taps(sbase + rel[e + 1], selv[e + 1], sbase1 + relb[e + 1]);
                    blend_px2(tp, tq, w00[hh], w10[hh], w01[hh], w11[hh], rgb_p, rgb_q, dm[hh]);
                }
                const uint32_t np_ = __shfl_down_sync(0xffffffffu, rgb_p, 1);
                const uint32_t nq_ = __shfl_down_sync(0xffffffffu, rgb_q, 1);
                const bool st_ok = lq != 3;
                stcs_if(st_ok, ow, __byte_perm(rgb_p, np_, wsel));
                stcs_if(st_ok, reinterpret_cast<uint32_t*>(reinterpret_cast<uint8_t*>(ow) + pitch3), __byte_perm(rgb_q, nq_, wsel));
                ow = reinterpret_cast<uint32_t*>(reinterpret_cast<uint8_t*>(ow) + 2 * pitch3);
            }
            if (EXACT) {
                float mx = 0.0f;
#pragma unroll
                for (int hh = 0; hh < NP; ++hh) mx = fmaxf(mx, fmaxf(dm[hh].x, dm[hh].y));
                if (__any_sync(0xffffffffu, mx > kCertThr)) {      // rare: certify by the FP64 blend, patch the bytes
                    __syncwarp();                                  // the word stores above are ordered before the patches
#pragma unroll
                    for (int hh = 0; hh < NP; ++hh) {
#pragma unroll
                        for (int j = 0; j < 2; ++j) {
                            const int e = 2 * hh + j;
                            if ((j ? dm[hh].y : dm[hh].x) > kCertThr) {
                                const uint32_t bo = rel[e] + (selv[e] & 3u);
                                store_rgb(oline + (long long)e * pitch3 + lane_id * 3,
                                          reblend_exact_u8(&pe, &gv, a, b0 + e, sbase + bo, sbase1 + bo));
                            }
                        }
                    }
                }
            }
        } else {
            // border tiles: staged and fill pixels unrolled over the map (static indices), byte stores;
            // then one rolled pass for the generic remainder (it needs no map entry).  A rolled loop that
            // selects the map entry through a compare chain costs ~100 instructions per pixel.
            uint8_t* o = oline + lane_id * 3;
#pragma unroll
            for (int e = 0; e < LPW; ++e, o += pitch3) {
                const uint32_t bit = 1u << e;
                if (m_skip & bit) continue;
                if (m_staged & bit) {
                    const uint32_t sel = selv[e];
                    if (IDP) {
                        store_rgb(o, blend_px_idp(lds6w(sbase + rel[e], sel), lds6w(sbase1 + rel[e], sel),
                                                  __float_as_uint((e & 1) ? w00[e / 2].y : w00[e / 2].x),
                                                  __float_as_uint((e & 1) ? w10[e / 2].y : w10[e / 2].x)));
                        continue;
                    }
                    const TapF t = load_taps(sbase + rel[e], sel, sbase1 + relb[e]);
                    const float f00 = (e & 1) ? w00[e / 2].y : w00[e / 2].x, f10 = (e & 1) ? w10[e / 2].y : w10[e / 2].x;
                    const float f01 = (e & 1) ? w01[e / 2].y : w01[e / 2].x, f11 = (e & 1) ? w11[e / 2].y : w11[e / 2].x;
                    uint32_t v, vq;
                    float2 dm1;
                    blend_px2(t, t, bc2(f00), bc2(f10), bc2(f01), bc2(f11), v, vq, dm1);
                    if (EXACT && dm1.x > kCertThr) {
                        const uint32_t bo = rel[e] + (sel & 3u);
                        v = reblend_exact_u8(&pe, &gv, a, b0 + e, sbase + bo, sbase1 + bo);
                    }
                    store_rgb(o, v);
                } else if (m_fill & bit) {
                    store_rgb(o, fill);
                }
            }
            const uint32_t m_gen = ~(m_staged | m_fill | m_skip) & ((1u << LPW) - 1u);
            if (m_gen) {
                RowTermD rtd;
                RowTermF rtf;
                if (EXACT) rtd = rect_row_term(pe, gv.axs0 + a); else rtf = rect_row_term(pf, gv.axs0 + a);
                uint8_t* og = oline + lane_id * 3;
#pragma unroll 1
                for (int e = 0; e < LPW; ++e, og += pitch3)
                    if ((m_gen >> e) & 1u)
                        store_rgb(og, sample_direct_u8<EXACT>(pe, pf, rtd, rtf, gv, sframe, pitch3, frame_bytes, b0 + e, fill));
            }
        }
        __syncwarp();
        if (elect_one()) mbar_arrive(&ring.empty[s]);
        frames_left = max(frames_left - 1, 0); ++frame_z;
        if (++s == cfg.stages) { s = 0; phase ^= 1; }
    }
}

template <bool EXACT>
__global__ void __launch_bounds__(kConsumerThreads + 32, EXACT ? kMinBlocksU8Exact : kMinBlocksU8)
rectify_u8c3_kernel(const __grid_constant__ CUtensorMap tmap, const __grid_constant__ RectExact pe,
                    const __grid_constant__ RectFast pf, const __grid_constant__ RectGeom g,
                    const __grid_constant__ TileCfg cfg, const TileHdr* __restrict__ plan,
                    const double* __restrict__ q2tab, RectSched* __restrict__ sched,
                    const uint8_t* __restrict__ src, uint8_t* __restrict__ dst, uchar3 fill3,
                    unsigned frame_bytes) {
    rectify_u8c3_body<EXACT, false>(tmap, pe, pf, g, cfg, plan, q2tab, sched, src, dst, fill3, frame_bytes, nullptr);
}
// frames with different views in one launch (cc_rectify_u8c3_views)
template <bool EXACT>
__global__ void __launch_bounds__(kConsumerThreads + 32, EXACT ? kMinBlocksU8Exact : 4)    // fast: 96 registers = 4 CTAs per SM, as the single-view kernel allocates
rectify_u8c3_views_kernel(const __grid_constant__ CUtensorMap tmap, const __grid_constant__ ViewTable vt,
                          const __grid_constant__ RectGeom g, const __grid_constant__ TileCfg cfg,
                          const TileHdr* __restrict__ plan, const double* __restrict__ q2tab,
                          RectSched* __restrict__ sched, const uint8_t* __restrict__ src, uint8_t* __restrict__ dst,
                          uchar3 fill3, unsigned frame_bytes) {
    rectify_u8c3_body<EXACT, true>(tmap, vt.v[0].pe, vt.v[0].pf, g, cfg, plan, q2tab, sched, src, dst, fill3, frame_bytes, &vt);
}

}  // namespace cc
