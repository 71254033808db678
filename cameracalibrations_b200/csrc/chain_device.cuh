// chain_device.cuh -- per-point arithmetic of the two chains, FP64 and FP32.
//
// FP64 world->pixel follows the normative operation order of the oracle
// (oracle/camcal_oracle.c) exactly -- same mul / fma / div sequence, compiled with
// -fmad=false so nothing else fuses -- because the rectification map must select
// bit-identical bilinear indices and weights.  FP64 pixel->world only has to agree
// to 1e-9 and solves the cubic differently (see inv_radial).
#pragma once

#include "common.cuh"

namespace cc {

// Rodrigues on the device (sincos: not bit-identical to rodrigues_host, so no point map or rectification uses it);
// returns theta^2.  tsc (optional): receives (theta, sin theta, cos theta) when theta >= DBL_EPSILON.
__device__ __forceinline__ double rodrigues(const double r[3], double R[9], double* tsc = nullptr) {
    const double th2 = fma(r[2], r[2], fma(r[1], r[1], r[0] * r[0]));
    const double th = sqrt(th2);
    if (th < 2.220446049250313e-16) {
#pragma unroll
        for (int i = 0; i < 9; ++i) R[i] = (i % 4 == 0) ? 1.0 : 0.0;
        return th2;
    }
    double s, c;
    sincos(th, &s, &c);
    if (tsc) { tsc[0] = th; tsc[1] = s; tsc[2] = c; }
    const double c1 = 1.0 - c, it = 1.0 / th;
    const double nx = r[0] * it, ny = r[1] * it, nz = r[2] * it;
    R[0] = fma(c1 * nx, nx, c);
    R[1] = fma(c1 * nx, ny, -(s * nz));
    R[2] = fma(c1 * nx, nz, s * ny);
    R[3] = fma(c1 * ny, nx, s * nz);
    R[4] = fma(c1 * ny, ny, c);
    R[5] = fma(c1 * ny, nz, -(s * nx));
    R[6] = fma(c1 * nz, nx, -(s * ny));
    R[7] = fma(c1 * nz, ny, s * nx);
    R[8] = fma(c1 * nz, nz, c);
    return th2;
}

// ---- world -> pixel: src/meta.jl:29  intrinsic o distort o Perspective o extrinsic o scale
__device__ __forceinline__ void world2img(const ChainD& ch, double x, double y, double z,
                                          double& row, double& col) {
    const double q1 = x * ch.inv_cs, q2 = y * ch.inv_cs, q3 = z * ch.inv_cs;
    const double P1 = fma(ch.R[1], q2, fma(ch.R[0], q1, fma(ch.R[2], q3, ch.t[0])));
    const double P2 = fma(ch.R[4], q2, fma(ch.R[3], q1, fma(ch.R[5], q3, ch.t[1])));
    const double P3 = fma(ch.R[7], q2, fma(ch.R[6], q1, fma(ch.R[8], q3, ch.t[2])));
    const double s = 1.0 / P3;                        // PerspectiveMap: scale = 1/v[3]
    double u = P1 * s, v = P2 * s;
    if (ch.k != 0.0) {                                // lens_distortion, src/meta.jl:39-44
        const double r2 = fma(v, v, u * u);
        const double radial = fma(ch.k, r2, 1.0);
        u = radial * u;
        v = radial * v;
    }
    row = fma(ch.frow, u, ch.crow);
    col = fma(ch.fcol, v, ch.ccol);
}

__device__ __forceinline__ void world2img(const ChainF& ch, float x, float y, float z,
                                          float& row, float& col) {
    const float q1 = x * ch.inv_cs, q2 = y * ch.inv_cs, q3 = z * ch.inv_cs;
    const float P1 = fmaf(ch.R[1], q2, fmaf(ch.R[0], q1, fmaf(ch.R[2], q3, ch.t[0])));
    const float P2 = fmaf(ch.R[4], q2, fmaf(ch.R[3], q1, fmaf(ch.R[5], q3, ch.t[1])));
    const float P3 = fmaf(ch.R[7], q2, fmaf(ch.R[6], q1, fmaf(ch.R[8], q3, ch.t[2])));
    const float s = __frcp_rn(P3);
    float u = P1 * s, v = P2 * s;
    if (ch.k != 0.0f) {
        const float r2 = fmaf(v, v, u * u);
        const float radial = fmaf(ch.k, r2, 1.0f);
        u = radial * u;
        v = radial * v;
    }
    row = fmaf(ch.frow, u, ch.crow);
    col = fmaf(ch.fcol, v, ch.ccol);
}

// ---- inverse radial distortion: src/meta.jl:50-57 ---------------------------------
// The reference divides by x*, the largest real root of x^3 - x^2 - c = 0 (companion
// eigenvalues, |imag| < 1e-10, maximum real part).  With y = 1/x* the same root solves
//     g(y) = c y^3 + y - 1 = 0 ,   g'(y) = 3 c y^2 + 1 ,
// and the chain needs exactly y (v2 / x* = v2 * y), so no division is left.
//   c > 0          : g convex increasing, y* in (0,1): Newton from y0 = 1 descends onto it
//   -4/27 <= c < 0 : g concave increasing on [1, 1.5], y* in (1, 1.5]: Newton from y0 = 1
//                    ascends onto it (the x-root in [2/3, 1) is the largest one)
//   c < -4/27      : only real root is negative (model not invertible there; the
//                    reference still uses it): g convex decreasing left of it, Newton
//                    from y0 = -max(2, sqrt(2/|c|)) ascends onto it
// returns y = 1/x*.
// `three_real`: c >= -4/27, decided by the caller in ITS precision (the branch must not flip when
// a double c just above -4/27 narrows to a float just below it: the result changes sign)
__device__ __forceinline__ float inv_radial_seed(float c, bool three_real) {
    float y;
    if (three_real) {
        y = 1.0f;
    } else {
        y = -fmaxf(2.0f, sqrtf(__fdividef(2.0f, -c)));
    }
    const float c3 = 3.0f * c;
    for (int it = 0; it < 64; ++it) {
        const float t = y * y;
        const float g = fmaf(c * t, y, y - 1.0f);
        const float gp = fmaf(c3, t, 1.0f);
        const float dy = __fdividef(g, gp);
        y -= dy;
        if (!(fabsf(dy) > 2e-4f * fabsf(y))) break;   // next step would be below FP32 eps
    }
    return y;
}

// Common range -0.12 <= c <= 1 (every sane lens: |k| r^2 well inside the invertible region): a
// FIXED schedule -- the Newton step from y = 1 in closed form, (1 + 2c) / (1 + 3c), then three
// full steps with SFU reciprocals -- reaches FP32 accuracy (max relative error 8e-8 over the
// range, checked against the companion-matrix roots) without a data-dependent loop, so the
// points a thread holds interleave.  Returns false outside the range.
__device__ __forceinline__ float rcp_sfu(float a) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(a));
    return r;
}
__device__ __forceinline__ bool inv_radial_fixed(float c, float& y) {
    const float c3 = 3.0f * c;
    y = fmaf(-c, rcp_sfu(c3 + 1.0f), 1.0f);
#pragma unroll
    for (int it = 0; it < 3; ++it) {
        const float t = y * y;
        const float g = fmaf(c * t, y, y - 1.0f);
        const float gp = fmaf(c3, t, 1.0f);
        y = fmaf(-g, rcp_sfu(gp), y);
    }
    return (c >= -0.12f) & (c <= 1.0f);
}

__device__ __forceinline__ float inv_radial_generic(float c) {
    if (c == 0.0f) return 1.0f;
    float y = inv_radial_seed(c, c >= -4.0f / 27.0f);
    // one more step at full FP32 accuracy
    const float t = y * y;
    const float g = fmaf(c * t, y, y - 1.0f);
    const float gp = fmaf(3.0f * c, t, 1.0f);
    return y - g / gp;
}

__device__ __forceinline__ float inv_radial(float c) {
    float y;
    if (!inv_radial_fixed(c, y)) y = inv_radial_generic(c);      // rare
    return y;
}

__device__ __forceinline__ double inv_radial(double c) {
    if (c == 0.0) return 1.0;                 // roots {0,0,1}
    // FP32 seed (error <~ 1e-6 relative away from the double root), then FP64 Newton
    // with an SFU reciprocal refined by one Newton-Schulz step: two polish steps give
    // e1 ~ K e0^2 + 2^-23 e0, e2 ~ K e1^2 + 1e-12 e1  -> full FP64 accuracy.
    float ys;
    const float cf = (float)c;
    const bool three_real = c >= -4.0 / 27.0;
    if (!inv_radial_fixed(cf, ys))                                           // rare
        // c within a float ulp above -4/27 narrows below it: no FP32 root to seed from, start at 1
        ys = (three_real && !(cf >= -4.0f / 27.0f)) ? 1.0f : inv_radial_seed(cf, three_real);
    double y = (double)ys;
    const double c3 = 3.0 * c;
    double t = y * y;
    double g = fma(c * t, y, y - 1.0);
    double gp = fma(c3, t, 1.0);
    double r = rcp_approx(gp);
    y = fma(-g, r, y);
    t = y * y;
    g = fma(c * t, y, y - 1.0);
    gp = fma(c3, t, 1.0);
    r = fma(r, fma(-gp, r, 1.0), r);
    double dy = g * r;
    y -= dy;
    // near the double root (c -> -4/27, gp -> 0) or for a poor seed keep iterating with
    // true divisions until the step stalls
    if (fabs(dy) > 1e-11 * fabs(y)) {
        for (int it = 0; it < 100; ++it) {
            t = y * y;
            g = fma(c * t, y, y - 1.0);
            gp = fma(c3, t, 1.0);
            dy = g / gp;
            const double yn = y - dy;
            if (!(fabs(dy) > 4e-16 * fabs(yn)) || yn == y) { y = yn; break; }
            y = yn;
        }
    }
    return y;
}

// ---- pixel -> world: src/meta.jl:31 ----------------------------------------------
template <typename T>
__device__ __forceinline__ T fma_t(T a, T b, T c);
template <> __device__ __forceinline__ double fma_t<double>(double a, double b, double c) { return fma(a, b, c); }
template <> __device__ __forceinline__ float fma_t<float>(float a, float b, float c) { return fmaf(a, b, c); }

__device__ __forceinline__ double div_t(double a, double b) { return a / b; }
__device__ __forceinline__ float div_t(float a, float b) { return __fdividef(a, b); }

template <typename T>
__device__ __forceinline__ void img2world(const Chain<T>& ch, T row, T col, T& x, T& y, T& z) {
    T u = fma_t(ch.a_row, row, ch.b_row);             // inv(intrinsic)
    T v = fma_t(ch.a_col, col, ch.b_col);
    if (ch.k != T(0)) {                               // inv_lens_distortion
        const T c = ch.k * fma_t(v, v, u * u);
        const T ir = inv_radial(c);
        u *= ir;
        v *= ir;
    }
    // get_inv_prespective_map, src/meta.jl:60-69: rc1 = (u,v,1), l = Rinv[3,:]
    const T den = fma_t(ch.Rinv[6], u, fma_t(ch.Rinv[7], v, ch.Rinv[8]));
    const T d = div_t(-ch.tinv[2], den);
    const T w1 = d * u, w2 = d * v, w3 = d;
    // inv(extrinsic), then inv(scale)
    x = ch.cs_back * fma_t(ch.Rinv[0], w1, fma_t(ch.Rinv[1], w2, fma_t(ch.Rinv[2], w3, ch.tinv[0])));
    y = ch.cs_back * fma_t(ch.Rinv[3], w1, fma_t(ch.Rinv[4], w2, fma_t(ch.Rinv[5], w3, ch.tinv[1])));
    z = ch.cs_back * fma_t(ch.Rinv[6], w1, fma_t(ch.Rinv[7], w2, fma_t(ch.Rinv[8], w3, ch.tinv[2])));
}

}  // namespace cc
