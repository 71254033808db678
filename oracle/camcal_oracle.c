/*
 * camcal_oracle.c -- see camcal_oracle.h.  TEST INFRASTRUCTURE ONLY.
 *
 * Plain C99 + optional OpenMP.  Compile with -ffp-contract=off: the only fused
 * operations are the explicit fma() calls, and their placement is the normative
 * operation order the CUDA kernels reproduce bit for bit in FP64.
 *
 * Reference = /root/reference (yakir12/CameraCalibrations v0.7.3); citations are
 * file:line in that tree.  No reference source text is copied; the reference is
 * Julia built on CoordinateTransformations/Rotations/Polynomials closures, this is
 * a scalar restatement of the arithmetic those closures perform.
 */
#include "camcal_oracle.h"

#include <float.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

static int cco_threads(int nthreads)
{
#ifdef _OPENMP
    return nthreads > 0 ? nthreads : omp_get_max_threads();
#else
    (void)nthreads;
    return 1;
#endif
}

/* ------------------------------------------------------------------------- */
/* Rotation vector -> matrix.  The reference stores Rotations.RotationVec      */
/* (src/buildcalibrations.jl:3) and applies it per call; here it is expanded   */
/* once (Rodrigues):  R = c I + (1-c) n n' + s [n]x ,  n = r/theta.            */
/* ------------------------------------------------------------------------- */
void cco_rodrigues(const double r[3], double R[9])
{
    double th2 = fma(r[2], r[2], fma(r[1], r[1], r[0] * r[0]));
    double th = sqrt(th2);
    if (th < DBL_EPSILON) {
        R[0] = 1; R[1] = 0; R[2] = 0;
        R[3] = 0; R[4] = 1; R[5] = 0;
        R[6] = 0; R[7] = 0; R[8] = 1;
        return;
    }
    double c = cos(th), s = sin(th), c1 = 1.0 - c, it = 1.0 / th;
    double nx = r[0] * it, ny = r[1] * it, nz = r[2] * it;
    R[0] = fma(c1 * nx, nx, c);
    R[1] = fma(c1 * nx, ny, -(s * nz));
    R[2] = fma(c1 * nx, nz, s * ny);
    R[3] = fma(c1 * ny, nx, s * nz);
    R[4] = fma(c1 * ny, ny, c);
    R[5] = fma(c1 * ny, nz, -(s * nx));
    R[6] = fma(c1 * nz, nx, -(s * ny));
    R[7] = fma(c1 * nz, ny, s * nx);
    R[8] = fma(c1 * nz, nz, c);
}

/* Calibration(...) constructor + img2obj: src/meta.jl:27-33, 71-76.
 * inv(AffineMap(M, v)) = AffineMap(inv(M), inv(M) * (-v))  (CoordinateTransformations). */
void cco_chain_build(const cco_intr *in, const cco_view *vw, cco_chain *ch)
{
    cco_rodrigues(vw->rvec, ch->R);
    for (int i = 0; i < 3; ++i) ch->t[i] = vw->tvec[i];
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) ch->Rinv[3 * i + j] = ch->R[3 * j + i];
    for (int i = 0; i < 3; ++i) {
        const double *m = ch->Rinv + 3 * i;
        double nt0 = -ch->t[0], nt1 = -ch->t[1], nt2 = -ch->t[2];
        ch->tinv[i] = fma(m[2], nt2, fma(m[1], nt1, m[0] * nt0));
    }
    ch->frow = in->frow; ch->fcol = in->fcol;
    ch->crow = in->crow; ch->ccol = in->ccol; ch->k = in->k;
    ch->a_row = 1.0 / in->frow;            /* inv(SDiagonal(frow, fcol))          */
    ch->a_col = 1.0 / in->fcol;
    ch->b_row = ch->a_row * (-in->crow);   /* inv(M) * (-translation)             */
    ch->b_col = ch->a_col * (-in->ccol);
    ch->inv_cs = 1.0 / in->checker_size;   /* src/buildcalibrations.jl:4          */
    ch->cs_back = 1.0 / ch->inv_cs;        /* inv(scale), src/meta.jl:75          */
}

/* ------------------------------------------------------------------------- */
/* src/meta.jl:50-57.  roots(Polynomial([c,0,1,-1])) = roots of x^3 - x^2 - c,  */
/* keep |imag| < 1e-10, take the maximum real part.                            */
/*   c == 0          -> roots {0,0,1}            -> 1                          */
/*   c > 0           -> one real root, > 1                                     */
/*   -4/27 <= c < 0  -> three real roots, largest in [2/3, 1)                  */
/*   c < -4/27       -> one real root, negative (the model is not invertible   */
/*                      there; the reference still divides by it)              */
/* f is convex for x > 1/3, so Newton from a point with f >= 0 right of the    */
/* largest root decreases monotonically onto it; iterate until it stalls.      */
/* ------------------------------------------------------------------------- */
double cco_cubic_root(double c)
{
    if (c == 0.0) return 1.0;
    if (c != c) return c;
    double x;
    if (c >= -4.0 / 27.0) {
        x = c > 0.0 ? 1.0 + fmin(c, cbrt(c)) : 1.0;
        for (int it = 0; it < 200; ++it) {
            double x2 = x * x;
            double f = fma(x2, x - 1.0, -c);
            double fp = x * fma(3.0, x, -2.0);
            if (!(fp > 0.0)) break;
            double xn = x - f / fp;
            if (!(xn < x)) break;
            x = xn;
        }
        /* c rounded to just above -4/27 can leave f > 0 everywhere right of 2/3 in
         * floating point: the iteration then stalls at the double root 2/3. */
        return x;
    }
    /* single negative root: f concave and increasing for x < 0, start left of it */
    x = -cbrt(-c);
    for (int it = 0; it < 200; ++it) {
        double x2 = x * x;
        double f = fma(x2, x - 1.0, -c);
        double fp = x * fma(3.0, x, -2.0);
        double xn = x - f / fp;
        if (!(xn > x)) break;
        x = xn;
    }
    return x;
}

/* src/meta.jl:29: intrinsic o distort o PerspectiveMap o extrinsic o scale */
void cco_world2img(const cco_chain *ch, double x, double y, double z,
                   double *row, double *col)
{
    /* scale: LinearMap(SDiagonal(1/cs)) */
    double q1 = x * ch->inv_cs, q2 = y * ch->inv_cs, q3 = z * ch->inv_cs;
    /* extrinsic: R q + t */
    const double *R = ch->R;
    /* order: z term, then the first world axis, then the second (the rectification
     * kernels keep the first-axis term per thread and add the second per pixel) */
    double P1 = fma(R[1], q2, fma(R[0], q1, fma(R[2], q3, ch->t[0])));
    double P2 = fma(R[4], q2, fma(R[3], q1, fma(R[5], q3, ch->t[1])));
    double P3 = fma(R[7], q2, fma(R[6], q1, fma(R[8], q3, ch->t[2])));
    /* PerspectiveMap: scale = 1/v[3]; (v[1]*scale, v[2]*scale) */
    double s = 1.0 / P3;
    double u = P1 * s, v = P2 * s;
    /* lens_distortion, src/meta.jl:39-44 */
    if (ch->k != 0.0) {
        double r2 = fma(v, v, u * u);
        double radial = fma(ch->k, r2, 1.0);
        u = radial * u;
        v = radial * v;
    }
    /* intrinsic: AffineMap(SDiagonal(frow,fcol), (crow,ccol)) */
    *row = fma(ch->frow, u, ch->crow);
    *col = fma(ch->fcol, v, ch->ccol);
}

/* src/meta.jl:31: inv_scale o inv_extrinsic o inv_perspective o inv_distort o inv_intrinsic */
void cco_img2world(const cco_chain *ch, double row, double col,
                   double *x, double *y, double *z)
{
    double u = fma(ch->a_row, row, ch->b_row);
    double v = fma(ch->a_col, col, ch->b_col);
    /* inv_lens_distortion, src/meta.jl:50-57 */
    if (ch->k != 0.0) {
        double c = ch->k * fma(v, v, u * u);
        double ir = 1.0 / cco_cubic_root(c);
        u = u * ir;
        v = v * ir;
    }
    /* get_inv_prespective_map, src/meta.jl:60-69: rc1=(u,v,1), l = Rinv[3,:] */
    const double *Ri = ch->Rinv;
    double den = fma(Ri[6], u, fma(Ri[7], v, Ri[8]));
    double d = (-ch->tinv[2]) / den;
    double w1 = d * u, w2 = d * v, w3 = d;
    /* inv_extrinsic: Rinv w + tinv */
    double p1 = fma(Ri[0], w1, fma(Ri[1], w2, fma(Ri[2], w3, ch->tinv[0])));
    double p2 = fma(Ri[3], w1, fma(Ri[4], w2, fma(Ri[5], w3, ch->tinv[1])));
    double p3 = fma(Ri[6], w1, fma(Ri[7], w2, fma(Ri[8], w3, ch->tinv[2])));
    /* inv_scale */
    *x = ch->cs_back * p1;
    *y = ch->cs_back * p2;
    *z = ch->cs_back * p3;
}

void cco_world2img_batch(const cco_chain *ch, const double *x, const double *y,
                         const double *z, double *row, double *col, size_t n,
                         int nthreads)
{
    int nt = cco_threads(nthreads);
    (void)nt;
#pragma omp parallel for num_threads(nt) schedule(static)
    for (long long i = 0; i < (long long)n; ++i)
        cco_world2img(ch, x[i], y[i], z ? z[i] : 0.0, row + i, col + i);
}

void cco_img2world_batch(const cco_chain *ch, const double *row, const double *col,
                         double *x, double *y, double *z, size_t n, int nthreads)
{
    int nt = cco_threads(nthreads);
    (void)nt;
#pragma omp parallel for num_threads(nt) schedule(static)
    for (long long i = 0; i < (long long)n; ++i) {
        double zz;
        cco_img2world(ch, row[i], col[i], x + i, y + i, &zz);
        if (z) z[i] = zz;
    }
}

/* src/plot_calibration.jl:8-13 */
double cco_get_ratio(const double *rows, const double *cols, int n1, int n2,
                     double checker_size)
{
    double s1 = 0.0, s2 = 0.0;
    /* diff(imgpoints; dims=1): (n1-1) x n2, column-major traversal */
    for (int b = 0; b < n2; ++b)
        for (int a = 0; a + 1 < n1; ++a) {
            double dr = rows[a + 1 + n1 * b] - rows[a + n1 * b];
            double dc = cols[a + 1 + n1 * b] - cols[a + n1 * b];
            s1 += sqrt(dr * dr + dc * dc);
        }
    for (int b = 0; b + 1 < n2; ++b)
        for (int a = 0; a < n1; ++a) {
            double dr = rows[a + n1 * (b + 1)] - rows[a + n1 * b];
            double dc = cols[a + n1 * (b + 1)] - cols[a + n1 * b];
            s2 += sqrt(dr * dr + dc * dc);
        }
    double m1 = s1 / (double)((n1 - 1) * n2);
    double m2 = s2 / (double)(n1 * (n2 - 1));
    double l = (m1 + m2) / 2.0;
    return l / checker_size;
}

/* src/plot_calibration.jl:1-6; round(Int, .) is round-half-even = rint() */
void cco_get_axes(double ratio, double checker_size, int n1, int n2, int sz1,
                  int sz2, long long axs_min[2])
{
    double w1 = rint(ratio * checker_size * (double)(n1 - 1));
    double w2 = rint(ratio * checker_size * (double)(n2 - 1));
    axs_min[0] = (long long)rint((w1 - (double)sz1) / 2.0);
    axs_min[1] = (long long)rint((w2 - (double)sz2) / 2.0);
}

/* tform = real2image[i] o push(.,0) o inv(LinearMap(ratio*I)),
 * src/plot_calibration.jl:17-18 */
void cco_rectify_coord(const cco_chain *ch, double inv_ratio, long long I1,
                       long long I2, double *row, double *col)
{
    double x = (double)I1 * inv_ratio;
    double y = (double)I2 * inv_ratio;
    cco_world2img(ch, x, y, 0.0, row, col);
}

/* Bilinear rule of warp() -> Interpolations BSpline(Linear()) OnGrid with a
 * filled extrapolation (src/plot_calibration.jl:40; third-party; pinned to
 * scipy.ndimage.map_coordinates and cv2.remap, not to Julia output: PARITY
 * UNPINNED against the reference itself): sample at (row, col) in the image's own 1-based axes;
 * outside [1,n] on either axis -> fill; i = floor(x), pulled back by one when
 * i > n-1 (x == n); delta = x - i; weights (1-delta, delta).
 * Returns 0 if out of bounds, else fills i0 (0-based), d. */
static inline int cco_lin_pos(double x, int n, int *i0, double *d)
{
    if (!(x >= 1.0 && x <= (double)n)) return 0;
    double xf = floor(x);
    if (xf > (double)(n - 1)) xf -= 1.0;
    *d = x - xf;
    *i0 = (int)xf - 1;
    return 1;
}

void cco_rectify_map(const cco_chain *ch, double inv_ratio,
                     const long long axs_min[2], double *map_row, double *map_col,
                     int sz1, int sz2, size_t pitch, int nthreads)
{
    int nt = cco_threads(nthreads);
    (void)nt;
#pragma omp parallel for num_threads(nt) schedule(static)
    for (int b = 0; b < sz2; ++b)
        for (int a = 0; a < sz1; ++a)
            cco_rectify_coord(ch, inv_ratio, axs_min[0] + a, axs_min[1] + b,
                              map_row + (size_t)b * pitch + a,
                              map_col + (size_t)b * pitch + a);
}

void cco_rectify_f32c1(const cco_chain *ch, double inv_ratio,
                       const long long axs_min[2], const float *src, float *dst,
                       int sz1, int sz2, size_t pitch, size_t frame_stride,
                       int nframes, float fill, int nthreads)
{
    int nt = cco_threads(nthreads);
    (void)nt;
#pragma omp parallel for num_threads(nt) schedule(static) collapse(2)
    for (int f = 0; f < nframes; ++f)
        for (int b = 0; b < sz2; ++b) {
            const float *s = src + (size_t)f * frame_stride;
            float *o = dst + (size_t)f * frame_stride + (size_t)b * pitch;
            for (int a = 0; a < sz1; ++a) {
                double row, col, d1, d2;
                int i1, i2;
                cco_rectify_coord(ch, inv_ratio, axs_min[0] + a, axs_min[1] + b,
                                  &row, &col);
                if (!cco_lin_pos(row, sz1, &i1, &d1) ||
                    !cco_lin_pos(col, sz2, &i2, &d2)) {
                    o[a] = fill;
                    continue;
                }
                const float *p = s + (size_t)i2 * pitch + i1;
                double a00 = p[0], a10 = p[1], a01 = p[pitch], a11 = p[pitch + 1];
                double e1 = 1.0 - d1, e2 = 1.0 - d2;
                double lo = fma(d2, a01, e2 * a00);   /* first-axis offset 0 */
                double hi = fma(d2, a11, e2 * a10);   /* first-axis offset 1 */
                o[a] = (float)fma(d1, hi, e1 * lo);
            }
        }
}

/* RGB{N0f8}: blend the raw 0..255 values in FP64, store round-half-even.  (The
 * reference blends value/255 and re-quantises on store; same real number, the two
 * can differ by 1 LSB only at exact .5 ties.) */
void cco_rectify_u8c3(const cco_chain *ch, double inv_ratio,
                      const long long axs_min[2], const uint8_t *src, uint8_t *dst,
                      int sz1, int sz2, size_t pitch, size_t frame_stride,
                      int nframes, const uint8_t fill[3], int nthreads)
{
    int nt = cco_threads(nthreads);
    (void)nt;
#pragma omp parallel for num_threads(nt) schedule(static) collapse(2)
    for (int f = 0; f < nframes; ++f)
        for (int b = 0; b < sz2; ++b) {
            const uint8_t *s = src + (size_t)f * frame_stride * 3;
            uint8_t *o = dst + ((size_t)f * frame_stride + (size_t)b * pitch) * 3;
            for (int a = 0; a < sz1; ++a) {
                double row, col, d1, d2;
                int i1, i2;
                cco_rectify_coord(ch, inv_ratio, axs_min[0] + a, axs_min[1] + b,
                                  &row, &col);
                if (!cco_lin_pos(row, sz1, &i1, &d1) ||
                    !cco_lin_pos(col, sz2, &i2, &d2)) {
                    o[3 * a] = fill[0]; o[3 * a + 1] = fill[1]; o[3 * a + 2] = fill[2];
                    continue;
                }
                const uint8_t *p = s + ((size_t)i2 * pitch + i1) * 3;
                double e1 = 1.0 - d1, e2 = 1.0 - d2;
                for (int ch3 = 0; ch3 < 3; ++ch3) {
                    double a00 = p[ch3], a10 = p[3 + ch3];
                    double a01 = p[3 * pitch + ch3], a11 = p[3 * pitch + 3 + ch3];
                    double lo = fma(d2, a01, e2 * a00);
                    double hi = fma(d2, a11, e2 * a10);
                    double val = rint(fma(d1, hi, e1 * lo));
                    if (val < 0.0) val = 0.0;
                    if (val > 255.0) val = 255.0;
                    o[3 * a + ch3] = (uint8_t)val;
                }
            }
        }
}

/* ------------------------------------------------------------------------- */
/* Row a7: residual, Jacobian, normal-equation blocks.                         */
/* dR/dr_i = ( r_i [r]x + [ r x w_i ]x ) R / theta^2          (theta > 0)      */
/*         = [e_i]x                                (theta < DBL_EPSILON)      */
/* w_i = (I - R) e_i = c1 (e_i - n n_i) - s (n x e_i),  n = r / theta,        */
/* s = sin theta, c1 = 1 - cos theta formed as s^2 / (1 + cos theta) while    */
/* cos theta > 0.  Formed as e_i - R e_i instead, w_i loses its c1 part to     */
/* rounding and the division by theta^2 magnifies the loss: ~2e-8 relative at */
/* theta = 1e-8; so does 1 - cos theta for small theta.                        */
/* ------------------------------------------------------------------------- */
static void skew(const double v[3], double S[9])
{
    S[0] = 0;     S[1] = -v[2]; S[2] = v[1];
    S[3] = v[2];  S[4] = 0;     S[5] = -v[0];
    S[6] = -v[1]; S[7] = v[0];  S[8] = 0;
}

static void matmul3(const double A[9], const double B[9], double C[9])
{
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j)
            C[3 * i + j] = A[3 * i] * B[j] + A[3 * i + 1] * B[3 + j] +
                           A[3 * i + 2] * B[6 + j];
}

static void rodrigues_jac(const double r[3], const double R[9], double dR[3][9])
{
    double th2 = fma(r[2], r[2], fma(r[1], r[1], r[0] * r[0]));
    double th = sqrt(th2);
    if (th < DBL_EPSILON) {
        for (int i = 0; i < 3; ++i) {
            double e[3] = {0, 0, 0};
            e[i] = 1.0;
            skew(e, dR[i]);
        }
        return;
    }
    double s = sin(th), c = cos(th), it = 1.0 / th;
    double c1 = c > 0.0 ? s * s / (1.0 + c) : 1.0 - c;
    double n[3] = {r[0] * it, r[1] * it, r[2] * it};
    double S[9], Sn[9];
    skew(r, S);
    skew(n, Sn);
    for (int i = 0; i < 3; ++i) {
        /* w = c1 (e_i - n n_i) - s (n x e_i);  n x e_i is column i of [n]x */
        double w[3];
        for (int j = 0; j < 3; ++j) w[j] = -(c1 * (n[j] * n[i])) - s * Sn[3 * j + i];
        w[i] += c1;
        double cr[3] = {r[1] * w[2] - r[2] * w[1], r[2] * w[0] - r[0] * w[2],
                        r[0] * w[1] - r[1] * w[0]};
        double C[9], M[9];
        skew(cr, C);
        for (int j = 0; j < 9; ++j) M[j] = (r[i] * S[j] + C[j]) / th2;
        matmul3(M, R, dR[i]);
    }
}

/* residual (2) and Jacobian (2 x 10) of one corner */
static void corner_jac(const double R[9], const double dR[3][9], const double t[3],
                       double frow, double fcol, double crow, double ccol, double k,
                       double aspect, double inv_cs, const double X[3],
                       const double obs[2], double res[2], double J[2][10])
{
    double q[3] = {X[0] * inv_cs, X[1] * inv_cs, X[2] * inv_cs};
    double P[3];
    for (int i = 0; i < 3; ++i)
        P[i] = fma(R[3 * i + 1], q[1], fma(R[3 * i], q[0], fma(R[3 * i + 2], q[2], t[i])));
    double s = 1.0 / P[2];
    double u = P[0] * s, v = P[1] * s;
    double r2 = fma(v, v, u * u);
    double radial = fma(k, r2, 1.0);
    double ud = radial * u, vd = radial * v;
    res[0] = fma(frow, ud, crow) - obs[0];
    res[1] = fma(fcol, vd, ccol) - obs[1];
    /* d(ud,vd)/d(u,v) */
    double a11 = radial + 2.0 * k * u * u, a12 = 2.0 * k * u * v;
    double a22 = radial + 2.0 * k * v * v;
    /* d(u,v)/dP */
    double du[3] = {s, 0.0, -u * s}, dv[3] = {0.0, s, -v * s};
    double gr[3], gc[3]; /* d row / dP, d col / dP */
    for (int i = 0; i < 3; ++i) {
        gr[i] = frow * (a11 * du[i] + a12 * dv[i]);
        gc[i] = fcol * (a12 * du[i] + a22 * dv[i]);
    }
    for (int i = 0; i < 3; ++i) {
        double dP[3];
        for (int j = 0; j < 3; ++j)
            dP[j] = dR[i][3 * j] * q[0] + dR[i][3 * j + 1] * q[1] + dR[i][3 * j + 2] * q[2];
        J[0][i] = gr[0] * dP[0] + gr[1] * dP[1] + gr[2] * dP[2];
        J[1][i] = gc[0] * dP[0] + gc[1] * dP[1] + gc[2] * dP[2];
        J[0][3 + i] = gr[i];
        J[1][3 + i] = gc[i];
    }
    J[0][6] = aspect * ud; J[1][6] = vd;         /* d/df, frow = aspect*f, fcol = f */
    J[0][7] = 1.0;         J[1][7] = 0.0;        /* d/dcrow */
    J[0][8] = 0.0;         J[1][8] = 1.0;        /* d/dccol */
    J[0][9] = frow * u * r2; J[1][9] = fcol * v * r2; /* d/dk */
}

void cco_reproj_jtj(const cco_intr *in, double aspect, const cco_view *views,
                    int nviews, const double *obj, const double *img, int ncorners,
                    double *per_view, double *shared, double *jac, int nthreads)
{
    int nt = cco_threads(nthreads);
    (void)nt;
    double inv_cs = 1.0 / in->checker_size;
    double *sh_all = (double *)calloc((size_t)nviews * CCO_SHARED, sizeof(double));
#pragma omp parallel for num_threads(nt) schedule(static)
    for (int vi = 0; vi < nviews; ++vi) {
        double R[9], dR[3][9];
        cco_rodrigues(views[vi].rvec, R);
        rodrigues_jac(views[vi].rvec, R, dR);
        double *pv = per_view + (size_t)vi * CCO_PER_VIEW;
        double *sh = sh_all + (size_t)vi * CCO_SHARED;
        memset(pv, 0, CCO_PER_VIEW * sizeof(double));
        for (int ci = 0; ci < ncorners; ++ci) {
            double res[2], J[2][10];
            corner_jac(R, dR, views[vi].tvec, in->frow, in->fcol, in->crow, in->ccol,
                       in->k, aspect, inv_cs, obj + 3 * ci,
                       img + 2 * ((size_t)vi * ncorners + ci), res, J);
            if (jac)
                memcpy(jac + ((size_t)vi * ncorners + ci) * 20, J, 20 * sizeof(double));
            for (int rr = 0; rr < 2; ++rr) {
                const double *j = J[rr];
                for (int a = 0; a < 6; ++a) {
                    for (int b = 0; b < 6; ++b) pv[6 * a + b] += j[a] * j[b];
                    for (int b = 0; b < 4; ++b) pv[36 + 4 * a + b] += j[a] * j[6 + b];
                    pv[60 + a] += j[a] * res[rr];
                }
                for (int a = 0; a < 4; ++a) {
                    for (int b = 0; b < 4; ++b) sh[4 * a + b] += j[6 + a] * j[6 + b];
                    sh[16 + a] += j[6 + a] * res[rr];
                }
                sh[20] += res[rr] * res[rr];
            }
        }
    }
    for (int j = 0; j < CCO_SHARED; ++j) shared[j] = 0.0;
    for (int vi = 0; vi < nviews; ++vi)
        for (int j = 0; j < CCO_SHARED; ++j) shared[j] += sh_all[(size_t)vi * CCO_SHARED + j];
    free(sh_all);
}

/* src/buildcalibrations.jl:37-67 */
void cco_calculate_error_sums(const cco_intr *in, const cco_view *views, int nviews,
                              const double *obj, const double *img, int n1, int n2,
                              const double *inv_rows, const double *inv_cols,
                              int inverse_samples, double sums[4])
{
    int nc = n1 * n2;
    double reprojection = 0.0, projection = 0.0, distance = 0.0, inverse = 0.0;
    double *px = (double *)malloc(sizeof(double) * 3 * (size_t)nc);
    for (int vi = 0; vi < nviews; ++vi) {
        cco_chain ch;
        cco_chain_build(in, &views[vi], &ch);
        const double *im = img + 2 * (size_t)vi * nc;
        double sr = 0.0, sp = 0.0;
        for (int ci = 0; ci < nc; ++ci) {
            double row, col;
            cco_world2img(&ch, obj[3 * ci], obj[3 * ci + 1], obj[3 * ci + 2], &row, &col);
            double dr = row - im[2 * ci], dc = col - im[2 * ci + 1];
            sr += dr * dr + dc * dc;                               /* :29-30 */
            double *p = px + 3 * ci;
            cco_img2world(&ch, im[2 * ci], im[2 * ci + 1], p, p + 1, p + 2);   /* :46 */
            double ex = p[0] - obj[3 * ci], ey = p[1] - obj[3 * ci + 1],
                   ez = p[2] - obj[3 * ci + 2];
            sp += ex * ex + ey * ey + ez * ez;                     /* :47 */
        }
        reprojection += sr;
        projection += sp;
        double sd = 0.0;                                           /* :49-51 */
        for (int b = 0; b < n2; ++b)
            for (int a = 0; a + 1 < n1; ++a) {
                const double *p0 = px + 3 * (a + n1 * b), *p1 = px + 3 * (a + 1 + n1 * b);
                double e = sqrt((p1[0] - p0[0]) * (p1[0] - p0[0]) +
                                (p1[1] - p0[1]) * (p1[1] - p0[1]) +
                                (p1[2] - p0[2]) * (p1[2] - p0[2])) - in->checker_size;
                sd += e * e;
            }
        for (int b = 0; b + 1 < n2; ++b)
            for (int a = 0; a < n1; ++a) {
                const double *p0 = px + 3 * (a + n1 * b), *p1 = px + 3 * (a + n1 * (b + 1));
                double e = sqrt((p1[0] - p0[0]) * (p1[0] - p0[0]) +
                                (p1[1] - p0[1]) * (p1[1] - p0[1]) +
                                (p1[2] - p0[2]) * (p1[2] - p0[2])) - in->checker_size;
                sd += e * e;
            }
        distance += sd;
        double si = 0.0;                                           /* :53-58 */
        for (int s = 0; s < inverse_samples; ++s) {
            double r0 = inv_rows[(size_t)vi * inverse_samples + s];
            double c0 = inv_cols[(size_t)vi * inverse_samples + s];
            double x, y, z, r1, c1;
            cco_img2world(&ch, r0, c0, &x, &y, &z);
            cco_world2img(&ch, x, y, z, &r1, &c1);
            si += (r0 - r1) * (r0 - r1) + (c0 - c1) * (c0 - c1);
        }
        inverse += si;
    }
    free(px);
    sums[0] = reprojection; sums[1] = projection; sums[2] = distance; sums[3] = inverse;
}

void cco_calculate_errors(const cco_intr *in, const cco_view *views, int nviews,
                          const double *obj, const double *img, int n1, int n2,
                          const double *inv_rows, const double *inv_cols,
                          int inverse_samples, double out[4])
{
    double s[4];
    cco_calculate_error_sums(in, views, nviews, obj, img, n1, n2, inv_rows, inv_cols,
                             inverse_samples, s);
    double n = (double)n1 * n2 * nviews;                           /* :60-65 */
    out[0] = sqrt(s[0] / n);
    out[1] = sqrt(s[1] / n);
    out[2] = sqrt(s[2] / (double)((n1 - 1) * (n2 - 1)) / nviews);
    out[3] = sqrt(s[3] / inverse_samples / nviews);
}
