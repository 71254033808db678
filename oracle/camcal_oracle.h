/*
 * camcal_oracle.h -- CPU restatement (plain C, FP64) of the calibration-object
 * evaluation path of yakir12/CameraCalibrations v0.7.3.
 *
 * THIS IS TEST INFRASTRUCTURE, NOT PRODUCT CODE.  Only tests/, the smoke check in
 * __graft_entry__.py and the cpu_baseline / --impl reference legs of bench.py may
 * call it.  The product path (cameracalibrations_b200/ + libcamcal_b200.so) never
 * links, imports or falls back to anything in oracle/.
 *
 * PARITY STATUS: the reference is Julia and Julia is not installed in this image,
 * so the oracle cannot be checked against the reference executed here.  It is
 * pinned against (1) the reference's own test bounds (test/runtests.jl:73-85) on a
 * cv2 4.13 fit of the reference's example images, (2) cv2.projectPoints /
 * cv2.undistortPoints outputs and Jacobians (the OpenCV the reference calls at
 * src/detect_fit.jl:47), (3) a numpy twin that finds the cubic root the way
 * src/meta.jl:53-55 does (companion-matrix eigenvalues).  The warp's third-party
 * bilinear rule (ImageTransformations/Interpolations, src/plot_calibration.jl:40)
 * has no reference test at all; since round 2 it is pinned to two independent
 * stand-ins (scipy.ndimage.map_coordinates(order=1): index, weights, edges, fill;
 * cv2.remap: tap selection -- tests/test_oracle.py), but NOT to output of the real
 * Julia package: against the reference itself that part stays "parity unpinned"
 * until julia/make_golden.jl has been run (tests/test_julia_golden.py consumes it).
 *
 * Every function cites the reference lines it follows.  The ORDER OF FLOATING
 * POINT OPERATIONS below is normative for the bit-exact FP64 remap parity tests:
 * the CUDA kernels use the same sequence of mul / fma / div.  All sources must be
 * compiled with -ffp-contract=off so that only the explicit fma() calls fuse.
 */
#ifndef CAMCAL_ORACLE_H
#define CAMCAL_ORACLE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Parameter block of `Calibration` (src/meta.jl:17-25) as filled by `obj2img`
 * (src/buildcalibrations.jl:1-6): intrinsic AffineMap diag + translation, k,
 * and checker_size (scale = I/checker_size). */
typedef struct {
    double frow, fcol, crow, ccol, k, checker_size;
} cco_intr;

/* One extrinsic: rotation VECTOR (Rotations.RotationVec) + translation
 * (src/buildcalibrations.jl:3). */
typedef struct {
    double rvec[3], tvec[3];
} cco_view;

/* Everything `Calibration(...)` / `img2obj` derive once per view
 * (src/meta.jl:27-33, 71-76).  Row-major 3x3. */
typedef struct {
    double R[9];      /* extrinsics[i].linear as a matrix            */
    double t[3];      /* extrinsics[i].translation                   */
    double Rinv[9];   /* inv(extrinsic).linear  = R'                 */
    double tinv[3];   /* inv(extrinsic).translation = R' * (-t)      */
    double a_row, b_row, a_col, b_col; /* inv(intrinsic): u = a*rc + b */
    double frow, fcol, crow, ccol, k;
    double inv_cs;    /* scale.linear.diag      = 1/checker_size     */
    double cs_back;   /* inv(scale).linear.diag = 1/(1/checker_size) */
} cco_chain;

void cco_rodrigues(const double rvec[3], double R[9]);
void cco_chain_build(const cco_intr *in, const cco_view *vw, cco_chain *ch);

/* src/meta.jl:50-57: max real root of x^3 - x^2 - c = 0 (see .c for branches) */
double cco_cubic_root(double c);

/* src/meta.jl:88 / :29   world -> pixel */
void cco_world2img(const cco_chain *ch, double x, double y, double z,
                   double *row, double *col);
/* src/meta.jl:82 / :31   pixel -> world */
void cco_img2world(const cco_chain *ch, double row, double col,
                   double *x, double *y, double *z);

/* Bulk forms = the Julia broadcasts c.(pts, i) (src/buildcalibrations.jl:29,46).
 * SoA; z may be NULL for img2world (rectification(c,i) = pop o image2real,
 * src/meta.jl:99) and NULL for world2img inputs meaning z = 0.
 * nthreads <= 0 -> all OpenMP threads. */
void cco_world2img_batch(const cco_chain *ch, const double *x, const double *y,
                         const double *z, double *row, double *col, size_t n,
                         int nthreads);
void cco_img2world_batch(const cco_chain *ch, const double *row, const double *col,
                         double *x, double *y, double *z, size_t n, int nthreads);

/* src/plot_calibration.jl:8-13 and :1-6.  imgpoints: n1*n2 corners, corner
 * (a,b) (0-based, a fastest) at rows[a + n1*b], cols[a + n1*b]. */
double cco_get_ratio(const double *rows, const double *cols, int n1, int n2,
                     double checker_size);
/* axs_min[0] = first index of the output's first axis, axs_min[1] = second. */
void cco_get_axes(double ratio, double checker_size, int n1, int n2,
                  int sz1, int sz2, long long axs_min[2]);

/* Source coordinate of output index (I1, I2): tform(I) of
 * src/plot_calibration.jl:17-18 = real2image o push(.,0) o inv(s). */
void cco_rectify_coord(const cco_chain *ch, double inv_ratio, long long I1,
                       long long I2, double *row, double *col);

/* warp(img, tform, axs) (src/plot_calibration.jl:40) for a batch of frames that
 * share one view.  Frames are stored the way Julia stores them: pixel (r, c)
 * 1-based at  frame_base + (c-1)*pitch + (r-1)   (pitch in pixels, r contiguous),
 * frames nframes apart by frame_stride pixels.  Output has the same size. */
void cco_rectify_f32c1(const cco_chain *ch, double inv_ratio,
                       const long long axs_min[2], const float *src, float *dst,
                       int sz1, int sz2, size_t pitch, size_t frame_stride,
                       int nframes, float fill, int nthreads);
void cco_rectify_u8c3(const cco_chain *ch, double inv_ratio,
                      const long long axs_min[2], const uint8_t *src, uint8_t *dst,
                      int sz1, int sz2, size_t pitch, size_t frame_stride,
                      int nframes, const uint8_t fill[3], int nthreads);
/* the map itself (row/col of the source sample per output pixel), same layout */
void cco_rectify_map(const cco_chain *ch, double inv_ratio,
                     const long long axs_min[2], double *map_row, double *map_col,
                     int sz1, int sz2, size_t pitch, int nthreads);

/* Reprojection residual + Jacobian + normal-equation blocks for row a7:
 * src/buildcalibrations.jl:28-31 (residual) and the arithmetic
 * OpenCV.calibrateCamera reduces (src/detect_fit.jl:40,47) with
 * ZERO_TANGENT + FIX_K2 + FIX_K3 + FIX_ASPECT_RATIO: free parameters per view
 * e = (rvec, tvec) and shared i = (f, crow, ccol, k), frow = aspect * f,
 * fcol = f.  obj: ncorners x 3 (AoS), img: nviews x ncorners x 2 (AoS).
 *   per_view: nviews x 66 doubles = [JtJ_ee 6x6 | JtJ_ei 6x4 | Jtr_e 6]
 *   shared:   21 doubles          = [JtJ_ii 4x4 | Jtr_i 4 | sse]
 * jac (optional, may be NULL): nviews x ncorners x 2 x 10 row-major. */
#define CCO_PER_VIEW 66
#define CCO_SHARED 21
void cco_reproj_jtj(const cco_intr *in, double aspect, const cco_view *views,
                    int nviews, const double *obj, const double *img, int ncorners,
                    double *per_view, double *shared, double *jac, int nthreads);

/* calculate_errors (src/buildcalibrations.jl:37-67).  The `inverse` metric draws
 * rand() in the reference; here the caller supplies the samples
 * (inv_rows/inv_cols: nviews x inverse_samples, already mapped to [1, sz]).
 * out = {reprojection, projection, distance, inverse}. */
void cco_calculate_errors(const cco_intr *in, const cco_view *views, int nviews,
                          const double *obj, const double *img, int n1, int n2,
                          const double *inv_rows, const double *inv_cols,
                          int inverse_samples, double out[4]);
/* The four raw sums over all views that cco_calculate_errors normalises (what
 * cc_calculate_errors_f64 returns): squared reprojection, projection, distance
 * and inverse errors. */
void cco_calculate_error_sums(const cco_intr *in, const cco_view *views, int nviews,
                              const double *obj, const double *img, int n1, int n2,
                              const double *inv_rows, const double *inv_cols,
                              int inverse_samples, double sums[4]);

#ifdef __cplusplus
}
#endif
#endif
