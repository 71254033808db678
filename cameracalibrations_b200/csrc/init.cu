// init.cu -- starting values of the fit on the device, for views that live in device memory
// (sharded over the ranks of the context's communicator or not).
//
// The reference gets its starting values inside OpenCV.calibrateCamera (src/detect_fit.jl:47):
// principal point at the image centre (src/detect_fit.jl:34-36 passes only the aspect ratio), focal
// length from the homographies' vanishing-point constraints (cvInitIntrinsicParams2D), one pose per
// view from the homography (cvFindExtrinsicCameraParams2's planar branch).  Same construction here:
//   init_homography_kernel  one warp per view: Hartley-normalised DLT, 9x9 normal matrix by
//                           warp-shuffle sums, smallest eigenvector by cyclic Jacobi in shared
//                           memory; the view's two linear equations in (1/frow^2, 1/fcol^2)
//   (fixed-order reduction over views, all-reduce over ranks: 5 doubles; 2x2 solve on the host)
//   init_pose_kernel        one thread per view: K^-1 H -> (r1, r2, t), nearest rotation by the
//                           Newton iteration of the polar decomposition, rotation vector
// These are STARTING values: the LM loop (lm.cu) refines them; tests compare the converged fit.
#include <algorithm>
#include <cmath>

#include "lm_state.cuh"

namespace cc {

constexpr int kInitWarps = 4;

// mean and isotropic scale (mean distance sqrt(2)) of n 2-D points with stride `stride` doubles
__device__ __forceinline__ void hartley(const double* p, int n, int stride, int lane, double& mx, double& my, double& s) {
    double sx = 0.0, sy = 0.0;
    for (int i = lane; i < n; i += 32) { sx += p[(size_t)i * stride]; sy += p[(size_t)i * stride + 1]; }
    mx = warp_sum(sx) / n; my = warp_sum(sy) / n;
    double sd = 0.0;
    for (int i = lane; i < n; i += 32) {
        const double dx = p[(size_t)i * stride] - mx, dy = p[(size_t)i * stride + 1] - my;
        sd += sqrt(dx * dx + dy * dy);
    }
    sd = warp_sum(sd) / n;
    s = 1.4142135623730951 / fmax(sd, 1e-300);
}

// Cyclic Jacobi on a symmetric 9x9 matrix in shared memory (lanes 0..8 each own one row/column
// index k); returns in `h` (all lanes) the eigenvector of the smallest eigenvalue.
__device__ void smallest_eigvec9(double* A, double* V, int lane, double h[9]) {
    if (lane < 9)
        for (int j = 0; j < 9; ++j) V[9 * lane + j] = (lane == j) ? 1.0 : 0.0;
    __syncwarp();
    for (int sweep = 0; sweep < 30; ++sweep) {
        double off = 0.0, dia = 0.0;
        for (int i = 0; i < 9; ++i)
            for (int j = 0; j < 9; ++j) { const double a = A[9 * i + j]; if (i == j) dia += a * a; else off += a * a; }
        if (off <= 1e-30 * dia) break;
        for (int p = 0; p < 8; ++p)
            for (int q = p + 1; q < 9; ++q) {
                const double apq = A[9 * p + q];
                const double app = A[9 * p + p], aqq = A[9 * q + q];
                __syncwarp();
                if (fabs(apq) <= 1e-300) continue;               // warp-uniform (same shared values)
                const double theta = (aqq - app) / (2.0 * apq);
                const double t = copysign(1.0, theta) / (fabs(theta) + sqrt(fma(theta, theta, 1.0)));
                const double c = 1.0 / sqrt(fma(t, t, 1.0)), s = t * c;
                if (lane < 9) {                                  // A <- A J,  V <- V J  (row `lane`)
                    const double akp = A[9 * lane + p], akq = A[9 * lane + q];
                    A[9 * lane + p] = c * akp - s * akq;
                    A[9 * lane + q] = s * akp + c * akq;
                    const double vkp = V[9 * lane + p], vkq = V[9 * lane + q];
                    V[9 * lane + p] = c * vkp - s * vkq;
                    V[9 * lane + q] = s * vkp + c * vkq;
                }
                __syncwarp();
                if (lane < 9) {                                  // A <- J' A      (column `lane`)
                    const double apk = A[9 * p + lane], aqk = A[9 * q + lane];
                    A[9 * p + lane] = c * apk - s * aqk;
                    A[9 * q + lane] = s * apk + c * aqk;
                }
                __syncwarp();
            }
    }
    int best = 0;
    double ev = A[0];
    for (int i = 1; i < 9; ++i)
        if (A[10 * i] < ev) { ev = A[10 * i]; best = i; }
    for (int i = 0; i < 9; ++i) h[i] = V[9 * i + best];
    __syncwarp();
}

// obj: ncorners x 3 (z ignored: the board plane), img: nviews x ncorners x 2 (row, col)
// Hout: nviews x 9 homographies (x, y, 1) -> (row, col, 1), H[8] == 1
// scratch: [5][nviews] this view's share of the normal equations for (1/frow^2, 1/fcol^2)
__global__ void __launch_bounds__(32 * kInitWarps)
init_homography_kernel(const double* __restrict__ obj, const double* __restrict__ img, int nviews, int ncorners,
                       double c0, double c1, double* __restrict__ Hout, double* __restrict__ scratch) {
    __shared__ double smA[kInitWarps][81], smV[kInitWarps][81];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int view = blockIdx.x * kInitWarps + warp;
    if (view >= nviews) return;
    const double* im = img + (size_t)view * ncorners * 2;
    double amx, amy, as, bmx, bmy, bs;
    hartley(obj, ncorners, 3, lane, amx, amy, as);
    hartley(im, ncorners, 2, lane, bmx, bmy, bs);
    // N = A'A, upper triangle (45 sums), two rows per corner
    double acc[45];
#pragma unroll
    for (int i = 0; i < 45; ++i) acc[i] = 0.0;
    for (int ci = lane; ci < ncorners; ci += 32) {
        const double a0 = (obj[3 * ci] - amx) * as, a1 = (obj[3 * ci + 1] - amy) * as;
        const double b0 = (im[2 * ci] - bmx) * bs, b1 = (im[2 * ci + 1] - bmy) * bs;
        const double r0[9] = {a0, a1, 1.0, 0.0, 0.0, 0.0, -b0 * a0, -b0 * a1, -b0};
        const double r1[9] = {0.0, 0.0, 0.0, a0, a1, 1.0, -b1 * a0, -b1 * a1, -b1};
        int k = 0;
#pragma unroll
        for (int i = 0; i < 9; ++i)
#pragma unroll
            for (int j = i; j < 9; ++j) { acc[k] = fma(r0[i], r0[j], fma(r1[i], r1[j], acc[k])); ++k; }
    }
    {
        int k = 0;
#pragma unroll
        for (int i = 0; i < 9; ++i)
#pragma unroll
            for (int j = i; j < 9; ++j) {
                const double v = warp_sum(acc[k]);
                if (lane == 0) { smA[warp][9 * i + j] = v; smA[warp][9 * j + i] = v; }
                ++k;
            }
    }
    __syncwarp();
    double h[9];
    smallest_eigvec9(smA[warp], smV[warp], lane, h);
    // H = Tb^-1 h Ta  with T = [s 0 -s m0; 0 s -s m1; 0 0 1]
    double G[9];                    // h Ta
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        G[3 * i] = h[3 * i] * as;
        G[3 * i + 1] = h[3 * i + 1] * as;
        G[3 * i + 2] = h[3 * i + 2] - as * (h[3 * i] * amx + h[3 * i + 1] * amy);
    }
    double H[9];                    // Tb^-1 = [1/s 0 m0; 0 1/s m1; 0 0 1]
    const double ibs = 1.0 / bs;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        H[j] = G[j] * ibs + bmx * G[6 + j];
        H[3 + j] = G[3 + j] * ibs + bmy * G[6 + j];
        H[6 + j] = G[6 + j];
    }
    const double n = 1.0 / H[8];
#pragma unroll
    for (int i = 0; i < 9; ++i) H[i] *= n;
    if (lane == 0) {
#pragma unroll
        for (int i = 0; i < 9; ++i) Hout[(size_t)view * 9 + i] = H[i];
        // cvInitIntrinsicParams2D: principal point removed; columns h, v and their half sum / half
        // difference, each normalised: two equations  x0 * p0 q0 + x1 * p1 q1 = -p2 q2
        double hc[3] = {H[0] - H[6] * c0, H[3] - H[6] * c1, H[6]};
        double vc[3] = {H[1] - H[7] * c0, H[4] - H[7] * c1, H[7]};
        double d1[3], d2[3];
#pragma unroll
        for (int i = 0; i < 3; ++i) { d1[i] = 0.5 * (hc[i] + vc[i]); d2[i] = 0.5 * (hc[i] - vc[i]); }
        auto unit = [](double* v) {
            const double n = 1.0 / sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]);
            v[0] *= n; v[1] *= n; v[2] *= n;
        };
        unit(hc); unit(vc); unit(d1); unit(d2);
        const double A0[2] = {hc[0] * vc[0], hc[1] * vc[1]}, b0 = -hc[2] * vc[2];
        const double A1[2] = {d1[0] * d2[0], d1[1] * d2[1]}, b1 = -d1[2] * d2[2];
        scratch[view] = A0[0] * A0[0] + A1[0] * A1[0];
        scratch[(size_t)nviews + view] = A0[0] * A0[1] + A1[0] * A1[1];
        scratch[(size_t)2 * nviews + view] = A0[1] * A0[1] + A1[1] * A1[1];
        scratch[(size_t)3 * nviews + view] = A0[0] * b0 + A1[0] * b1;
        scratch[(size_t)4 * nviews + view] = A0[1] * b0 + A1[1] * b1;
    }
}

// pose of every view from its homography and the intrinsics (frow, fcol, c0, c1)
__global__ void __launch_bounds__(128)
init_pose_kernel(const double* __restrict__ Hs, int nviews, double frow, double fcol, double c0, double c1,
                 cc_view* __restrict__ views) {
    const int v = blockIdx.x * 128 + threadIdx.x;
    if (v >= nviews) return;
    const double* H = Hs + (size_t)v * 9;
    double M[9];                                           // K^-1 H
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        M[j] = (H[j] - c0 * H[6 + j]) / frow;
        M[3 + j] = (H[3 + j] - c1 * H[6 + j]) / fcol;
        M[6 + j] = H[6 + j];
    }
    const double n0 = sqrt(M[0] * M[0] + M[3] * M[3] + M[6] * M[6]);
    const double n1 = sqrt(M[1] * M[1] + M[4] * M[4] + M[7] * M[7]);
    double lam = 2.0 / (n0 + n1);
    if (M[8] * lam < 0.0) lam = -lam;                      // board in front of the camera
    double R[9];
    const double r1[3] = {M[0] * lam, M[3] * lam, M[6] * lam}, r2[3] = {M[1] * lam, M[4] * lam, M[7] * lam};
    const double r3[3] = {r1[1] * r2[2] - r1[2] * r2[1], r1[2] * r2[0] - r1[0] * r2[2], r1[0] * r2[1] - r1[1] * r2[0]};
#pragma unroll
    for (int i = 0; i < 3; ++i) { R[3 * i] = r1[i]; R[3 * i + 1] = r2[i]; R[3 * i + 2] = r3[i]; }
    // nearest rotation: Newton iteration of the polar decomposition, R <- (R + R^-T) / 2
    for (int it = 0; it < 12; ++it) {
        const double c00 = R[4] * R[8] - R[5] * R[7], c01 = R[5] * R[6] - R[3] * R[8], c02 = R[3] * R[7] - R[4] * R[6];
        const double det = R[0] * c00 + R[1] * c01 + R[2] * c02;
        if (!(fabs(det) > 1e-300)) break;
        const double id = 1.0 / det;
        // R^-T = cofactor matrix / det
        const double C[9] = {c00, c01, c02,
                             R[2] * R[7] - R[1] * R[8], R[0] * R[8] - R[2] * R[6], R[1] * R[6] - R[0] * R[7],
                             R[1] * R[5] - R[2] * R[4], R[2] * R[3] - R[0] * R[5], R[0] * R[4] - R[1] * R[3]};
        double diff = 0.0;
#pragma unroll
        for (int i = 0; i < 9; ++i) {
            const double nr = 0.5 * (R[i] + C[i] * id);
            diff = fmax(diff, fabs(nr - R[i]));
            R[i] = nr;
        }
        if (diff < 1e-15) break;
    }
    // rotation vector (inverse Rodrigues)
    const double tr = R[0] + R[4] + R[8];
    const double th = acos(fmin(1.0, fmax(-1.0, 0.5 * (tr - 1.0))));
    const double w[3] = {R[7] - R[5], R[2] - R[6], R[3] - R[1]};
    double rv[3];
    if (th < 1e-12) {
#pragma unroll
        for (int i = 0; i < 3; ++i) rv[i] = 0.5 * w[i];
    } else if (3.141592653589793 - th < 1e-6) {            // near pi: axis from the symmetric part
        const double B[3] = {0.5 * (R[0] + 1.0), 0.5 * (R[4] + 1.0), 0.5 * (R[8] + 1.0)};
        const int i = (B[0] >= B[1] && B[0] >= B[2]) ? 0 : (B[1] >= B[2] ? 1 : 2);
        double ax[3];
        const double d = sqrt(fmax(B[i], 0.0));
#pragma unroll
        for (int j = 0; j < 3; ++j) ax[j] = 0.5 * (R[3 * i + j] + R[3 * j + i] + (i == j ? 2.0 : 0.0)) * 0.5 / d;
        const double n = 1.0 / sqrt(ax[0] * ax[0] + ax[1] * ax[1] + ax[2] * ax[2]);
#pragma unroll
        for (int j = 0; j < 3; ++j) rv[j] = th * ax[j] * n;
    } else {
        const double f = th / (2.0 * sin(th));
#pragma unroll
        for (int i = 0; i < 3; ++i) rv[i] = f * w[i];
    }
#pragma unroll
    for (int i = 0; i < 3; ++i) { views[v].rvec[i] = rv[i]; views[v].tvec[i] = M[3 * i + 2] * lam; }
}

struct InitBuf {
    void* p = nullptr;
    ~InitBuf() { if (p) cudaFree(p); }
};

int launch_initial_guess(cc_ctx* ctx, const double* obj, const double* img, int nviews, int ncorners, int sz1,
                         int sz2, double aspect, cc_intr* intr, cc_view* views, cudaStream_t st) {
    const int nv1 = nviews > 0 ? nviews : 1;
    InitBuf hs, scr, red;
    CC_CUDA(cudaMalloc(&hs.p, (size_t)nv1 * 9 * sizeof(double)));
    CC_CUDA(cudaMalloc(&scr.p, (size_t)nv1 * 5 * sizeof(double)));
    CC_CUDA(cudaMalloc(&red.p, 8 * sizeof(double)));
    const double c0 = 0.5 * (sz1 - 1), c1 = 0.5 * (sz2 - 1);
    if (nviews > 0) {
        init_homography_kernel<<<(nviews + kInitWarps - 1) / kInitWarps, 32 * kInitWarps, 0, st>>>(
            obj, img, nviews, ncorners, c0, c1, static_cast<double*>(hs.p), static_cast<double*>(scr.p));
        ctx->launches++;
    }
    int rc = launch_reduce(ctx, nullptr, static_cast<double*>(scr.p), 5, nviews, static_cast<double*>(red.p), st);
    if (rc || (rc = comm_allreduce_sum(ctx, static_cast<double*>(red.p), 5, st))) return rc;
    double n[5];
    CC_CUDA(cudaMemcpyAsync(n, red.p, sizeof(n), cudaMemcpyDeviceToHost, st));
    CC_CUDA(cudaStreamSynchronize(st));
    // least squares for x = (1/frow^2, 1/fcol^2)
    const double det = n[0] * n[2] - n[1] * n[1];
    CC_REQUIRE(std::isfinite(det) && det != 0.0, "degenerate views: cannot initialise the focal length");
    const double x0 = (n[2] * n[3] - n[1] * n[4]) / det, x1 = (n[0] * n[4] - n[1] * n[3]) / det;
    double fr = std::sqrt(std::fabs(1.0 / x0)), fc = std::sqrt(std::fabs(1.0 / x1));
    if (aspect > 0.0) {                                    // CALIB_FIX_ASPECT_RATIO
        const double tf = (fr + fc) / (aspect + 1.0);
        fr = aspect * tf; fc = tf;
    }
    CC_REQUIRE(std::isfinite(fr) && std::isfinite(fc) && fr > 0.0 && fc > 0.0, "focal length initialisation failed");
    intr->frow = fr; intr->fcol = fc; intr->crow = c0; intr->ccol = c1; intr->k = 0.0;
    if (nviews > 0) {
        init_pose_kernel<<<(nviews + 127) / 128, 128, 0, st>>>(static_cast<double*>(hs.p), nviews, fr, fc, c0, c1, views);
        ctx->launches++;
        CC_CUDA(cudaGetLastError());
        CC_CUDA(cudaStreamSynchronize(st));                // hs is freed on return
    }
    return CC_OK;
}

}  // namespace cc
