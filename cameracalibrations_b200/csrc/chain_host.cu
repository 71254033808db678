// chain_host.cu -- host-side expansion of the parameter block, once per call.
//
// This is what the reference's `Calibration(...)` constructor and `img2obj` build
// as closures (src/meta.jl:27-33, 71-76; parameters packed by `obj2img`,
// src/buildcalibrations.jl:1-6): the rotation matrix of the RotationVec, the inverse
// extrinsic inv(AffineMap(R,t)) = (R', R'*(-t)), the inverse intrinsic
// inv(AffineMap(diag(f), c)) = (diag(1/f), (1/f)*(-c)), scale = 1/checker_size and its
// inverse.  No trigonometry is left for the kernels.
//
// Compiled with -ffp-contract=off; fusion happens only in the explicit fma() calls so
// the matrices are bit-identical run to run and platform to platform.
#include <cfloat>
#include <cmath>

#include "common.cuh"

namespace cc {

void rodrigues_host(const double r[3], double R[9]) {
    const double th2 = std::fma(r[2], r[2], std::fma(r[1], r[1], r[0] * r[0]));
    const double th = std::sqrt(th2);
    if (th < DBL_EPSILON) {
        for (int i = 0; i < 9; ++i) R[i] = (i % 4 == 0) ? 1.0 : 0.0;
        return;
    }
    const double c = std::cos(th), s = std::sin(th), c1 = 1.0 - c, it = 1.0 / th;
    const double nx = r[0] * it, ny = r[1] * it, nz = r[2] * it;
    R[0] = std::fma(c1 * nx, nx, c);
    R[1] = std::fma(c1 * nx, ny, -(s * nz));
    R[2] = std::fma(c1 * nx, nz, s * ny);
    R[3] = std::fma(c1 * ny, nx, s * nz);
    R[4] = std::fma(c1 * ny, ny, c);
    R[5] = std::fma(c1 * ny, nz, -(s * nx));
    R[6] = std::fma(c1 * nz, nx, -(s * ny));
    R[7] = std::fma(c1 * nz, ny, s * nx);
    R[8] = std::fma(c1 * nz, nz, c);
}

void build_chain(const cc_intr* in, const cc_view* vw, ChainD* ch) {
    rodrigues_host(vw->rvec, ch->R);
    for (int i = 0; i < 3; ++i) ch->t[i] = vw->tvec[i];
    complete_chain(*in, *ch);
}

void narrow_chain(const ChainD& d, ChainF* f) {
    for (int i = 0; i < 9; ++i) { f->R[i] = (float)d.R[i]; f->Rinv[i] = (float)d.Rinv[i]; }
    for (int i = 0; i < 3; ++i) { f->t[i] = (float)d.t[i]; f->tinv[i] = (float)d.tinv[i]; }
    f->a_row = (float)d.a_row; f->b_row = (float)d.b_row;
    f->a_col = (float)d.a_col; f->b_col = (float)d.b_col;
    f->frow = (float)d.frow; f->fcol = (float)d.fcol;
    f->crow = (float)d.crow; f->ccol = (float)d.ccol;
    f->k = (float)d.k; f->inv_cs = (float)d.inv_cs; f->cs_back = (float)d.cs_back;
}

}  // namespace cc
