// lm_state.cuh -- device-resident state of the Levenberg-Marquardt loop (lm.cu, residual.cu), and the
// launchers of the fit path (residual.cu, lm.cu, init.cu), which abi.cu calls after its argument checks.
//
// The loop of cc_lm_fit_f64 never returns to the host between iterations: damping, the
// accept / reject decision and the stopping rule live in this block in device memory; every kernel
// of an iteration reads what it needs from it (which of the two view / block buffers is current,
// lambda, the candidate intrinsics) and returns at once when `done` is set.
#pragma once

#include "common.cuh"

namespace cc {

struct LmState {
    double par[4];        // current shared parameters (f, crow, ccol, k); frow = aspect * f
    double cand[4];       // candidate = par + di of the last update
    double lambda;        // Marquardt damping (CvLevMarq: starts at 1e-3, /10 accepted, *10 rejected)
    double sse;           // sum |residual|^2 at `par` over ALL ranks
    double npoints;       // residual points over all ranks (views * corners)
    double step2, size2;  // |step|^2, |parameters|^2 of the last accepted step
    int cur;              // index of the current view / per-view-block buffers
    int done;             // stopping rule met, or max_iter reached
    int iterations, accepted;
    int step_ok;          // the 4x4 solve of the last update succeeded
    int pad[3];
};

// the two generations of per-rank arrays the loop ping-pongs between
struct LmBufs {
    cc_view* views[2];
    double* pv[2];        // per-view blocks, nviews x CC_PER_VIEW
};

// The context's scratch ([components][views] partials) is shared by reproj_jtj, calc_errors and the LM
// kernels.  A hold brackets one launcher's use of it on stream st: acquire() grows the buffer and, when the
// previous user was another stream, makes st wait for the event that user recorded.  The event is recorded on
// st by release(), or when the hold goes out of scope after an error, so kernels already enqueued are always
// covered.  Holds nest on one stream: lm_fit_device holds the scratch around launchers that take it again.
class ScratchHold {
  public:
    ScratchHold(cc_ctx* ctx, cudaStream_t st) : ctx_(ctx), st_(st) {}
    ~ScratchHold() { if (held_) record(); }     // error path: the caller's status and message stand
    int acquire(size_t elems);
    int release();
  private:
    cudaError_t record();
    cc_ctx* ctx_;
    cudaStream_t st_;
    bool held_ = false;
};

// residual.cu.  The caller checks the arguments: img 16-byte aligned, calc_errors_smem(n1, n2) at most
// kCalcErrorsSmemMax.
constexpr size_t kCalcErrorsSmemMax = 200 * 1024;
size_t calc_errors_smem(int n1, int n2);
int launch_reproj_jtj(cc_ctx* ctx, const cc_intr* intr, double aspect, const cc_view* views, int nviews,
                      const double* obj, const double* img, int ncorners, double* per_view, double* shared,
                      cudaStream_t st);
int launch_reproj_jtj_state(cc_ctx* ctx, const LmState* st, int which, const LmBufs& b, double aspect,
                            double checker_size, int nviews, const double* obj, const double* img,
                            int ncorners, double* shared_out, cudaStream_t stream);
int launch_calc_errors(cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews, const double* obj,
                       const double* img, int n1, int n2, const double* inv_rows, const double* inv_cols,
                       int inverse_samples, double* sums, cudaStream_t st);
// out[c] = sum_v parts[c][v] for c < ncomp in a fixed order (bit-reproducible); skipped when gate->done,
// always run when gate == nullptr
int launch_reduce(cc_ctx* ctx, const LmState* gate, const double* parts, int ncomp, int nviews, double* out,
                  cudaStream_t st);
// lm.cu
int launch_lm_schur(cc_ctx* ctx, const double* per_view, int nviews, double lambda, double* yz, double* schur,
                    cudaStream_t st);
int launch_lm_update(cc_ctx* ctx, const double* shared, const double* schur, double lambda, unsigned free_mask,
                     const double* yz, const cc_view* views_in, int nviews, cc_view* views_out, double* delta,
                     cudaStream_t st);
int lm_fit_device(cc_ctx* ctx, cc_intr* intr, double aspect, unsigned free_mask, cc_view* views, int nviews,
                  const double* obj, const double* img, int ncorners, int max_iter, double eps, double* rms,
                  int* iterations, cudaStream_t st);
// init.cu
int launch_initial_guess(cc_ctx* ctx, const double* obj, const double* img, int nviews, int ncorners, int sz1,
                         int sz2, double aspect, cc_intr* intr, cc_view* views, cudaStream_t st);
// comm.cu
int comm_allreduce_sum(cc_ctx* ctx, double* buf, size_t count, cudaStream_t st);

}  // namespace cc
