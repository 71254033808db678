// lm.cu -- one Levenberg-Marquardt step on the normal equations that reproj_jtj_kernel
// accumulates (SURVEY 8f rank 2: the solve that OpenCV.calibrateCamera runs inside the
// reference's fit, src/detect_fit.jl:47, flags :40, criteria src/CameraCalibrations.jl:16).
//
// The system is an arrowhead: per view a 6x6 block A_v (rvec, tvec), a 6x4 coupling B_v to the
// shared intrinsics (f, crow, ccol, k) and the shared 4x4 block C:
//     [ A  B ] [de]     [ge]          A_v' = A_v + lambda*diag(A_v)   (Marquardt damping, as
//     [ B' C ] [di] = - [gi]          C'   = C   + lambda*diag(C)      CvLevMarq scales the diagonal)
// Phase 1 (lm_schur_kernel, one thread per view): Cholesky of A_v', Y_v = A_v'^-1 B_v,
//   z_v = A_v'^-1 ge_v, and the view's share of the Schur complement S = sum B_v' Y_v,
//   s = sum B_v' z_v (reduced over views in a fixed order; all-reduced over ranks by the host
//   layer when views are sharded across GPUs -- 20 doubles).
// Phase 2 (lm_update_kernel): (C' - S) di = -(gi - s);  de_v = -(z_v + Y_v di);  candidate
//   parameters = parameters + delta; step and parameter norms for the stopping rule.
// Fixed shared parameters (CALIB_FIX_K1 when with_distortion == false) are masked out.
#include <algorithm>
#include <cmath>

#include "lm_state.cuh"

namespace cc {

constexpr int kLmThreads = 128;

// in-place Cholesky of a symmetric positive definite N x N matrix (lower triangle); false if a
// pivot is not positive
template <int N>
__device__ __forceinline__ bool cholesky(double (&a)[N][N]) {
    bool ok = true;
#pragma unroll
    for (int j = 0; j < N; ++j) {
        double d = a[j][j];
#pragma unroll
        for (int k = 0; k < j; ++k) d -= a[j][k] * a[j][k];
        ok &= d > 0.0;
        const double l = sqrt(d), il = 1.0 / l;
        a[j][j] = l;
#pragma unroll
        for (int i = j + 1; i < N; ++i) {
            double s = a[i][j];
#pragma unroll
            for (int k = 0; k < j; ++k) s -= a[i][k] * a[j][k];
            a[i][j] = s * il;
        }
    }
    return ok;
}

// solve L L' x = b in place
template <int N>
__device__ __forceinline__ void chol_solve(const double (&a)[N][N], double (&x)[N]) {
#pragma unroll
    for (int i = 0; i < N; ++i) {
        double s = x[i];
#pragma unroll
        for (int k = 0; k < i; ++k) s -= a[i][k] * x[k];
        x[i] = s / a[i][i];
    }
#pragma unroll
    for (int i = N - 1; i >= 0; --i) {
        double s = x[i];
#pragma unroll
        for (int k = i + 1; k < N; ++k) s -= a[k][i] * x[k];
        x[i] = s / a[i][i];
    }
}

// scratch layout (component-major, like reproj_jtj_kernel): [0,16) S, [16,20) s, [20] failed views
constexpr int kSchurComponents = 21;

// Eight lanes per view: every lane factors the (same) damped 6x6 block, then lane r solves ONE right-hand
// side -- r < 4: column r of B (-> column r of Y and of the view's Schur share), r == 4: g (-> z and the
// share of s) -- instead of one thread walking five solves in a row.  The kernel is pure latency (10 000
// views are 79 warps on 148 SMs): the serial chain per view drops from Cholesky + 5 solves + 20 dot
// products to Cholesky + 1 solve + 4 dot products; every entry is computed by the same sequence of
// operations as before, so the values are unchanged.
constexpr int kSchurLanes = 8;
__device__ __forceinline__ void
lm_schur_view(const double* __restrict__ per_view, int nviews, double lambda, double* __restrict__ yz,
              double* __restrict__ scratch) {
    const int t = blockIdx.x * kLmThreads + threadIdx.x;
    const int v = t / kSchurLanes, r = t % kSchurLanes;
    if (v >= nviews || r > 4) return;
    const double* pv = per_view + (size_t)v * CC_PER_VIEW;
    double A[6][6], B[6][4], x[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) {
#pragma unroll
        for (int j = 0; j < 6; ++j) A[i][j] = pv[6 * i + j];
#pragma unroll
        for (int j = 0; j < 4; ++j) B[i][j] = pv[36 + 4 * i + j];
    }
#pragma unroll
    for (int i = 0; i < 6; ++i) x[i] = r < 4 ? pv[36 + 4 * i + r] : pv[60 + i];      // column r of B, or g
#pragma unroll
    for (int i = 0; i < 6; ++i) A[i][i] = fma(lambda, A[i][i], A[i][i]);
    const bool ok = cholesky<6>(A);
    chol_solve<6>(A, x);
    double* o = yz + (size_t)v * 30;
#pragma unroll
    for (int i = 0; i < 6; ++i) o[r < 4 ? 4 * i + r : 24 + i] = ok ? x[i] : 0.0;
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        double s = 0.0;
#pragma unroll
        for (int i = 0; i < 6; ++i) s = fma(B[i][a], x[i], s);
        scratch[(size_t)(r < 4 ? 4 * a + r : 16 + a) * nviews + v] = ok ? s : 0.0;
    }
    if (r == 4) scratch[(size_t)20 * nviews + v] = ok ? 0.0 : 1.0;
}

__global__ void __launch_bounds__(kLmThreads)
lm_schur_kernel(const double* __restrict__ per_view, int nviews, double lambda, double* __restrict__ yz,
                double* __restrict__ scratch) {
    lm_schur_view(per_view, nviews, lambda, yz, scratch);
}
// inside the device-resident loop: blocks and damping from the loop state
__global__ void __launch_bounds__(kLmThreads)
lm_schur_state_kernel(const LmState* __restrict__ st, const LmBufs b, int nviews, double* __restrict__ yz,
                      double* __restrict__ scratch) {
    if (st->done) return;
    lm_schur_view(b.pv[st->cur], nviews, st->lambda, yz, scratch);
}

// delta layout: [0,4) di | [4] sum |de|^2 | [5] sum |pe|^2 | [6] 1 if the 4x4 solve succeeded | [7] spare
__device__ __forceinline__ void
lm_update_view(const double* __restrict__ shared, const double* __restrict__ schur, double lambda,
               unsigned free_mask, const double* __restrict__ yz, const cc_view* __restrict__ vin,
               int nviews, cc_view* __restrict__ vout, double* __restrict__ delta,
               double* __restrict__ scratch) {
    __shared__ double di_sm[4];
    __shared__ int ok_sm;
    if (threadIdx.x == 0) {
        double M[4][4], rhs[4];
#pragma unroll
        for (int a = 0; a < 4; ++a) {
#pragma unroll
            for (int b = 0; b < 4; ++b) M[a][b] = shared[4 * a + b] - schur[4 * a + b];
            M[a][a] = fma(lambda, shared[5 * a], M[a][a]);
            rhs[a] = -(shared[16 + a] - schur[16 + a]);
        }
#pragma unroll
        for (int a = 0; a < 4; ++a)
            if (!((free_mask >> a) & 1u)) {
#pragma unroll
                for (int b = 0; b < 4; ++b) { M[a][b] = 0.0; M[b][a] = 0.0; }
                M[a][a] = 1.0;
                rhs[a] = 0.0;
            }
        const bool ok = cholesky<4>(M);
        chol_solve<4>(M, rhs);
#pragma unroll
        for (int a = 0; a < 4; ++a) di_sm[a] = ok ? rhs[a] : 0.0;
        ok_sm = ok ? 1 : 0;
        if (blockIdx.x == 0) {
#pragma unroll
            for (int a = 0; a < 4; ++a) delta[a] = di_sm[a];
            delta[6] = ok ? 1.0 : 0.0;
            delta[7] = 0.0;
        }
    }
    __syncthreads();
    const int v = blockIdx.x * kLmThreads + threadIdx.x;
    if (v >= nviews) return;
    const double* o = yz + (size_t)v * 30;
    const double p[6] = {vin[v].rvec[0], vin[v].rvec[1], vin[v].rvec[2],
                         vin[v].tvec[0], vin[v].tvec[1], vin[v].tvec[2]};
    double de[6], n_de = 0.0, n_p = 0.0;
#pragma unroll
    for (int i = 0; i < 6; ++i) {
        double s = o[24 + i];
#pragma unroll
        for (int j = 0; j < 4; ++j) s = fma(o[4 * i + j], di_sm[j], s);
        de[i] = ok_sm ? -s : 0.0;
        n_de = fma(de[i], de[i], n_de);
        n_p = fma(p[i], p[i], n_p);
    }
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        vout[v].rvec[i] = p[i] + de[i];
        vout[v].tvec[i] = p[3 + i] + de[3 + i];
    }
    scratch[v] = n_de;
    scratch[(size_t)nviews + v] = n_p;
}

__global__ void __launch_bounds__(kLmThreads)
lm_update_kernel(const double* __restrict__ shared, const double* __restrict__ schur, double lambda,
                 unsigned free_mask, const double* __restrict__ yz, const cc_view* __restrict__ vin,
                 int nviews, cc_view* __restrict__ vout, double* __restrict__ delta,
                 double* __restrict__ scratch) {
    lm_update_view(shared, schur, lambda, free_mask, yz, vin, nviews, vout, delta, scratch);
}
// inside the device-resident loop: current views -> candidate views (the other buffer); the
// candidate intrinsics are published by lm_candidate_kernel once delta is complete
__global__ void __launch_bounds__(kLmThreads)
lm_update_state_kernel(const LmState* __restrict__ st, const double* __restrict__ shared,
                       const double* __restrict__ schur, unsigned free_mask, const double* __restrict__ yz,
                       const LmBufs b, int nviews, double* __restrict__ delta, double* __restrict__ scratch) {
    if (st->done) return;
    lm_update_view(shared, schur, st->lambda, free_mask, yz, b.views[st->cur], nviews, b.views[st->cur ^ 1],
                   delta, scratch);
}
__global__ void lm_candidate_kernel(LmState* __restrict__ st, const double* __restrict__ delta) {
    if (st->done) return;
#pragma unroll
    for (int a = 0; a < 4; ++a) st->cand[a] = st->par[a] + delta[a];
    st->step_ok = delta[6] != 0.0;
}

// first evaluation: red = all-reduced [shared block 21 | residual points 1]
__global__ void lm_init_kernel(LmState* __restrict__ st, double f, double crow, double ccol, double k,
                               const double* __restrict__ red, double* __restrict__ sh_cur) {
    st->par[0] = f; st->par[1] = crow; st->par[2] = ccol; st->par[3] = k;
#pragma unroll
    for (int a = 0; a < 4; ++a) st->cand[a] = st->par[a];
    st->lambda = 1e-3;
    st->sse = red[20];
    st->npoints = red[21];
    st->step2 = 0.0; st->size2 = 0.0;
    st->cur = 0; st->done = 0; st->iterations = 0; st->accepted = 0; st->step_ok = 0;
    for (int i = 0; i < CC_SHARED; ++i) sh_cur[i] = red[i];
}
__global__ void lm_count_kernel(double* __restrict__ red, double npoints) { red[21] = npoints; }

// The accept / reject select and the stopping rule, on the device (one thread).
//   red   : all-reduced [candidate's shared block 21 | sum |de|^2 | sum |pe|^2]
//   schur : all-reduced Schur share; [20] = views (any rank) whose 6x6 block was not positive definite
// Every rank sees the same all-reduced numbers and therefore takes the same decision.
__global__ void lm_decide_kernel(LmState* __restrict__ st, const double* __restrict__ red,
                                 const double* __restrict__ schur, double* __restrict__ sh_cur, double eps,
                                 int max_iter) {
    if (st->done) return;
    st->iterations++;
    double d2 = 0.0, p2 = 0.0;
    bool bad = schur[20] > 0.0 || !st->step_ok;
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        const double di = st->cand[a] - st->par[a];
        bad = bad || !isfinite(di);
        d2 = fma(di, di, d2);
        p2 = fma(st->par[a], st->par[a], p2);
    }
    const double sse_c = red[20];
    bad = bad || !isfinite(red[21]) || !isfinite(sse_c) || !(sse_c < st->sse);
    if (bad) {
        st->lambda = fmin(st->lambda * 10.0, 1e16);
    } else {
        st->step2 = red[21] + d2;
        st->size2 = red[22] + p2;
#pragma unroll
        for (int a = 0; a < 4; ++a) st->par[a] = st->cand[a];
        st->sse = sse_c;
        for (int i = 0; i < CC_SHARED; ++i) sh_cur[i] = red[i];
        st->cur ^= 1;
        st->lambda = fmax(st->lambda / 10.0, 1e-16);
        st->accepted++;
        if (sqrt(st->step2) < eps * sqrt(st->size2)) st->done = 1;
    }
    if (st->iterations >= max_iter) st->done = 1;
}


int launch_lm_schur(cc_ctx* ctx, const double* per_view, int nviews, double lambda, double* yz,
                    double* schur, cudaStream_t st) {
    const int nv = nviews > 0 ? nviews : 1;
    ScratchHold hold(ctx, st);
    int rc = hold.acquire((size_t)kSchurComponents * nv);
    if (rc) return rc;
    if (nviews > 0) {
        lm_schur_kernel<<<(nviews * kSchurLanes + kLmThreads - 1) / kLmThreads, kLmThreads, 0, st>>>(per_view, nviews, lambda, yz,
                                                                                   ctx->jtj_scratch);
        ctx->launches++;
        CC_CUDA(cudaGetLastError());
    }
    if ((rc = launch_reduce(ctx, nullptr, ctx->jtj_scratch, kSchurComponents, nviews, schur, st))) return rc;
    return hold.release();
}

int launch_lm_update(cc_ctx* ctx, const double* shared, const double* schur, double lambda,
                     unsigned free_mask, const double* yz, const cc_view* views_in, int nviews,
                     cc_view* views_out, double* delta, cudaStream_t st) {
    const int nv = nviews > 0 ? nviews : 1;
    ScratchHold hold(ctx, st);
    int rc = hold.acquire((size_t)kSchurComponents * nv);
    if (rc) return rc;
    // at least one block: block 0 publishes the shared-parameter step even without local views
    const int blocks = std::max(1, (nviews + kLmThreads - 1) / kLmThreads);
    lm_update_kernel<<<blocks, kLmThreads, 0, st>>>(shared, schur, lambda, free_mask, yz, views_in, nviews,
                                                    views_out, delta, ctx->jtj_scratch);
    ctx->launches++;
    CC_CUDA(cudaGetLastError());
    if ((rc = launch_reduce(ctx, nullptr, ctx->jtj_scratch, 2, nviews, delta + 4, st))) return rc;
    return hold.release();
}

// ---------------------------------------------------------------------------------------------
// The fit as one device-resident loop (cc_lm_fit_f64): replaces the OpenCV.calibrateCamera call of
// src/detect_fit.jl:47 (flags :40, CRITERIA src/CameraCalibrations.jl:16) for views that already
// live in device memory, sharded over the ranks of the context's communicator or not.
//
// Per iteration the host enqueues, without ever waiting:
//   lm_schur_state  (+ fixed-order reduce)          -> schur[21]          | all-reduce (21 doubles)
//   lm_update_state (+ reduce of the two norms)     -> candidate views, di
//   reproj_jtj_state on the candidate (+ reduce)    -> red[0..21)          | all-reduce (23 doubles)
//   lm_decide                                       -> accept / reject, lambda, stopping rule
// i.e. TWO small all-reduces (the Schur share must be global before the step exists; the candidate's
// blocks need the step) and ZERO host synchronisations.  The host copies the 128-byte state to
// pinned memory after every iteration and looks at it three iterations later (event query, never a
// wait) to stop enqueueing once `done` is set; kernels of iterations enqueued past that point
// return immediately.
// ---------------------------------------------------------------------------------------------
struct LmWorkspace {
    int cap_views = 0;
    cc_view* views1 = nullptr;
    double* pv[2] = {nullptr, nullptr};
    double* yz = nullptr;
    double* small = nullptr;       // [schur 21 | pad 3 | red 24 | sh_cur 21 | pad 3 | delta 8]
    LmState* state = nullptr;
    LmState* host_state = nullptr; // pinned ring
    cudaEvent_t ev[8] = {};
    static constexpr int kRing = 8;
};

void lm_free_workspace(cc_ctx* ctx) {
    LmWorkspace* w = static_cast<LmWorkspace*>(ctx->lm_ws);
    if (!w) return;
    cudaFree(w->views1); cudaFree(w->pv[0]); cudaFree(w->pv[1]); cudaFree(w->yz); cudaFree(w->small);
    cudaFree(w->state);
    if (w->host_state) cudaFreeHost(w->host_state);
    for (auto& e : w->ev) if (e) cudaEventDestroy(e);
    delete w;
    ctx->lm_ws = nullptr;
}

static int lm_workspace(cc_ctx* ctx, int nviews, LmWorkspace** out) {
    LmWorkspace* w = static_cast<LmWorkspace*>(ctx->lm_ws);
    if (!w) {
        w = new (std::nothrow) LmWorkspace();
        if (!w) return set_error(CC_ERR_NOMEM, "out of host memory");
        ctx->lm_ws = w;
        CC_CUDA(cudaMalloc(&w->small, 80 * sizeof(double)));
        CC_CUDA(cudaMalloc(&w->state, sizeof(LmState)));
        CC_CUDA(cudaHostAlloc(&w->host_state, LmWorkspace::kRing * sizeof(LmState), cudaHostAllocDefault));
        for (auto& e : w->ev) CC_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
    const int need = nviews > 0 ? nviews : 1;
    if (w->cap_views < need) {
        cudaFree(w->views1); cudaFree(w->pv[0]); cudaFree(w->pv[1]); cudaFree(w->yz);
        w->views1 = nullptr; w->pv[0] = w->pv[1] = w->yz = nullptr; w->cap_views = 0;
        CC_CUDA(cudaMalloc(&w->views1, (size_t)need * sizeof(cc_view)));
        CC_CUDA(cudaMalloc(&w->pv[0], (size_t)need * CC_PER_VIEW * sizeof(double)));
        CC_CUDA(cudaMalloc(&w->pv[1], (size_t)need * CC_PER_VIEW * sizeof(double)));
        CC_CUDA(cudaMalloc(&w->yz, (size_t)need * CC_LM_YZ * sizeof(double)));
        w->cap_views = need;
    }
    *out = w;
    return CC_OK;
}

int lm_fit_device(cc_ctx* ctx, cc_intr* intr, double aspect, unsigned free_mask, cc_view* views, int nviews,
                  const double* obj, const double* img, int ncorners, int max_iter, double eps, double* rms,
                  int* iterations, cudaStream_t st) {
    LmWorkspace* w = nullptr;
    int rc = lm_workspace(ctx, nviews, &w);
    if (rc) return rc;
    const int nv1 = nviews > 0 ? nviews : 1;
    ScratchHold hold(ctx, st);                       // the whole loop; the launchers below take it again
    if ((rc = hold.acquire((size_t)kSchurComponents * nv1))) return rc;
    double* schur = w->small;
    double* red = w->small + 24;
    double* sh_cur = w->small + 48;
    double* delta = w->small + 72;
    LmBufs b;
    b.views[0] = views; b.views[1] = w->views1;
    b.pv[0] = w->pv[0]; b.pv[1] = w->pv[1];

    // first evaluation at the starting values
    cc_intr in = *intr;
    const double k0 = (free_mask & 8u) ? intr->k : 0.0;
    in.frow = aspect * intr->fcol; in.k = k0;
    if ((rc = launch_reproj_jtj(ctx, &in, aspect, views, nviews, obj, img, ncorners, b.pv[0], red, st))) return rc;
    lm_count_kernel<<<1, 1, 0, st>>>(red, (double)nviews * (double)ncorners);
    if ((rc = comm_allreduce_sum(ctx, red, 22, st))) return rc;
    lm_init_kernel<<<1, 1, 0, st>>>(w->state, intr->fcol, intr->crow, intr->ccol, k0, red, sh_cur);
    ctx->launches += 2;
    CC_CUDA(cudaGetLastError());

    const int blocks_v = std::max(1, (nviews + kLmThreads - 1) / kLmThreads);
    constexpr int kLag = 3;
    int enq = 0;
    for (; enq < max_iter; ++enq) {
        if (enq >= kLag) {                               // look at the state of iteration enq - kLag, if it has arrived
            const int slot = (enq - kLag) % LmWorkspace::kRing;
            if (cudaEventQuery(w->ev[slot]) == cudaSuccess && w->host_state[slot].done) break;
            cudaGetLastError();                          // cudaErrorNotReady is not an error
        }
        // phase 1: per-view Cholesky, Schur share
        if (nviews > 0) {
            lm_schur_state_kernel<<<(nviews * kSchurLanes + kLmThreads - 1) / kLmThreads, kLmThreads, 0, st>>>(w->state, b, nviews, w->yz, ctx->jtj_scratch);
            ctx->launches++;
        }
        if ((rc = launch_reduce(ctx, w->state, ctx->jtj_scratch, kSchurComponents, nviews, schur, st))) return rc;
        if ((rc = comm_allreduce_sum(ctx, schur, CC_LM_SCHUR, st))) return rc;
        // phase 2: shared step, candidate views, step norms
        lm_update_state_kernel<<<blocks_v, kLmThreads, 0, st>>>(w->state, sh_cur, schur, free_mask, w->yz, b, nviews,
                                                               delta, ctx->jtj_scratch);
        ctx->launches++;
        if ((rc = launch_reduce(ctx, w->state, ctx->jtj_scratch, 2, nviews, red + 21, st))) return rc;
        lm_candidate_kernel<<<1, 1, 0, st>>>(w->state, delta);
        ctx->launches++;
        // candidate's residual and blocks
        if ((rc = launch_reproj_jtj_state(ctx, w->state, 1, b, aspect, intr->checker_size, nviews, obj, img,
                                          ncorners, red, st))) return rc;
        if ((rc = comm_allreduce_sum(ctx, red, 23, st))) return rc;
        lm_decide_kernel<<<1, 1, 0, st>>>(w->state, red, schur, sh_cur, eps, max_iter);
        ctx->launches++;
        CC_CUDA(cudaGetLastError());
        const int slot = enq % LmWorkspace::kRing;
        CC_CUDA(cudaMemcpyAsync(&w->host_state[slot], w->state, sizeof(LmState), cudaMemcpyDeviceToHost, st));
        CC_CUDA(cudaEventRecord(w->ev[slot], st));
    }
    if ((rc = hold.release())) return rc;
    // the one wait of the call: the caller gets the intrinsics back on the host
    LmState fin;
    CC_CUDA(cudaMemcpyAsync(&w->host_state[0], w->state, sizeof(LmState), cudaMemcpyDeviceToHost, st));
    CC_CUDA(cudaStreamSynchronize(st));
    fin = w->host_state[0];
    if (fin.cur == 1 && nviews > 0) {
        CC_CUDA(cudaMemcpyAsync(views, w->views1, (size_t)nviews * sizeof(cc_view), cudaMemcpyDeviceToDevice, st));
        CC_CUDA(cudaStreamSynchronize(st));
    }
    intr->frow = aspect * fin.par[0]; intr->fcol = fin.par[0]; intr->crow = fin.par[1]; intr->ccol = fin.par[2];
    intr->k = fin.par[3];
    if (rms) *rms = std::sqrt(fin.sse / std::max(1.0, fin.npoints));
    if (iterations) *iterations = fin.iterations;
    return CC_OK;
}

}  // namespace cc
