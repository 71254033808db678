// residual.cu -- reprojection residual, analytic Jacobian and normal-equation blocks;
// fused calculate_errors.
//
// Residual: _reprojection, src/buildcalibrations.jl:28-31 (sum ||c(obj,i) - img||^2).
// Jacobian / J'J: the reference has no Jacobian code of its own -- this is the
// arithmetic OpenCV.calibrateCamera reduces (src/detect_fit.jl:40,47) for the flags
// ZERO_TANGENT + FIX_K2 + FIX_K3 + FIX_ASPECT_RATIO: per view e = (rvec, tvec), shared
// i = (f, crow, ccol, k), frow = aspect * f, fcol = f.
//
// One warp per view.  Each lane walks corners lane, lane+32, ...; image points are read
// as one coalesced 16-byte (row,col) pair per lane; 66 FP64 accumulators per lane
// (upper triangles only) are combined with xor-shuffle butterflies.  The shared 21-value
// block is written per view, component-major, and reduced over views by a second
// kernel in a fixed order (bit-reproducible; no atomics).  Across GPUs the 21 doubles
// are all-reduced with NCCL by the host layer.
#include "chain_device.cuh"
#include "lm_state.cuh"

namespace cc {

constexpr int kResWarps = 4;
constexpr int kResThreads = 32 * kResWarps;

struct ViewGeom {
    double R[9];
    double dR[3][9];   // dR/dr_i
};

__device__ __forceinline__ void skew(const double v[3], double S[9]) {
    S[0] = 0;     S[1] = -v[2]; S[2] = v[1];
    S[3] = v[2];  S[4] = 0;     S[5] = -v[0];
    S[6] = -v[1]; S[7] = v[0];  S[8] = 0;
}

// Rodrigues and its derivative:
//   dR/dr_i = ( r_i [r]x + [ r x ((I - R) e_i) ]x ) R / theta^2 ,  -> [e_i]x as theta -> 0
__device__ void view_geom(const double r[3], ViewGeom& g) {
    const double th2 = rodrigues(r, g.R);
    if (th2 < 1e-24) {
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            double e[3] = {0.0, 0.0, 0.0};
            e[i] = 1.0;
            skew(e, g.dR[i]);
        }
        return;
    }
    double S[9];
    skew(r, S);
    const double ith2 = 1.0 / th2;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        double w[3] = {-g.R[i], -g.R[3 + i], -g.R[6 + i]};
        w[i] += 1.0;
        const double cr[3] = {r[1] * w[2] - r[2] * w[1], r[2] * w[0] - r[0] * w[2],
                              r[0] * w[1] - r[1] * w[0]};
        double C[9], M[9];
        skew(cr, C);
#pragma unroll
        for (int j = 0; j < 9; ++j) M[j] = (r[i] * S[j] + C[j]) * ith2;
#pragma unroll
        for (int a = 0; a < 3; ++a)
#pragma unroll
            for (int b = 0; b < 3; ++b)
                g.dR[i][3 * a + b] = M[3 * a] * g.R[b] + M[3 * a + 1] * g.R[3 + b] + M[3 * a + 2] * g.R[6 + b];
    }
}

struct SharedIntr {
    double frow, fcol, crow, ccol, k, aspect, inv_cs;
};

// residual (2) and Jacobian rows (2 x 10) of one corner
__device__ __forceinline__ void corner_jac(const ViewGeom& g, const double t[3], const SharedIntr& in,
                                           double X0, double X1, double X2, double obs_r,
                                           double obs_c, double res[2], double J[2][10]) {
    const double q0 = X0 * in.inv_cs, q1 = X1 * in.inv_cs, q2 = X2 * in.inv_cs;
    const double P0 = fma(g.R[1], q1, fma(g.R[0], q0, fma(g.R[2], q2, t[0])));
    const double P1 = fma(g.R[4], q1, fma(g.R[3], q0, fma(g.R[5], q2, t[1])));
    const double P2 = fma(g.R[7], q1, fma(g.R[6], q0, fma(g.R[8], q2, t[2])));
    const double s = 1.0 / P2;
    const double u = P0 * s, v = P1 * s;
    const double r2 = fma(v, v, u * u);
    const double radial = fma(in.k, r2, 1.0);
    const double ud = radial * u, vd = radial * v;
    res[0] = fma(in.frow, ud, in.crow) - obs_r;
    res[1] = fma(in.fcol, vd, in.ccol) - obs_c;
    const double a11 = radial + 2.0 * in.k * u * u, a12 = 2.0 * in.k * u * v;
    const double a22 = radial + 2.0 * in.k * v * v;
    const double du[3] = {s, 0.0, -u * s}, dv[3] = {0.0, s, -v * s};
    double gr[3], gc[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        gr[i] = in.frow * (a11 * du[i] + a12 * dv[i]);
        gc[i] = in.fcol * (a12 * du[i] + a22 * dv[i]);
    }
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        double dP[3];
#pragma unroll
        for (int j = 0; j < 3; ++j)
            dP[j] = g.dR[i][3 * j] * q0 + g.dR[i][3 * j + 1] * q1 + g.dR[i][3 * j + 2] * q2;
        J[0][i] = gr[0] * dP[0] + gr[1] * dP[1] + gr[2] * dP[2];
        J[1][i] = gc[0] * dP[0] + gc[1] * dP[1] + gc[2] * dP[2];
        J[0][3 + i] = gr[i];
        J[1][3 + i] = gc[i];
    }
    J[0][6] = in.aspect * ud; J[1][6] = vd;
    J[0][7] = 1.0;            J[1][7] = 0.0;
    J[0][8] = 0.0;            J[1][8] = 1.0;
    J[0][9] = in.frow * u * r2; J[1][9] = in.fcol * v * r2;
}

// Sum 64 per-lane partials over the warp with a HALVING butterfly: at the step with partner mask m a
// lane keeps one half of its values, sends the other half and adds what its partner sent, so the
// steps move 32 + 16 + 8 + 4 + 2 = 62 doubles instead of 64 x 5 = 320 (the plain xor butterfly of
// round 1 spent 660 SHFLs per view: a quarter of the kernel, ncu round 2).  Afterwards lane l holds
// the warp totals of entries 2l and 2l+1 in v[0], v[1].  Fixed order: bit-reproducible.
template <int N, int MASK>
__device__ __forceinline__ void halve_step(double (&v)[64], bool up) {
#pragma unroll
    for (int i = 0; i < N / 2; ++i) {
        const double keep = up ? v[i + N / 2] : v[i];
        const double send = up ? v[i] : v[i + N / 2];
        v[i] = keep + __shfl_xor_sync(0xffffffffu, send, MASK);
    }
}
__device__ __forceinline__ void warp_sum64(double (&v)[64], int lane_id) {
    halve_step<64, 16>(v, (lane_id & 16) != 0);
    halve_step<32, 8>(v, (lane_id & 8) != 0);
    halve_step<16, 4>(v, (lane_id & 4) != 0);
    halve_step<8, 2>(v, (lane_id & 2) != 0);
    halve_step<4, 1>(v, (lane_id & 1) != 0);
}

// acc layout: [0,21) JtJ_ee upper | [21,45) JtJ_ei | [45,51) Jtr_e | [51,61) JtJ_ii upper |
//             [61,65) Jtr_i | [65] sse
// The Jacobian columns of crow / ccol are the constants (1, 0) / (0, 1): their products are written
// out as additions (or nothing) instead of FMAs with 1.0 / 0.0 -- 108 instead of 132 accumulation
// instructions per corner, same values (x * 1 and x * 0 + acc are exact).
__device__ __forceinline__ void
reproj_jtj_view(const SharedIntr& in, const cc_view* __restrict__ views, int nviews,
                const double* __restrict__ obj, const double* __restrict__ img, int ncorners,
                double* __restrict__ per_view, double* __restrict__ scratch) {
    __shared__ double red[kResWarps][66];
    const int lane_id = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int view = blockIdx.x * kResWarps + warp;
    if (view >= nviews) return;
    double r[3], t[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) { r[i] = views[view].rvec[i]; t[i] = views[view].tvec[i]; }
    ViewGeom g;
    view_geom(r, g);

    double acc[64];            // entries 0..63; 64 (Jtr_i[3]) and 65 (sse) separately
    double acc64 = 0.0, acc65 = 0.0;
#pragma unroll
    for (int i = 0; i < 64; ++i) acc[i] = 0.0;
    int mine = 0;              // corners of this lane: J'J entries (crow,crow) and (ccol,ccol)
    const double2* im = reinterpret_cast<const double2*>(img) + (size_t)view * ncorners;
    for (int ci = lane_id; ci < ncorners; ci += 32) {
        const double2 ob = im[ci];
        const double X0 = __ldg(obj + 3 * ci), X1 = __ldg(obj + 3 * ci + 1), X2 = __ldg(obj + 3 * ci + 2);
        double res[2], J[2][10];
        corner_jac(g, t, in, X0, X1, X2, ob.x, ob.y, res, J);
        ++mine;
#pragma unroll
        for (int rr = 0; rr < 2; ++rr) {
            int k = 0;
#pragma unroll
            for (int a = 0; a < 6; ++a)
#pragma unroll
                for (int b = a; b < 6; ++b) { acc[k] = fma(J[rr][a], J[rr][b], acc[k]); ++k; }
#pragma unroll
            for (int a = 0; a < 6; ++a) {
                acc[21 + 4 * a + 0] = fma(J[rr][a], J[rr][6], acc[21 + 4 * a + 0]);
                acc[21 + 4 * a + 1 + rr] += J[rr][a];                 // column crow (rr = 0) / ccol (rr = 1) is 1
                acc[21 + 4 * a + 3] = fma(J[rr][a], J[rr][9], acc[21 + 4 * a + 3]);
                acc[45 + a] = fma(J[rr][a], res[rr], acc[45 + a]);
            }
            acc[51] = fma(J[rr][6], J[rr][6], acc[51]);               // (f, f)
            acc[52 + rr] += J[rr][6];                                 // (f, crow) / (f, ccol)
            acc[54] = fma(J[rr][6], J[rr][9], acc[54]);               // (f, k)
            if (rr == 0) acc[57] += J[0][9]; else acc[59] += J[1][9]; // (crow, k) / (ccol, k)
            acc[60] = fma(J[rr][9], J[rr][9], acc[60]);               // (k, k)
            acc[61] = fma(J[rr][6], res[rr], acc[61]);
            if (rr == 0) acc[62] += res[0]; else acc[63] += res[1];
            acc64 = fma(J[rr][9], res[rr], acc64);
            acc65 = fma(res[rr], res[rr], acc65);
        }
    }
    acc[55] = acc[58] = (double)mine;                                 // (crow, crow), (ccol, ccol); [56] (crow, ccol) stays 0
    warp_sum64(acc, lane_id);
    acc64 = warp_sum(acc64);
    acc65 = warp_sum(acc65);
    red[warp][2 * lane_id] = acc[0];
    red[warp][2 * lane_id + 1] = acc[1];
    if (lane_id == 0) { red[warp][64] = acc64; red[warp][65] = acc65; }
    __syncwarp();
    const double* rd = red[warp];
    double* pv = per_view + (size_t)view * CC_PER_VIEW;
    for (int idx = lane_id; idx < CC_PER_VIEW; idx += 32) {
        int k;
        if (idx < 36) {
            const int a0 = idx / 6, b0 = idx - 6 * a0, a = min(a0, b0), b = max(a0, b0);
            k = 6 * a - (a * (a - 1)) / 2 + (b - a);
        } else if (idx < 60) {
            k = 21 + (idx - 36);
        } else {
            k = 45 + (idx - 60);
        }
        pv[idx] = rd[k];
    }
    if (lane_id < 21) {
        int k;
        if (lane_id < 16) {
            const int a0 = lane_id >> 2, b0 = lane_id & 3, a = min(a0, b0), b = max(a0, b0);
            k = 51 + 4 * a - (a * (a - 1)) / 2 + (b - a);
        } else {
            k = 61 + (lane_id - 16);
        }
        scratch[(size_t)lane_id * nviews + view] = rd[k];
    }
}

__global__ void __launch_bounds__(kResThreads)
reproj_jtj_kernel(const SharedIntr in, const cc_view* __restrict__ views, int nviews,
                  const double* __restrict__ obj, const double* __restrict__ img, int ncorners,
                  double* __restrict__ per_view, double* __restrict__ scratch) {
    reproj_jtj_view(in, views, nviews, obj, img, ncorners, per_view, scratch);
}

// The same blocks inside the device-resident LM loop (lm.cu): intrinsics and buffers come from
// the loop state -- which == 0: current parameters and buffers; 1: the candidate of the last update.
__global__ void __launch_bounds__(kResThreads)
reproj_jtj_state_kernel(const LmState* __restrict__ st, int which, const LmBufs b, double aspect, double inv_cs,
                        int nviews, const double* __restrict__ obj, const double* __restrict__ img,
                        int ncorners, double* __restrict__ scratch) {
    if (st->done) return;
    const double* p = which ? st->cand : st->par;
    const SharedIntr in{aspect * p[0], p[0], p[1], p[2], p[3], aspect, inv_cs};
    const int slot = st->cur ^ which;
    reproj_jtj_view(in, b.views[slot], nviews, obj, img, ncorners, b.pv[slot], scratch);
}

// out[c] = sum_v parts[c][v] (blockIdx.x = c) in a fixed order: strided serial partials, then a tree.  Inside the
// device-resident LM loop the kernel returns at once when gate->done; gate == nullptr: it always runs.
__global__ void __launch_bounds__(256)
reduce_components_kernel(const LmState* __restrict__ gate, const double* __restrict__ parts, int nviews,
                         double* __restrict__ out) {
    if (gate && gate->done) return;
    __shared__ double sm[256];
    const double* col = parts + (size_t)blockIdx.x * nviews;
    double s = 0.0;
    for (int v = threadIdx.x; v < nviews; v += 256) s += col[v];
    sm[threadIdx.x] = s;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) sm[threadIdx.x] += sm[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) out[blockIdx.x] = sm[0];
}

// ---------------------------------------------------------------------------------
// calculate_errors, src/buildcalibrations.jl:37-67: per view the four raw sums
//   reprojection :29-30,44 | projection :46-47 | distance :49-51 | inverse :53-58
// One warp per view; projected world points are staged in shared memory for the
// adjacent-corner differences.
// ---------------------------------------------------------------------------------
__global__ void __launch_bounds__(kResThreads)
calc_errors_kernel(const cc_intr intr, const cc_view* __restrict__ views, int nviews,
                   const double* __restrict__ obj, const double* __restrict__ img, int n1, int n2,
                   const double* __restrict__ inv_rows, const double* __restrict__ inv_cols,
                   int inverse_samples, double* __restrict__ scratch) {
    extern __shared__ double proj_sm[];           // [kResWarps][ncorners*3]
    const int lane_id = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int view = blockIdx.x * kResWarps + warp;
    if (view >= nviews) return;
    const int nc = n1 * n2;
    double* pw = proj_sm + (size_t)warp * nc * 3;

    // expand the chain on the device (views live in device memory here)
    ChainD ch;
    double r[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) { r[i] = views[view].rvec[i]; ch.t[i] = views[view].tvec[i]; }
    rodrigues(r, ch.R);
    complete_chain(intr, ch);

    double s_rep = 0.0, s_pro = 0.0, s_dis = 0.0, s_inv = 0.0;
    const double2* im = reinterpret_cast<const double2*>(img) + (size_t)view * nc;
    for (int ci = lane_id; ci < nc; ci += 32) {
        const double2 ob = im[ci];
        const double X0 = __ldg(obj + 3 * ci), X1 = __ldg(obj + 3 * ci + 1), X2 = __ldg(obj + 3 * ci + 2);
        double row, col;
        world2img(ch, X0, X1, X2, row, col);
        const double dr = row - ob.x, dc = col - ob.y;
        s_rep += dr * dr + dc * dc;
        double x, y, z;
        img2world(ch, ob.x, ob.y, x, y, z);
        pw[3 * ci] = x; pw[3 * ci + 1] = y; pw[3 * ci + 2] = z;
        const double ex = x - X0, ey = y - X1, ez = z - X2;
        s_pro += ex * ex + ey * ey + ez * ez;
    }
    __syncwarp();
    for (int ci = lane_id; ci < nc; ci += 32) {
        const int a = ci % n1, b = ci / n1;
        const double* p0 = pw + 3 * ci;
        if (a + 1 < n1) {
            const double* p1 = p0 + 3;
            const double e = sqrt((p1[0] - p0[0]) * (p1[0] - p0[0]) + (p1[1] - p0[1]) * (p1[1] - p0[1]) +
                                  (p1[2] - p0[2]) * (p1[2] - p0[2])) - intr.checker_size;
            s_dis += e * e;
        }
        if (b + 1 < n2) {
            const double* p1 = p0 + 3 * n1;
            const double e = sqrt((p1[0] - p0[0]) * (p1[0] - p0[0]) + (p1[1] - p0[1]) * (p1[1] - p0[1]) +
                                  (p1[2] - p0[2]) * (p1[2] - p0[2])) - intr.checker_size;
            s_dis += e * e;
        }
    }
    for (int si = lane_id; si < inverse_samples; si += 32) {
        const double r0 = inv_rows[(size_t)view * inverse_samples + si];
        const double c0 = inv_cols[(size_t)view * inverse_samples + si];
        double x, y, z, r1, c1;
        img2world(ch, r0, c0, x, y, z);
        world2img(ch, x, y, z, r1, c1);
        s_inv += (r0 - r1) * (r0 - r1) + (c0 - c1) * (c0 - c1);
    }
    s_rep = warp_sum(s_rep); s_pro = warp_sum(s_pro);
    s_dis = warp_sum(s_dis); s_inv = warp_sum(s_inv);
    if (lane_id == 0) {
        scratch[view] = s_rep;
        scratch[(size_t)nviews + view] = s_pro;
        scratch[(size_t)2 * nviews + view] = s_dis;
        scratch[(size_t)3 * nviews + view] = s_inv;
    }
}

cudaError_t ScratchHold::record() {
    cudaError_t e = ctx_->scratch_event ? cudaSuccess : cudaEventCreateWithFlags(&ctx_->scratch_event,
                                                                                  cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventRecord(ctx_->scratch_event, st_);
    if (e == cudaSuccess) { ctx_->scratch_stream = st_; ctx_->scratch_used = 1; }
    return e;
}
int ScratchHold::acquire(size_t elems) {
    if (ctx_->scratch_used && ctx_->scratch_stream != st_ && ctx_->scratch_event)
        CC_CUDA(cudaStreamWaitEvent(st_, ctx_->scratch_event, 0));
    held_ = true;
    if (ctx_->jtj_scratch_elems >= elems) return CC_OK;
    if (ctx_->jtj_scratch) { CC_CUDA(cudaFree(ctx_->jtj_scratch)); ctx_->jtj_scratch = nullptr; }
    ctx_->jtj_scratch_elems = 0;
    CC_CUDA(cudaMalloc(&ctx_->jtj_scratch, elems * sizeof(double)));
    ctx_->jtj_scratch_elems = elems;
    return CC_OK;
}
int ScratchHold::release() {
    held_ = false;
    const cudaError_t e = record();
    return e == cudaSuccess ? CC_OK : cuda_fail(e, "scratch event");
}

int launch_reduce(cc_ctx* ctx, const LmState* gate, const double* parts, int ncomp, int nviews, double* out,
                  cudaStream_t st) {
    reduce_components_kernel<<<ncomp, 256, 0, st>>>(gate, parts, nviews, out);
    ctx->launches++;
    CC_CUDA(cudaGetLastError());
    return CC_OK;
}

int launch_reproj_jtj(cc_ctx* ctx, const cc_intr* intr, double aspect, const cc_view* views,
                      int nviews, const double* obj, const double* img, int ncorners,
                      double* per_view, double* shared, cudaStream_t st) {
    ScratchHold hold(ctx, st);
    int rc = hold.acquire((size_t)CC_SHARED * (size_t)(nviews > 0 ? nviews : 1));
    if (rc) return rc;
    if (nviews > 0) {
        SharedIntr in{intr->frow, intr->fcol, intr->crow, intr->ccol, intr->k, aspect,
                      1.0 / intr->checker_size};
        reproj_jtj_kernel<<<(nviews + kResWarps - 1) / kResWarps, kResThreads, 0, st>>>(
            in, views, nviews, obj, img, ncorners, per_view, ctx->jtj_scratch);
        ctx->launches++;
        CC_CUDA(cudaGetLastError());
    }
    if ((rc = launch_reduce(ctx, nullptr, ctx->jtj_scratch, CC_SHARED, nviews, shared, st))) return rc;
    return hold.release();
}

int launch_reproj_jtj_state(cc_ctx* ctx, const LmState* st, int which, const LmBufs& b, double aspect,
                            double checker_size, int nviews, const double* obj, const double* img,
                            int ncorners, double* shared_out, cudaStream_t stream) {
    ScratchHold hold(ctx, stream);
    int rc = hold.acquire((size_t)CC_SHARED * (size_t)(nviews > 0 ? nviews : 1));
    if (rc) return rc;
    if (nviews > 0) {
        reproj_jtj_state_kernel<<<(nviews + kResWarps - 1) / kResWarps, kResThreads, 0, stream>>>(
            st, which, b, aspect, 1.0 / checker_size, nviews, obj, img, ncorners, ctx->jtj_scratch);
        ctx->launches++;
        CC_CUDA(cudaGetLastError());
    }
    if ((rc = launch_reduce(ctx, st, ctx->jtj_scratch, CC_SHARED, nviews, shared_out, stream))) return rc;
    return hold.release();
}

size_t calc_errors_smem(int n1, int n2) { return (size_t)kResWarps * n1 * n2 * 3 * sizeof(double); }

int launch_calc_errors(cc_ctx* ctx, const cc_intr* intr, const cc_view* views, int nviews,
                       const double* obj, const double* img, int n1, int n2, const double* inv_rows,
                       const double* inv_cols, int inverse_samples, double* sums, cudaStream_t st) {
    const size_t smem = calc_errors_smem(n1, n2);
    ScratchHold hold(ctx, st);
    int rc = hold.acquire((size_t)CC_SHARED * (size_t)(nviews > 0 ? nviews : 1));
    if (rc) return rc;
    if (nviews > 0) {
        if (smem > 48 * 1024)
            CC_CUDA(cudaFuncSetAttribute(calc_errors_kernel,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        calc_errors_kernel<<<(nviews + kResWarps - 1) / kResWarps, kResThreads, smem, st>>>(
            *intr, views, nviews, obj, img, n1, n2, inv_rows, inv_cols, inverse_samples,
            ctx->jtj_scratch);
        ctx->launches++;
        CC_CUDA(cudaGetLastError());
    }
    if ((rc = launch_reduce(ctx, nullptr, ctx->jtj_scratch, 4, nviews, sums, st))) return rc;
    return hold.release();
}

}  // namespace cc
