// Low-rank (Burer-Monteiro) solve of max-cut-type SDPs (an extension: the reference has no low-rank path).
//
//   min C . X  s.t.  X_ii = b_i (b_i > 0),  X >= 0,   with X = V V^T, V n x r (row-major, row i = v_i).
//
// The block-coordinate "mixing" update minimizes C . V V^T over v_i on the sphere ||v_i||^2 = b_i with the other rows
// fixed: v_i <- -sqrt(b_i) w_i / ||w_i||, w_i = sum_{j != i} C_ij v_j.  Vertices of one colour of a proper colouring of
// C's off-diagonal pattern are not adjacent, so updating a whole colour at once is the sequential method in colour order
// and the objective never rises (up to rounding).
//  * Rows: the CSR of the one-flip search (ls_rows_upload): off-diagonal entries of C from both triangles, increasing
//    columns, duplicates summed in input order.  Colouring: greedy in increasing vertex index (vertex i takes the
//    smallest colour none of its lower-index neighbours has), on the host; within a colour, vertices ascend.
//  * Start: row i of V_0 is sample i of round_normal_kernel with n = r (ldb = r), scaled to norm sqrt(b_i).
//  * w_i is summed in row order one component at a time with separately rounded products and sums (__dmul_rn /
//    __dadd_rn: no FMA contraction), so a NumPy restatement reproduces the bits.  A row norm or dot product of a warp:
//    lane l sums components l, l + 32, ... in order, then an xor butterfly over offsets 16, 8, 4, 2, 1.
//  * Objective f = sum_i e_i with e_i = C_ii b_i + <v_i, w_i>: per-vertex terms, partial sums of LR_OBJ_VB consecutive
//    vertices in vertex order, then the partials in order.  Evaluated at the start (f_0) and after every sweep.  The run
//    stops after the first sweep k with f_{k-1} - f_k <= tol max(1, |f_k|), or after max_sweeps sweeps; then
//    y_i = e_i / b_i (at a stationary point (C - Diag(y)) V = 0).
//  * The host enqueues LR_GROUP sweeps at a time and reads the stop flag once per group.  Every kernel of a sweep or an
//    evaluation first reads that flag (set by the evaluation that stops the run) and returns at once when it is set, so
//    the results do not depend on the group size.
#include "internal.cuh"
#include <algorithm>
#include <chrono>
#include <cmath>

#define LR_MAX_RANK 512      // w lives in registers: up to 16 doubles per lane
#define LR_WARPS 8           // warps per block of the sweep and start kernels
#define LR_OBJ_VB 64         // vertices per block of the objective
#define LR_GROUP 16          // sweeps enqueued between two reads of the stop flag

struct LrState {
    int done;                // the run has stopped: every later kernel returns at once
    int converged;           // the stopping criterion held
    long long sweeps;
};

__device__ __forceinline__ double lr_warp_sum(double s) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s = __dadd_rn(s, __shfl_xor_sync(0xffffffffu, s, o));
    return s;
}

// lane's components q (32 q + lane < r) of w_i = sum_{j != i} C_ij v_j, in row order
template <int NQ>
__device__ __forceinline__ void lr_w(int i, int r, int lane, const long long *__restrict__ rp, const int *__restrict__ col,
                                     const double *__restrict__ val, const double *V, double (&w)[NQ]) {
#pragma unroll
    for (int q = 0; q < NQ; ++q) w[q] = 0.0;
    for (long long p = rp[i]; p < rp[i + 1]; ++p) {
        const double c = val[p];
        const double *vj = V + (long long)col[p] * r + lane;
#pragma unroll
        for (int q = 0; q < NQ; ++q)
            if (32 * q + lane < r) w[q] = __dadd_rn(w[q], __dmul_rn(c, vj[32 * q]));
    }
}

// start: row i <- (sqrt(b_i) / ||v_i||) v_i, one warp per vertex
template <int NQ>
__global__ void __launch_bounds__(32 * LR_WARPS) lowrank_start_kernel(int n, int r, const double *__restrict__ sb, double *V) {
    const int lane = threadIdx.x & 31;
    const int i = blockIdx.x * LR_WARPS + (threadIdx.x >> 5);
    if (i >= n) return;
    double *vi = V + (long long)i * r + lane;
    double v[NQ], ss = 0.0;
#pragma unroll
    for (int q = 0; q < NQ; ++q) {
        v[q] = 32 * q + lane < r ? vi[32 * q] : 0.0;
        if (32 * q + lane < r) ss = __dadd_rn(ss, __dmul_rn(v[q], v[q]));
    }
    ss = lr_warp_sum(ss);
    if (!(ss > 0.0)) return;
    const double a = sb[i] / sqrt(ss);
#pragma unroll
    for (int q = 0; q < NQ; ++q)
        if (32 * q + lane < r) vi[32 * q] = __dmul_rn(a, v[q]);
}

// one colour of a sweep: the cnt vertices verts[0 .. cnt), one warp each, v_i <- (-sqrt(b_i) / ||w_i||) w_i when w_i != 0.
// No vertex of the colour is a neighbour of another, so no warp reads a row that another writes.
template <int NQ>
__global__ void __launch_bounds__(32 * LR_WARPS) lowrank_sweep_kernel(const LrState *st, const int *__restrict__ verts, int cnt,
                                                                      int r, const long long *__restrict__ rp,
                                                                      const int *__restrict__ col, const double *__restrict__ val,
                                                                      const double *__restrict__ sb, double *V) {
    if (st->done) return;
    const int lane = threadIdx.x & 31;
    const int g = blockIdx.x * LR_WARPS + (threadIdx.x >> 5);
    if (g >= cnt) return;
    const int i = verts[g];
    double w[NQ];
    lr_w<NQ>(i, r, lane, rp, col, val, V, w);
    double ss = 0.0;
#pragma unroll
    for (int q = 0; q < NQ; ++q)
        if (32 * q + lane < r) ss = __dadd_rn(ss, __dmul_rn(w[q], w[q]));
    ss = lr_warp_sum(ss);
    if (!(ss > 0.0)) return;
    const double a = -sb[i] / sqrt(ss);
    double *vi = V + (long long)i * r + lane;
#pragma unroll
    for (int q = 0; q < NQ; ++q)
        if (32 * q + lane < r) vi[32 * q] = __dmul_rn(a, w[q]);
}

// e_i = C_ii b_i + <v_i, w_i> of the LR_OBJ_VB vertices of the block and their sum in vertex order into part[blockIdx.x]
template <int NQ>
__global__ void __launch_bounds__(32 * LR_WARPS) lowrank_obj_kernel(const LrState *st, int n, int r, const long long *__restrict__ rp,
                                                                    const int *__restrict__ col, const double *__restrict__ val,
                                                                    const double *__restrict__ cd, const double *__restrict__ b,
                                                                    const double *V, double *__restrict__ e,
                                                                    double *__restrict__ part) {
    if (st->done) return;
    __shared__ double se[LR_OBJ_VB];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int i0 = blockIdx.x * LR_OBJ_VB, cnt = min(LR_OBJ_VB, n - i0);
    for (int k = warp; k < cnt; k += LR_WARPS) {
        const int i = i0 + k;
        double w[NQ];
        lr_w<NQ>(i, r, lane, rp, col, val, V, w);
        const double *vi = V + (long long)i * r + lane;
        double d = 0.0;
#pragma unroll
        for (int q = 0; q < NQ; ++q)
            if (32 * q + lane < r) d = __dadd_rn(d, __dmul_rn(vi[32 * q], w[q]));
        d = lr_warp_sum(d);
        if (lane == 0) {
            const double ei = __dadd_rn(__dmul_rn(cd[i], b[i]), d);
            se[k] = ei;
            e[i] = ei;
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int k = 0; k < cnt; ++k) s = __dadd_rn(s, se[k]);
        part[blockIdx.x] = s;
    }
}

// f_k = sum of the nb partials in order into fh[k]; stops the run when the criterion holds or k = max_sweeps, and then
// writes y = e / b.  One block.
__global__ void lowrank_sum_kernel(LrState *st, int nb, const double *__restrict__ part, long long k, long long max_sweeps,
                                   double tol, double *fh, int n, const double *__restrict__ e, const double *__restrict__ b,
                                   double *__restrict__ y) {
    __shared__ int fin;
    if (st->done) return;
    if (threadIdx.x == 0) {
        double f = 0.0;
        for (int p = 0; p < nb; ++p) f = __dadd_rn(f, part[p]);
        fh[k] = f;
        const bool conv = k > 0 && __dsub_rn(fh[k - 1], f) <= __dmul_rn(tol, fmax(1.0, fabs(f)));
        fin = conv || k >= max_sweeps;
        if (fin) {
            st->converged = conv;
            st->sweeps = k;
        }
    }
    __syncthreads();
    if (!fin) return;
    for (int i = threadIdx.x; i < n; i += blockDim.x) y[i] = e[i] / b[i];
    __syncthreads();
    if (threadIdx.x == 0) st->done = 1;
}

// the kernel instance for NQ = ceil(r / 32)
#define LR_DISPATCH(NQ_, CALL)                                                                                               \
    switch (NQ_) {                                                                                                           \
    case 1: CALL(1); break;   case 2: CALL(2); break;   case 3: CALL(3); break;   case 4: CALL(4); break;                    \
    case 5: CALL(5); break;   case 6: CALL(6); break;   case 7: CALL(7); break;   case 8: CALL(8); break;                    \
    case 9: CALL(9); break;   case 10: CALL(10); break; case 11: CALL(11); break; case 12: CALL(12); break;                  \
    case 13: CALL(13); break; case 14: CALL(14); break; case 15: CALL(15); break; default: CALL(16); break;                  \
    }

// greedy colouring in increasing vertex index of the CSR pattern; returns the number of colours, colour[i] per vertex
static int lowrank_colour(int n, const LsRowsHost &h, std::vector<int> &colour) {
    colour.assign((size_t)n, 0);
    std::vector<int> mark;              // mark[c] == i: colour c is taken by a lower-index neighbour of i
    int nc = 0;
    for (int i = 0; i < n; ++i) {
        for (long long p = h.rp[i]; p < h.rp[i + 1]; ++p) {
            const int j = h.col[p];
            if (j >= i) break;          // columns ascend
            if ((size_t)colour[j] >= mark.size()) mark.resize((size_t)colour[j] + 1, -1);
            mark[colour[j]] = i;
        }
        int c = 0;
        while ((size_t)c < mark.size() && mark[c] == i) ++c;
        colour[i] = c;
        nc = std::max(nc, c + 1);
    }
    return nc;
}

int k_lowrank_solve(smcp_ctx *ctx, int64_t n, int64_t r, int64_t nc, const int64_t *crow, const int64_t *ccol, const double *cval,
                    const double *b, uint64_t seed, int64_t max_sweeps, double tol, double *V_host, double *f_host, double *y_host,
                    int64_t *sweeps_out, int64_t *colors_out) {
    const char *fn = "smcp_lowrank_solve";
    if (n < 1 || n > INT32_MAX || r < 1 || r > LR_MAX_RANK || nc < 0 || max_sweeps < 0 || !(tol >= 0.0) || !std::isfinite(tol)) {
        smcp_set_error("%s: need 1 <= n < 2^31, 1 <= r <= %d, nc >= 0, max_sweeps >= 0 and a finite tol >= 0 "
                       "(got %lld, %lld, %lld, %lld, %g)", fn, LR_MAX_RANK, (long long)n, (long long)r, (long long)nc,
                       (long long)max_sweeps, tol);
        return -2;
    }
    if (!b || !V_host || !f_host || !y_host || !sweeps_out || !colors_out || (nc > 0 && (!crow || !ccol || !cval))) {
        smcp_set_error("%s: null argument", fn);
        return -2;
    }
    for (int64_t i = 0; i < n; ++i)
        if (!(b[i] > 0.0) || !std::isfinite(b[i])) {
            smcp_set_error("%s: b[%lld] = %g is not finite and positive", fn, (long long)i, b[i]);
            return -2;
        }
    for (int64_t q = 0; q < nc; ++q)
        if (crow[q] < 0 || crow[q] >= n || ccol[q] < 0 || ccol[q] >= n) {
            smcp_set_error("%s: objective entry %lld at (%lld, %lld) is outside 0..%lld", fn, (long long)q, (long long)crow[q],
                           (long long)ccol[q], (long long)n - 1);
            return -2;
        }
    CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const int N = (int)n, R = (int)r, NQ = (R + 31) / 32;
    RoundWs ws{ctx, fn, {}};
    LsRows d;
    LsRowsHost h;
    if (ls_rows_upload(ws, N, nc, crow, ccol, cval, 0.0, d, &h)) return -1;

    // colours (host time recorded as the region "lowrank_colour_host"), then the vertices by colour, ascending within
    const auto c0 = std::chrono::steady_clock::now();
    std::vector<int> colour;
    const int ncol = lowrank_colour(N, h, colour);
    std::vector<int> cptr((size_t)ncol + 1, 0), verts((size_t)N);
    for (int i = 0; i < N; ++i) ++cptr[colour[i] + 1];
    for (int c = 0; c < ncol; ++c) cptr[c + 1] += cptr[c];
    {
        std::vector<int> fill(cptr.begin(), cptr.end() - 1);
        for (int i = 0; i < N; ++i) verts[fill[colour[i]]++] = i;
    }
    RegionAcc &cacc = ctx->regions["lowrank_colour_host"];
    cacc.ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - c0).count();
    cacc.calls += 1;

    std::vector<double> cd((size_t)N, 0.0), sb((size_t)N);
    for (int64_t q = 0; q < nc; ++q)
        if (crow[q] == ccol[q]) cd[crow[q]] += cval[q];
    for (int i = 0; i < N; ++i) sb[i] = std::sqrt(b[i]);
    const int nb = (N + LR_OBJ_VB - 1) / LR_OBJ_VB;
    double *V = (double *)ws.alloc((size_t)N * R * sizeof(double));
    double *dcd = (double *)ws.alloc((size_t)N * sizeof(double));
    double *db = (double *)ws.alloc((size_t)N * sizeof(double));
    double *dsb = (double *)ws.alloc((size_t)N * sizeof(double));
    double *e = (double *)ws.alloc((size_t)N * sizeof(double));
    double *y = (double *)ws.alloc((size_t)N * sizeof(double));
    double *part = (double *)ws.alloc((size_t)nb * sizeof(double));
    double *fh = (double *)ws.alloc((size_t)(max_sweeps + 1) * sizeof(double));
    int *dverts = (int *)ws.alloc((size_t)N * sizeof(int));
    LrState *state = (LrState *)ws.alloc(sizeof(LrState));
    if (!V || !dcd || !db || !dsb || !e || !y || !part || !fh || !dverts || !state) return -1;
    CUDA_TRY(cudaMemcpyAsync(dcd, cd.data(), (size_t)N * sizeof(double), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(db, b, (size_t)N * sizeof(double), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(dsb, sb.data(), (size_t)N * sizeof(double), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(dverts, verts.data(), (size_t)N * sizeof(int), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemsetAsync(state, 0, sizeof(LrState), st));

    if (launch_round_normals(ctx, seed, 0, R, V, R, n)) return -1;
    const unsigned vgrid = (unsigned)((N + LR_WARPS - 1) / LR_WARPS);
    {
        LaunchScope ls(ctx, "lowrank_sweep");
#define LR_START(Q) lowrank_start_kernel<Q><<<vgrid, 32 * LR_WARPS, 0, st>>>(N, R, dsb, V)
        LR_DISPATCH(NQ, LR_START)
#undef LR_START
    }
    CUDA_TRY(cudaGetLastError());
    // evaluation k: f_k, the stopping test and, when the run stops, y
    auto evaluate = [&](long long k) -> int {
        LaunchScope ls(ctx, "lowrank_obj", 2);
#define LR_OBJ(Q) lowrank_obj_kernel<Q><<<(unsigned)nb, 32 * LR_WARPS, 0, st>>>(state, N, R, d.rp, d.col, d.val, dcd, db, V, e, part)
        LR_DISPATCH(NQ, LR_OBJ)
#undef LR_OBJ
        lowrank_sum_kernel<<<1, 256, 0, st>>>(state, nb, part, k, (long long)max_sweeps, tol, fh, N, e, db, y);
        CUDA_TRY(cudaGetLastError());
        return 0;
    };
    LrState hs{0, 0, 0};
    {
        RegionScope rs(ctx, "lowrank_loop");
        if (evaluate(0)) return -1;
        for (long long k0 = 1; k0 <= max_sweeps; k0 += LR_GROUP) {
            const long long k1 = std::min<long long>(max_sweeps, k0 + LR_GROUP - 1);
            for (long long k = k0; k <= k1; ++k) {
                for (int c = 0; c < ncol; ++c) {
                    const int cnt = cptr[c + 1] - cptr[c];
                    const unsigned grid = (unsigned)((cnt + LR_WARPS - 1) / LR_WARPS);
                    LaunchScope ls(ctx, "lowrank_sweep");
#define LR_SWEEP(Q) lowrank_sweep_kernel<Q><<<grid, 32 * LR_WARPS, 0, st>>>(state, dverts + cptr[c], cnt, R, d.rp, d.col, d.val, dsb, V)
                    LR_DISPATCH(NQ, LR_SWEEP)
#undef LR_SWEEP
                }
                CUDA_TRY(cudaGetLastError());
                if (evaluate(k)) return -1;
            }
            CUDA_TRY(cudaMemcpyAsync(&hs, state, sizeof(hs), cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaStreamSynchronize(st));
            if (hs.done) break;
        }
    }
    CUDA_TRY(cudaMemcpyAsync(&hs, state, sizeof(hs), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (!hs.done) {
        smcp_set_error("%s: the run did not stop after %lld sweeps", fn, (long long)max_sweeps);
        return -1;
    }
    CUDA_TRY(cudaMemcpyAsync(V_host, V, (size_t)N * R * sizeof(double), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(f_host, fh, (size_t)(hs.sweeps + 1) * sizeof(double), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(y_host, y, (size_t)N * sizeof(double), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    *sweeps_out = hs.sweeps;
    *colors_out = ncol;
    return 0;
}
