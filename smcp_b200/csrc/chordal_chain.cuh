// Segment-parallel kernels for CHAIN clique trees with single-column supernodes (band SDPs:
// the benchmark's n = 5000, bandwidth 5 pattern is a chain of 4994 blocks of 6 x 1 plus a
// 6 x 6 root).  Included by chordal_small.cu.
//
// Why.  On a chain the level schedule has no parallelism at all: every recursion of the
// barrier Hessian (chompack.hessian, reference call sites src/python/solvers.py:483, 524, 531,
// 405) is a 5000-step sequential recurrence, ~0.5 us per step for one warp, and a single
// Hessian costs milliseconds no matter how few flops it has.  But both sweeps of the Hessian
// are LINEAR recurrences whose coefficients depend only on the scaling point (L):
//     up   (App. A.4 step 1):  U_k  = F_aa - Lt F_an^T - K_an Lt^T,   F = block_k + shift(U_{k-1})
//     down (App. A.4 step 3):  Z_an = M_an - Z_aa Lt,  Z_nn = M_nn - Lt^T (M_an + Z_an)
// so the chain is cut into P segments of SEG nodes and every sweep becomes
//   (1) PROBE : one THREAD per (matrix, segment) runs its segment with zero incoming state
//               and keeps only the outgoing state g_s                      (all in parallel)
//   (2) SCAN  : b_{s+1} = g_s + Phi_s b_s over the P boundaries, Phi_s = the D x D propagator
//               of segment s (D = W(W+1)/2 entries of the symmetric W x W state), computed
//               once per scaling point by running the same recurrence on unit states
//   (3) FINAL : every (matrix, segment) thread reruns its segment from the true incoming
//               state b_s and writes the result in place                   (all in parallel)
// Latency drops from N steps to 2*SEG steps + P tiny mat-vecs, and a batch of B matrices
// exposes B*P independent threads instead of B warps.  Inside a segment the arithmetic is
// the sequential recurrence itself; only the D boundary values go through the superposition
// (Phi_s is a contraction for positive definite scaling points — products of the entries of
// L_an L_nn^{-1} — measured difference to the sequential sweep <= 1e-10 relative at
// cond(S) = 5e11, see DESIGN.md).  Sums are formed in a fixed order: bitwise reproducible.
//
// The inverse Hessian and llt need no recurrence at all on a chain: the update matrix of a
// node leaves the front after W steps, so every entry of the result is a sum of at most W+1
// local-front entries (chain_add_kernel).
#pragma once

struct ChainArgs {
    int N, P, SEG, B, D;
    long long nblk;            // stride between the matrices of a batch
    double *X;                 // B x nblk
    const double *Lt;          // factor: [l0, lt_1..lt_W] per node
    double *state;             // B x P x D : probe writes g_s, scan turns it into b_s, final reads b_s
    double *phi;               // P x D x (D+1): phi[(s*D + c)*(D+1) + r] = d state_out[r] / d state_in[c]
    const double *F;           // add kernel: B x nsq local fronts
    long long nsq;
    int root_off, root_nj, root_sq;
    const double *Yaa;         // up-final: fused Hessian scaling (Y_aa per node, W x W)
    double *psi;               // two-level scan: G x D x (D+1) group propagators
    int G, gs;                 // groups of gs consecutive boundaries
};

enum { CH_PROBE = 0, CH_FINAL = 1, CH_BASIS = 2 };

#define TRI(p, q) ((p) * ((p) + 1) / 2 + (q))

__device__ __forceinline__ void chain_cp_async8(void *smem, const void *gmem) {
    unsigned sa = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(sa), "l"(gmem));
}

// PF = how many nodes ahead the block / factor entries are fetched: 4 for the propagators (one thread per
// (segment, basis vector) straight from global memory), 1 for the staged kernels (entries in shared memory).
// One segment of the up sweep for matrix / basis vector b.  x, l and yaa are indexed by the ABSOLUTE
// node number: global arrays, or shared-memory copies of the segment shifted by its first node.
template <int W, int MODE, int PF>
__device__ __forceinline__ void chain_up_body(const ChainArgs &a, const int s, const int b, double *x, const double *l, const double *yaa) {
    constexpr int D = W * (W + 1) / 2, NJ = W + 1;
    double u[W][W];
#pragma unroll
    for (int p = 0; p < W; ++p)
#pragma unroll
        for (int q = 0; q <= p; ++q) {
            if (MODE == CH_PROBE) u[p][q] = 0.0;
            else if (MODE == CH_FINAL) u[p][q] = a.state[((long long)b * a.P + s) * D + TRI(p, q)];
            else u[p][q] = (TRI(p, q) == b) ? 1.0 : 0.0;
        }
    const int k0 = s * a.SEG, k1 = min(a.N, k0 + a.SEG);
    double xb[PF][NJ], lb[PF][W];
#pragma unroll
    for (int t = 0; t < PF; ++t) {
        const bool in = k0 + t < k1;
#pragma unroll
        for (int i = 0; i < NJ; ++i) xb[t][i] = (MODE != CH_BASIS && in) ? x[(long long)(k0 + t) * NJ + i] : 0.0;
#pragma unroll
        for (int i = 0; i < W; ++i) lb[t][i] = in ? l[(long long)(k0 + t) * NJ + 1 + i] : 0.0;
    }
    for (int kk = k0; kk < k1; kk += PF) {
#pragma unroll
        for (int t = 0; t < PF; ++t) {
            const int k = kk + t;
            if (k < k1) {
                double xv[NJ], lt[W];
#pragma unroll
                for (int i = 0; i < NJ; ++i) xv[i] = xb[t][i];
#pragma unroll
                for (int i = 0; i < W; ++i) lt[i] = lb[t][i];
                if (k + PF < k1) {
#pragma unroll
                    for (int i = 0; i < NJ; ++i) xb[t][i] = (MODE != CH_BASIS) ? x[(long long)(k + PF) * NJ + i] : 0.0;
#pragma unroll
                    for (int i = 0; i < W; ++i) lb[t][i] = l[(long long)(k + PF) * NJ + 1 + i];
                }
                const double f0 = xv[0] + u[0][0];
                double fa[W], ka[W];
#pragma unroll
                for (int i = 0; i < W; ++i) {
                    fa[i] = (i + 1 < W) ? xv[1 + i] + u[i + 1][0] : xv[1 + i];
                    ka[i] = fma(-lt[i], f0, fa[i]);
                }
                double un[W][W];
#pragma unroll
                for (int i = 0; i < W; ++i)
#pragma unroll
                    for (int j = 0; j <= i; ++j) {
                        const double faa = (i + 1 < W) ? u[i + 1][j + 1] : 0.0;
                        un[i][j] = fma(-ka[i], lt[j], fma(-lt[i], fa[j], faa));
                    }
                if (MODE == CH_FINAL) {
                    double *o = x + (long long)k * NJ;
                    if (yaa) {
                        // fused scaling (App. A.4 step 2, single-column supernode):
                        // M_nn = K_nn / l^4, M_an = Y_aa (K_an / l^2)
                        const double l0 = l[(long long)k * NJ];
                        const double *yp = yaa + (long long)k * W * W;
                        const double inv = 1.0 / (l0 * l0);
                        double kv[W];
#pragma unroll
                        for (int i = 0; i < W; ++i) kv[i] = ka[i] * inv;
                        o[0] = f0 * inv * inv;
#pragma unroll
                        for (int r = 0; r < W; ++r) {
                            double acc = 0.0;
#pragma unroll
                            for (int c = 0; c < W; ++c) acc = fma(yp[r + c * W], kv[c], acc);
                            o[1 + r] = acc;
                        }
                    } else {
                        o[0] = f0;
#pragma unroll
                        for (int i = 0; i < W; ++i) o[1 + i] = ka[i];
                    }
                }
#pragma unroll
                for (int i = 0; i < W; ++i)
#pragma unroll
                    for (int j = 0; j <= i; ++j) u[i][j] = un[i][j];
            }
        }
    }
    if (MODE == CH_PROBE) {
        double *g = a.state + ((long long)b * a.P + s) * D;
#pragma unroll
        for (int p = 0; p < W; ++p)
#pragma unroll
            for (int q = 0; q <= p; ++q) g[TRI(p, q)] = u[p][q];
    } else if (MODE == CH_BASIS) {
        double *g = a.phi + ((long long)s * D + b) * (D + 1);
#pragma unroll
        for (int p = 0; p < W; ++p)
#pragma unroll
            for (int q = 0; q <= p; ++q) g[TRI(p, q)] = u[p][q];
    }
}

// propagators Phi_s of the up sweep: one thread per (segment, basis vector)
template <int W>
__global__ void __launch_bounds__(128) chain_up_kernel(ChainArgs a) {
    constexpr int D = W * (W + 1) / 2;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int s = (int)(idx / D), b = (int)(idx - (long long)s * D);
    if (s >= a.P) return;
    chain_up_body<W, CH_BASIS, 4>(a, s, b, a.X + (long long)b * a.nblk, a.Lt, a.Yaa);
}

// Few matrices (Newton solves, line-search steps): one WARP per (segment, matrix) copies the
// segment's entries of X, L (and Y_aa for the fused scaling) into shared memory with coalesced
// loads -- one round trip to memory instead of one per node --, lane 0 runs the recurrence on
// the copies, and the warp writes the segment back.  (Thread-per-segment straight from global
// memory paid ~4 us per node: 129 us for the 32-node final pass of one matrix.)
#define CHAIN_SEG 32
template <int W, int MODE, bool UP>
__global__ void __launch_bounds__(128) chain_staged_kernel(ChainArgs a);

template <int W, int MODE, int PF>
__device__ __forceinline__ void chain_down_body(const ChainArgs &a, const int s, const int b, double *x, const double *l) {
    constexpr int D = W * (W + 1) / 2, NJ = W + 1;
    double z[W][W];
#pragma unroll
    for (int p = 0; p < W; ++p)
#pragma unroll
        for (int q = 0; q <= p; ++q) {
            if (MODE == CH_PROBE) z[p][q] = 0.0;
            else if (MODE == CH_FINAL) z[p][q] = a.state[((long long)b * a.P + s) * D + TRI(p, q)];
            else z[p][q] = (TRI(p, q) == b) ? 1.0 : 0.0;
        }
    const int k0 = s * a.SEG, k1 = min(a.N, k0 + a.SEG);
    double xb[PF][NJ], lb[PF][W];
#pragma unroll
    for (int t = 0; t < PF; ++t) {
        const bool in = k1 - 1 - t >= k0;
#pragma unroll
        for (int i = 0; i < NJ; ++i) xb[t][i] = (MODE != CH_BASIS && in) ? x[(long long)(k1 - 1 - t) * NJ + i] : 0.0;
#pragma unroll
        for (int i = 0; i < W; ++i) lb[t][i] = in ? l[(long long)(k1 - 1 - t) * NJ + 1 + i] : 0.0;
    }
    for (int kk = k1 - 1; kk >= k0; kk -= PF) {
#pragma unroll
        for (int t = 0; t < PF; ++t) {
            const int k = kk - t;
            if (k >= k0) {
                double m[NJ], lt[W];
#pragma unroll
                for (int i = 0; i < NJ; ++i) m[i] = xb[t][i];
#pragma unroll
                for (int i = 0; i < W; ++i) lt[i] = lb[t][i];
                if (k - PF >= k0) {
#pragma unroll
                    for (int i = 0; i < NJ; ++i) xb[t][i] = (MODE != CH_BASIS) ? x[(long long)(k - PF) * NJ + i] : 0.0;
#pragma unroll
                    for (int i = 0; i < W; ++i) lb[t][i] = l[(long long)(k - PF) * NJ + 1 + i];
                }
                double za[W], tt[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) tt[i] = 0.0;
#pragma unroll
                for (int i = 0; i < W; ++i) {
                    double a0 = m[1 + i], a1 = 0.0;
#pragma unroll
                    for (int r = 0; r < W; ++r) {
                        const double zir = (i >= r) ? z[i][r] : z[r][i];
                        if (r & 1) a1 = fma(-zir, lt[r], a1);
                        else a0 = fma(-zir, lt[r], a0);
                    }
                    za[i] = a0 + a1;
                    tt[1 + i] = lt[i] * (m[1 + i] + za[i]);
                }
                const double z0 = m[0] - (((tt[0] + tt[1]) + (tt[2] + tt[3])) + ((tt[4] + tt[5]) + (tt[6] + tt[7])));
                if (MODE == CH_FINAL) {
                    double *o = x + (long long)k * NJ;
                    o[0] = z0;
#pragma unroll
                    for (int i = 0; i < W; ++i) o[1 + i] = za[i];
                }
                // state of the child: its separator = [this node's vertex, alpha_0 .. alpha_{W-2}]
#pragma unroll
                for (int p = W - 1; p >= 1; --p)
#pragma unroll
                    for (int q = p; q >= 1; --q) z[p][q] = z[p - 1][q - 1];
#pragma unroll
                for (int p = 1; p < W; ++p) z[p][0] = za[p - 1];
                z[0][0] = z0;
            }
        }
    }
    if (MODE == CH_PROBE) {
        double *g = a.state + ((long long)b * a.P + s) * D;
#pragma unroll
        for (int p = 0; p < W; ++p)
#pragma unroll
            for (int q = 0; q <= p; ++q) g[TRI(p, q)] = z[p][q];
    } else if (MODE == CH_BASIS) {
        double *g = a.phi + ((long long)s * D + b) * (D + 1);
#pragma unroll
        for (int p = 0; p < W; ++p)
#pragma unroll
            for (int q = 0; q <= p; ++q) g[TRI(p, q)] = z[p][q];
    }
}

// propagators Phi_s of the down sweep
template <int W>
__global__ void __launch_bounds__(128) chain_down_kernel(ChainArgs a) {
    constexpr int D = W * (W + 1) / 2;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int s = (int)(idx / D), b = (int)(idx - (long long)s * D);
    if (s >= a.P) return;
    chain_down_body<W, CH_BASIS, 4>(a, s, b, a.X + (long long)b * a.nblk, a.Lt);
}

template <int W, int MODE, bool UP>
__global__ void __launch_bounds__(128) chain_staged_kernel(ChainArgs a) {
    constexpr int NJ = W + 1;
    constexpr int WPC = (W <= 5) ? 4 : 2;                       // warps (items) per CTA: static shared memory < 48 KB
    constexpr bool YS = UP && MODE == CH_FINAL;
    __shared__ double xs[WPC][CHAIN_SEG * NJ], ls[WPC][CHAIN_SEG * NJ], ys[WPC][YS ? CHAIN_SEG * W * W : 1];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp >= WPC) return;
    const long long item = (long long)blockIdx.x * WPC + warp;   // item = s * B + b
    if (item >= (long long)a.P * a.B) return;
    const int s = (int)(item / a.B), b = (int)(item - (long long)s * a.B);
    const int k0 = s * a.SEG, k1 = min(a.N, k0 + a.SEG), cnt = (k1 - k0) * NJ;
    double *xg = a.X + (long long)b * a.nblk + (long long)k0 * NJ;
    const double *lg = a.Lt + (long long)k0 * NJ;
    for (int i = lane; i < cnt; i += 32) {
        xs[warp][i] = xg[i];
        ls[warp][i] = lg[i];
    }
    const bool scale = YS && a.Yaa != nullptr;
    if (scale) {
        const double *yg = a.Yaa + (long long)k0 * W * W;
        for (int i = lane; i < (k1 - k0) * W * W; i += 32) ys[warp][i] = yg[i];
    }
    __syncwarp();
    if (lane == 0) {
        double *xv = xs[warp] - (long long)k0 * NJ;
        const double *lv = ls[warp] - (long long)k0 * NJ;
        if (UP) chain_up_body<W, MODE, 1>(a, s, b, xv, lv, scale ? ys[warp] - (long long)k0 * W * W : nullptr);
        else chain_down_body<W, MODE, 1>(a, s, b, xv, lv);
    }
    __syncwarp();
    if (MODE == CH_FINAL)
        for (int i = lane; i < cnt; i += 32) xg[i] = xs[warp][i];
}

// Large batches (Schur assembly: one matrix per constraint): a warp takes 32 matrices of ONE segment,
// lane = matrix.  Thread-per-(matrix, segment) straight from global memory makes every load
// instruction touch 32 different lines (the matrices are nblk*8 bytes apart): ncu showed the
// kernels stalled on the load/store queue (lg_throttle) at 12 % of the HBM rate.  Here the warp
// copies each matrix's segment (SEG*NJ contiguous doubles) into shared memory with coalesced
// cp.async, every lane runs the recurrence on its row (odd row stride: conflict-free), and the
// rows are written back coalesced.  L and Y_aa are read by all lanes at the same address
// (broadcast, L1-resident).
template <int W, int MODE, bool UP>
__global__ void __launch_bounds__(32) chain_staged_batch_kernel(ChainArgs a) {
    constexpr int NJ = W + 1, RS = (CHAIN_SEG * NJ) | 1;
    constexpr bool YS = UP && MODE == CH_FINAL;
    extern __shared__ double csb[];                               // 32 x RS | L segment | Y_aa segment
    double *lsm = csb + 32 * RS, *ysm = lsm + CHAIN_SEG * NJ;
    const int lane = threadIdx.x;
    const int ngrp = (a.B + 31) / 32;
    const int s = blockIdx.x / ngrp, g = blockIdx.x - s * ngrp;
    const int b0 = g * 32, nmat = min(32, a.B - b0);
    const int k0 = s * a.SEG, k1 = min(a.N, k0 + a.SEG), cnt = (k1 - k0) * NJ;
    for (int mm = 0; mm < nmat; ++mm) {
        const double *src = a.X + (long long)(b0 + mm) * a.nblk + (long long)k0 * NJ;
        double *dst = csb + mm * RS;
        for (int i = lane; i < cnt; i += 32) chain_cp_async8(dst + i, src + i);
    }
    // the factor (and Y_aa for the fused scaling) of the segment: shared by the 32 matrices
    for (int i = lane; i < cnt; i += 32) chain_cp_async8(lsm + i, a.Lt + (long long)k0 * NJ + i);
    const bool scale = YS && a.Yaa != nullptr;
    if (scale)
        for (int i = lane; i < (k1 - k0) * W * W; i += 32) chain_cp_async8(ysm + i, a.Yaa + (long long)k0 * W * W + i);
    asm volatile("cp.async.commit_group;");
    asm volatile("cp.async.wait_group 0;");
    __syncwarp();
    if (lane < nmat) {
        double *xv = csb + lane * RS - (long long)k0 * NJ;
        const double *lv = lsm - (long long)k0 * NJ;
        if (UP) chain_up_body<W, MODE, 1>(a, s, b0 + lane, xv, lv, scale ? ysm - (long long)k0 * W * W : nullptr);
        else chain_down_body<W, MODE, 1>(a, s, b0 + lane, xv, lv);
    }
    __syncwarp();
    if (MODE == CH_FINAL) {
        for (int mm = 0; mm < nmat; ++mm) {
            double *dst = a.X + (long long)(b0 + mm) * a.nblk + (long long)k0 * NJ;
            const double *src = csb + mm * RS;
            for (int i = lane; i < cnt; i += 32) dst[i] = src[i];
        }
    }
}

// Boundary scan, one warp per matrix, lane r < D owns entry r of the state.
//   UP  : b_0 = 0, b_{s+1} = g_s + Phi_s b_s; the last state is added into the root block.
//   DOWN: b_{P-1} = Z_aa gathered from the root block, b_{s-1} = g_s + Phi_s b_s.
// state[b][s] holds g_s on entry and b_s (the incoming state of segment s) on exit.
// phi layout: phi[(s*D + c)*(D+1) + r], r < D (row D of every column is padding).  The D + 1
// values a lane needs for a segment (its row of Phi_s and g_s) do not depend on the recurrence,
// so they are fetched PD segments ahead into registers; the recurrence itself is D shuffles + D
// FMAs (three partial sums) per boundary.
template <int W, bool UP>
__global__ void __launch_bounds__(128) chain_scan_kernel(ChainArgs a) {
    constexpr int D = W * (W + 1) / 2, PD = 3;
    const int lane = threadIdx.x & 31;
    const int b = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    if (b >= a.B) return;
    int p = 0, q = 0;
    if (lane < D) {
        while (TRI(p + 1, 0) <= lane) ++p;
        q = lane - TRI(p, 0);
    }
    const int r = lane < D ? lane : 0;
    double *root = a.X + (long long)b * a.nblk + a.root_off;
    double *st = a.state + (long long)b * a.P * D;
    double bv = 0.0;
    if (!UP && lane < D) bv = root[p + q * a.root_nj];
    double ph[PD][D], g[PD];
#pragma unroll
    for (int t = 0; t < PD; ++t) {
        const int it = t, s = UP ? it : a.P - 1 - it;
        const bool in = it < a.P;
        const double *src = a.phi + (long long)(in ? s : 0) * D * (D + 1) + r;
#pragma unroll
        for (int c = 0; c < D; ++c) ph[t][c] = in ? src[c * (D + 1)] : 0.0;
        g[t] = in ? st[(long long)s * D + r] : 0.0;
    }
    for (int it0 = 0; it0 < a.P; it0 += PD) {
#pragma unroll
        for (int t = 0; t < PD; ++t) {
            const int it = it0 + t;
            if (it < a.P) {
                const int s = UP ? it : a.P - 1 - it;
                double pc[D];
#pragma unroll
                for (int c = 0; c < D; ++c) pc[c] = ph[t][c];
                double acc0 = g[t], acc1 = 0.0, acc2 = 0.0;
                if (it + PD < a.P) {
                    const int sn = UP ? it + PD : a.P - 1 - (it + PD);
                    const double *src = a.phi + (long long)sn * D * (D + 1) + r;
#pragma unroll
                    for (int c = 0; c < D; ++c) ph[t][c] = src[c * (D + 1)];
                    g[t] = st[(long long)sn * D + r];
                }
                if (lane < D) st[(long long)s * D + lane] = bv;
#pragma unroll
                for (int c = 0; c < D; ++c) {
                    const double bc = __shfl_sync(0xffffffffu, bv, c);
                    if (c % 3 == 0) acc0 = fma(pc[c], bc, acc0);
                    else if (c % 3 == 1) acc1 = fma(pc[c], bc, acc1);
                    else acc2 = fma(pc[c], bc, acc2);
                }
                bv = acc0 + (acc1 + acc2);
            }
        }
    }
    if (UP && lane < D) root[p + q * a.root_nj] += bv;
}

// ---- two-level scan for a single matrix (or a handful): the P boundaries are cut into G groups,
// warp w scans its group from a zero state (level 1), warp 0 carries the group states across with
// the group propagators Psi_w (level 2, G steps), every warp rescans its group from its true
// incoming state and stores the b_s (level 3): 2*P/G + G dependent steps instead of P.
#define SCAN_G 8

template <int W, bool UP, bool WRITE, bool GZERO>
__device__ __forceinline__ double chain_scan_range(const ChainArgs &a, double *st, int it_lo, int it_hi, double bv, int lane) {
    constexpr int D = W * (W + 1) / 2, PD = 3;
    const int r = lane < D ? lane : 0;
    double ph[PD][D], g[PD];
#pragma unroll
    for (int t = 0; t < PD; ++t) {
        const int it = it_lo + t, s = UP ? it : a.P - 1 - it;
        const bool in = it < it_hi;
        const double *src = a.phi + (long long)(in ? s : 0) * D * (D + 1) + r;
#pragma unroll
        for (int c = 0; c < D; ++c) ph[t][c] = in ? src[c * (D + 1)] : 0.0;
        g[t] = (in && !GZERO) ? st[(long long)s * D + r] : 0.0;
    }
    for (int it0 = it_lo; it0 < it_hi; it0 += PD) {
#pragma unroll
        for (int t = 0; t < PD; ++t) {
            const int it = it0 + t;
            if (it < it_hi) {
                const int s = UP ? it : a.P - 1 - it;
                double pc[D];
#pragma unroll
                for (int c = 0; c < D; ++c) pc[c] = ph[t][c];
                double acc0 = g[t], acc1 = 0.0, acc2 = 0.0;
                if (it + PD < it_hi) {
                    const int sn = UP ? it + PD : a.P - 1 - (it + PD);
                    const double *src = a.phi + (long long)sn * D * (D + 1) + r;
#pragma unroll
                    for (int c = 0; c < D; ++c) ph[t][c] = src[c * (D + 1)];
                    if (!GZERO) g[t] = st[(long long)sn * D + r];
                }
                if (WRITE && lane < D) st[(long long)s * D + lane] = bv;
#pragma unroll
                for (int c = 0; c < D; ++c) {
                    const double bc = __shfl_sync(0xffffffffu, bv, c);
                    if (c % 3 == 0) acc0 = fma(pc[c], bc, acc0);
                    else if (c % 3 == 1) acc1 = fma(pc[c], bc, acc1);
                    else acc2 = fma(pc[c], bc, acc2);
                }
                bv = acc0 + (acc1 + acc2);
            }
        }
    }
    return bv;
}

// Psi_w[:, c] = state after group w when entering it with the unit state e_c and g = 0
template <int W, bool UP>
__global__ void __launch_bounds__(128) chain_psi_kernel(ChainArgs a) {
    constexpr int D = W * (W + 1) / 2;
    const int lane = threadIdx.x & 31;
    const int wid = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    if (wid >= a.G * D) return;
    const int w = wid / D, c = wid - w * D;
    const int lo = w * a.gs, hi = min(a.P, lo + a.gs);
    double bv = (lane == c) ? 1.0 : 0.0;
    bv = chain_scan_range<W, UP, false, true>(a, nullptr, lo, hi, bv, lane);
    if (lane < D) a.psi[((long long)w * D + c) * (D + 1) + lane] = bv;
}

template <int W, bool UP>
__global__ void __launch_bounds__(32 * SCAN_G) chain_scan2_kernel(ChainArgs a) {
    constexpr int D = W * (W + 1) / 2;
    __shared__ double gam[SCAN_G][32], bst[SCAN_G][32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int b = blockIdx.x;
    double *root = a.X + (long long)b * a.nblk + a.root_off;
    double *st = a.state + (long long)b * a.P * D;
    const int lo = min(a.P, w * a.gs), hi = min(a.P, lo + a.gs);
    gam[w][lane] = chain_scan_range<W, UP, false, false>(a, st, lo, hi, 0.0, lane);
    __syncthreads();
    if (w == 0) {
        int p = 0, q = 0;
        if (lane < D) {
            while (TRI(p + 1, 0) <= lane) ++p;
            q = lane - TRI(p, 0);
        }
        double bv = 0.0;
        if (!UP && lane < D) bv = root[p + q * a.root_nj];
        for (int g = 0; g < a.G; ++g) {
            bst[g][lane] = bv;
            const double *ps = a.psi + (long long)g * D * (D + 1) + (lane < D ? lane : 0);
            double acc0 = gam[g][lane], acc1 = 0.0, acc2 = 0.0;
#pragma unroll
            for (int c = 0; c < D; ++c) {
                const double bc = __shfl_sync(0xffffffffu, bv, c);
                const double pv = ps[c * (D + 1)];
                if (c % 3 == 0) acc0 = fma(pv, bc, acc0);
                else if (c % 3 == 1) acc1 = fma(pv, bc, acc1);
                else acc2 = fma(pv, bc, acc2);
            }
            bv = acc0 + (acc1 + acc2);
        }
        if (UP && lane < D) root[p + q * a.root_nj] += bv;
    }
    __syncthreads();
    chain_scan_range<W, UP, true, false>(a, st, lo, hi, bst[w][lane], lane);
}

// inverse Hessian / llt on a chain: X = sum over nodes of the scattered local fronts
// (App. A.5 stage 1^-1, App. A.6).  Thread per (matrix, block entry); the sum runs from the
// oldest contributing front to the node's own one, the order of the sequential sweep.
template <int W>
__global__ void __launch_bounds__(256) chain_add_kernel(ChainArgs a) {
    constexpr int NJ = W + 1, SQ = NJ * NJ;
    const long long per = (long long)a.N * NJ + (long long)a.root_nj * a.root_nj;
    const long long total = per * a.B;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const int b = (int)(idx / per);
        const long long e = idx - (long long)b * per;
        const double *F = a.F + (long long)b * a.nsq;
        double *X = a.X + (long long)b * a.nblk;
        if (e < (long long)a.N * NJ) {
            const int k = (int)(e / NJ), i = (int)(e - (long long)k * NJ);
            int tmax = W - i;
            if (tmax > k) tmax = k;
            double acc = F[(long long)(k - tmax) * SQ + (i + tmax) + tmax * NJ];
            for (int t = tmax - 1; t >= 0; --t) acc = F[(long long)(k - t) * SQ + (i + t) + t * NJ] + acc;
            X[e] = acc;
        } else {
            const int r = (int)(e - (long long)a.N * NJ);
            const int p = r % a.root_nj, q = r / a.root_nj;
            double v = 0.0;
            if (p >= q) {
                // carried part: node N-1-t contributes its front entry (p+1+t, q+1+t)
                int tmax = W - 1 - p;
                if (tmax > a.N - 1) tmax = a.N - 1;
                double acc = 0.0;
                bool any = false;
                for (int t = tmax; t >= 0; --t) {
                    const double f = F[(long long)(a.N - 1 - t) * SQ + (p + 1 + t) + (q + 1 + t) * NJ];
                    acc = any ? f + acc : f;
                    any = true;
                }
                const double loc = F[a.root_sq + p + q * a.root_nj];
                v = any ? acc + loc : loc;
            }
            X[a.root_off + r] = v;
        }
    }
}

// root of a chain: dense nn x nn front = root block + carried update (positions < W), right-looking
template <int W>
__device__ __forceinline__ bool chain_chol_root(const ChainArgs &a, double *x, double (&u)[W][W]) {
    bool anybad = false;
    const int nn = a.root_nj;
    double *rb = x + a.root_off;
    double f[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            double v = 0.0;
            if (i < nn && j <= i) {
                v = rb[i + j * nn];
                if (i < W) v = u[i < W ? i : 0][j < W ? j : 0] + v;
            }
            f[i][j] = v;
        }
#pragma unroll
    for (int r = 0; r < 8; ++r) {
        if (r < nn) {
            const double d = f[r][r];
            const bool bad = !(d > 0.0);
            anybad |= bad;
            const double rs = bad ? 1.0 : rsqrt(d);
            double l[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) l[i] = (i > r) ? f[i][r] * rs : 0.0;
            double dg = d * rs;
            dg = fma(fma(-dg, dg, d), 0.5 * rs, dg);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                if (i < nn) {
                    if (i == r) rb[i + r * nn] = bad ? 1.0 : dg;
                    else if (i > r) rb[i + r * nn] = l[i];
                    else rb[i + r * nn] = 0.0;
                }
            }
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j <= i; ++j)
                    if (j > r) f[i][j] = fma(-l[i], l[j], f[i][j]);
        }
    }
    return anybad;
}

// one node of the chain Cholesky: xn[0..W] in -> L column out (in place), u = carried update matrix
template <int W>
__device__ __forceinline__ bool chain_chol_node(double *xn, double (&u)[W][W]) {
    const double f0 = xn[0] + u[0][0];
    const bool bad = !(f0 > 0.0);
    const double rs = bad ? 1.0 : rsqrt(f0);
    double li[W];
#pragma unroll
    for (int i = 0; i < W; ++i) {
        const double fa = (i + 1 < W) ? xn[1 + i] + u[i + 1][0] : xn[1 + i];
        li[i] = fa * rs;
    }
    double un[W][W];
#pragma unroll
    for (int i = 0; i < W; ++i)
#pragma unroll
        for (int j = 0; j <= i; ++j) {
            const double faa = (i + 1 < W) ? u[i + 1][j + 1] : 0.0;
            un[i][j] = fma(-li[i], li[j], faa);
        }
#pragma unroll
    for (int i = 0; i < W; ++i)
#pragma unroll
        for (int j = 0; j <= i; ++j) u[i][j] = un[i][j];
    double dg = f0 * rs;
    dg = fma(fma(-dg, dg, f0), 0.5 * rs, dg);
    xn[0] = bad ? 1.0 : dg;
#pragma unroll
    for (int i = 0; i < W; ++i) xn[1 + i] = li[i];
    return bad;
}

// Cholesky on a chain (chompack.cholesky, solvers.py:640, 884, 1218): the recurrence is NOT linear
// (the pivot depends on the incoming update), so it stays sequential — but one THREAD per matrix
// with the W x W update matrix in registers has a critical path of one rsqrt + three FP64 ops per
// node (~60 cycles) instead of the ~400 cycles of a warp that exchanges the front through shared
// memory, and a batch of line-search candidates costs the same latency as one matrix.  Same
// operation order as the warp sweep (chordal_small.cu, SW_CHOL): bitwise identical factors.
// A warp owns up to 32 matrices (one per lane).  The chain is cut into chunks of C nodes; the warp
// copies the chunk of every one of its matrices into shared memory with coalesced cp.async (each
// matrix's chunk is contiguous), double-buffered so that the next chunk is in flight while the
// lanes run the recurrence on the current one, and writes the factor back coalesced.  Straight
// from global memory, every lane would issue one uncoalesced 8-byte load per entry, i.e. a DRAM
// round trip per node (0.3 - 0.6 us): 1.7 ms for one matrix, 2.9 ms for 255 candidates.
template <int W>
__global__ void __launch_bounds__(32) chain_chol_staged_kernel(ChainArgs a, int *fail, int C, int R) {
    constexpr int NJ = W + 1;
    extern __shared__ double chsm[];
    const int lane = threadIdx.x;
    const int b0 = blockIdx.x * R;                      // R matrices per warp (lanes >= R idle): few matrices per
    const int nmat = min(R, a.B - b0);                  // warp = long chunks = little copy overhead per node
    const int rs = (C * NJ) | 1;                        // odd row stride: conflict-free lane access
    double *buf0 = chsm, *buf1 = chsm + (size_t)R * rs;          // R = rows (matrices) per buffer
    const int nchunks = (a.N + C - 1) / C;
    double u[W][W];
#pragma unroll
    for (int p = 0; p < W; ++p)
#pragma unroll
        for (int q = 0; q <= p; ++q) u[p][q] = 0.0;
    bool anybad = false;
    auto stage = [&](int c, double *buf) {
        const int k0 = c * C, cnt = min(C, a.N - k0) * NJ;
        for (int mm = 0; mm < nmat; ++mm) {
            const double *src = a.X + (long long)(b0 + mm) * a.nblk + (long long)k0 * NJ;
            for (int i = lane; i < cnt; i += 32) chain_cp_async8(buf + (size_t)mm * rs + i, src + i);
        }
        asm volatile("cp.async.commit_group;");
    };
    if (nchunks > 0) stage(0, buf0);
    for (int c = 0; c < nchunks; ++c) {
        double *cur = (c & 1) ? buf1 : buf0;
        if (c + 1 < nchunks) {
            stage(c + 1, (c & 1) ? buf0 : buf1);
            asm volatile("cp.async.wait_group 1;");
        } else {
            asm volatile("cp.async.wait_group 0;");
        }
        __syncwarp();
        const int k0 = c * C, nk = min(C, a.N - k0);
        if (lane < nmat) {
            double *row = cur + (size_t)lane * rs;
            for (int k = 0; k < nk; ++k) anybad |= chain_chol_node<W>(row + k * NJ, u);
        }
        __syncwarp();
        for (int mm = 0; mm < nmat; ++mm) {
            double *dst = a.X + (long long)(b0 + mm) * a.nblk + (long long)k0 * NJ;
            for (int i = lane; i < nk * NJ; i += 32) dst[i] = cur[(size_t)mm * rs + i];
        }
        __syncwarp();
    }
    if (lane < nmat) {
        anybad |= chain_chol_root<W>(a, a.X + (long long)(b0 + lane) * a.nblk, u);
        if (anybad) fail[b0 + lane] = 1;
    }
}

// completion on a chain (chompack.completion, solvers.py:625, 874; App. A.3): every node is
// independent — one THREAD per (matrix, node) with the W x W separator block in registers:
// R = chol(X_aa), w = X_aa^{-1} X_an, delta = X_nn - X_an^T w, L_nn = delta^{-1/2}, L_an = -w L_nn.
// Same operation order as the warp version (op_compl), which still handles the root supernode.
template <int W>
__global__ void __launch_bounds__(128) chain_compl_kernel(ChainArgs a, const double *__restrict__ Xin, const int *__restrict__ aaidx, int *fail) {
    const long long total = (long long)a.N * a.B;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const int b = (int)(idx / a.N), k = (int)(idx - (long long)b * a.N);
        const double *xi = Xin + (long long)b * a.nblk;
        const int *ai = aaidx + (long long)k * W * W;
        double R[W][W], z[W];
#pragma unroll
        for (int i = 0; i < W; ++i)
#pragma unroll
            for (int j = 0; j <= i; ++j) R[i][j] = xi[ai[i + j * W]];
        const double *blk = xi + (long long)k * (W + 1);
#pragma unroll
        for (int i = 0; i < W; ++i) z[i] = blk[1 + i];
        double dl = blk[0];
        bool bad = false;
#pragma unroll
        for (int j = 0; j < W; ++j) {
            const double d = R[j][j];
            const bool bj = !(d > 0.0);
            bad |= bj;
            const double sq = bj ? 1.0 : sqrt(d);
#pragma unroll
            for (int i = j + 1; i < W; ++i) R[i][j] /= sq;
            R[j][j] = sq;
#pragma unroll
            for (int c = j + 1; c < W; ++c)
#pragma unroll
                for (int i = c; i < W; ++i) R[i][c] = fma(-R[i][j], R[c][j], R[i][c]);
        }
#pragma unroll
        for (int j = 0; j < W; ++j) {          // z <- R^{-1} z
            z[j] /= R[j][j];
#pragma unroll
            for (int i = j + 1; i < W; ++i) z[i] = fma(-R[i][j], z[j], z[i]);
        }
        double ss = 0.0;
#pragma unroll
        for (int i = 0; i < W; ++i) ss = fma(z[i], z[i], ss);
        dl = dl + (-1.0) * ss;
#pragma unroll
        for (int j = W - 1; j >= 0; --j) {     // z <- R^{-T} z
            z[j] /= R[j][j];
#pragma unroll
            for (int i = 0; i < j; ++i) z[i] = fma(-R[j][i], z[j], z[i]);
        }
        const bool bd = !(dl > 0.0);
        bad |= bd;
        const double sq = bd ? 1.0 : sqrt(dl);
        const double li = 1.0 / sq;
        double *o = a.X + (long long)b * a.nblk + (long long)k * (W + 1);
        o[0] = li;
#pragma unroll
        for (int i = 0; i < W; ++i) o[1 + i] = -fma(z[i], li, 0.0);
        if (bad) fail[b] = 1;
    }
}

// ---------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------

// chain structure test (called from small_setup)
static void chain_detect(smcp_sym *s, const smcp_sym_desc *D, const std::vector<int> &nn, const std::vector<int> &na) {
    s->chain = false;
    const int nsn = (int)D->nsn;
    if (nsn < 2 || getenv("SMCP_B200_NO_CHAIN")) return;
    const int W = na[0], root = nsn - 1;
    if (W < 1 || W > 7) return;
    if (D->snpar[root] != -1 || na[root] != 0 || nn[root] < W) return;
    for (int k = 0; k < root; ++k) {
        if (nn[k] != 1 || na[k] != W || D->snpar[k] != k + 1) return;
        if (D->blkptr[k] != (int64_t)k * (W + 1)) return;
        for (int q = 0; q < W; ++q)
            if (D->relidx[D->relptr[k] + q] != q) return;
    }
    if (D->blkptr[root] != (int64_t)root * (W + 1)) return;
    s->chain = true;
    s->chW = W;
    s->chN = root;
    s->chP = (root + CHAIN_SEG - 1) / CHAIN_SEG;
    s->ch_root_off = (int)D->blkptr[root];
    s->ch_root_nj = nn[root];
}

static int chain_fill(smcp_sym *s, ChainArgs &a, double *X, const double *Lt, int64_t batch) {
    const int W = s->chW;
    a.N = s->chN;
    a.P = s->chP;
    a.SEG = CHAIN_SEG;
    a.B = (int)batch;
    a.D = W * (W + 1) / 2;
    a.nblk = s->d.nblk;
    a.X = X;
    a.Lt = Lt;
    a.root_off = s->ch_root_off;
    a.root_nj = s->ch_root_nj;
    a.root_sq = (int)((long long)s->chN * (W + 1) * (W + 1));
    a.nsq = s->sm.nsq;
    a.G = SCAN_G;
    a.gs = (a.P + SCAN_G - 1) / SCAN_G;
    if (grow((void **)&s->ch_state, &s->ch_state_cap, (size_t)batch * a.P * a.D * sizeof(double) + 64)) return -1;
    a.state = s->ch_state;
    return 0;
}

template <int W, int MODE>
static void chain_launch_dir(bool up, const ChainArgs &a, cudaStream_t st) {
    if (MODE == CH_BASIS) {
        const unsigned grid = (unsigned)(((long long)a.P * a.D + 127) / 128);
        if (up) chain_up_kernel<W><<<grid, 128, 0, st>>>(a);
        else chain_down_kernel<W><<<grid, 128, 0, st>>>(a);
    } else if (a.B < 32) {
        constexpr int WPC = (W <= 5) ? 4 : 2;
        const unsigned g2 = (unsigned)(((long long)a.P * a.B + WPC - 1) / WPC);
        if (up) chain_staged_kernel<W, MODE, true><<<g2, 32 * WPC, 0, st>>>(a);
        else chain_staged_kernel<W, MODE, false><<<g2, 32 * WPC, 0, st>>>(a);
    } else {
        constexpr int RS = (CHAIN_SEG * (W + 1)) | 1;
        const int smem = (32 * RS + CHAIN_SEG * (W + 1) + CHAIN_SEG * W * W) * (int)sizeof(double);
        const unsigned g3 = (unsigned)((long long)a.P * ((a.B + 31) / 32));
        if (up) {
            cudaFuncSetAttribute(chain_staged_batch_kernel<W, MODE, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
            chain_staged_batch_kernel<W, MODE, true><<<g3, 32, smem, st>>>(a);
        } else {
            cudaFuncSetAttribute(chain_staged_batch_kernel<W, MODE, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
            chain_staged_batch_kernel<W, MODE, false><<<g3, 32, smem, st>>>(a);
        }
    }
}

template <int W>
static void chain_scan_dir(bool up, const ChainArgs &a, cudaStream_t st) {
    if (a.psi && a.B <= 8 && a.P >= 2 * SCAN_G) {
        if (up) chain_scan2_kernel<W, true><<<a.B, 32 * SCAN_G, 0, st>>>(a);
        else chain_scan2_kernel<W, false><<<a.B, 32 * SCAN_G, 0, st>>>(a);
        return;
    }
    const unsigned grid = (unsigned)(((long long)a.B * 32 + 127) / 128);
    if (up) chain_scan_kernel<W, true><<<grid, 128, 0, st>>>(a);
    else chain_scan_kernel<W, false><<<grid, 128, 0, st>>>(a);
}

template <int W>
static void chain_psi_dir(bool up, const ChainArgs &a, cudaStream_t st) {
    const unsigned grid = (unsigned)(((long long)a.G * a.D * 32 + 127) / 128);
    if (up) chain_psi_kernel<W, true><<<grid, 128, 0, st>>>(a);
    else chain_psi_kernel<W, false><<<grid, 128, 0, st>>>(a);
}

static void chain_psi(int W, bool up, const ChainArgs &a, cudaStream_t st) {
    switch (W) {
        case 1: chain_psi_dir<1>(up, a, st); break;
        case 2: chain_psi_dir<2>(up, a, st); break;
        case 3: chain_psi_dir<3>(up, a, st); break;
        case 4: chain_psi_dir<4>(up, a, st); break;
        case 5: chain_psi_dir<5>(up, a, st); break;
        case 6: chain_psi_dir<6>(up, a, st); break;
        default: chain_psi_dir<7>(up, a, st); break;
    }
}

static void chain_scan(int W, bool up, const ChainArgs &a, cudaStream_t st) {
    switch (W) {
        case 1: chain_scan_dir<1>(up, a, st); break;
        case 2: chain_scan_dir<2>(up, a, st); break;
        case 3: chain_scan_dir<3>(up, a, st); break;
        case 4: chain_scan_dir<4>(up, a, st); break;
        case 5: chain_scan_dir<5>(up, a, st); break;
        case 6: chain_scan_dir<6>(up, a, st); break;
        default: chain_scan_dir<7>(up, a, st); break;
    }
}

template <int MODE>
static void chain_launch(int W, bool up, const ChainArgs &a, cudaStream_t st) {
    switch (W) {
        case 1: chain_launch_dir<1, MODE>(up, a, st); break;
        case 2: chain_launch_dir<2, MODE>(up, a, st); break;
        case 3: chain_launch_dir<3, MODE>(up, a, st); break;
        case 4: chain_launch_dir<4, MODE>(up, a, st); break;
        case 5: chain_launch_dir<5, MODE>(up, a, st); break;
        case 6: chain_launch_dir<6, MODE>(up, a, st); break;
        default: chain_launch_dir<7, MODE>(up, a, st); break;
    }
}

// largest |entry| of the segment propagators (rows r < D of every column)
__global__ void chain_gamma_kernel(const double *__restrict__ phi, long long ncol, int D, unsigned long long *out) {
    double mx = 0.0;
    const long long total = ncol * D;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const long long c = idx / D;
        const int r = (int)(idx - c * D);
        const double v = fabs(phi[c * (D + 1) + r]);
        mx = (v > mx || v != v) ? (v != v ? 1e300 : v) : mx;
    }
    for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if ((threadIdx.x & 31) == 0) atomicMax(out, (unsigned long long)__double_as_longlong(mx));    // non-negative doubles order like integers
}

// largest |entry| of the segment propagators for which the segment-parallel sweeps are used
static const double CHAIN_GAMMA_MAX = 1e3;

// propagators of both sweeps for the scaling point of `h` (once per smcp_hess)
static int chain_prepare(smcp_hess *h) {
    smcp_sym *s = h->sym;
    smcp_ctx *ctx = s->ctx;
    if (h->have_phi) return 0;
    const int W = s->chW, D = W * (W + 1) / 2;
    const size_t bytes = (size_t)s->chP * D * (D + 1) * sizeof(double);
    const size_t pbytes = (size_t)SCAN_G * D * (D + 1) * sizeof(double);
    if (!h->phi_up) CUDA_TRY(cudaMalloc(&h->phi_up, 2 * (bytes + pbytes)));      // reused from the pool of the symbolic object
    h->phi_dn = h->phi_up + bytes / sizeof(double);
    h->psi_up = h->phi_dn + bytes / sizeof(double);
    h->psi_dn = h->psi_up + pbytes / sizeof(double);
    ChainArgs a = {};
    if (chain_fill(s, a, nullptr, h->Lt, 1)) return -1;
    {
        LaunchScope ls(ctx, "hessian_chain_prep", 4);
        a.phi = h->phi_up;
        a.psi = h->psi_up;
        chain_launch<CH_BASIS>(W, true, a, ctx->stream);
        chain_psi(W, true, a, ctx->stream);
        a.phi = h->phi_dn;
        a.psi = h->psi_dn;
        chain_launch<CH_BASIS>(W, false, a, ctx->stream);
        chain_psi(W, false, a, ctx->stream);
    }
    CUDA_TRY(cudaGetLastError());
    h->have_phi = true;
    // Accuracy guard.  The boundary recurrence b_{s+1} = g_s + Phi_s b_s is exact in exact arithmetic, but
    // when the entries of Phi_s (products of L_an L_nn^{-1} over a segment) grow, g_s and Phi_s b_s cancel
    // and the boundary states lose digits: on the benchmark problem the Schur complement assembled through
    // the segment-parallel sweeps was only ~1e-2 accurate in the last iterations (cond(S) > 1e12) and the
    // solver stalled at a primal residual of 3e-5.  Scaling points whose propagators exceed CHAIN_GAMMA_MAX use
    // the sequential warp-per-chain sweeps instead (exact recurrences, ~2x slower per iteration).
    {
        unsigned long long *dv = (unsigned long long *)s->counter + 2;       // scratch next to the work-queue head (64 bytes)
        CUDA_TRY(cudaMemsetAsync(dv, 0, sizeof(unsigned long long), ctx->stream));
        {
            LaunchScope ls(ctx, "hessian_chain_prep", 2);
            chain_gamma_kernel<<<64, 256, 0, ctx->stream>>>(h->phi_up, (long long)s->chP * D, D, dv);
            chain_gamma_kernel<<<64, 256, 0, ctx->stream>>>(h->phi_dn, (long long)s->chP * D, D, dv);
        }
        unsigned long long hv = 0;
        CUDA_TRY(cudaMemcpyAsync(&hv, dv, sizeof(hv), cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_TRY(cudaStreamSynchronize(ctx->stream));
        double g;
        memcpy(&g, &hv, sizeof(g));
        h->chain_gamma = g;
        h->chain_ok = g <= CHAIN_GAMMA_MAX;
        if (getenv("SMCP_B200_CHAIN_DEBUG")) fprintf(stderr, "[smcp_b200] chain propagators: max |Phi| = %.3e -> %s\n", g, h->chain_ok ? "segment-parallel sweeps" : "sequential sweeps");
    }
    return 0;
}

// one linear sweep (probe, scan, final) on `batch` matrices
static int chain_sweep(smcp_sym *s, bool up, double *X, const double *Lt, double *phi, double *psi, const double *Yaa, int64_t batch, const char *name) {
    smcp_ctx *ctx = s->ctx;
    ChainArgs a = {};
    if (chain_fill(s, a, X, Lt, batch)) return -1;
    a.phi = phi;
    a.psi = psi;
    a.Yaa = Yaa;
    {
        LaunchScope ls(ctx, name, 3, (double)batch);
        chain_launch<CH_PROBE>(s->chW, up, a, ctx->stream);
        chain_scan(s->chW, up, a, ctx->stream);
        chain_launch<CH_FINAL>(s->chW, up, a, ctx->stream);
    }
    CUDA_TRY(cudaGetLastError());
    return 0;
}

static int chain_add(smcp_sym *s, double *X, const double *F, int64_t batch, const char *name) {
    smcp_ctx *ctx = s->ctx;
    ChainArgs a = {};
    if (chain_fill(s, a, X, nullptr, batch)) return -1;
    a.F = F;
    const long long total = ((long long)a.N * (s->chW + 1) + (long long)a.root_nj * a.root_nj) * batch;
    long long grid = (total + 255) / 256;
    if (grid > (long long)ctx->num_sms * 16) grid = (long long)ctx->num_sms * 16;
    {
        LaunchScope ls(ctx, name, 1, (double)batch);
        switch (s->chW) {
            case 1: chain_add_kernel<1><<<(unsigned)grid, 256, 0, ctx->stream>>>(a); break;
            case 2: chain_add_kernel<2><<<(unsigned)grid, 256, 0, ctx->stream>>>(a); break;
            case 3: chain_add_kernel<3><<<(unsigned)grid, 256, 0, ctx->stream>>>(a); break;
            case 4: chain_add_kernel<4><<<(unsigned)grid, 256, 0, ctx->stream>>>(a); break;
            case 5: chain_add_kernel<5><<<(unsigned)grid, 256, 0, ctx->stream>>>(a); break;
            case 6: chain_add_kernel<6><<<(unsigned)grid, 256, 0, ctx->stream>>>(a); break;
            default: chain_add_kernel<7><<<(unsigned)grid, 256, 0, ctx->stream>>>(a); break;
        }
    }
    CUDA_TRY(cudaGetLastError());
    return 0;
}

static int chain_cholesky(smcp_sym *s, double *X, int64_t batch, const char *name) {
    smcp_ctx *ctx = s->ctx;
    ChainArgs a = {};
    if (chain_fill(s, a, X, nullptr, batch)) return -1;
    // chunk length: 2 buffers x 32 rows of C*NJ doubles within ~96 KB; fewer matrices -> longer chunks
    // the recurrence costs ~300 cycles per node whatever the number of active lanes, so a batch is
    // spread over many warps: 8 matrices per warp (255 line-search candidates -> 32 SMs)
    const int NJ = s->chW + 1, nmat = (int)std::min<int64_t>(batch >= 64 ? 8 : 32, batch);
    int C = 6000 / (nmat * NJ);
    C = std::max(8, std::min(C, 512));
    const size_t smem = (size_t)2 * nmat * ((C * NJ) | 1) * sizeof(double);
    const unsigned g2 = (unsigned)((batch + nmat - 1) / nmat);
    {
        LaunchScope ls(ctx, name, 1, (double)batch);
#define CHOL_ST(W_)                                                                                                         \
    do {                                                                                                                    \
        CUDA_TRY(cudaFuncSetAttribute(chain_chol_staged_kernel<W_>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024)); \
        chain_chol_staged_kernel<W_><<<g2, 32, smem, ctx->stream>>>(a, s->fail, C, nmat);                                    \
    } while (0)
        switch (s->chW) {
            case 1: CHOL_ST(1); break;
            case 2: CHOL_ST(2); break;
            case 3: CHOL_ST(3); break;
            case 4: CHOL_ST(4); break;
            case 5: CHOL_ST(5); break;
            case 6: CHOL_ST(6); break;
            default: CHOL_ST(7); break;
        }
#undef CHOL_ST
    }
    CUDA_TRY(cudaGetLastError());
    return 0;
}

static int chain_completion(smcp_sym *s, double *X, const double *Xin, int64_t batch, const char *name) {
    smcp_ctx *ctx = s->ctx;
    ChainArgs a = {};
    if (chain_fill(s, a, X, nullptr, batch)) return -1;
    long long grid = ((long long)a.N * batch + 127) / 128;
    if (grid > (long long)ctx->num_sms * 32) grid = (long long)ctx->num_sms * 32;
    {
        LaunchScope ls(ctx, name, 1, (double)batch);
        switch (s->chW) {
            case 1: chain_compl_kernel<1><<<(unsigned)grid, 128, 0, ctx->stream>>>(a, Xin, s->d.aaidx, s->fail); break;
            case 2: chain_compl_kernel<2><<<(unsigned)grid, 128, 0, ctx->stream>>>(a, Xin, s->d.aaidx, s->fail); break;
            case 3: chain_compl_kernel<3><<<(unsigned)grid, 128, 0, ctx->stream>>>(a, Xin, s->d.aaidx, s->fail); break;
            case 4: chain_compl_kernel<4><<<(unsigned)grid, 128, 0, ctx->stream>>>(a, Xin, s->d.aaidx, s->fail); break;
            case 5: chain_compl_kernel<5><<<(unsigned)grid, 128, 0, ctx->stream>>>(a, Xin, s->d.aaidx, s->fail); break;
            case 6: chain_compl_kernel<6><<<(unsigned)grid, 128, 0, ctx->stream>>>(a, Xin, s->d.aaidx, s->fail); break;
            default: chain_compl_kernel<7><<<(unsigned)grid, 128, 0, ctx->stream>>>(a, Xin, s->d.aaidx, s->fail); break;
        }
    }
    CUDA_TRY(cudaGetLastError());
    return 0;
}
