// Warp-per-chain kernels for chordal patterns with tiny cliques (every clique has at most 8
// vertices: band SDPs, sparse-graph relaxations with small separators).
//
// Same routines and contracts as chordal.cu (cholesky, completion, projected_inverse, llt,
// barrier Hessian and its inverse; reference call sites src/python/solvers.py:874, 884, 891,
// 904, 483, 405), different execution model.  With 6 x 1 blocks a CTA per supernode wastes
// the machine and a long clique-tree chain (band n=5000: 4995 supernodes in a row) is a
// pure latency problem.  Here
//   * every recursion is split into a FLAT part (no dependency between supernodes: the
//     scaling of the Hessian, the local fronts of llt / inverse Hessian, the factor
//     preparation, completion) that runs with one warp per (supernode, matrix), and a SWEEP
//     that carries only the recurrence along the tree (extend-add + congruence with the
//     elimination matrix, or the Cholesky pivot), one warp per (task, matrix);
//   * in a sweep the 8 x 8 frontal matrix lives in shared memory (two ping-pong tiles per
//     warp); the update matrix handed from a child to its parent never goes through global
//     memory when the parent is the next supernode of the chain (the common case), so the
//     sweep's traffic is one read and one write of each matrix entry;
//   * everything a step needs from global memory (step descriptor, its own entries of the
//     block, the factor, relative indices) is fetched one step ahead into registers, so
//     the critical path of a step is two shared-memory round trips and a few FMAs;
//   * tasks are claimed from an atomic queue in topological order and cross-task
//     dependencies use release/acquire flags exactly like chordal.cu (all warps of the grid
//     are co-resident, so the scheme cannot deadlock);
//   * sums are formed in a fixed order (no floating-point atomics): results are bitwise
//     reproducible from run to run.
#include "internal.cuh"
#include <algorithm>
#include <cstdio>
#include <cstdlib>

#include "chordal_ops.cuh"

#define FULLMASK 0xffffffffu
#define WTID ((int)(threadIdx.x & 31))

enum { SW_CHOL = 0, SW_HUP, SW_ADD };
enum { FL_COMPL = 0, FL_HPREP, FL_HPREP_INV, FL_HSCALE, FL_HINV_LOCAL, FL_LLT_LOCAL, FL_PINV_PREP };

struct SmallArgs {
    TreeArgs t;            // S, T, X, Xin, upd, Lt, Yaa, Raa, L0, Y0, Lt_out, Yaa_out, B, counter, done, epoch, fail
    SmallDev M;
    double *F;             // B x nsq local fronts
    long long ltstride;    // 0: one factor for the whole batch (Hessian); nblk: one per matrix
    const int *list;       // flat kernels: restrict to these supernodes (nullptr = all)
    int nlist;
};

// ---------------------------------------------------------------------------------------
// flat part: new per-supernode steps (warp scope)
// ---------------------------------------------------------------------------------------
#define TID WTID
#define NT 32
#define SYNC() __syncwarp()

// Hessian scaling (App. A.4 step 2): blk holds K_nn (lower) and K_an after the up sweep;
// M_nn = D^{-1} K_nn D^{-1}, M_an = Y_aa K_an D^{-1}, D = L_nn L_nn^T.
__device__ void fl_hscale(const TreeArgs &a, const Node &q, int b, double *ws) {
    const SymDev &S = a.S;
    double *blk = a.X + (long long)b * S.nblk + q.boff;
    const double *Lb = a.Lt + q.boff;
    const double *Yaa = a.Yaa + q.uoff;
    const int nn = q.nn, na = q.na, nj = q.nj;
    double *Fnn = ws;               // nn x nn full
    double *Fan = Fnn + nn * nn;    // na x nn
    for (int idx = TID; idx < nn * nn; idx += NT) {
        int i = idx % nn, j = idx / nn;
        Fnn[idx] = (i >= j) ? blk[i + (long long)j * nj] : blk[j + (long long)i * nj];
    }
    for (int idx = TID; idx < na * nn; idx += NT) Fan[idx] = blk[nn + idx % na + (long long)(idx / na) * nj];
    SYNC();
    trsm_ll<true>(Lb, nj, nn, Fnn, nn, nn);
    trsm_rlt<true>(Lb, nj, nn, Fnn, nn, nn);
    trsm_llt<true>(Lb, nj, nn, Fnn, nn, nn);
    trsm_rl<true>(Lb, nj, nn, Fnn, nn, nn);
    if (na) {
        trsm_rlt<true>(Lb, nj, nn, Fan, na, na);
        trsm_rl<true>(Lb, nj, nn, Fan, na, na);
        mm<true>(blk + nn, nj, na, nn, na, 1.0, Yaa, 1, na, Fan, 1, na, false, false);
    }
    for (int idx = TID; idx < nn * nn; idx += NT) {
        int i = idx % nn, j = idx / nn;
        blk[i + (long long)j * nj] = (i >= j) ? 0.5 * (Fnn[idx] + Fnn[j + i * nn]) : 0.0;
    }
    SYNC();
}

// local front of the inverse Hessian (App. A.5 stages 3^-1, 2^-1 and the congruence of
// 1^-1): F = T^{-1} [K_nn K_an^T; K_an 0] T^{-T}, written as a full nj x nj matrix.
__device__ void fl_hinv_local(const TreeArgs &a, const Node &q, int b, double *ws, double *Fout) {
    const SymDev &S = a.S;
    const double *Xb = a.X + (long long)b * S.nblk;
    const double *blk = Xb + q.boff;
    const double *Lb = a.Lt + q.boff;
    const double *Ltan = Lb + q.nn;
    const int nn = q.nn, na = q.na, nj = q.nj;
    double *T1 = ws;                 // na x nn : M_an, later F_an
    double *T2 = T1 + na * nn;       // nn x nn : M_nn, later K_nn
    double *T3 = T2 + nn * nn;       // na x na : Z_aa, later F_aa
    double *T4 = T3 + na * na;       // nn x nn : D
    double *T5 = T4 + nn * nn;       // nn x nn : temp
    double *T6 = T5 + nn * nn;       // na x nn : K_an
    gather_aa<true>(S, q, Xb, T3);
    for (int idx = TID; idx < nn * nn; idx += NT) {
        int i = idx % nn, j = idx / nn;
        int kmax = i < j ? i : j;
        double s = 0.0;
        for (int r = 0; r <= kmax; ++r) s = fma(Lb[i + (long long)r * nj], Lb[j + (long long)r * nj], s);
        T4[idx] = s;
    }
    SYNC();
    for (int idx = TID; idx < na * nn; idx += NT) {
        int i = idx % na, c = idx / na;
        double s = 0.0;
        for (int r = 0; r < na; ++r) s = fma(T3[i + r * na], Ltan[r + (long long)c * nj], s);
        T1[idx] = blk[nn + i + (long long)c * nj] + s;
    }
    SYNC();
    for (int idx = TID; idx < nn * nn; idx += NT) {
        int i = idx % nn, j = idx / nn;
        double s = (i >= j) ? blk[i + (long long)j * nj] : blk[j + (long long)i * nj];
        for (int r = 0; r < na; ++r) {
            s = fma(Ltan[r + (long long)i * nj], blk[nn + r + (long long)j * nj], s);
            s = fma(T1[r + i * na], Ltan[r + (long long)j * nj], s);
        }
        T2[idx] = s;
    }
    SYNC();
    mm<true>(T5, nn, nn, nn, nn, 1.0, T4, 1, nn, T2, 1, nn, false, false);
    mm<true>(T2, nn, nn, nn, nn, 1.0, T5, 1, nn, T4, 1, nn, false, false);
    if (na) {
        mm<true>(T6, na, na, nn, nn, 1.0, T1, 1, na, T4, 1, nn, false, false);
        const double *R = a.Raa + q.uoff;
        trsm_ll<true>(R, na, na, T6, na, nn);
        trsm_llt<true>(R, na, na, T6, na, nn);
        for (int idx = TID; idx < na * nn; idx += NT) {
            int i = idx % na, c = idx / na;
            double s = 0.0;
            for (int r = 0; r < nn; ++r) s = fma(Ltan[i + (long long)r * nj], T2[r + c * nn], s);
            T1[idx] = T6[idx] + s;
        }
        SYNC();
        for (int idx = TID; idx < na * na; idx += NT) {
            int i = idx % na, j = idx / na;
            double s = 0.0;
            for (int r = 0; r < nn; ++r) {
                s = fma(Ltan[i + (long long)r * nj], T6[j + r * na], s);
                s = fma(T1[i + r * na], Ltan[j + (long long)r * nj], s);
            }
            T3[idx] = s;
        }
        SYNC();
    }
    for (int idx = TID; idx < nj * nj; idx += NT) {
        int i = idx % nj, j = idx / nj;
        double v;
        if (i < nn && j < nn) v = 0.5 * (T2[i + j * nn] + T2[j + i * nn]);
        else if (i >= nn && j < nn) v = T1[(i - nn) + j * na];
        else if (i < nn) v = T1[(j - nn) + i * na];
        else v = T3[(i - nn) + (j - nn) * na];
        Fout[idx] = v;
    }
    SYNC();
}

// local front of llt (App. A.6): F = [L_nn; L_an] [L_nn; L_an]^T, full nj x nj
__device__ void fl_llt_local(const TreeArgs &a, const Node &q, int b, double *Fout) {
    const SymDev &S = a.S;
    const double *blk = a.X + (long long)b * S.nblk + q.boff;
    const int nn = q.nn, nj = q.nj;
    for (int idx = TID; idx < nj * nj; idx += NT) {
        int i = idx % nj, j = idx / nj;
        int hi = i > j ? i : j, lo = i > j ? j : i;
        int kmax = lo < nn ? lo : nn - 1;
        double s = 0.0;
        for (int c = 0; c <= kmax; ++c) s = fma(blk[hi + (long long)c * nj], blk[lo + (long long)c * nj], s);
        Fout[idx] = s;
    }
    SYNC();
}

// projected inverse, flat part: Lt_out(alpha, nu) = L_an L_nn^{-1}; X_nn <- D^{-1}, X_an <- 0
__device__ void fl_pinv_prep(const TreeArgs &a, const Node &q, int b, double *ws) {
    const SymDev &S = a.S;
    double *blk = a.X + (long long)b * S.nblk + q.boff;
    double *Ob = a.Lt_out + (long long)b * S.nblk + q.boff;
    const int nn = q.nn, na = q.na, nj = q.nj;
    double *Lw = ws;                // nn x nn  L_nn
    double *T1 = Lw + nn * nn;      // na x nn  L_an -> Lt
    double *T2 = T1 + na * nn;      // nn x nn  L_nn^{-1}
    for (int idx = TID; idx < nn * nn; idx += NT) {
        int i = idx % nn, j = idx / nn;
        Lw[idx] = (i >= j) ? blk[i + (long long)j * nj] : 0.0;
        T2[idx] = (i == j) ? 1.0 : 0.0;
    }
    for (int idx = TID; idx < na * nn; idx += NT) T1[idx] = blk[nn + idx % na + (long long)(idx / na) * nj];
    SYNC();
    if (na) trsm_rl<true>(Lw, nn, nn, T1, na, na);
    trsm_ll<true>(Lw, nn, nn, T2, nn, nn);
    for (int idx = TID; idx < nn * nn; idx += NT) {
        int i = idx % nn, j = idx / nn;
        double s = 0.0;
        if (i >= j)
            for (int r = i; r < nn; ++r) s = fma(T2[r + i * nn], T2[r + j * nn], s);
        blk[i + (long long)j * nj] = s;
        Ob[i + (long long)j * nj] = Lw[idx];
    }
    for (int idx = TID; idx < na * nn; idx += NT) {
        int i = idx % na, c = idx / na;
        blk[nn + i + (long long)c * nj] = 0.0;
        Ob[nn + i + (long long)c * nj] = T1[idx];
    }
    SYNC();
}

#undef TID
#undef NT
#undef SYNC

// Hessian scaling for supernodes with a single column, one THREAD per (supernode, matrix):
// M_nn = K_nn / l^4, M_an = Y_aa (K_an / l^2), l = L_nn.  Used for batches (Schur-complement
// assembly), where one warp per supernode would be issue-bound; consecutive lanes take
// consecutive supernodes of the same matrix so the block entries they touch are contiguous.
__global__ void __launch_bounds__(256) hscale_nn1_kernel(SmallArgs a) {
    const TreeArgs &t = a.t;
    const long long nsn = t.S.nsn, total = nsn * t.B;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const int b = (int)(idx / nsn), k = (int)(idx - (long long)b * nsn);
        if (t.S.nn[k] != 1) continue;
        const int na = t.S.na[k];
        const long long boff = t.S.blkptr[k];
        double *blk = t.X + (long long)b * t.S.nblk + boff;
        const double *Y = t.Yaa + t.S.updptr[k];
        const double l = t.Lt[boff];
        const double inv = 1.0 / (l * l);
        double kv[7];
#pragma unroll
        for (int q = 0; q < 7; ++q) kv[q] = (q < na) ? blk[1 + q] * inv : 0.0;
        blk[0] = blk[0] * inv * inv;
#pragma unroll
        for (int r = 0; r < 7; ++r) {
            if (r < na) {
                double s = 0.0;
#pragma unroll
                for (int q = 0; q < 7; ++q)
                    if (q < na) s = fma(Y[r + q * na], kv[q], s);
                blk[1 + r] = s;
            }
        }
    }
}

#define FLAT_THREADS 128
#define FLAT_WS (4 * 64 + 8)

template <int OP>
__global__ void __launch_bounds__(FLAT_THREADS) flat_small_kernel(SmallArgs a) {
    __shared__ double smem[(FLAT_THREADS / 32) * FLAT_WS];
    double *ws = smem + (threadIdx.x >> 5) * FLAT_WS;
    const TreeArgs &t = a.t;
    const long long nsn = a.list ? a.nlist : t.S.nsn;     // all supernodes, or only those in `list`
    const long long total = nsn * t.B;
    const long long nwarps = (long long)gridDim.x * (FLAT_THREADS / 32);
    for (long long item = (long long)blockIdx.x * (FLAT_THREADS / 32) + (threadIdx.x >> 5); item < total; item += nwarps) {
        const int b = (int)(item / nsn);
        int k = (int)(item - (long long)b * nsn);
        if (a.list) k = a.list[k];
        Node q = node_of(t.S, k);
        if (OP == FL_COMPL) op_compl<true>(t, q, b, ws);
        else if (OP == FL_HPREP) op_hprep<true>(t, q);
        else if (OP == FL_HPREP_INV) op_hprep_inv<true>(t, q);
        else if (OP == FL_HSCALE) fl_hscale(t, q, b, ws);
        else if (OP == FL_HINV_LOCAL) fl_hinv_local(t, q, b, ws, a.F + (long long)b * a.M.nsq + a.M.sqptr[k]);
        else if (OP == FL_LLT_LOCAL) fl_llt_local(t, q, b, a.F + (long long)b * a.M.nsq + a.M.sqptr[k]);
        else if (OP == FL_PINV_PREP) fl_pinv_prep(t, q, b, ws);
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------
// sweeps
//
// Slot colouring.  Every vertex gets a slot in 0..7 such that the vertices of a clique have
// distinct slots (a chordal graph with cliques of at most 8 vertices is 8-colourable; the
// colouring is built top-down over the clique tree by small_setup).  A frontal matrix is
// then held at tile position (slot(row), slot(col)) of an 8 x 8 tile, and because the
// separator of a child is contained in the clique of its parent, extend-add is
// position-preserving: the update matrix computed at a child already sits where the parent
// needs it.  In the bottom-up sweeps the tile lives in registers (lane = i + 8*(j & 3) holds
// entries (i, j) and (i, j + 4), j = lane >> 3), the pivot column is broadcast with warp
// shuffles and nothing is exchanged through memory between consecutive supernodes of a
// chain.  The top-down sweep keeps the tile in shared memory (every entry of Z_aa is read
// by several lanes).
//
// Staging.  A single warp has no memory-level parallelism of its own and an L2 hit costs
// ~310 cycles, so a sweep never loads from global memory inside a step: the steps of a task
// are cut into chunks (at most 32 steps, 256 block entries); all lanes fetch the
// descriptors, matrix entries and factor entries of chunk c+1 with coalesced loads while
// chunk c is being processed, park them in registers and drop them into the other half of
// a double-buffered shared-memory stage at the chunk boundary.
// ---------------------------------------------------------------------------------------
#define SW_THREADS 128
#define SW_WARPS (SW_THREADS / 32)
#define CH_STEPS 32
#define CH_BLK 256       // doubles of matrix / factor entries per chunk
#define CH_SQ 512        // doubles of local fronts per chunk (add sweep)
#define F_CARRY 1        // the previous step of the task is a child (up) / the parent (down)
#define F_WR 2           // write the update matrix to its global tile
#define F_OCH 4          // children other than the previous step contribute through global tiles

// per-warp shared memory (doubles): descriptors [2][32 x 8 ints], X stage [2][256],
// Y stage [2][256 or 512] (factor / local fronts), then the Z tile [64] (down sweep) or two
// ping-pong tiles with zero pads [2][80] (up sweeps)
__host__ __device__ constexpr int sweep_ws(int ybuf, bool down) { return 256 + 512 + 2 * ybuf + (down ? 64 : 160); }

struct ChunkRegs {
    int4 d0, d1;
    double x[8];
};

template <int NY>
struct YRegs {
    double y[NY > 0 ? NY : 1];
};

__device__ __forceinline__ void chunk_load(const int4 *steps, const int4 c0, const double *xsrc, int lane, ChunkRegs &r) {
    // c0 = {p_begin, p_end, blk_lo, blk_hi}
    r.d0 = make_int4(0, 0, 0, 0);
    r.d1 = r.d0;
    if (c0.x + lane < c0.y) {
        r.d0 = steps[2 * (c0.x + lane)];
        r.d1 = steps[2 * (c0.x + lane) + 1];
    }
#pragma unroll
    for (int t = 0; t < 8; ++t) {
        const int o = c0.z + lane + 32 * t;
        r.x[t] = (o < c0.w) ? xsrc[o] : 0.0;
    }
}

template <int NY>
__device__ __forceinline__ void chunk_load_y(const double *ysrc, int lo, int hi, int lane, YRegs<NY> &r) {
#pragma unroll
    for (int t = 0; t < NY; ++t) {
        const int o = lo + lane + 32 * t;
        r.y[t] = (o < hi) ? ysrc[o] : 0.0;
    }
}

__device__ __forceinline__ void chunk_store(int *descS, double *xS, int lane, const ChunkRegs &r) {
    reinterpret_cast<int4 *>(descS)[2 * lane] = r.d0;
    reinterpret_cast<int4 *>(descS)[2 * lane + 1] = r.d1;
#pragma unroll
    for (int t = 0; t < 8; ++t) xS[lane + 32 * t] = r.x[t];
}

template <int NY>
__device__ __forceinline__ void chunk_store_y(double *yS, int lane, const YRegs<NY> &r) {
#pragma unroll
    for (int t = 0; t < NY; ++t) yS[lane + 32 * t] = r.y[t];
}

__device__ __forceinline__ void wait_deps(const TaskSched &T, const unsigned *done, int t, int B, int b, unsigned epoch, int lane) {
    if (lane == 0) {
        for (int d = T.dep_ptr[t]; d < T.dep_ptr[t + 1]; ++d) {
            const unsigned *flag = done + (long long)T.dep_idx[d] * B + b;
            while (ld_acquire(flag) != epoch) __nanosleep(32);
        }
    }
    __syncwarp();
}

// new lane (i, j) takes the old entry (mi, mj) of the register tile; indices >= 8 give zero
__device__ __forceinline__ void tile_permute(double &uA, double &uB, int mi, int mjA, int mjB) {
    const int sA = (mi & 7) + 8 * (mjA & 3), sB = (mi & 7) + 8 * (mjB & 3);
    const double a1 = __shfl_sync(FULLMASK, uA, sA), a2 = __shfl_sync(FULLMASK, uB, sA);
    const double b1 = __shfl_sync(FULLMASK, uA, sB), b2 = __shfl_sync(FULLMASK, uB, sB);
    uA = (mi < 8 && mjA < 8) ? ((mjA & 4) ? a2 : a1) : 0.0;
    uB = (mi < 8 && mjB < 8) ? ((mjB & 4) ? b2 : b1) : 0.0;
}

struct UpCtx {
    double *xb, *ug;          // this matrix: blocks, update-matrix tiles
    const double *xsb, *ysb;  // staged inputs of the chunk, biased so that [blkptr] / [sqptr] index them
    const int *och;
    int *fail;
    int lane, i, jA, jB, eA, eB;
};

// One supernode of a bottom-up sweep.  (pi, pjA, pjB) = positions inside the clique of the
// rows this lane holds, rowslot = tile row of every position.  In the slot layout these come
// from the step descriptor; in the position layout of a uniform run they are the lane's own
// coordinates and the identity, i.e. loop invariants that the compiler hoists.
template <int OP>
__device__ __forceinline__ void up_step(const UpCtx &c, int nn, int na, int flags, int boff, unsigned rowslot, int pi, int pjA,
                                        int pjB, const int4 e1, double &uA, double &uB) {
    const int nj = nn + na;
    const int i = c.i, jA = c.jA, jB = c.jB;
    const bool vi = pi < nj, vA = vi && pjA < nj, vB = vi && pjB < nj;
    double *blk = c.xb + boff;
    double bA = 0.0, bB = 0.0;
    if (OP == SW_ADD) {
        const double *fl = c.ysb + e1.w;
        if (vA) bA = fl[pi + pjA * nj];
        if (vB) bB = fl[pi + pjB * nj];
    } else {
        const double *xs = c.xsb + boff;
        if (vA) {
            const int lo = min(pi, pjA), hi = max(pi, pjA);
            if (lo < nn) bA = xs[hi + lo * nj];
        }
        if (vB) {
            const int lo = min(pi, pjB), hi = max(pi, pjB);
            if (lo < nn) bB = xs[hi + lo * nj];
        }
    }
    if (!(flags & F_CARRY)) uA = uB = 0.0;
    if (flags & F_OCH) {
        for (int q = 0; q < e1.z; ++q) {
            const double *tile = c.ug + (long long)c.och[e1.y + q] * 64;
            uA += __ldcg(tile + c.eA);
            uB += __ldcg(tile + c.eB);
        }
    }
    double fA = uA + bA, fB = uB + bB;
    if (OP == SW_ADD) {
        if (vA && pjA < nn) blk[pi + pjA * nj] = (pi >= pjA) ? fA : 0.0;
        if (vB && pjB < nn) blk[pi + pjB * nj] = (pi >= pjB) ? fB : 0.0;
        uA = (vA && pi >= nn && pjA >= nn) ? fA : 0.0;
        uB = (vB && pi >= nn && pjB >= nn) ? fB : 0.0;
    } else if (OP == SW_HUP) {
        const double *ls = c.ysb + boff;
        double accA = fA, accB = fB;
        const bool ri = vi && pi >= nn, rA = pjA >= nn && pjA < nj, rB = pjB >= nn && pjB < nj;
        for (int r = 0; r < nn; ++r) {
            const int sr = (rowslot >> (4 * r)) & 15, src = (sr & 3) * 8;
            const double x = (sr & 4) ? fB : fA;
            const double Fi = __shfl_sync(FULLMASK, x, i + src);
            const double FjA = __shfl_sync(FULLMASK, x, jA + src);
            const double FjB = __shfl_sync(FULLMASK, x, jB + src);
            const double lI = ri ? ls[pi + r * nj] : 0.0;
            const double lJA = rA ? ls[pjA + r * nj] : 0.0;
            const double lJB = rB ? ls[pjB + r * nj] : 0.0;
            double kar = Fi;
            for (int s2 = 0; s2 < nn; ++s2) {
                const int ss = (rowslot >> (4 * s2)) & 15;
                const double Fsr = __shfl_sync(FULLMASK, x, ss + src);
                const double lIs = ri ? ls[pi + s2 * nj] : 0.0;
                kar = fma(-lIs, Fsr, kar);
            }
            accA = fma(-lI, FjA, accA);
            accA = fma(-kar, lJA, accA);
            accB = fma(-lI, FjB, accB);
            accB = fma(-kar, lJB, accB);
            if (vi && (jA == sr || jB == sr)) blk[pi + r * nj] = (pi >= nn) ? kar : (pi >= r ? Fi : 0.0);
        }
        uA = (vA && ri && rA) ? accA : 0.0;
        uB = (vB && ri && rB) ? accB : 0.0;
    } else {   // SW_CHOL, right-looking over the pivots of the supernode
        for (int r = 0; r < nn; ++r) {
            const int sr = (rowslot >> (4 * r)) & 15, src = (sr & 3) * 8;
            const double x = (sr & 4) ? fB : fA;
            const double d = __shfl_sync(FULLMASK, x, sr + src);
            const double Fi = __shfl_sync(FULLMASK, x, i + src);
            const double FjA = __shfl_sync(FULLMASK, x, jA + src);
            const double FjB = __shfl_sync(FULLMASK, x, jB + src);
            const bool bad = !(d > 0.0);
            if (bad && c.lane == 0) *c.fail = 1;
            const double rs = bad ? 1.0 : rsqrt(d);
            const double li = Fi * rs, ljA = FjA * rs, ljB = FjB * rs;
            if (vi && (jA == sr || jB == sr)) {
                double dg = d * rs;
                dg = fma(fma(-dg, dg, d), 0.5 * rs, dg);      // one Newton step: sqrt(d) to < 1 ulp
                blk[pi + r * nj] = (pi == r) ? (bad ? 1.0 : dg) : (pi > r ? li : 0.0);
            }
            fA = fma(-li, ljA, fA);
            fB = fma(-li, ljB, fB);
            if (i == sr || jA == sr) fA = 0.0;
            if (i == sr || jB == sr) fB = 0.0;
        }
        uA = vA ? fA : 0.0;
        uB = vB ? fB : 0.0;
    }
    if (flags & F_WR) {
        double *tile = c.ug + (long long)e1.x * 64;
        tile[c.eA] = uA;
        tile[c.eB] = uB;
    }
}

// Uniform run with one column per supernode (band matrices, trees of small separators): the
// hot case.  Position layout in two ping-pong shared-memory tiles (entry 64.. of a tile is a
// zero pad used instead of masks); every lane's role, offsets and predicates are fixed for
// the whole run, so a step is ~30 instructions: P0 front = own block entry + child's update
// matrix shifted by one, P1 the rank-2 (Hessian) / rank-1 (Cholesky) update with the pivot
// column read back from the tile.
template <int OP>
__device__ __forceinline__ void up_run_fast(const UpCtx &c, double *T, int na, int run, int boff, int sqoff,
                                            unsigned slotpos_head, unsigned slotpos_last, double &uA, double &uB) {
    const int lane = c.lane, i = c.i, jA = c.jA, jB = c.jB, eA = c.eA, eB = c.eB;
    const int nj = na + 1;
    double *T0 = T, *T1 = T + 80;
    // the child's update matrix (slot registers) -> T1 in the child's position layout
    T1[lane] = 0.0;
    T1[lane + 32] = 0.0;
    __syncwarp();
    {
        const int pi = (slotpos_head >> (4 * i)) & 15, pA = (slotpos_head >> (4 * jA)) & 15, pB = (slotpos_head >> (4 * jB)) & 15;
        if (pi < na && pA < na) T1[(1 + pi) + 8 * (1 + pA)] = uA;
        if (pi < na && pB < na) T1[(1 + pi) + 8 * (1 + pB)] = uB;
    }
    __syncwarp();
    const bool in = i < nj, inA = in && jA < nj, inB = in && jB < nj;
    const bool pbA = inA && (i == 0 || jA == 0), pbB = inB && i == 0;
    const int obA = max(i, jA), obB = max(i, jB);
    const int fA_off = i + jA * nj, fB_off = i + jB * nj;
    const int sA = (i + 1 <= na && jA + 1 <= na) ? (i + 1) + 8 * (jA + 1) : 64;
    const int sB = (i + 1 <= na && jB + 1 <= na) ? (i + 1) + 8 * (jB + 1) : 64;
    const int ci = in ? i : 64, cA = (jA < nj) ? jA : 64, cB = (jB < nj) ? jB : 64;
    const bool li_ok = in && i >= 1, lA_ok = jA >= 1 && jA < nj, lB_ok = jB < nj;
    const bool wA = inA && jA != 0, wB = inB;
    const bool outK = in && jA == 0;
    const double *xs = c.xsb + boff, *ys = c.ysb + (OP == SW_ADD ? sqoff : boff);
    double *blk = c.xb + boff;
    const int ystep = (OP == SW_ADD) ? nj * nj : nj;
    for (int q = 0; q < run; ++q) {
        double *cur = (q & 1) ? T1 : T0;
        const double *prev = (q & 1) ? T0 : T1;
        double bA = 0.0, bB = 0.0;
        if (OP == SW_ADD) {
            if (inA) bA = ys[fA_off];
            if (inB) bB = ys[fB_off];
        } else {
            if (pbA) bA = xs[obA];
            if (pbB) bB = xs[obB];
        }
        const double fA = bA + prev[sA], fB = bB + prev[sB];
        cur[eA] = fA;
        cur[eB] = fB;
        __syncwarp();
        if (OP == SW_ADD) {
            if (outK) blk[i] = fA;
        } else if (OP == SW_HUP) {
            const double F0 = cur[0], Fi = cur[ci], FA = cur[cA], FB = cur[cB];
            const double li = li_ok ? ys[i] : 0.0, lA = lA_ok ? ys[jA] : 0.0, lB = lB_ok ? ys[jB] : 0.0;
            const double kar = fma(-li, F0, Fi);
            double vA = fma(-li, FA, fA), vB = fma(-li, FB, fB);
            vA = fma(-kar, lA, vA);
            vB = fma(-kar, lB, vB);
            if (wA) cur[eA] = vA;
            if (wB) cur[eB] = vB;
            if (outK) blk[i] = kar;
            __syncwarp();
        } else {
            const double d = cur[0], Fi = cur[ci], FA = cur[cA], FB = cur[cB];
            const bool bad = !(d > 0.0);
            if (bad && lane == 0) *c.fail = 1;
            const double rs = bad ? 1.0 : rsqrt(d);
            const double li = Fi * rs, lA = FA * rs, lB = FB * rs;
            if (wA) cur[eA] = fma(-li, lA, fA);
            if (wB) cur[eB] = fma(-li, lB, fB);
            if (outK) {
                double dg = d * rs;
                dg = fma(fma(-dg, dg, d), 0.5 * rs, dg);
                blk[i] = (i == 0) ? (bad ? 1.0 : dg) : li;
            }
            __syncwarp();
        }
        xs += nj;
        ys += ystep;
        blk += nj;
    }
    // the last update matrix back into slot registers
    {
        const double *last = ((run - 1) & 1) ? T1 : T0;
        const int pi = (slotpos_last >> (4 * i)) & 15, pA = (slotpos_last >> (4 * jA)) & 15, pB = (slotpos_last >> (4 * jB)) & 15;
        const bool ok = pi >= 1 && pi < nj;
        uA = (ok && pA >= 1 && pA < nj) ? last[pi + 8 * pA] : 0.0;
        uB = (ok && pB >= 1 && pB < nj) ? last[pi + 8 * pB] : 0.0;
    }
    __syncwarp();
}

template <int OP>
__global__ void __launch_bounds__(SW_THREADS) sweep_up_kernel(SmallArgs a) {
    extern __shared__ double dsm[];
    constexpr int YB = (OP == SW_ADD) ? CH_SQ : CH_BLK;
    constexpr int NY = (OP == SW_ADD) ? 16 : (OP == SW_HUP ? 8 : 0);
    constexpr int WS = sweep_ws(OP == SW_CHOL ? 0 : YB, false);
    const int lane = threadIdx.x & 31;
    double *w = dsm + (threadIdx.x >> 5) * WS;
    int *descS = reinterpret_cast<int *>(w);
    double *xS = w + 256, *yS = w + 768;
    double *tiles = w + WS - 160;      // two 8 x 8 tiles + zero pads
    tiles[64 + (lane & 15)] = 0.0;
    tiles[144 + (lane & 15)] = 0.0;
    __syncwarp();
    const TreeArgs &t = a.t;
    const int total = t.T.ntask * t.B;
    const int4 *steps = a.M.up_steps;
    const int4 *chunks = (OP == SW_ADD) ? a.M.add_chunks : a.M.up_chunks;
    const int *chunk_ptr = (OP == SW_ADD) ? a.M.add_chunk_ptr : a.M.up_chunk_ptr;
    UpCtx c;
    c.lane = lane;
    c.i = lane & 7; c.jA = lane >> 3; c.jB = c.jA + 4;
    c.eA = c.i + 8 * c.jA; c.eB = c.i + 8 * c.jB;
    c.och = a.M.och;
    const int i = c.i, jA = c.jA, jB = c.jB;
    for (;;) {
        int item = 0;
        if (lane == 0) item = (int)atomicAdd(t.counter, 1u);
        item = __shfl_sync(FULLMASK, item, 0);
        if (item >= total) break;
        const int tk = item / t.B, b = item - tk * t.B;
        wait_deps(t.T, t.done, tk, t.B, b, t.epoch, lane);
        c.xb = t.X + (long long)b * t.S.nblk;
        c.ug = t.upd + (long long)b * a.M.ntiles * 64;
        c.fail = t.fail + b;
        const double *ysrc = (OP == SW_ADD) ? a.F + (long long)b * a.M.nsq : t.Lt;
        const int c0 = chunk_ptr[tk], c1 = chunk_ptr[tk + 1];
        ChunkRegs R;
        YRegs<NY> RY;
        {
            const int4 ch = chunks[2 * c0], ch2 = chunks[2 * c0 + 1];
            chunk_load(steps, ch, c.xb, lane, R);
            if (OP == SW_HUP) chunk_load_y<NY>(ysrc, ch.z, ch.w, lane, RY);
            if (OP == SW_ADD) chunk_load_y<NY>(ysrc, ch2.x, ch2.y, lane, RY);
            chunk_store(descS, xS, lane, R);
            if (NY) chunk_store_y<NY>(yS, lane, RY);
            __syncwarp();
        }
        double uA = 0.0, uB = 0.0;
        for (int cc = c0; cc < c1; ++cc) {
            const int buf = (cc - c0) & 1;
            const int4 ch = chunks[2 * cc], ch2 = chunks[2 * cc + 1];
            if (cc + 1 < c1) {
                const int4 nh = chunks[2 * cc + 2], nh2 = chunks[2 * cc + 3];
                chunk_load(steps, nh, c.xb, lane, R);
                if (OP == SW_HUP) chunk_load_y<NY>(ysrc, nh.z, nh.w, lane, RY);
                if (OP == SW_ADD) chunk_load_y<NY>(ysrc, nh2.x, nh2.y, lane, RY);
            }
            const int *dsb = descS + buf * 256;
            c.xsb = xS + buf * 256 - ch.z;
            c.ysb = yS + buf * YB - ((OP == SW_ADD) ? ch2.x : ch.z);
            int p = ch.x;
            while (p < ch.y) {
                const int4 e0 = reinterpret_cast<const int4 *>(dsb)[2 * (p - ch.x)];
                const int4 e1 = reinterpret_cast<const int4 *>(dsb)[2 * (p - ch.x) + 1];
                // e0 = {nn | na<<4 | flags<<8 | run<<16, blkptr, rowslot, slotpos}, e1 = {upd tile, och_beg, och_cnt, sqptr}
                const int nn = e0.x & 15, na = (e0.x >> 4) & 15, flags = (e0.x >> 8) & 255;
                const unsigned rowslot = (unsigned)e0.z, slotpos = (unsigned)e0.w;
                int run = e0.x >> 16;
                if (run > ch.y - p) run = ch.y - p;
                if (run >= 2 && nn == 1) {
                    const int4 l0 = reinterpret_cast<const int4 *>(dsb)[2 * (p + run - 1 - ch.x)];
                    up_run_fast<OP>(c, tiles, na, run, e0.y, e1.w, slotpos, (unsigned)l0.w, uA, uB);
                    p += run;
                } else {
                    const int pi = (slotpos >> (4 * i)) & 15, pjA = (slotpos >> (4 * jA)) & 15, pjB = (slotpos >> (4 * jB)) & 15;
                    up_step<OP>(c, nn, na, flags, e0.y, rowslot, pi, pjA, pjB, e1, uA, uB);
                    ++p;
                }
            }
            if (cc + 1 < c1) {
                chunk_store(descS + (buf ^ 1) * 256, xS + (buf ^ 1) * 256, lane, R);
                if (NY) chunk_store_y<NY>(yS + (buf ^ 1) * YB, lane, RY);
            }
            __syncwarp();
        }
        __threadfence();
        __syncwarp();
        if (lane == 0) st_release(t.done + (long long)tk * t.B + b, t.epoch);
    }
}

struct DnCtx {
    double *xb;
    const double *xsb, *ysb;
    const int *aaidx;
    double *Z;
    int lane, i, jA, jB;
};

// One supernode of the top-down sweep.  Z tile index of (row slot a, column slot b) is
// (o + a + 8 b) & 63: o = 0 in the slot layout; in the position layout of a uniform run the
// tile is addressed by clique positions and moving to the child is o -= 9 nn.
__device__ __forceinline__ void down_step(const DnCtx &c, int nn, int na, int flags, int boff, unsigned rowslot, int pi, int pjA,
                                          int pjB, int uoff, int o) {
    const int nj = nn + na;
    const int i = c.i;
    const bool vi = pi < nj, vA = vi && pjA < nj, vB = vi && pjB < nj;
    double *blk = c.xb + boff;
    const double *xs = c.xsb + boff, *ls = c.ysb + boff;
    double *Z = c.Z;
    if (!(flags & F_CARRY) && na) {
        // Z_aa of the ancestors from global memory (another task / an earlier subtree)
        const int *ai = c.aaidx + uoff;
        if (vA && pi >= nn && pjA >= nn) Z[(o + i + 8 * c.jA) & 63] = __ldcg(c.xb + ai[(pi - nn) + (pjA - nn) * na]);
        if (vB && pi >= nn && pjB >= nn) Z[(o + i + 8 * c.jB) & 63] = __ldcg(c.xb + ai[(pi - nn) + (pjB - nn) * na]);
        __syncwarp();
    }
    // ---- P0: Z_an for the entries (alpha row, nu column)
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int j = h ? c.jB : c.jA, pj = h ? pjB : pjA;
        if (vi && pi >= nn && pj < nn) {
            double acc = xs[pi + pj * nj];
            for (int q = 0; q < na; ++q) {
                const int sq = (rowslot >> (4 * (nn + q))) & 15;
                acc = fma(-Z[(o + i + 8 * sq) & 63], ls[nn + q + pj * nj], acc);
            }
            Z[(o + i + 8 * j) & 63] = acc;
            Z[(o + j + 8 * i) & 63] = acc;
            blk[pi + pj * nj] = acc;
        }
    }
    __syncwarp();
    // ---- P1: Z_nn, evaluated for the (larger, smaller) position pair so that both triangles agree
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int j = h ? c.jB : c.jA, pj = h ? pjB : pjA;
        if (pi < nn && pj < nn) {
            const bool ge = pi >= pj;
            const int ph = ge ? pi : pj, pl = ge ? pj : pi;
            const int sh = ge ? i : j, sl = ge ? j : i;
            double s = 0.0;
            for (int q = 0; q < na; ++q) {
                const int sq = (rowslot >> (4 * (nn + q))) & 15;
                const double lh = ls[nn + q + ph * nj], ll = ls[nn + q + pl * nj];
                s = fma(lh, xs[nn + q + pl * nj], s);
                s = fma(Z[(o + sq + 8 * sh) & 63], ll, s);
                s = fma(ll, xs[nn + q + ph * nj], s);
                s = fma(Z[(o + sq + 8 * sl) & 63], lh, s);
            }
            const double z = xs[ph + pl * nj] - 0.5 * s;
            Z[(o + i + 8 * j) & 63] = z;
            if (ge) blk[pi + pj * nj] = z;
        }
    }
    __syncwarp();
}

// move the shared-memory tile between layouts: new entry (i, j) <- old entry (mi, mj) read with
// offset o_old, written with offset o_new (indices >= 8: entry left untouched)
__device__ __forceinline__ void ztile_permute(double *Z, int i, int jA, int jB, int mi, int mjA, int mjB, int o_old, int o_new) {
    double vA = 0.0, vB = 0.0;
    const bool okA = mi < 8 && mjA < 8, okB = mi < 8 && mjB < 8;
    if (okA) vA = Z[(o_old + mi + 8 * mjA) & 63];
    if (okB) vB = Z[(o_old + mi + 8 * mjB) & 63];
    __syncwarp();
    if (okA) Z[(o_new + i + 8 * jA) & 63] = vA;
    if (okB) Z[(o_new + i + 8 * jB) & 63] = vB;
    __syncwarp();
}

// Uniform run with one column per supernode, top-down: position layout with a rotating tile
// offset, fixed lane roles.  Lanes (i, 0), i = 1..na, compute Z_an(i) = M_an(i) - sum_q
// Z_aa(i, q) Lt(q); the pivot entry Z_nn = M_nn - sum_q Lt(q) (M_an(q) + Z_an(q)) is a
// shuffle reduction over the same lanes.
__device__ __forceinline__ void down_run_fast(const DnCtx &c, int na, int run, int boff, unsigned rowslot_head, unsigned slotpos_last) {
    const int lane = c.lane, i = c.i, jA = c.jA, jB = c.jB;
    const int nj = na + 1;
    double *Z = c.Z;
    ztile_permute(Z, i, jA, jB, (i >= 1 && i < nj) ? (int)((rowslot_head >> (4 * i)) & 15) : 15,
                  (jA >= 1 && jA < nj) ? (int)((rowslot_head >> (4 * jA)) & 15) : 15,
                  (jB < nj) ? (int)((rowslot_head >> (4 * jB)) & 15) : 15, 0, 0);
    const bool col0 = jA == 0 && i < nj, p0 = col0 && i >= 1;
    const double *xs = c.xsb + boff, *ls = c.ysb + boff;
    double *blk = c.xb + boff;
    int o = 0;
    for (int q = 0; q < run; ++q) {
        double m = 0.0, acc = 0.0, tsum = 0.0;
        if (col0) m = xs[i];
        if (p0) {
            // all loads first (independent of each other), then the FMA chain
            const int zb = o + i + 8;
            double zr[7], lr[7];
#pragma unroll
            for (int r = 0; r < 7; ++r) {
                zr[r] = (r < na) ? Z[(zb + 8 * r) & 63] : 0.0;
                lr[r] = (r < na) ? ls[1 + r] : 0.0;
            }
            const double lself = ls[i];
            double a0 = m, a1 = 0.0;
#pragma unroll
            for (int r = 0; r < 7; r += 2) {
                a0 = fma(-zr[r], lr[r], a0);
                if (r + 1 < 7) a1 = fma(-zr[r + 1], lr[r + 1], a1);
            }
            acc = a0 + a1;
            tsum = lself * (m + acc);
        }
        tsum += __shfl_xor_sync(FULLMASK, tsum, 1);
        tsum += __shfl_xor_sync(FULLMASK, tsum, 2);
        tsum += __shfl_xor_sync(FULLMASK, tsum, 4);
        if (p0) {
            Z[(o + i) & 63] = acc;
            Z[(o + 8 * i) & 63] = acc;
            blk[i] = acc;
        }
        if (lane == 0) {
            const double z = m - tsum;
            Z[o & 63] = z;
            blk[0] = z;
        }
        __syncwarp();
        o = (o - 9) & 63;
        xs -= nj;
        ls -= nj;
        blk -= nj;
    }
    o = (o + 9) & 63;
    ztile_permute(Z, i, jA, jB, (slotpos_last >> (4 * i)) & 15, (slotpos_last >> (4 * jA)) & 15, (slotpos_last >> (4 * jB)) & 15, o, 0);
}

// top-down sweep: Z_an = M_an - Z_aa Lt, Z_nn = M_nn - Lt^T M_an - Z_an^T Lt (App. A.4 step 3;
// with M = (D^{-1}, 0) this is the projected inverse, App. A.2)
__global__ void __launch_bounds__(SW_THREADS) sweep_down_kernel(SmallArgs a) {
    extern __shared__ double dsm[];
    constexpr int WS = sweep_ws(CH_BLK, true);
    const int lane = threadIdx.x & 31;
    double *w = dsm + (threadIdx.x >> 5) * WS;
    int *descS = reinterpret_cast<int *>(w);
    double *xS = w + 256, *yS = w + 768;
    const TreeArgs &t = a.t;
    const int total = t.T.ntask * t.B;
    const int4 *steps = a.M.down_steps;
    const int4 *chunks = a.M.down_chunks;
    DnCtx c;
    c.lane = lane;
    c.i = lane & 7; c.jA = lane >> 3; c.jB = c.jA + 4;
    c.Z = w + 1280;
    c.aaidx = t.S.aaidx;
    const int i = c.i, jA = c.jA, jB = c.jB;
    for (;;) {
        int item = 0;
        if (lane == 0) item = (int)atomicAdd(t.counter, 1u);
        item = __shfl_sync(FULLMASK, item, 0);
        if (item >= total) break;
        const int tk = item / t.B, b = item - tk * t.B;
        wait_deps(t.T, t.done, tk, t.B, b, t.epoch, lane);
        c.xb = t.X + (long long)b * t.S.nblk;
        const double *lsrc = t.Lt + (long long)b * a.ltstride;
        const int c0 = a.M.down_chunk_ptr[tk], c1 = a.M.down_chunk_ptr[tk + 1];
        ChunkRegs R;
        YRegs<8> RY;
        {
            const int4 ch = chunks[2 * c0];
            chunk_load(steps, ch, c.xb, lane, R);
            chunk_load_y<8>(lsrc, ch.z, ch.w, lane, RY);
            chunk_store(descS, xS, lane, R);
            chunk_store_y<8>(yS, lane, RY);
            __syncwarp();
        }
        for (int cc = c0; cc < c1; ++cc) {
            const int buf = (cc - c0) & 1;
            const int4 ch = chunks[2 * cc];
            if (cc + 1 < c1) {
                const int4 nh = chunks[2 * cc + 2];
                chunk_load(steps, nh, c.xb, lane, R);
                chunk_load_y<8>(lsrc, nh.z, nh.w, lane, RY);
            }
            const int *dsb = descS + buf * 256;
            c.xsb = xS + buf * 256 - ch.z;
            c.ysb = yS + buf * 256 - ch.z;
            int p = ch.x;
            while (p < ch.y) {
                const int4 e0 = reinterpret_cast<const int4 *>(dsb)[2 * (p - ch.x)];
                const int4 e1 = reinterpret_cast<const int4 *>(dsb)[2 * (p - ch.x) + 1];
                // e0 = {nn | na<<4 | flags<<8 | run<<16, blkptr, rowslot, slotpos}, e1 = {updptr (aaidx offset), 0, 0, 0}
                const int nn = e0.x & 15, na = (e0.x >> 4) & 15, flags = (e0.x >> 8) & 255;
                const unsigned rowslot = (unsigned)e0.z, slotpos = (unsigned)e0.w;
                int run = e0.x >> 16;
                if (run > ch.y - p) run = ch.y - p;
                if (run >= 2 && nn == 1) {
                    const int4 l0 = reinterpret_cast<const int4 *>(dsb)[2 * (p + run - 1 - ch.x)];
                    down_run_fast(c, na, run, e0.y, rowslot, (unsigned)l0.w);
                    p += run;
                } else {
                    const int pi = (slotpos >> (4 * i)) & 15, pjA = (slotpos >> (4 * jA)) & 15, pjB = (slotpos >> (4 * jB)) & 15;
                    down_step(c, nn, na, flags, e0.y, rowslot, pi, pjA, pjB, e1.x, 0);
                    ++p;
                }
            }
            if (cc + 1 < c1) {
                chunk_store(descS + (buf ^ 1) * 256, xS + (buf ^ 1) * 256, lane, R);
                chunk_store_y<8>(yS + (buf ^ 1) * 256, lane, RY);
            }
            __syncwarp();
        }
        __threadfence();
        __syncwarp();
        if (lane == 0) st_release(t.done + (long long)tk * t.B + b, t.epoch);
    }
}

// ---------------------------------------------------------------------------------------
// host: tables, launchers, dispatch
// ---------------------------------------------------------------------------------------
#include "chordal_chain.cuh"

template <class T>
static int up_vec(smcp_sym *s, const std::vector<T> &v, const T **out) {
    void *d = nullptr;
    size_t n = v.size() ? v.size() : 1;
    CUDA_TRY(cudaMalloc(&d, n * sizeof(T)));
    if (v.size()) CUDA_TRY(cudaMemcpy(d, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
    s->allocs.push_back(d);
    *out = (const T *)d;
    return 0;
}

// cut the steps [tp[t], tp[t+1]) of every task into chunks
static void build_chunks(const std::vector<int> &tp, const std::vector<int> &ts, const smcp_sym_desc *D,
                         const std::vector<long long> &sq, bool limit_sq, std::vector<int> &chunk_ptr, std::vector<int4> &chunks) {
    const int nt = (int)tp.size() - 1;
    chunk_ptr.assign(nt + 1, 0);
    for (int t = 0; t < nt; ++t) {
        int p = tp[t];
        while (p < tp[t + 1]) {
            const int pb = p;
            long long blo = D->blkptr[ts[p]], bhi = D->blkptr[ts[p] + 1];
            long long slo = sq[ts[p]], shi = sq[ts[p] + 1];
            ++p;
            while (p < tp[t + 1] && p - pb < CH_STEPS) {
                const int k = ts[p];
                const long long nblo = std::min<long long>(blo, D->blkptr[k]), nbhi = std::max<long long>(bhi, D->blkptr[k + 1]);
                const long long nslo = std::min(slo, sq[k]), nshi = std::max(shi, sq[k + 1]);
                if (nbhi - nblo > CH_BLK || (limit_sq && nshi - nslo > CH_SQ)) break;
                blo = nblo; bhi = nbhi; slo = nslo; shi = nshi;
                ++p;
            }
            chunks.push_back(make_int4(pb, p, (int)blo, (int)bhi));
            chunks.push_back(make_int4((int)slo, (int)shi, 0, 0));
        }
        chunk_ptr[t + 1] = (int)(chunks.size() / 2);
    }
}

int small_setup(smcp_sym *s, const smcp_sym_desc *D, const std::vector<int> &tp, const std::vector<int> &ts,
                const std::vector<int> &tp2, const std::vector<int> &ts2) {
    const int nsn = (int)D->nsn;
    std::vector<int> nn(nsn), na(nsn), nj(nsn);
    for (int k = 0; k < nsn; ++k) {
        nn[k] = (int)(D->snptr[k + 1] - D->snptr[k]);
        nj[k] = (int)(D->rowptr[k + 1] - D->rowptr[k]);
        na[k] = nj[k] - nn[k];
    }
    chain_detect(s, D, nn, na);
    // slot colouring, root to leaves: the separator rows are coloured already (they belong to
    // the parent's clique), the supernode's own vertices take the free slots
    std::vector<int> slot(D->n, -1);
    std::vector<unsigned> rowslot(nsn), slotpos(nsn);
    for (int k = nsn - 1; k >= 0; --k) {
        const int64_t *rows = D->rowidx + D->rowptr[k];
        unsigned used = 0;
        for (int q = nn[k]; q < nj[k]; ++q) used |= 1u << slot[rows[q]];
        for (int q = 0; q < nn[k]; ++q) {
            int c = 0;
            while (used & (1u << c)) ++c;
            if (c >= 8) { smcp_set_error("slot colouring failed (clique larger than 8?)"); return -2; }
            slot[rows[q]] = c;
            used |= 1u << c;
        }
        unsigned rs = 0, sp = 0xffffffffu;
        for (int q = 0; q < nj[k]; ++q) {
            const unsigned c = (unsigned)slot[rows[q]];
            rs |= c << (4 * q);
            sp = (sp & ~(15u << (4 * c))) | ((unsigned)q << (4 * c));
        }
        rowslot[k] = rs;
        slotpos[k] = sp;
    }
    std::vector<long long> sq(nsn + 1, 0);
    for (int k = 0; k < nsn; ++k) sq[k + 1] = sq[k] + (long long)nj[k] * nj[k];
    if (sq[nsn] >= (1LL << 31)) { smcp_set_error("pattern too large for the tiny-clique kernels"); return -2; }
    const int nt = (int)tp.size() - 1;
    // which supernodes hand their update matrix over through a global tile
    std::vector<int> tile(nsn, -1);
    int ntiles = 0;
    for (int t = 0; t < nt; ++t)
        for (int p = tp[t]; p < tp[t + 1]; ++p) {
            const int k = ts[p], par = (int)D->snpar[k];
            if (par >= 0 && !(p + 1 < tp[t + 1] && ts[p + 1] == par)) tile[k] = ntiles++;
        }
    std::vector<int4> up(2 * (size_t)nsn), down(2 * (size_t)nsn);
    std::vector<int> och;
    for (int t = 0; t < nt; ++t)
        for (int p = tp[t]; p < tp[t + 1]; ++p) {
            const int k = ts[p];
            const int prev = p > tp[t] ? ts[p - 1] : -1;
            int flags = 0;
            if (prev >= 0 && D->snpar[prev] == k) flags |= F_CARRY;
            if (tile[k] >= 0) flags |= F_WR;
            const int ob = (int)och.size();
            for (int64_t q = D->chptr[k]; q < D->chptr[k + 1]; ++q) {
                const int c = (int)D->chidx[q];
                if ((flags & F_CARRY) && c == prev) continue;
                och.push_back(tile[c]);
            }
            if ((int)och.size() > ob) flags |= F_OCH;
            up[2 * (size_t)p] = make_int4(nn[k] | (na[k] << 4) | (flags << 8), (int)D->blkptr[k], (int)rowslot[k], (int)slotpos[k]);
            up[2 * (size_t)p + 1] = make_int4(tile[k], ob, (int)och.size() - ob, (int)sq[k]);
        }
    for (int t = 0; t < nt; ++t)
        for (int p = tp2[t]; p < tp2[t + 1]; ++p) {
            const int k = ts2[p];
            const int prev = p > tp2[t] ? ts2[p - 1] : -1;
            int flags = 0;
            if (prev >= 0 && D->snpar[k] == prev) flags |= F_CARRY;
            down[2 * (size_t)p] = make_int4(nn[k] | (na[k] << 4) | (flags << 8), (int)D->blkptr[k], (int)rowslot[k], (int)slotpos[k]);
            down[2 * (size_t)p + 1] = make_int4((int)D->updptr[k], 0, 0, 0);
        }
    // uniform runs (see the kernels): remaining run length of every step, bits 16.. of word 0
    auto ident_prefix = [&](int c) {      // separator of c = leading rows of its parent's clique
        for (int q = 0; q < na[c]; ++q)
            if (D->relidx[D->relptr[c] + q] != q) return false;
        return true;
    };
    auto mark_runs = [&](const std::vector<int> &tpx, const std::vector<int> &tsx, std::vector<int4> &st, bool upward) {
        for (int t = 0; t < nt; ++t) {
            int rem = 0;
            for (int p = tpx[t + 1] - 1; p >= tpx[t]; --p) {
                bool uni = false;
                if (p > tpx[t]) {
                    const int k = tsx[p], q = tsx[p - 1];
                    const int fl = (st[2 * (size_t)p].x >> 8) & 255;
                    const int child = upward ? q : k;
                    uni = fl == F_CARRY && nn[k] == nn[q] && na[k] == na[q] && (upward ? k == q + 1 : k == q - 1) &&
                          D->snpar[child] == (upward ? k : q) && ident_prefix(child);
                }
                rem = uni ? std::min(rem + 1, 32767) : 0;
                st[2 * (size_t)p].x |= rem << 16;
            }
        }
    };
    mark_runs(tp, ts, up, true);
    mark_runs(tp2, ts2, down, false);
    std::vector<int> ucp, dcp, acp;
    std::vector<int4> uch, dch, ach;
    build_chunks(tp, ts, D, sq, false, ucp, uch);
    build_chunks(tp, ts, D, sq, true, acp, ach);
    build_chunks(tp2, ts2, D, sq, false, dcp, dch);
    SmallDev &M = s->sm;
    if (up_vec(s, up, &M.up_steps) || up_vec(s, down, &M.down_steps) || up_vec(s, och, &M.och) ||
        up_vec(s, sq, &M.sqptr) || up_vec(s, ucp, &M.up_chunk_ptr) || up_vec(s, uch, &M.up_chunks) ||
        up_vec(s, dcp, &M.down_chunk_ptr) || up_vec(s, dch, &M.down_chunks) || up_vec(s, acp, &M.add_chunk_ptr) ||
        up_vec(s, ach, &M.add_chunks))
        return -1;
    std::vector<int> wide;
    for (int k = 0; k < nsn; ++k)
        if (nn[k] != 1) wide.push_back(k);
    if (up_vec(s, wide, &M.wide_sn)) return -1;
    M.nwide = (int)wide.size();
    M.nsq = sq[nsn];
    M.ntiles = ntiles;
    s->small = true;
    return 0;
}

static void fill_common(smcp_sym *s, SmallArgs &a, const TaskSched &T, int64_t batch) {
    a.t.S = s->d;
    a.t.T = T;
    a.t.B = (int)batch;
    a.t.counter = s->counter;
    a.t.done = s->done;
    a.t.fail = s->fail;
    a.t.upd = s->upd;
    a.M = s->sm;
}

template <int OP>
static int launch_flat(smcp_sym *s, SmallArgs &a, int64_t batch, const char *name) {
    smcp_ctx *ctx = s->ctx;
    fill_common(s, a, s->flat, batch);
    long long items = (long long)(a.list ? a.nlist : s->d.nsn) * batch;
    if (items == 0) return 0;
    long long grid = (items + (FLAT_THREADS / 32) - 1) / (FLAT_THREADS / 32);
    long long cap = (long long)ctx->num_sms * 16;
    if (grid > cap) grid = cap;
    if (grid < 1) grid = 1;
    {
        LaunchScope ls(ctx, name, 1, (double)batch);
        flat_small_kernel<OP><<<(unsigned)grid, FLAT_THREADS, 0, ctx->stream>>>(a);
    }
    CUDA_TRY(cudaGetLastError());
    return 0;
}

template <class K>
static int launch_sweep(smcp_sym *s, K kern, int ws_doubles, SmallArgs &a, const TaskSched &T, int64_t batch, const char *name) {
    smcp_ctx *ctx = s->ctx;
    fill_common(s, a, T, batch);
    a.t.epoch = ++s->epoch;
    const size_t smem = (size_t)SW_WARPS * ws_doubles * sizeof(double);
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, SW_THREADS, smem));
    if (per_sm < 1) { smcp_set_error("sweep kernel does not fit on an SM"); return -1; }
    long long items = (long long)T.ntask * batch;
    long long grid = (items + SW_WARPS - 1) / SW_WARPS;
    long long cap = (long long)per_sm * ctx->num_sms;
    if (grid > cap) grid = cap;
    if (grid < 1) grid = 1;
    CUDA_TRY(cudaMemsetAsync(s->counter, 0, sizeof(unsigned), ctx->stream));
    {
        LaunchScope ls(ctx, name, 1, (double)batch);
        kern<<<(unsigned)grid, SW_THREADS, smem, ctx->stream>>>(a);
    }
    CUDA_TRY(cudaGetLastError());
    return 0;
}

static const int WS_CHOL = sweep_ws(0, false), WS_HUP = sweep_ws(CH_BLK, false), WS_ADD = sweep_ws(CH_SQ, false),
                 WS_DOWN = sweep_ws(CH_BLK, true);

static int ensure_fbuf(smcp_sym *s, int64_t batch) {
    return grow((void **)&s->fbuf, &s->fbuf_cap, (size_t)batch * (size_t)(s->sm.nsq + 1) * sizeof(double));
}

// matrices per launch of the routines that need the nj x nj local fronts
static int64_t fbuf_chunk(smcp_sym *s, int64_t batch) {
    int64_t per = (int64_t)(s->sm.nsq + 1) * 8;
    int64_t c = ((int64_t)2 << 30) / per;
    if (c < 1) c = 1;
    return c < batch ? c : batch;
}

int ks_cholesky(smcp_sym *s, double *x, int64_t batch, int32_t *info_host) {
    if (sym_ensure(s, batch, false)) return -1;
    CUDA_TRY(cudaMemsetAsync(s->fail, 0, (size_t)batch * sizeof(int), s->ctx->stream));
    SmallArgs a = {};
    a.t.X = x;
    if (s->chain) {
        if (chain_cholesky(s, x, batch, batch > 1 ? "cholesky_chain_batch" : "cholesky_chain")) return -1;
    } else if (launch_sweep(s, sweep_up_kernel<SW_CHOL>, WS_CHOL, a, s->up, batch, batch > 1 ? "cholesky_batch" : "cholesky")) return -1;
    if (info_host) return fetch_fail(s, batch, info_host);
    return 0;
}

int ks_completion(smcp_sym *s, double *x, int64_t batch, int32_t *info_host) {
    if (sym_ensure(s, batch, true)) return -1;
    smcp_ctx *ctx = s->ctx;
    CUDA_TRY(cudaMemsetAsync(s->fail, 0, (size_t)batch * sizeof(int), ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(s->tmp, x, (size_t)batch * s->d.nblk * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
    SmallArgs a = {};
    a.t.X = x;
    a.t.Xin = s->tmp;
    if (s->chain && batch >= 8) {
        // chain nodes: one thread per (matrix, node); the root supernode keeps the warp kernel
        if (chain_completion(s, x, s->tmp, batch, "completion_chain_batch")) return -1;
        a.list = s->sm.wide_sn;
        a.nlist = s->sm.nwide;
        if (launch_flat<FL_COMPL>(s, a, batch, "completion_root_batch")) return -1;
    } else if (launch_flat<FL_COMPL>(s, a, batch, batch > 1 ? "completion_batch" : "completion")) return -1;
    if (info_host) return fetch_fail(s, batch, info_host);
    return 0;
}

int ks_llt(smcp_sym *s, double *x, int64_t batch) {
    if (sym_ensure(s, batch, false)) return -1;
    const int64_t chunk = fbuf_chunk(s, batch);
    if (ensure_fbuf(s, chunk)) return -1;
    for (int64_t b0 = 0; b0 < batch; b0 += chunk) {
        const int64_t nb = std::min(chunk, batch - b0);
        SmallArgs a = {};
        a.t.X = x + b0 * s->d.nblk;
        a.F = s->fbuf;
        if (launch_flat<FL_LLT_LOCAL>(s, a, nb, "llt_local")) return -1;
        if (s->chain) {
            if (chain_add(s, a.t.X, s->fbuf, nb, "llt_chain")) return -1;
        } else if (launch_sweep(s, sweep_up_kernel<SW_ADD>, WS_ADD, a, s->up, nb, "llt")) return -1;
    }
    return 0;
}

int ks_projinv(smcp_sym *s, double *x, int64_t batch) {
    if (sym_ensure(s, batch, true)) return -1;
    SmallArgs a = {};
    a.t.X = x;
    a.t.Lt_out = s->tmp;
    if (launch_flat<FL_PINV_PREP>(s, a, batch, "projected_inverse_prep")) return -1;
    a.t.Lt = s->tmp;
    a.ltstride = s->d.nblk;
    return launch_sweep(s, sweep_down_kernel, WS_DOWN, a, s->down, batch, "projected_inverse");
}

int ks_hess_prep(smcp_hess *h, const double *L, const double *Y) {
    smcp_sym *s = h->sym;
    if (sym_ensure(s, 1, false)) return -1;
    SmallArgs a = {};
    a.t.L0 = L;
    a.t.Y0 = Y;
    a.t.Lt_out = h->Lt;
    a.t.Yaa_out = h->Yaa;
    return launch_flat<FL_HPREP>(s, a, 1, "hessian_prep");
}

int ks_hess_prep_inv(smcp_hess *h) {
    smcp_sym *s = h->sym;
    if (sym_ensure(s, 1, false)) return -1;
    CUDA_TRY(cudaMemsetAsync(s->fail, 0, sizeof(int), s->ctx->stream));
    SmallArgs a = {};
    a.t.Yaa = h->Yaa;
    a.t.Raa = h->Raa;
    return launch_flat<FL_HPREP_INV>(s, a, 1, "hessian_prep_inv");
}

int ks_hess_apply(smcp_hess *h, double *U, int64_t batch, int inv) {
    smcp_sym *s = h->sym;
    if (sym_ensure(s, batch, false)) return -1;
    const bool big = batch >= 32;
    if (!inv) {
        SmallArgs a = {};
        a.t.X = U;
        a.t.Lt = h->Lt;
        a.t.Yaa = h->Yaa;
        bool ch = s->chain;
        if (ch) {
            if (chain_prepare(h)) return -1;
            ch = h->chain_ok;          // accuracy guard: see chain_prepare
        }
        if (ch) {
            if (chain_sweep(s, true, U, h->Lt, h->phi_up, h->psi_up, h->Yaa, batch, big ? "hessian_up_chain_batch" : "hessian_up_chain")) return -1;
        } else if (launch_sweep(s, sweep_up_kernel<SW_HUP>, WS_HUP, a, s->up, batch, big ? "hessian_up_batch" : "hessian_up")) return -1;
        if (big || ch) {
            // one thread per (supernode, matrix) for the single-column supernodes, warps for the rest
            smcp_ctx *ctx = s->ctx;
            fill_common(s, a, s->flat, batch);
            long long items = (long long)s->d.nsn * batch;
            long long grid = std::min<long long>((items + 255) / 256, (long long)ctx->num_sms * 16);
            if (!ch) {      // chain: fused into the final pass of the up sweep
                LaunchScope ls(ctx, "hessian_scale_batch", 1, (double)batch);
                hscale_nn1_kernel<<<(unsigned)grid, 256, 0, ctx->stream>>>(a);
            }
            CUDA_TRY(cudaGetLastError());
            a.list = s->sm.wide_sn;
            a.nlist = s->sm.nwide;
            if (launch_flat<FL_HSCALE>(s, a, batch, "hessian_scale_wide_batch")) return -1;
            a.list = nullptr;
            a.nlist = 0;
        } else if (launch_flat<FL_HSCALE>(s, a, batch, "hessian_scale")) return -1;
        if (ch) return chain_sweep(s, false, U, h->Lt, h->phi_dn, h->psi_dn, nullptr, batch, big ? "hessian_down_chain_batch" : "hessian_down_chain");
        return launch_sweep(s, sweep_down_kernel, WS_DOWN, a, s->down, batch, big ? "hessian_down_batch" : "hessian_down");
    }
    if (!h->have_Raa) {
        if (ks_hess_prep_inv(h)) return -1;
        h->have_Raa = true;
    }
    const int64_t chunk = fbuf_chunk(s, batch);
    if (ensure_fbuf(s, chunk)) return -1;
    for (int64_t b0 = 0; b0 < batch; b0 += chunk) {
        const int64_t nb = std::min(chunk, batch - b0);
        SmallArgs a = {};
        a.t.X = U + b0 * s->d.nblk;
        a.t.Lt = h->Lt;
        a.t.Yaa = h->Yaa;
        a.t.Raa = h->Raa;
        a.F = s->fbuf;
        if (launch_flat<FL_HINV_LOCAL>(s, a, nb, big ? "hessian_inv_local_batch" : "hessian_inv_local")) return -1;
        if (s->chain) {
            if (chain_add(s, a.t.X, s->fbuf, nb, big ? "hessian_inv_chain_batch" : "hessian_inv_chain")) return -1;
        } else if (launch_sweep(s, sweep_up_kernel<SW_ADD>, WS_ADD, a, s->up, nb, big ? "hessian_inv_batch" : "hessian_inv")) return -1;
    }
    return 0;
}
