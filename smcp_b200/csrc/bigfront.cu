// Large frontal matrices as dense multi-CTA kernels on the FP64 tensor cores (north star (1):
// "large frontal updates run as FP64 tensor-core (DMMA) tiles").
//
// The persistent tree kernels (chordal.cu) give one supernode to ONE CTA and keep its frontal matrix
// in shared memory (nj <= 79) or in a per-CTA global scratch.  On patterns with real fill (rand_SDP,
// max-cut embeddings, mtxnorm) a handful of supernodes near the root carry > 99 % of the flops
// (rand_SDP n = 2000: root 1186 x 1186; max-cut n = 5000: a 679-column supernode with a 1-row
// separator under a chain of 600-row separators), and a single CTA needs 0.1 .. 1 s for them.
// For single matrices (Newton solves, line-search factorisations, scaling points) those supernodes
// are taken out of the tree kernel: the "top set" T = {supernodes with nj >= threshold} plus all
// their ancestors is processed here, supernode by supernode in (reverse) post-order, with dense
// building blocks that use the whole GPU:
//   * DMMA GEMM (dense.cu) for every congruence / Schur-complement product,
//   * blocked triangular solves (front.cu: 64 x 64 diagonal blocks + DMMA updates),
//   * the blocked Cholesky of dense.cu, as a PARTIAL factorisation of the frontal matrix: the
//     leading nn columns become L, the trailing na x na block the update matrix.
// The block formulas are those of chordal_ops.cuh / oracle/supernodal.py (SURVEY App. A); reference
// call sites: src/python/solvers.py:884 (cholesky), 874 (completion), 891 (projected_inverse),
// 904 (llt), 483/524/531 (hessian), 405 (inverse hessian).
// Children's update matrices are added through a precomputed inverse relative-index map so that
// every entry of a frontal matrix is summed by one thread in child order (deterministic).
#include "internal.cuh"
#include <algorithm>
#include <cstdlib>

// thin supernodes: at most THIN_NN columns (the thin_* kernels below)
#define THIN_NN 8
#define THIN_TS 32         // tile of the alpha x alpha passes (thin_up / thin_hinv_sweep / thin_chol): 32 x 32 per CTA of 256 threads (64 x 64 was slower: 20.5 -> 30.8 us, latency bound)

// ---------------------------------------------------------------------------------------
// elementwise kernels
// ---------------------------------------------------------------------------------------
struct BigArgs {
    int nn, na, nj, nch;
    const int *ch;           // children
    const int *inv;          // nch x nj: position of row p of this supernode in the child's separator, or -1
    const int *na_all;       // per supernode
    const long long *updptr;
    const double *ub;        // update matrices of this matrix
};

__device__ __forceinline__ double big_children(const BigArgs &r, int i, int j, bool lower_stored) {
    double acc = 0.0;
    for (int q = 0; q < r.nch; ++q) {
        const int a = r.inv[(long long)q * r.nj + i], b = r.inv[(long long)q * r.nj + j];
        if (a >= 0 && b >= 0) {
            const int c = r.ch[q], nac = r.na_all[c];
            const double *Uc = r.ub + r.updptr[c];
            acc += lower_stored ? Uc[max(a, b) + (long long)min(a, b) * nac] : Uc[a + (long long)b * nac];
        }
    }
    return acc;
}

// children's contributions to the entries (i, j[0..3]) of a frontal matrix: the row lookup is done once per child and the
// four column lookups / gathers are independent loads (big_children does two dependent lookups per entry)
__device__ __forceinline__ void big_children_row4(const BigArgs &r, int i, const int (&j)[4], const bool (&live)[4], bool lower_stored,
                                                  double (&acc)[4]) {
#pragma unroll
    for (int e = 0; e < 4; ++e) acc[e] = 0.0;
    for (int q = 0; q < r.nch; ++q) {
        const int *invq = r.inv + (long long)q * r.nj;
        const int a = invq[i];
        if (a < 0) continue;
        const int c = r.ch[q], nac = r.na_all[c];
        const double *Uc = r.ub + r.updptr[c];
        int b[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) b[e] = live[e] ? invq[j[e]] : -1;
        double u[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            u[e] = 0.0;
            if (b[e] >= 0) u[e] = lower_stored ? Uc[max(a, b[e]) + (long long)min(a, b[e]) * nac] : Uc[a + (long long)b[e] * nac];
        }
#pragma unroll
        for (int e = 0; e < 4; ++e) acc[e] += u[e];
    }
}

#define BIG_LOOP(total) for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < (total); idx += (long long)gridDim.x * blockDim.x)

// F (nj x nj, lower) = [blk_nn(lower) ; blk_an ; 0] + children (lower-stored); upper <- 0        (cholesky)
__global__ void big_front_lower_kernel(BigArgs r, const double *__restrict__ blk, double *__restrict__ F) {
    const int nj = r.nj, nn = r.nn;
    BIG_LOOP((long long)nj * nj) {
        const int i = (int)(idx % nj), j = (int)(idx / nj);
        double v = 0.0;
        if (i >= j) {
            if (j < nn) v = blk[i + (long long)j * nj];
            v += big_children(r, i, j, true);
        }
        F[idx] = v;
    }
}

// F (nj x nj, full symmetric) = sym([blk_nn blk_an^T; blk_an 0]) + children (full)               (hessian pass 1)
__global__ void big_front_full_kernel(BigArgs r, const double *__restrict__ blk, double *__restrict__ F) {
    const int nj = r.nj, nn = r.nn;
    BIG_LOOP((long long)nj * nj) {
        const int i = (int)(idx % nj), j = (int)(idx / nj);
        const int hi = max(i, j), lo = min(i, j);
        double v = (lo < nn) ? blk[hi + (long long)lo * nj] : 0.0;
        F[idx] = v + big_children(r, i, j, false);
    }
}

// copy the leading nn columns of F (ld nj) to blk: lower part of the nn x nn block, zero above
__global__ void big_store_cols_kernel(const double *__restrict__ F, double *__restrict__ blk, int nn, int nj) {
    BIG_LOOP((long long)nj * nn) {
        const int i = (int)(idx % nj), j = (int)(idx / nj);
        blk[idx] = (i >= j) ? F[idx] : 0.0;
    }
}

// U (na x na, ld na) = S (ld lds); lower: only i >= j is written, the rest is zeroed
__global__ void big_copy_mat_kernel(const double *__restrict__ S, long long lds, double *__restrict__ U, long long ldu, int rows, int cols, int lower) {
    BIG_LOOP((long long)rows * cols) {
        const int i = (int)(idx % rows), j = (int)(idx / rows);
        U[i + (long long)j * ldu] = (!lower || i >= j) ? S[i + (long long)j * lds] : 0.0;
    }
}

// llt: blk(lower nn cols) = P + children(lower), U(lower) = P_aa + children
__global__ void big_llt_store_kernel(BigArgs r, const double *__restrict__ P, double *__restrict__ blk, double *__restrict__ U) {
    const int nj = r.nj, nn = r.nn, na = r.na;
    BIG_LOOP((long long)nj * nj) {
        const int i = (int)(idx % nj), j = (int)(idx / nj);
        if (j < nn) {
            blk[i + (long long)j * nj] = (i >= j) ? P[idx] + big_children(r, i, j, true) : 0.0;
        } else if (i >= j) {
            U[(i - nn) + (long long)(j - nn) * na] = P[idx] + big_children(r, i, j, true);
        }
    }
}

// T (n x n, ld ldt) <- full symmetric copy of the lower-stored n x n block S (ld lds)
__global__ void big_sym_copy_kernel(const double *__restrict__ S, long long lds, double *__restrict__ T, long long ldt, int n) {
    BIG_LOOP((long long)n * n) {
        const int i = (int)(idx % n), j = (int)(idx / n);
        T[i + (long long)j * ldt] = (i >= j) ? S[i + (long long)j * lds] : S[j + (long long)i * lds];
    }
}

// blk_nn (lower, ld nj) = alpha * blk_nn + beta * 0.5 (T(i,j) + T(j,i)) ; upper <- 0
__global__ void big_sym_store_kernel(const double *__restrict__ T, long long ldt, double *__restrict__ blk, long long ldb, int n, double alpha, double beta) {
    BIG_LOOP((long long)n * n) {
        const int i = (int)(idx % n), j = (int)(idx / n);
        double *d = blk + i + (long long)j * ldb;
        if (i >= j) {
            const double t = 0.5 * (T[i + (long long)j * ldt] + T[j + (long long)i * ldt]);
            *d = (alpha != 0.0 ? alpha * *d : 0.0) + beta * t;
        } else *d = 0.0;
    }
}

// B (cols x rows, ld ldb) = A^T, A rows x cols (ld lda)
__global__ void big_transpose_kernel(const double *__restrict__ A, long long lda, int rows, int cols, double *__restrict__ Bt, long long ldb) {
    __shared__ double tile[32][33];
    const int bx = blockIdx.x * 32, by = blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int i = bx + threadIdx.x, j = by + r;
        tile[r][threadIdx.x] = (i < rows && j < cols) ? A[i + (long long)j * lda] : 0.0;
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int i = by + threadIdx.x, j = bx + r;      // Bt(i, j) = A(j, i)
        if (i < cols && j < rows) Bt[i + (long long)j * ldb] = tile[threadIdx.x][r];
    }
}

__global__ void big_identity_kernel(double *A, long long lda, int n) {
    BIG_LOOP((long long)n * n) {
        const int i = (int)(idx % n), j = (int)(idx / n);
        A[i + (long long)j * lda] = (i == j) ? 1.0 : 0.0;
    }
}

// dst (na x na, ld na) = X[aaidx]: the alpha x alpha entries of the ancestors, full symmetric
__global__ void big_gather_aa_kernel(const int *__restrict__ aaidx, const double *__restrict__ Xb, double *__restrict__ dst, long long total) {
    BIG_LOOP(total) dst[idx] = Xb[aaidx[idx]];
}

// reversed symmetric copy (mode 0) and M = (P Lc P)^T (mode 1) for the "reverse" Cholesky of completion
__global__ void big_reverse_kernel(const double *__restrict__ S, long long lds, double *__restrict__ T, int n, int mode) {
    BIG_LOOP((long long)n * n) {
        const int i = (int)(idx % n), j = (int)(idx / n);
        if (mode == 0) {
            const int ri = n - 1 - i, rj = n - 1 - j;
            T[idx] = (ri >= rj) ? S[ri + (long long)rj * lds] : S[rj + (long long)ri * lds];
        } else {
            T[idx] = (i >= j) ? S[(n - 1 - j) + (long long)(n - 1 - i) * lds] : 0.0;
        }
    }
}

// completion: the clique matrix in the order [alpha; nu], lower triangle:
//   T[0:na, 0:na] = X_aa (gathered from the ancestors), T[na:, 0:na] = X_an^T, T[na:, na:] = X_nn
__global__ void big_compl_front_kernel(const int *__restrict__ aaidx, const double *__restrict__ Xb, const double *__restrict__ bin,
                                       double *__restrict__ T, int nn, int na, int nj) {
    BIG_LOOP((long long)nj * nj) {
        const int i = (int)(idx % nj), j = (int)(idx / nj);
        double v = 0.0;
        if (j < na) {
            if (i < na) v = Xb[aaidx[i + (long long)j * na]];
            else v = bin[(nn + j) + (long long)(i - na) * nj];
        } else if (i >= j) {
            v = bin[(i - na) + (long long)(j - na) * nj];
        }
        T[idx] = v;
    }
}

// inverse Hessian, final assembly: children (full) are added to (K_nn, F_an, F_aa)
__global__ void big_hinv_store_kernel(BigArgs r, const double *__restrict__ Knn, const double *__restrict__ Fan, const double *__restrict__ Faa,
                                      double *__restrict__ blk, double *__restrict__ U) {
    const int nj = r.nj, nn = r.nn, na = r.na;
    BIG_LOOP((long long)nj * nj) {
        const int i = (int)(idx % nj), j = (int)(idx / nj);
        if (j < nn) {
            if (i < nn) {
                if (i >= j) {
                    const double a = Knn[i + (long long)j * nn] + big_children(r, i, j, false);
                    const double b = Knn[j + (long long)i * nn] + big_children(r, j, i, false);
                    blk[i + (long long)j * nj] = 0.5 * (a + b);
                } else blk[i + (long long)j * nj] = 0.0;
            } else {
                blk[i + (long long)j * nj] = Fan[(i - nn) + (long long)j * na] + big_children(r, i, j, false);
            }
        } else if (i >= nn) {
            U[(i - nn) + (long long)(j - nn) * na] = Faa[(i - nn) + (long long)(j - nn) * na] + big_children(r, i, j, false);
        }
    }
}

__global__ void big_flag_kernel(const int *info, int *fail) {
    if (*info) *fail = 1;
}

// ---------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------
// frontal factorisations are profiled as their own family ("front_potrf"), apart from the Cholesky of H ("potrf_dmma")
static int front_potrf(smcp_ctx *ctx, double *H, int64_t ld, int64_t m, int64_t ncols, int32_t *info_dev) {
    const char *prev = ctx->potrf_family;
    ctx->potrf_family = "front_potrf";
    const int rc = d_potrf(ctx, H, ld, m, ncols, info_dev, 0, 1);
    ctx->potrf_family = prev;
    return rc;
}
static unsigned egrid(smcp_sym *s, long long total) {
    long long g = (total + 255) / 256;
    return (unsigned)std::max<long long>(1, std::min<long long>(g, (long long)s->ctx->num_sms * 8));
}

int big_setup(smcp_sym *s, const smcp_sym_desc *D) {
    s->big.clear();
    s->big_flag = nullptr;
    const int nsn = (int)D->nsn;
    if (nsn < 1) return 0;
    // a supernode goes to the dense path when its share of a Hessian evaluation
    // (4 nn^3 + 6 na nn^2 + 6 na^2 nn flops, SURVEY 8d) is too much for one CTA;
    // SMCP_B200_BIG_FLOPS overrides the threshold (0 disables the path), SMCP_B200_BIG_NJ adds a
    // criterion on the front size (tests force tiny fronts through the dense path with it)
    // A third criterion covers the completion (and the inverse-Hessian factor): both need the Cholesky
    // factor of the na x na separator block whatever nn is (na^3/3 flops, SURVEY 8a a3) -- a 1-column
    // supernode under a 500-row separator is 4e7 flops that one CTA of the tree kernel needs 20 ms for
    // (rand_SDP n = 2000: 43 ms per completion before this rule).  SMCP_B200_BIG_COMPL_FLOPS overrides.
    const char *envf = getenv("SMCP_B200_BIG_FLOPS"), *envn = getenv("SMCP_B200_BIG_NJ"), *envc = getenv("SMCP_B200_BIG_COMPL_FLOPS");
    const double thr_flops = envf ? atof(envf) : 2.0e6;
    // 6e5 (na >= 122) since the thin-supernode kernels: a larger top set costs the sweeps little now and takes the
    // separator factorisations off the one-CTA-per-supernode tree kernels (rand_SDP n = 2000: 128 -> 119 ms per iteration
    // against 6e6, gpurun_out/r02_v23_thresholds.log)
    const double thr_compl = envc ? atof(envc) : (thr_flops > 0.0 ? 6.0e5 : 0.0);
    const int thr_nj = envn ? atoi(envn) : 0;
    if (thr_flops <= 0.0 && thr_nj <= 0) return 0;
    std::vector<int> flag(nsn, 0);
    bool any = false;
    for (int k = 0; k < nsn; ++k) {
        const double nj = (double)(D->rowptr[k + 1] - D->rowptr[k]), nn = (double)(D->snptr[k + 1] - D->snptr[k]), na = nj - nn;
        const double fl = 4.0 * nn * nn * nn + 6.0 * na * nn * nn + 6.0 * na * na * nn;
        if ((thr_flops > 0.0 && fl >= thr_flops) || (thr_nj > 0 && nj >= thr_nj) || (thr_compl > 0.0 && na * na * na / 3.0 >= thr_compl)) { flag[k] = 1; any = true; }
    }
    if (!any) return 0;
    // ancestor closure: post-order => parents have larger indices
    for (int k = 0; k < nsn; ++k)
        if (flag[k] && D->snpar[k] >= 0) flag[D->snpar[k]] = 1;
    int max_nj_small = 1, max_nj_big = 1;
    size_t inv_total = 0, ch_total = 0;
    for (int k = 0; k < nsn; ++k) {
        const int nj = (int)(D->rowptr[k + 1] - D->rowptr[k]);
        if (flag[k]) {
            max_nj_big = std::max(max_nj_big, nj);
            const size_t nch = (size_t)(D->chptr[k + 1] - D->chptr[k]);
            inv_total += nch * (size_t)nj;
            ch_total += nch;
        } else max_nj_small = std::max(max_nj_small, nj);
    }
    std::vector<int> inv(std::max<size_t>(1, inv_total), -1), ch(std::max<size_t>(1, ch_total), 0);
    size_t io = 0, co = 0;
    for (int k = 0; k < nsn; ++k) {
        if (!flag[k]) continue;
        BigNode b;
        b.k = k;
        b.nn = (int)(D->snptr[k + 1] - D->snptr[k]);
        b.nj = (int)(D->rowptr[k + 1] - D->rowptr[k]);
        b.na = b.nj - b.nn;
        b.nch = (int)(D->chptr[k + 1] - D->chptr[k]);
        b.boff = D->blkptr[k];
        b.uoff = D->updptr[k];
        b.rowoff = D->rowptr[k];
        b.r0 = (int)D->rowidx[D->rowptr[k]];
        b.inv_off = (long long)io;
        b.ch_off = (long long)co;
        for (int q = 0; q < b.nch; ++q) {
            const int c = (int)D->chidx[D->chptr[k] + q];
            ch[co + q] = c;
            const int nac = (int)(D->relptr[c + 1] - D->relptr[c]);
            for (int a = 0; a < nac; ++a) inv[io + (size_t)q * b.nj + D->relidx[D->relptr[c] + a]] = a;
        }
        io += (size_t)b.nch * b.nj;
        co += b.nch;
        s->big.push_back(b);
    }
    void *d = nullptr;
    CUDA_TRY(cudaMalloc(&d, inv.size() * sizeof(int)));
    CUDA_TRY(cudaMemcpy(d, inv.data(), inv.size() * sizeof(int), cudaMemcpyHostToDevice));
    s->allocs.push_back(d);
    s->big_inv = (const int *)d;
    CUDA_TRY(cudaMalloc(&d, ch.size() * sizeof(int)));
    CUDA_TRY(cudaMemcpy(d, ch.data(), ch.size() * sizeof(int), cudaMemcpyHostToDevice));
    s->allocs.push_back(d);
    s->big_ch = (const int *)d;
    CUDA_TRY(cudaMalloc(&d, (size_t)nsn * sizeof(int)));
    CUDA_TRY(cudaMemcpy(d, flag.data(), (size_t)nsn * sizeof(int), cudaMemcpyHostToDevice));
    s->allocs.push_back(d);
    s->big_flag = (const int *)d;
    // levels of the top set's own tree: supernodes of equal height (depth) are independent in the
    // leaves-to-root (root-to-leaves) sweeps -- each reads its children's update matrices (its ancestors'
    // blocks) and writes its own block only
    {
        const int nb = (int)s->big.size();
        std::vector<int> pos(nsn, -1), ht(nb, 0), dp(nb, 0);
        for (int i = 0; i < nb; ++i) pos[s->big[i].k] = i;
        int maxh = 0, maxd = 0;
        for (int i = 0; i < nb; ++i) {
            const int p = (int)D->snpar[s->big[i].k];
            if (p >= 0) { ht[pos[p]] = std::max(ht[pos[p]], ht[i] + 1); maxh = std::max(maxh, ht[pos[p]]); }
        }
        for (int i = nb - 1; i >= 0; --i) {
            const int p = (int)D->snpar[s->big[i].k];
            if (p >= 0) { dp[i] = dp[pos[p]] + 1; maxd = std::max(maxd, dp[i]); }
        }
        s->big_up.assign(maxh + 1, std::vector<int>());
        s->big_down.assign(maxd + 1, std::vector<int>());
        for (int i = 0; i < nb; ++i) s->big_up[ht[i]].push_back(i);
        for (int i = nb - 1; i >= 0; --i) s->big_down[dp[i]].push_back(i);
    }
    // lanes: the independent per-supernode operations of a top set of moderate fronts run on a few streams at once
    // (one of the ~1100-row factorisations of the rand_SDP separators keeps at most 18 of the 148 SMs busy in
    // its panel phase); SMCP_B200_LANES = 1 turns this off
    {
        const char *envl = getenv("SMCP_B200_LANES");
        int nl = envl ? atoi(envl) : 8;
        const size_t per_lane = (size_t)BIG_NWS * max_nj_big * max_nj_big * sizeof(double);
        if (nl < 1 || s->big.size() < 2) nl = 1;
        if (!envl && (s->big.size() < 4 || max_nj_big > 2560 || max_nj_big < 128)) nl = 1;    // an explicit setting is obeyed (tests)
        while (nl > 1 && per_lane * nl > ((size_t)4 << 30)) --nl;
        s->big_nlanes = std::min(nl, 16);
    }
    CUDA_TRY(cudaMalloc(&d, (size_t)s->big_nlanes * BIG_NWS * max_nj_big * max_nj_big * sizeof(double) + 64));
    s->allocs.push_back(d);
    s->big_ws = (double *)d;
    s->big_ws_stride = (size_t)max_nj_big * max_nj_big;
    CUDA_TRY(cudaMalloc(&d, 64));
    s->allocs.push_back(d);
    s->big_info = (int *)d;
    s->max_nj_small = max_nj_small;
    return 0;
}

static BigArgs big_args(smcp_sym *s, const BigNode &q, int64_t b) {
    BigArgs r;
    r.nn = q.nn; r.na = q.na; r.nj = q.nj; r.nch = q.nch;
    r.ch = s->big_ch + q.ch_off;
    r.inv = s->big_inv + q.inv_off;
    r.na_all = s->d.na;
    r.updptr = s->d.updptr;
    r.ub = s->upd + (size_t)b * s->d.nupd;
    return r;
}

#define WS(i) (s->big_ws + ((size_t)s->big_lane * BIG_NWS + (i)) * s->big_ws_stride)
#define BIG_INFO (s->big_info + s->big_lane)
#define ELEM(name, total, ...)                                                      \
    do {                                                                            \
        LaunchScope ls_(ctx, "front_elem");                                         \
        name<<<egrid(s, (total)), 256, 0, ctx->stream>>>(__VA_ARGS__);              \
    } while (0)

static int big_transpose(smcp_sym *s, const double *A, int64_t lda, int rows, int cols, double *Bt, int64_t ldb) {
    if (rows <= 0 || cols <= 0) return 0;
    smcp_ctx *ctx = s->ctx;
    dim3 grid((rows + 31) / 32, (cols + 31) / 32), block(32, 8);
    LaunchScope ls(ctx, "front_elem");
    big_transpose_kernel<<<grid, block, 0, ctx->stream>>>(A, lda, rows, cols, Bt, ldb);
    return 0;
}

// C = [C +] alpha op(A) op(B)^T in launch_gemm's convention, family "front_gemm_dmma"
static int G(smcp_sym *s, bool ta, bool tb, const double *A, int64_t lda, const double *B, int64_t ldb, double *C, int64_t ldc,
             int64_t M, int64_t N, int64_t K, double alpha, int acc, int tri = 0) {
    if (M <= 0 || N <= 0) return 0;
    if (K <= 0) {
        if (acc) return 0;
        smcp_ctx *ctx = s->ctx;
        CUDA_TRY(cudaMemset2DAsync(C, (size_t)ldc * sizeof(double), 0, (size_t)M * sizeof(double), (size_t)N, ctx->stream));
        return 0;
    }
    return launch_gemm(s->ctx, ta, tb, A, lda, B, ldb, C, ldc, M, N, K, alpha, acc, tri, 0, "front_gemm_dmma");
}

// ---- lanes over the top set ---------------------------------------------------------------------
int big_lanes_begin(smcp_sym *s) {
    const int nl = (s->ctx->prof || s->ctx->lanes_active) ? 1 : s->big_nlanes;
    if (nl > 1 && lanes_fork(s->ctx, nl)) return -1;
    return nl;
}
void big_lane_pick(smcp_sym *s, int lane) {
    s->big_lane = lane;
    lane_select(s->ctx, lane);
}
int big_lanes_end(smcp_sym *s) {
    s->big_lane = 0;
    return lanes_join(s->ctx);
}

// Cholesky of a thin supernode's frontal matrix in ONE launch: every CTA factors F_nn (block + children, nn <= 8) itself,
// forms L_an(i, :) = F_an(i, :) L_nn^-T for its 32 rows i and 32 rows j of alpha and writes the 32 x 32 tile
// U(i, j) = children(i, j) - L_an(i, :) L_an(j, :)^T of the update matrix (lower triangle; zero above, like the generic
// path).  The CTA that finishes last -- every CTA has read the block by then -- overwrites the block with L_nn, L_an
// and raises the verdict.  Generic path: front assembly, a cooperative partial factorisation with nn pivots, flag,
// two copies (5 launches).
__global__ void __launch_bounds__(256) thin_chol_kernel(BigArgs r, double *__restrict__ blk, double *__restrict__ U, int *__restrict__ fail,
                                                        unsigned *__restrict__ counter) {
    __shared__ double Li[THIN_NN][THIN_TS + 1], Lj[THIN_NN][THIN_TS + 1];
    __shared__ double Lnn[THIN_NN * THIN_NN];
    __shared__ int bad_s;
    __shared__ bool last_s;
    const int nn = r.nn, na = r.na, nj = r.nj, tid = threadIdx.x;
    const int i0 = blockIdx.x * THIN_TS, j0 = blockIdx.y * THIN_TS;
    if (tid < THIN_NN * THIN_NN) {
        const int a = tid % THIN_NN, b = tid / THIN_NN;
        Lnn[tid] = (a < nn && b < nn && a >= b) ? blk[a + (long long)b * nj] + big_children(r, a, b, true) : 0.0;
    }
    __syncthreads();
    if (tid == 0) {
        int bad = 0;
        for (int c = 0; c < nn; ++c) {
            double d = Lnn[c + c * THIN_NN];
            if (!(d > 0.0)) { bad = 1; d = 1.0; }
            const double l = sqrt(d);
            Lnn[c + c * THIN_NN] = l;
            for (int a = c + 1; a < nn; ++a) Lnn[a + c * THIN_NN] /= l;
            for (int b = c + 1; b < nn; ++b)
                for (int a = b; a < nn; ++a) Lnn[a + b * THIN_NN] = fma(-Lnn[a + c * THIN_NN], Lnn[b + c * THIN_NN], Lnn[a + b * THIN_NN]);
        }
        bad_s = bad;
    }
    __syncthreads();
    // rows of L_an: x L_nn^T = f  (forward over the columns)
    if (tid < 2 * THIN_TS) {
        const int rr = tid % THIN_TS;
        const int row = (tid < THIN_TS ? i0 : j0) + rr;
        double x[THIN_NN];
#pragma unroll
        for (int k2 = 0; k2 < THIN_NN; ++k2)
            x[k2] = (k2 < nn && row < na) ? blk[(nn + row) + (long long)k2 * nj] + big_children(r, nn + row, k2, true) : 0.0;
#pragma unroll
        for (int k2 = 0; k2 < THIN_NN; ++k2)
            if (k2 < nn) {
                double t = x[k2];
#pragma unroll
                for (int p2 = 0; p2 < THIN_NN; ++p2)
                    if (p2 < k2) t = fma(-x[p2], Lnn[k2 + p2 * THIN_NN], t);
                x[k2] = t / Lnn[k2 + k2 * THIN_NN];
            }
#pragma unroll
        for (int k2 = 0; k2 < THIN_NN; ++k2) {
            if (tid < THIN_TS) Li[k2][rr] = x[k2];
            else Lj[k2][rr] = x[k2];
        }
    }
    __syncthreads();
    const int tx = tid & 31, ty = tid >> 5;
#pragma unroll
    for (int ri = 0; ri < THIN_TS / 32; ++ri) {
        const int ii = tx + 32 * ri, i = i0 + ii;
        if (i >= na) continue;
#pragma unroll
        for (int qg = 0; qg < THIN_TS / 32; ++qg) {
            int jc[4];
            bool live[4];
            double ch[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int j = j0 + ty + 8 * (4 * qg + q);
                jc[q] = nn + j;
                live[q] = j < na && i >= j;
            }
            big_children_row4(r, nn + i, jc, live, true, ch);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int jj = ty + 8 * (4 * qg + q), j = j0 + jj;
                if (j < na) {
                    double v = 0.0;
                    if (i >= j) {
                        v = ch[q];
                        for (int k2 = 0; k2 < nn; ++k2) v = fma(-Li[k2][ii], Lj[k2][jj], v);
                    }
                    U[i + (long long)j * na] = v;
                }
            }
        }
    }
    __threadfence();
    __syncthreads();
    if (tid == 0) {
        const unsigned done = atomicAdd(counter, 1u);
        last_s = (done == gridDim.x * gridDim.y - 1);
    }
    __syncthreads();
    if (!last_s) return;
    // the block: L_an rows (recomputed from the still untouched input), then L_nn
    for (int row = tid; row < na; row += 256) {
        double x[THIN_NN];
#pragma unroll
        for (int k2 = 0; k2 < THIN_NN; ++k2)
            x[k2] = (k2 < nn) ? blk[(nn + row) + (long long)k2 * nj] + big_children(r, nn + row, k2, true) : 0.0;
#pragma unroll
        for (int k2 = 0; k2 < THIN_NN; ++k2)
            if (k2 < nn) {
                double t = x[k2];
#pragma unroll
                for (int p2 = 0; p2 < THIN_NN; ++p2)
                    if (p2 < k2) t = fma(-x[p2], Lnn[k2 + p2 * THIN_NN], t);
                x[k2] = t / Lnn[k2 + k2 * THIN_NN];
                blk[(nn + row) + (long long)k2 * nj] = x[k2];
            }
    }
    if (tid < nn * nn) {
        const int a = tid % nn, b = tid / nn;
        blk[a + (long long)b * nj] = (a >= b) ? Lnn[a + b * THIN_NN] : 0.0;
    }
    if (tid == 0) {
        if (bad_s) *fail = 1;
        *counter = 0u;
    }
}

// ---- cholesky --------------------------------------------------------------------------
int big_cholesky(smcp_sym *s, const BigNode &q, double *X, int64_t b) {
    smcp_ctx *ctx = s->ctx;
    const int nn = q.nn, na = q.na, nj = q.nj;
    double *blk = X + (size_t)b * s->d.nblk + q.boff;
    double *Uk = s->upd + (size_t)b * s->d.nupd + q.uoff;
    double *F = WS(0);
    if (nn <= THIN_NN && na >= 1) {
        if (!s->thin_counters) {
            CUDA_TRY(cudaMalloc(&s->thin_counters, 64 * sizeof(unsigned)));
            CUDA_TRY(cudaMemset(s->thin_counters, 0, 64 * sizeof(unsigned)));
            s->allocs.push_back(s->thin_counters);
        }
        LaunchScope ls_(ctx, "thin_chol");
        thin_chol_kernel<<<dim3((unsigned)((na + THIN_TS - 1) / THIN_TS), (unsigned)((na + THIN_TS - 1) / THIN_TS)), 256, 0, ctx->stream>>>(big_args(s, q, b), blk, Uk, s->fail + b,
                                                                                                                s->thin_counters + s->big_lane);
        CUDA_TRY(cudaGetLastError());
        return 0;
    }
    ELEM(big_front_lower_kernel, (long long)nj * nj, big_args(s, q, b), blk, F);
    if (front_potrf(ctx, F, nj, nj, nn, BIG_INFO)) return -1;
    big_flag_kernel<<<1, 1, 0, ctx->stream>>>(BIG_INFO, s->fail + b);
    ELEM(big_store_cols_kernel, (long long)nj * nn, F, blk, nn, nj);
    if (na) ELEM(big_copy_mat_kernel, (long long)na * na, F + nn + (size_t)nn * nj, nj, Uk, na, na, na, 1);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// ---- llt -------------------------------------------------------------------------------
int big_llt(smcp_sym *s, const BigNode &q, double *X, int64_t b) {
    smcp_ctx *ctx = s->ctx;
    const int nn = q.nn, nj = q.nj;
    double *blk = X + (size_t)b * s->d.nblk + q.boff;
    double *Uk = s->upd + (size_t)b * s->d.nupd + q.uoff;
    double *P = WS(0);
    if (G(s, false, false, blk, nj, blk, nj, P, nj, nj, nj, nn, 1.0, 0, 1)) return -1;      // P = L L^T (lower)
    ELEM(big_llt_store_kernel, (long long)nj * nj, big_args(s, q, b), P, blk, Uk);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// ---- thin supernodes (nn <= THIN_NN columns under a large separator) ------------------------------
// rand_SDP n = 2000: 41 of the 43 top-set supernodes have ONE or two columns under ~1100-row separators,
// chained one per level.  Through the generic building blocks above one forward Hessian costs 22 launches
// per supernode (16 up, 6 down) of which all but two touch nj x nn = a few thousand numbers: the sweep is a
// chain of launch latencies (956 launches, 5.3 ms; the host cannot even issue them faster).  Here the nn-wide
// algebra of a supernode is done by the threads that own the rows: 3 launches up, 1 down.

// w <- (L L^T)^-1 w, L = Lnn (nn x nn lower, ld THIN_NN) in shared memory
__device__ __forceinline__ void thin_dsolve(const double *Lnn, int nn, double (&w)[THIN_NN]) {
#pragma unroll
    for (int a = 0; a < THIN_NN; ++a) {
        if (a < nn) {
            double t = w[a];
#pragma unroll
            for (int b = 0; b < THIN_NN; ++b)
                if (b < a) t = fma(-Lnn[a + b * THIN_NN], w[b], t);
            w[a] = t / Lnn[a + a * THIN_NN];
        }
    }
#pragma unroll
    for (int a = THIN_NN - 1; a >= 0; --a) {
        if (a < nn) {
            double t = w[a];
#pragma unroll
            for (int b = THIN_NN - 1; b >= 0; --b)
                if (b > a && b < nn) t = fma(-Lnn[b + a * THIN_NN], w[b], t);
            w[a] = t / Lnn[a + a * THIN_NN];
        }
    }
}

// Forward Hessian, leaves-to-root pass of a thin supernode in ONE launch over alpha x alpha (32 x 32 per CTA).  Every CTA
// forms F_nn (block + children) and, for its 32 rows i and 32 rows j of alpha, F_an (block + children) and
// K_an = F_an - Lt F_nn (a few hundred numbers: cheaper than a launch that would hand them over), then
//     U'(i, j) = children(i, j) - Lt(i, :) F_an(j, :)^T - K_an(i, :) Lt(j, :)^T.
// The CTAs of the first tile column leave W(:, i) = D^-1 K_an(i, :)^T for the product M_an = Y_aa W^T that follows;
// the CTA that finishes LAST (every CTA has read the block's nn x nn part by then) stores M_nn = D^-1 F_nn D^-1 into it.
__global__ void __launch_bounds__(256) thin_up_kernel(BigArgs r, const double *__restrict__ Lb, double *__restrict__ blk, double *__restrict__ U,
                                                      double *__restrict__ W, unsigned *__restrict__ counter) {
    __shared__ double Li[THIN_NN][THIN_TS + 1], Lj[THIN_NN][THIN_TS + 1], Fi[THIN_NN][THIN_TS + 1], Fj[THIN_NN][THIN_TS + 1], Ki[THIN_NN][THIN_TS + 1];
    __shared__ double Fnn[THIN_NN * THIN_NN], Lnn[THIN_NN * THIN_NN], T1[THIN_NN * THIN_NN], Msm[THIN_NN * THIN_NN];
    __shared__ bool last_s;
    const int nn = r.nn, na = r.na, nj = r.nj, tid = threadIdx.x;
    const int i0 = blockIdx.x * THIN_TS, j0 = blockIdx.y * THIN_TS;
    if (tid < nn * nn) {
        const int a = tid % nn, b = tid / nn;
        const int hi = max(a, b), lo = min(a, b);
        Fnn[a + b * THIN_NN] = blk[hi + (long long)lo * nj] + big_children(r, a, b, false);
        Lnn[a + b * THIN_NN] = (a >= b) ? Lb[a + (long long)b * nj] : 0.0;
    }
    for (int idx = tid; idx < THIN_TS * nn; idx += 256) {
        const int rr = idx % THIN_TS, k = idx / THIN_TS;
        const int i = i0 + rr, j = j0 + rr;
        Li[k][rr] = (i < na) ? Lb[(nn + i) + (long long)k * nj] : 0.0;
        Fi[k][rr] = (i < na) ? blk[(nn + i) + (long long)k * nj] + big_children(r, nn + i, k, false) : 0.0;
        Lj[k][rr] = (j < na) ? Lb[(nn + j) + (long long)k * nj] : 0.0;
        Fj[k][rr] = (j < na) ? blk[(nn + j) + (long long)k * nj] + big_children(r, nn + j, k, false) : 0.0;
    }
    __syncthreads();
    for (int idx = tid; idx < THIN_TS * nn; idx += 256) {
        const int rr = idx % THIN_TS, k = idx / THIN_TS;
        double t = Fi[k][rr];
        for (int l = 0; l < nn; ++l) t = fma(-Li[l][rr], Fnn[l + k * THIN_NN], t);
        Ki[k][rr] = t;
    }
    __syncthreads();
    const int tx = tid & 31, ty = tid >> 5;
#pragma unroll
    for (int ri = 0; ri < THIN_TS / 32; ++ri) {
        const int ii = tx + 32 * ri, i = i0 + ii;
        if (i >= na) continue;
#pragma unroll
        for (int qg = 0; qg < THIN_TS / 32; ++qg) {
            int jc[4];
            bool live[4];
            double ch[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) { jc[q] = nn + j0 + ty + 8 * (4 * qg + q); live[q] = j0 + ty + 8 * (4 * qg + q) < na; }
            big_children_row4(r, nn + i, jc, live, false, ch);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int jj = ty + 8 * (4 * qg + q), j = j0 + jj;
                if (j < na) {
                    double v = ch[q];
                    for (int k = 0; k < nn; ++k) v = fma(-Li[k][ii], Fj[k][jj], v);
                    for (int k = 0; k < nn; ++k) v = fma(-Ki[k][ii], Lj[k][jj], v);
                    U[i + (long long)j * na] = v;
                }
            }
        }
        if (blockIdx.y == 0 && ty == 0) {
            double w[THIN_NN];
#pragma unroll
            for (int k = 0; k < THIN_NN; ++k) w[k] = (k < nn) ? Ki[k][ii] : 0.0;
            thin_dsolve(Lnn, nn, w);
#pragma unroll
            for (int k = 0; k < THIN_NN; ++k)
                if (k < nn) W[k + (long long)i * nn] = w[k];
        }
    }
    __threadfence();
    __syncthreads();
    if (tid == 0) {
        const unsigned done = atomicAdd(counter, 1u);
        last_s = (done == gridDim.x * gridDim.y - 1);
    }
    __syncthreads();
    if (!last_s) return;
    // T1 = D^-1 F_nn (columns), M = T1 D^-1 (rows), stored symmetrised (lower; the upper part of the block is zero)
    if (tid < nn) {
        double c[THIN_NN];
#pragma unroll
        for (int a = 0; a < THIN_NN; ++a) c[a] = (a < nn) ? Fnn[a + tid * THIN_NN] : 0.0;
        thin_dsolve(Lnn, nn, c);
#pragma unroll
        for (int a = 0; a < THIN_NN; ++a)
            if (a < nn) T1[a + tid * THIN_NN] = c[a];
    }
    __syncthreads();
    if (tid < nn) {
        double c[THIN_NN];
#pragma unroll
        for (int b = 0; b < THIN_NN; ++b) c[b] = (b < nn) ? T1[tid + b * THIN_NN] : 0.0;
        thin_dsolve(Lnn, nn, c);
#pragma unroll
        for (int b = 0; b < THIN_NN; ++b)
            if (b < nn) Msm[tid + b * THIN_NN] = c[b];
    }
    __syncthreads();
    if (tid < nn * nn) {
        const int a = tid % nn, b = tid / nn;
        blk[a + (long long)b * nj] = (a >= b) ? 0.5 * (Msm[a + b * THIN_NN] + Msm[b + a * THIN_NN]) : 0.0;
    }
    if (tid == 0) *counter = 0u;
}

// Forward Hessian, root-to-leaves pass of a thin supernode in ONE launch: a CTA owns 16 rows of alpha,
// Z_an(i, :) = M_an(i, :) - sum_k Z_aa(i, k) Lt(k, :) with Z_aa gathered from the ancestors' blocks (32 slices
// of k per row; partial sums combined in a fixed order), then its share of S = Lt^T M_an + Z_an^T Lt; the
// CTA that finishes last adds the shares in CTA order and forms Z_nn = M_nn - sym(S)  (deterministic).
__global__ void __launch_bounds__(512) thin_down_kernel(int nn, int na, int nj, const int *__restrict__ aaidx, const double *__restrict__ Xb,
                                                        const double *__restrict__ Lb, double *__restrict__ blk, double *__restrict__ part,
                                                        unsigned *__restrict__ counter) {
    __shared__ double red[32][16][THIN_NN + 1];
    __shared__ double Ssm[THIN_NN * THIN_NN];
    __shared__ bool last_s;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int row = tid & 15, slice = tid >> 4;          // 16 rows x 32 slices of k
    const int i = blockIdx.x * 16 + row;
    const int kc = (na + 31) / 32, k0 = slice * kc, k1 = min(na, k0 + kc);
    double acc[THIN_NN];
#pragma unroll
    for (int l = 0; l < THIN_NN; ++l) acc[l] = 0.0;
    if (i < na) {
        const int *ai = aaidx + i;
        const double *Lt = Lb + nn;
#pragma unroll 4
        for (int k = k0; k < k1; ++k) {
            const double z = Xb[ai[(long long)k * na]];
#pragma unroll
            for (int l = 0; l < THIN_NN; ++l)
                if (l < nn) acc[l] = fma(z, __ldg(Lt + k + (long long)l * nj), acc[l]);
        }
    }
#pragma unroll
    for (int l = 0; l < THIN_NN; ++l) red[slice][row][l] = acc[l];
    __syncthreads();
    if (warp == 0) {
        double mold[THIN_NN], zan[THIN_NN], lt[THIN_NN];
#pragma unroll
        for (int l = 0; l < THIN_NN; ++l) {
            mold[l] = zan[l] = lt[l] = 0.0;
            if (l < nn && i < na && lane < 16) {
                double t = red[0][row][l];
#pragma unroll
                for (int w = 1; w < 32; ++w) t += red[w][row][l];
                double *p = blk + (nn + i) + (long long)l * nj;
                mold[l] = *p;
                zan[l] = mold[l] - t;
                *p = zan[l];
                lt[l] = Lb[(nn + i) + (long long)l * nj];
            }
        }
        // this CTA's share of S(a, b) = sum_i Lt(i, a) M_an(i, b) + Z_an(i, a) Lt(i, b)
#pragma unroll
        for (int a = 0; a < THIN_NN; ++a)
#pragma unroll
            for (int b = 0; b < THIN_NN; ++b)
                if (a < nn && b < nn) {
                    double v = fma(lt[a], mold[b], zan[a] * lt[b]);
                    for (int o = 8; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
                    if (lane == 0) part[(long long)blockIdx.x * (THIN_NN * THIN_NN) + a + b * THIN_NN] = v;
                }
    }
    __threadfence();
    __syncthreads();
    if (tid == 0) {
        const unsigned done = atomicAdd(counter, 1u);
        last_s = (done == gridDim.x - 1);
    }
    __syncthreads();
    if (!last_s) return;
    __threadfence();
    if (tid < nn * nn) {
        const int a = tid % nn, b = tid / nn;
        double sacc = 0.0;
        for (unsigned c = 0; c < gridDim.x; ++c) sacc += __ldcg(part + (long long)c * (THIN_NN * THIN_NN) + a + b * THIN_NN);
        Ssm[a + b * THIN_NN] = sacc;
    }
    __syncthreads();
    if (tid < nn * nn) {
        const int a = tid % nn, b = tid / nn;
        double *d = blk + a + (long long)b * nj;
        *d = (a >= b) ? *d - 0.5 * (Ssm[a + b * THIN_NN] + Ssm[b + a * THIN_NN]) : 0.0;
    }
    if (tid == 0) *counter = 0u;
}

// Inverse Hessian, per-supernode phase of a thin supernode in ONE launch (same layout as thin_down_kernel):
// M_an(i, :) = Z_an(i, :) + sum_k Z_aa(i, k) Lt(k, :), the row of M_an D goes to Kan (the two triangular solves with
// chol(Y_aa) follow), the CTA's share of Lt^T Z_an + M_an^T Lt to `part`; the last CTA forms K_nn = D (Z_nn + S) D.
__global__ void __launch_bounds__(512) thin_hinv_local_kernel(int nn, int na, int nj, const int *__restrict__ aaidx, const double *__restrict__ Xb,
                                                              const double *__restrict__ Lb, const double *__restrict__ blk,
                                                              double *__restrict__ Knn, double *__restrict__ Kan, double *__restrict__ part,
                                                              unsigned *__restrict__ counter) {
    __shared__ double red[32][16][THIN_NN + 1];
    __shared__ double Dsm[THIN_NN * THIN_NN], Msm[THIN_NN * THIN_NN], Tsm[THIN_NN * THIN_NN];
    __shared__ bool last_s;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int row = tid & 15, slice = tid >> 4;          // 16 rows x 32 slices of k
    const int i = blockIdx.x * 16 + row;
    const int kc = (na + 31) / 32, k0 = slice * kc, k1 = min(na, k0 + kc);
    if (tid < nn * nn) {
        // D = L L^T
        const int a = tid % nn, b = tid / nn;
        double t = 0.0;
        for (int c = 0; c <= min(a, b); ++c) t = fma(Lb[a + (long long)c * nj], Lb[b + (long long)c * nj], t);
        Dsm[a + b * THIN_NN] = t;
    }
    double acc[THIN_NN];
#pragma unroll
    for (int l = 0; l < THIN_NN; ++l) acc[l] = 0.0;
    if (i < na) {
        const int *ai = aaidx + i;
        const double *Lt = Lb + nn;
#pragma unroll 4
        for (int k = k0; k < k1; ++k) {
            const double z = Xb[ai[(long long)k * na]];
#pragma unroll
            for (int l = 0; l < THIN_NN; ++l)
                if (l < nn) acc[l] = fma(z, __ldg(Lt + k + (long long)l * nj), acc[l]);
        }
    }
#pragma unroll
    for (int l = 0; l < THIN_NN; ++l) red[slice][row][l] = acc[l];
    __syncthreads();
    if (warp == 0) {
        double zan[THIN_NN], man[THIN_NN], lt[THIN_NN];
#pragma unroll
        for (int l = 0; l < THIN_NN; ++l) {
            zan[l] = man[l] = lt[l] = 0.0;
            if (l < nn && i < na && lane < 16) {
                double t = red[0][row][l];
#pragma unroll
                for (int w = 1; w < 32; ++w) t += red[w][row][l];
                zan[l] = blk[(nn + i) + (long long)l * nj];
                man[l] = zan[l] + t;
                lt[l] = Lb[(nn + i) + (long long)l * nj];
            }
        }
        if (i < na && lane < 16) {
#pragma unroll
            for (int b = 0; b < THIN_NN; ++b)
                if (b < nn) {
                    double t = 0.0;
#pragma unroll
                    for (int a = 0; a < THIN_NN; ++a)
                        if (a < nn) t = fma(man[a], Dsm[a + b * THIN_NN], t);
                    Kan[i + (long long)b * na] = t;
                }
        }
#pragma unroll
        for (int a = 0; a < THIN_NN; ++a)
#pragma unroll
            for (int b = 0; b < THIN_NN; ++b)
                if (a < nn && b < nn) {
                    double v = fma(lt[a], zan[b], man[a] * lt[b]);
                    for (int o = 8; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
                    if (lane == 0) part[(long long)blockIdx.x * (THIN_NN * THIN_NN) + a + b * THIN_NN] = v;
                }
    }
    __threadfence();
    __syncthreads();
    if (tid == 0) {
        const unsigned done = atomicAdd(counter, 1u);
        last_s = (done == gridDim.x - 1);
    }
    __syncthreads();
    if (!last_s) return;
    __threadfence();
    if (tid < nn * nn) {
        const int a = tid % nn, b = tid / nn;
        const int hi = max(a, b), lo = min(a, b);
        double sacc = blk[hi + (long long)lo * nj];
        for (unsigned c = 0; c < gridDim.x; ++c) sacc += __ldcg(part + (long long)c * (THIN_NN * THIN_NN) + a + b * THIN_NN);
        Msm[a + b * THIN_NN] = sacc;
    }
    __syncthreads();
    if (tid < nn * nn) {
        const int a = tid % nn, b = tid / nn;
        double t = 0.0;
        for (int c = 0; c < nn; ++c) t = fma(Dsm[a + c * THIN_NN], Msm[c + b * THIN_NN], t);
        Tsm[a + b * THIN_NN] = t;
    }
    __syncthreads();
    if (tid < nn * nn) {
        const int a = tid % nn, b = tid / nn;
        double t = 0.0;
        for (int c = 0; c < nn; ++c) t = fma(Tsm[a + c * THIN_NN], Dsm[c + b * THIN_NN], t);
        Knn[a + b * nn] = t;
    }
    if (tid == 0) *counter = 0u;
}

// Inverse Hessian, leaves-to-root sweep of a thin supernode in ONE launch: F_an = K_an + Lt K_nn,
// U = Lt K_an^T + F_an Lt^T + children over alpha x alpha (32 x 32 per CTA); the CTAs of the first tile column
// also store F_an + children into the block, CTA (0, 0) the symmetrised K_nn + children.
__global__ void __launch_bounds__(256) thin_hinv_sweep_kernel(BigArgs r, const double *__restrict__ Lb, const double *__restrict__ Knn,
                                                              const double *__restrict__ Kan, double *__restrict__ blk, double *__restrict__ U) {
    __shared__ double Li[THIN_NN][THIN_TS + 1], Lj[THIN_NN][THIN_TS + 1], Kj[THIN_NN][THIN_TS + 1], Fi[THIN_NN][THIN_TS + 1], Ks[THIN_NN * THIN_NN];
    const int nn = r.nn, na = r.na, nj = r.nj, tid = threadIdx.x;
    const int i0 = blockIdx.x * THIN_TS, j0 = blockIdx.y * THIN_TS;
    if (tid < nn * nn) Ks[(tid % nn) + (tid / nn) * THIN_NN] = Knn[tid];
    for (int idx = tid; idx < THIN_TS * nn; idx += 256) {
        const int rr = idx % THIN_TS, k = idx / THIN_TS;
        const bool vi = i0 + rr < na, vj = j0 + rr < na;
        Li[k][rr] = vi ? Lb[(nn + i0 + rr) + (long long)k * nj] : 0.0;
        Lj[k][rr] = vj ? Lb[(nn + j0 + rr) + (long long)k * nj] : 0.0;
        Kj[k][rr] = vj ? Kan[(j0 + rr) + (long long)k * na] : 0.0;
    }
    __syncthreads();
    for (int idx = tid; idx < THIN_TS * nn; idx += 256) {
        const int rr = idx % THIN_TS, k = idx / THIN_TS;
        double t = (i0 + rr < na) ? Kan[(i0 + rr) + (long long)k * na] : 0.0;
        for (int c = 0; c < nn; ++c) t = fma(Li[c][rr], Ks[c + k * THIN_NN], t);
        Fi[k][rr] = t;
    }
    __syncthreads();
    const int tx = tid & 31, ty = tid >> 5;
#pragma unroll
    for (int ri = 0; ri < THIN_TS / 32; ++ri) {
        const int ii = tx + 32 * ri, i = i0 + ii;
        if (i >= na) continue;
#pragma unroll
        for (int qg = 0; qg < THIN_TS / 32; ++qg) {
            int jc[4];
            bool live[4];
            double ch[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) { jc[q] = nn + j0 + ty + 8 * (4 * qg + q); live[q] = j0 + ty + 8 * (4 * qg + q) < na; }
            big_children_row4(r, nn + i, jc, live, false, ch);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int jj = ty + 8 * (4 * qg + q), j = j0 + jj;
                if (j < na) {
                    double v = 0.0;
                    for (int k = 0; k < nn; ++k) v = fma(Li[k][ii], Kj[k][jj], v);
                    for (int k = 0; k < nn; ++k) v = fma(Fi[k][ii], Lj[k][jj], v);
                    U[i + (long long)j * na] = v + ch[q];
                }
            }
        }
        if (blockIdx.y == 0 && ty < nn) {
            for (int k = ty; k < nn; k += 8) blk[(nn + i) + (long long)k * nj] = Fi[k][ii] + big_children(r, nn + i, k, false);
        }
    }
    if (blockIdx.x == 0 && blockIdx.y == 0 && tid < nn * nn) {
        const int a = tid % nn, b = tid / nn;
        if (a >= b) {
            const double x = Ks[a + b * THIN_NN] + big_children(r, a, b, false);
            const double y = Ks[b + a * THIN_NN] + big_children(r, b, a, false);
            blk[a + (long long)b * nj] = 0.5 * (x + y);
        } else blk[a + (long long)b * nj] = 0.0;
    }
}

// ---- forward Hessian, pass 1 + scaling ---------------------------------------------------
int big_hess_up(smcp_sym *s, const BigNode &q, const double *Lt, const double *Yaa_all, double *X, int64_t b) {
    smcp_ctx *ctx = s->ctx;
    const int nn = q.nn, na = q.na, nj = q.nj;
    double *blk = X + (size_t)b * s->d.nblk + q.boff;
    double *Uk = s->upd + (size_t)b * s->d.nupd + q.uoff;
    const double *Lb = Lt + q.boff, *Ltan = Lb + nn, *Yaa = Yaa_all + q.uoff;
    double *F = WS(0), *T1 = WS(1), *T2 = WS(2);
    if (nn <= THIN_NN && na >= 1) {
        // W of this supernode outlives the launch on its lane (the product below runs on a side stream): own slot
        const size_t tidx = (size_t)(&q - s->big.data());
        if (s->thin_w_off.empty()) {
            size_t tot = 0;
            for (const BigNode &t : s->big) { s->thin_w_off.push_back(tot); if (t.nn <= THIN_NN) tot += (size_t)t.na * t.nn; }
            CUDA_TRY(cudaMalloc(&s->thin_w, std::max<size_t>(tot, 1) * sizeof(double)));
            s->allocs.push_back(s->thin_w);
        }
        double *W = s->thin_w + s->thin_w_off[tidx];
        if (!s->thin_counters) {
            CUDA_TRY(cudaMalloc(&s->thin_counters, 64 * sizeof(unsigned)));
            CUDA_TRY(cudaMemset(s->thin_counters, 0, 64 * sizeof(unsigned)));
            s->allocs.push_back(s->thin_counters);
        }
        {
            LaunchScope ls_(ctx, "thin_up");
            thin_up_kernel<<<dim3((unsigned)((na + THIN_TS - 1) / THIN_TS), (unsigned)((na + THIN_TS - 1) / THIN_TS)), 256, 0, ctx->stream>>>(big_args(s, q, b), Lb, blk, Uk, W,
                                                                                                                  s->thin_counters + s->big_lane);
        }
        // M_an = Y_aa W^T.  Y_aa is stored full and exactly symmetric (the alpha x alpha gather mirrors the lower entries), so
        // it is read as its transpose: a warp then owns a row and streams one contiguous column (na / 8 CTAs instead of na / 32)
        // Nothing in the rest of the leaves-to-root pass reads M_an (the parents take the update matrix): the product
        // leaves the chain of dependent launches and runs on a side stream; big_thin_join() waits for all of them before
        // the root-to-leaves pass
        if (ctx->prof) {
            if (G(s, true, false, Yaa, na, W, nn, blk + nn, nj, na, nn, na, 1.0, 0)) return -1;
        } else {
            if (s->thin_side.empty()) {
                for (int i = 0; i < 4; ++i) {
                    cudaStream_t st;
                    CUDA_TRY(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
                    s->thin_side.push_back(st);
                }
                for (size_t i = 0; i < 2 * s->big.size(); ++i) {
                    cudaEvent_t e;
                    CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
                    s->thin_ev.push_back(e);
                }
            }
            cudaStream_t side = s->thin_side[tidx % s->thin_side.size()];
            CUDA_TRY(cudaEventRecord(s->thin_ev[2 * tidx], ctx->stream));
            CUDA_TRY(cudaStreamWaitEvent(side, s->thin_ev[2 * tidx], 0));
            cudaStream_t saved = ctx->stream;
            ctx->stream = side;
            const int rc = G(s, true, false, Yaa, na, W, nn, blk + nn, nj, na, nn, na, 1.0, 0);
            ctx->stream = saved;
            if (rc) return -1;
            CUDA_TRY(cudaEventRecord(s->thin_ev[2 * tidx + 1], side));
            s->thin_pending.push_back((int)tidx);
        }
        CUDA_TRY(cudaGetLastError());
        return 0;
    }
    double *Fan = F + nn, *Faa = F + nn + (size_t)nn * nj, *Fna = F + (size_t)nn * nj;
    ELEM(big_front_full_kernel, (long long)nj * nj, big_args(s, q, b), blk, F);
    if (na) {
        // K_an = F_an - Lt F_nn
        if (G(s, false, true, Ltan, nj, F, nj, Fan, nj, na, nn, nn, -1.0, 1)) return -1;
        // U' = F_aa - Lt F_an(old)^T - K_an Lt^T ; F_na still holds F_an(old)^T
        if (G(s, false, true, Ltan, nj, Fna, nj, Faa, nj, na, na, nn, -1.0, 1)) return -1;
        if (G(s, false, false, Fan, nj, Ltan, nj, Faa, nj, na, na, nn, -1.0, 1)) return -1;
        ELEM(big_copy_mat_kernel, (long long)na * na, Faa, nj, Uk, na, na, na, 0);
    }
    // M_nn = D^{-1} F_nn D^{-1}
    if (nn >= 256) {
        // wide supernode (the root of rand_SDP: 1186 columns): D^-1 = L^-T L^-1 is formed ONCE per scaling point
        // (one triangular solve on the identity + one product) and every Hessian is two DMMA products instead of
        // four triangular solves with nn right-hand sides and two transposes (1.4 ms -> 0.4 ms at nn = 1186)
        const size_t idx = (size_t)(&q - s->big.data());
        if (s->big_dinv_off.empty()) {
            size_t tot = 0;
            for (const BigNode &t : s->big) { s->big_dinv_off.push_back(tot); if (t.nn >= 256) tot += (size_t)t.nn * t.nn; }
            s->big_dinv_gen.assign(s->big.size(), 0);
            CUDA_TRY(cudaMalloc(&s->big_dinv, std::max<size_t>(tot, 1) * sizeof(double)));
            s->allocs.push_back(s->big_dinv);
        }
        double *Dinv = s->big_dinv + s->big_dinv_off[idx];
        if (s->big_dinv_gen[idx] != s->lt_gen_cur) {
            ELEM(big_identity_kernel, (long long)nn * nn, T1, nn, nn);
            if (d_trsm_left_lower(ctx, false, Lb, nj, nn, T1, nn, nn)) return -1;                  // L^-1
            if (G(s, true, true, T1, nn, T1, nn, Dinv, nn, nn, nn, nn, 1.0, 0)) return -1;         // D^-1 = L^-T L^-1 (full)
            s->big_dinv_gen[idx] = s->lt_gen_cur;
        }
        if (G(s, true, true, Dinv, nn, F, nj, T1, nn, nn, nn, nn, 1.0, 0)) return -1;              // D^-1 F   (both symmetric)
        if (G(s, false, true, T1, nn, Dinv, nn, T2, nn, nn, nn, nn, 1.0, 0)) return -1;            // (D^-1 F) D^-1
    } else {
        if (d_trsm_left_lower(ctx, false, Lb, nj, nn, F, nj, nn)) return -1;          // L^-1 F
        big_transpose(s, F, nj, nn, nn, T1, nn);
        if (d_trsm_left_lower(ctx, false, Lb, nj, nn, T1, nn, nn)) return -1;         // L^-1 F L^-T
        if (d_trsm_left_lower(ctx, true, Lb, nj, nn, T1, nn, nn)) return -1;          // L^-T (.)
        big_transpose(s, T1, nn, nn, nn, T2, nn);
        if (d_trsm_left_lower(ctx, true, Lb, nj, nn, T2, nn, nn)) return -1;          // D^-1 F D^-1
    }
    if (na) {
        // M_an = Y_aa K_an D^{-1}: W = D^{-1} K_an^T, M_an = Y_aa W^T
        double *W = T1;
        big_transpose(s, Fan, nj, na, nn, W, nn);
        if (d_trsm_left_lower(ctx, false, Lb, nj, nn, W, nn, na)) return -1;
        if (d_trsm_left_lower(ctx, true, Lb, nj, nn, W, nn, na)) return -1;
        if (G(s, false, false, Yaa, na, W, nn, blk + nn, nj, na, nn, na, 1.0, 0)) return -1;
    }
    ELEM(big_sym_store_kernel, (long long)nn * nn, T2, nn, blk, nj, nn, 0.0, 1.0);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// the side-stream products of big_hess_up must have landed before anything reads M_an
int big_thin_join(smcp_sym *s) {
    for (int idx : s->thin_pending) CUDA_TRY(cudaStreamWaitEvent(s->ctx->stream, s->thin_ev[2 * (size_t)idx + 1], 0));
    s->thin_pending.clear();
    return 0;
}

// ---- forward Hessian, pass 3 (root to leaves) --------------------------------------------
int big_hess_down(smcp_sym *s, const BigNode &q, const double *Lt, double *X, int64_t b) {
    smcp_ctx *ctx = s->ctx;
    const int nn = q.nn, na = q.na, nj = q.nj;
    if (!na) return 0;
    double *Xb = X + (size_t)b * s->d.nblk;
    double *blk = Xb + q.boff;
    const double *Ltan = Lt + q.boff + nn;
    double *Zaa = WS(0), *Mold = WS(1), *S = WS(2);
    if (nn <= THIN_NN && na >= 1) {
        if (!s->thin_counters) {
            CUDA_TRY(cudaMalloc(&s->thin_counters, 64 * sizeof(unsigned)));
            CUDA_TRY(cudaMemset(s->thin_counters, 0, 64 * sizeof(unsigned)));
            s->allocs.push_back(s->thin_counters);
        }
        LaunchScope ls_(ctx, "thin_down");
        thin_down_kernel<<<(unsigned)((na + 15) / 16), 512, 0, ctx->stream>>>(nn, na, nj, s->d.aaidx + q.uoff, Xb, Lt + q.boff, blk, WS(0),
                                                                              s->thin_counters + s->big_lane);
        CUDA_TRY(cudaGetLastError());
        return 0;
    }
    ELEM(big_gather_aa_kernel, (long long)na * na, s->d.aaidx + q.uoff, Xb, Zaa, (long long)na * na);
    ELEM(big_copy_mat_kernel, (long long)na * nn, blk + nn, nj, Mold, na, na, nn, 0);
    // Z_an = M_an - Z_aa Lt
    if (G(s, false, true, Zaa, na, Ltan, nj, blk + nn, nj, na, nn, na, -1.0, 1)) return -1;
    // S = Lt^T M_an(old) + Z_an^T Lt ; Z_nn = M_nn - sym(S)
    if (G(s, true, true, Ltan, nj, Mold, na, S, nn, nn, nn, na, 1.0, 0)) return -1;
    if (G(s, true, true, blk + nn, nj, Ltan, nj, S, nn, nn, nn, na, 1.0, 1)) return -1;
    ELEM(big_sym_store_kernel, (long long)nn * nn, S, nn, blk, nj, nn, 1.0, -1.0);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// ---- inverse Hessian ----------------------------------------------------------------------
// Two phases (SURVEY App. A.5: every stage but the final extend-add is independent per supernode):
//   local: reads the supernode's own block and the still-untouched alpha x alpha entries of its ancestors,
//          leaves K_nn = D M_nn D and K_an = Y_aa^-1 M_an D in the scratch block KS (nn^2 | na x nn);
//          all supernodes at once, in any order -- with several ranks they are shared out (chordal.cu);
//   sweep: F_an = K_an + Lt K_nn, F_aa = Lt K_an^T + F_an Lt^T, children's update matrices added, leaves to root.
int big_hess_inv_local(smcp_sym *s, const BigNode &q, const double *Lt, const double *Raa_all, const double *X, int64_t b, double *KS) {
    smcp_ctx *ctx = s->ctx;
    const int nn = q.nn, na = q.na, nj = q.nj;
    const double *Xb = X + (size_t)b * s->d.nblk;
    const double *blk = Xb + q.boff;
    const double *Lb = Lt + q.boff, *Ltan = Lb + nn, *R = Raa_all + q.uoff;
    double *D = WS(0), *Zaa = WS(1), *Man = WS(2), *T = WS(4);
    double *Mnn = KS + q.boff, *Kan = Mnn + (size_t)nn * nn;
    if (nn <= THIN_NN && na >= 1) {
        if (!s->thin_counters) {
            CUDA_TRY(cudaMalloc(&s->thin_counters, 64 * sizeof(unsigned)));
            CUDA_TRY(cudaMemset(s->thin_counters, 0, 64 * sizeof(unsigned)));
            s->allocs.push_back(s->thin_counters);
        }
        {
            LaunchScope ls_(ctx, "thin_hinv_local");
            thin_hinv_local_kernel<<<(unsigned)((na + 15) / 16), 512, 0, ctx->stream>>>(nn, na, nj, s->d.aaidx + q.uoff, Xb, Lb, blk, Mnn, Kan, WS(0),
                                                                                        s->thin_counters + s->big_lane);
        }
        // K_an = Y_aa^-1 M_an D.  One or two columns against the ~1100-row factor R = chol(Y_aa): ONE cluster launch
        // for both substitutions; R's inverted 64 x 64 diagonal blocks are kept per supernode for the whole life of
        // the scaling point (they were rebuilt by a trtri launch in front of every solve)
        if (nn <= 2 && na >= 256 && na <= 16384) {
            const size_t idx = (size_t)(&q - s->big.data());
            if (s->thin_dinv_off.empty()) {
                size_t tot = 0;
                for (const BigNode &t : s->big) { s->thin_dinv_off.push_back(tot); tot += (size_t)((t.na + 63) / 64) * 4096; }
                s->thin_dinv_gen.assign(s->big.size(), 0);
                CUDA_TRY(cudaMalloc(&s->thin_dinv, std::max<size_t>(tot, 1) * sizeof(double)));
                s->allocs.push_back(s->thin_dinv);
            }
            double *Dinv = s->thin_dinv + s->thin_dinv_off[idx];
            if (s->thin_dinv_gen[idx] != s->raa_gen_cur) {
                if (d_potrs_prepare(ctx, R, na, na, Dinv)) return -1;
                s->thin_dinv_gen[idx] = s->raa_gen_cur;
            }
            if (d_trs_cluster(ctx, R, na, na, Dinv, Kan, na, nn, 1, 1, "trsm_cluster")) return -1;
        } else {
            if (d_trsm_left_lower(ctx, false, R, na, na, Kan, na, nn)) return -1;
            if (d_trsm_left_lower(ctx, true, R, na, na, Kan, na, nn)) return -1;
        }
        CUDA_TRY(cudaGetLastError());
        return 0;
    }
    if (G(s, false, false, Lb, nj, Lb, nj, D, nn, nn, nn, nn, 1.0, 0)) return -1;                 // D = L L^T (full)
    ELEM(big_sym_copy_kernel, (long long)nn * nn, blk, nj, Mnn, nn, nn);                          // Z_nn (full)
    if (na) {
        ELEM(big_gather_aa_kernel, (long long)na * na, s->d.aaidx + q.uoff, Xb, Zaa, (long long)na * na);
        ELEM(big_copy_mat_kernel, (long long)na * nn, blk + nn, nj, Man, na, na, nn, 0);
        if (G(s, false, true, Zaa, na, Ltan, nj, Man, na, na, nn, na, 1.0, 1)) return -1;          // M_an = Z_an + Z_aa Lt
        if (G(s, true, true, Ltan, nj, blk + nn, nj, Mnn, nn, nn, nn, na, 1.0, 1)) return -1;      // += Lt^T Z_an
        if (G(s, true, true, Man, na, Ltan, nj, Mnn, nn, nn, nn, na, 1.0, 1)) return -1;           // += M_an^T Lt
    }
    if (G(s, false, true, D, nn, Mnn, nn, T, nn, nn, nn, nn, 1.0, 0)) return -1;                   // D M
    if (G(s, false, true, T, nn, D, nn, Mnn, nn, nn, nn, nn, 1.0, 0)) return -1;                   // K_nn = D M D
    if (na) {
        if (G(s, false, true, Man, na, D, nn, Kan, na, na, nn, nn, 1.0, 0)) return -1;             // M_an D
        if (d_trsm_left_lower(ctx, false, R, na, na, Kan, na, nn)) return -1;                      // K_an = Y_aa^-1 M_an D
        if (d_trsm_left_lower(ctx, true, R, na, na, Kan, na, nn)) return -1;
    }
    CUDA_TRY(cudaGetLastError());
    return 0;
}

int big_hess_inv_sweep(smcp_sym *s, const BigNode &q, const double *Lt, double *X, int64_t b, const double *KS) {
    smcp_ctx *ctx = s->ctx;
    const int nn = q.nn, na = q.na, nj = q.nj;
    double *blk = X + (size_t)b * s->d.nblk + q.boff;
    double *Uk = s->upd + (size_t)b * s->d.nupd + q.uoff;
    const double *Ltan = Lt + q.boff + nn;
    const double *Mnn = KS + q.boff, *Kan = Mnn + (size_t)nn * nn;
    double *Zaa = WS(1), *Man = WS(2);
    if (nn <= THIN_NN && na >= 1) {
        LaunchScope ls_(ctx, "thin_hinv_sweep");
        thin_hinv_sweep_kernel<<<dim3((unsigned)((na + THIN_TS - 1) / THIN_TS), (unsigned)((na + THIN_TS - 1) / THIN_TS)), 256, 0, ctx->stream>>>(big_args(s, q, b), Lt + q.boff, Mnn,
                                                                                                                      Kan, blk, Uk);
        CUDA_TRY(cudaGetLastError());
        return 0;
    }
    if (na) {
        ELEM(big_copy_mat_kernel, (long long)na * nn, Kan, na, Man, na, na, nn, 0);
        if (G(s, false, true, Ltan, nj, Mnn, nn, Man, na, na, nn, nn, 1.0, 1)) return -1;          // F_an = K_an + Lt K_nn
        if (G(s, false, false, Ltan, nj, Kan, na, Zaa, na, na, na, nn, 1.0, 0)) return -1;         // F_aa = Lt K_an^T
        if (G(s, false, false, Man, na, Ltan, nj, Zaa, na, na, na, nn, 1.0, 1)) return -1;         //      + F_an Lt^T
    }
    ELEM(big_hinv_store_kernel, (long long)nj * nj, big_args(s, q, b), Mnn, Man, Zaa, blk, Uk);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// ---- projected inverse (root to leaves) ------------------------------------------------------
int big_projinv(smcp_sym *s, const BigNode &q, double *X, int64_t b) {
    smcp_ctx *ctx = s->ctx;
    const int nn = q.nn, na = q.na, nj = q.nj;
    double *Xb = X + (size_t)b * s->d.nblk;
    double *blk = Xb + q.boff;
    double *LtT = WS(0), *Li = WS(1), *Di = WS(2), *Yaa = WS(3), *S = WS(4);
    if (na) {
        big_transpose(s, blk + nn, nj, na, nn, LtT, nn);                                          // L_an^T
        if (d_trsm_left_lower(ctx, true, blk, nj, nn, LtT, nn, na)) return -1;                      // Lt^T = L_nn^-T L_an^T
    }
    ELEM(big_identity_kernel, (long long)nn * nn, Li, nn, nn);
    if (d_trsm_left_lower(ctx, false, blk, nj, nn, Li, nn, nn)) return -1;                          // L^-1
    if (G(s, true, true, Li, nn, Li, nn, Di, nn, nn, nn, nn, 1.0, 0)) return -1;                    // D^-1 = L^-T L^-1 (full)
    if (na) {
        ELEM(big_gather_aa_kernel, (long long)na * na, s->d.aaidx + q.uoff, Xb, Yaa, (long long)na * na);
        if (G(s, false, false, Yaa, na, LtT, nn, blk + nn, nj, na, nn, na, -1.0, 0)) return -1;     // Y_an = -Y_aa Lt
        if (G(s, false, true, LtT, nn, blk + nn, nj, S, nn, nn, nn, na, 1.0, 0)) return -1;          // S = Lt^T Y_an
        ELEM(big_copy_mat_kernel, (long long)nn * nn, Di, nn, blk, nj, nn, nn, 1);
        ELEM(big_sym_store_kernel, (long long)nn * nn, S, nn, blk, nj, nn, 1.0, -1.0);              // Y_nn = D^-1 - sym(S)
    } else {
        ELEM(big_copy_mat_kernel, (long long)nn * nn, Di, nn, blk, nj, nn, nn, 1);
    }
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// Completion of a thin supernode after the partial factorisation and the backward solve (W = X_aa^-1 X_an): the
// trailing nn x nn block Delta = M^T M (M lower: a Cholesky factorisation run from the last row up), L_nn = M^-1,
// L_an = -W L_nn, and the verdict of the factorisation -- one launch instead of nine (two of them cooperative
// launches for a 1 x 1 "matrix").  Every CTA redoes the nn x nn part (nn <= 8), a thread owns a row of alpha.
__global__ void __launch_bounds__(128) thin_compl_tail_kernel(int nn, int na, int nj, const double *__restrict__ T, const double *__restrict__ W,
                                                              double *__restrict__ bout, const int *__restrict__ info, int *__restrict__ fail) {
    __shared__ double Ms[THIN_NN * THIN_NN], Ls[THIN_NN * THIN_NN];
    __shared__ int bad_s;
    const int tid = threadIdx.x;
    if (tid < THIN_NN * THIN_NN) {
        const int a = tid % THIN_NN, b = tid / THIN_NN;
        Ms[tid] = (a < nn && b < nn && a >= b) ? T[(na + a) + (long long)(na + b) * nj] : 0.0;
        Ls[tid] = 0.0;
    }
    __syncthreads();
    if (tid == 0) {
        int bad = 0;
        // in place: M(j, i), i <= j, from the last row up; Delta(j, i) = sum_{k >= j} M(k, j) M(k, i)
        for (int j = nn - 1; j >= 0; --j) {
            double d = Ms[j + j * THIN_NN];
            for (int k2 = j + 1; k2 < nn; ++k2) d = fma(-Ms[k2 + j * THIN_NN], Ms[k2 + j * THIN_NN], d);
            if (!(d > 0.0)) { bad = 1; d = 1.0; }
            const double mjj = sqrt(d);
            Ms[j + j * THIN_NN] = mjj;
            for (int i = 0; i < j; ++i) {
                double t = Ms[j + i * THIN_NN];
                for (int k2 = j + 1; k2 < nn; ++k2) t = fma(-Ms[k2 + j * THIN_NN], Ms[k2 + i * THIN_NN], t);
                Ms[j + i * THIN_NN] = t / mjj;
            }
        }
        // L_nn = M^-1 (lower), column by column
        for (int c = 0; c < nn; ++c) {
            for (int r2 = c; r2 < nn; ++r2) {
                double t = (r2 == c) ? 1.0 : 0.0;
                for (int p2 = c; p2 < r2; ++p2) t = fma(-Ms[r2 + p2 * THIN_NN], Ls[p2 + c * THIN_NN], t);
                Ls[r2 + c * THIN_NN] = t / Ms[r2 + r2 * THIN_NN];
            }
        }
        bad_s = bad;
    }
    __syncthreads();
    const int i = blockIdx.x * 128 + tid;
    if (i < na) {
        double w[THIN_NN];
#pragma unroll
        for (int k2 = 0; k2 < THIN_NN; ++k2) w[k2] = (k2 < nn) ? W[i + (long long)k2 * na] : 0.0;
#pragma unroll
        for (int j = 0; j < THIN_NN; ++j)
            if (j < nn) {
                double t = 0.0;
#pragma unroll
                for (int k2 = 0; k2 < THIN_NN; ++k2)
                    if (k2 >= j && k2 < nn) t = fma(w[k2], Ls[k2 + j * THIN_NN], t);
                bout[(nn + i) + (long long)j * nj] = -t;
            }
    }
    if (blockIdx.x == 0) {
        if (tid < nn * nn) {
            const int a = tid % nn, b = tid / nn;
            bout[a + (long long)b * nj] = (a >= b) ? Ls[a + b * THIN_NN] : 0.0;
        }
        if (tid == 0 && (bad_s || *info)) *fail = 1;
    }
}

// ---- completion (independent per supernode, out of place) ---------------------------------------
int big_completion(smcp_sym *s, const BigNode &q, double *X, const double *Xin, int64_t b) {
    smcp_ctx *ctx = s->ctx;
    const int nn = q.nn, na = q.na, nj = q.nj;
    const double *Xi = Xin + (size_t)b * s->d.nblk;
    const double *bin = Xi + q.boff;
    double *bout = X + (size_t)b * s->d.nblk + q.boff;
    double *T = WS(0), *Z = WS(1), *T0 = WS(3), *M = WS(4), *Li = WS(5);
    // The clique reordered as [alpha; nu]: ONE partial factorisation of T = [X_aa . ; X_na X_nn] with na
    // pivots gives R = chol(X_aa), Z^T = X_na R^-T in the rows below it and Delta = X_nn - Z^T Z in
    // the trailing block (instead of potrf + a forward solve + a rank-na product per supernode)
    ELEM(big_compl_front_kernel, (long long)nj * nj, s->d.aaidx + q.uoff, Xi, bin, T, nn, na, nj);
    if (na) {
        if (front_potrf(ctx, T, nj, nj, na, BIG_INFO)) return -1;
        if (nn > THIN_NN) big_flag_kernel<<<1, 1, 0, ctx->stream>>>(BIG_INFO, s->fail + b);   // thin: in the tail kernel
        big_transpose(s, T + na, nj, nn, na, Z, na);                                                // Z = R^-1 X_an
        if (d_trsm_left_lower(ctx, true, T, nj, na, Z, na, nn)) return -1;                          // W = X_aa^-1 X_an
    }
    if (nn <= THIN_NN && na >= 1) {
        LaunchScope ls_(ctx, "thin_compl_tail");
        thin_compl_tail_kernel<<<(unsigned)((na + 127) / 128), 128, 0, ctx->stream>>>(nn, na, nj, T, Z, bout, BIG_INFO, s->fail + b);
        CUDA_TRY(cudaGetLastError());
        return 0;
    }
    ELEM(big_reverse_kernel, (long long)nn * nn, T + na + (size_t)na * nj, nj, T0, nn, 0);
    if (front_potrf(ctx, T0, nn, nn, nn, BIG_INFO)) return -1;
    big_flag_kernel<<<1, 1, 0, ctx->stream>>>(BIG_INFO, s->fail + b);
    ELEM(big_reverse_kernel, (long long)nn * nn, T0, nn, M, nn, 1);                                 // Delta = M^T M
    ELEM(big_identity_kernel, (long long)nn * nn, Li, nn, nn);
    if (d_trsm_left_lower(ctx, false, M, nn, nn, Li, nn, nn)) return -1;                            // L_nn = M^-1
    ELEM(big_copy_mat_kernel, (long long)nn * nn, Li, nn, bout, nj, nn, nn, 1);
    if (na && G(s, false, true, Z, na, Li, nn, bout + nn, nj, na, nn, nn, -1.0, 0)) return -1;      // L_an = -W L_nn
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// ---- chordal trsm with many right-hand sides: one supernode of the top set ------------------------
// forward : B_nu <- L_nn^-1 B_nu ; B_alpha -= L_an B_nu          (rows alpha scattered: rowidx)
// backward: B_nu -= L_an^T B_alpha ; B_nu <- L_nn^-T B_nu
__global__ void big_rows_gather_kernel(const double *__restrict__ B, long long ldb, const int *__restrict__ rows, int na, long long nrhs,
                                       double *__restrict__ G) {
    BIG_LOOP((long long)na * nrhs) {
        const int i = (int)(idx % na);
        const long long c = idx / na;
        G[idx] = B[rows[i] + c * ldb];
    }
}
__global__ void big_rows_sub_kernel(double *__restrict__ B, long long ldb, const int *__restrict__ rows, int na, long long nrhs,
                                    const double *__restrict__ T) {
    BIG_LOOP((long long)na * nrhs) {
        const int i = (int)(idx % na);
        const long long c = idx / na;
        B[rows[i] + c * ldb] -= T[idx];
    }
}

// Thin supernode (nn <= THIN_NN) against many right-hand sides in ONE launch per direction.
//   forward : warp = right-hand side c: x = L_nn^-1 B_nu(:, c) in registers, then B(rows_i, c) -= L_an(i, :) x with the
//             lanes striding over the separator rows (coalesced: the rows of a separator are runs of consecutive indices);
//   backward: warp = right-hand side: lanes stride over the separator rows, t = L_an^T B_alpha(:, c) by a fixed-order
//             shuffle tree, lane 0 finishes x = L_nn^-T (B_nu(:, c) - t).
// The generic path took a 128 x 128-tile DMMA GEMM with M = nn (145 us a supernode at 2000 right-hand sides).
__global__ void __launch_bounds__(256) thin_trsm_fwd_kernel(int nn, int na, int nj, const double *__restrict__ blk, const int *__restrict__ rows,
                                                            int r0, double *__restrict__ B, long long ldb, long long nrhs) {
    __shared__ double Lnn[THIN_NN * THIN_NN];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid < nn * nn) Lnn[(tid % nn) + (tid / nn) * THIN_NN] = blk[(tid % nn) + (long long)(tid / nn) * nj];
    __syncthreads();
    const long long c = (long long)blockIdx.x * 8 + warp;
    if (c >= nrhs) return;
    double *bc = B + c * ldb;
    // every lane solves the nn x nn system of its column (same arithmetic), lane 0 stores it
    double x[THIN_NN];
#pragma unroll
    for (int a = 0; a < THIN_NN; ++a) x[a] = (a < nn) ? bc[r0 + a] : 0.0;
    __syncwarp();
#pragma unroll
    for (int a = 0; a < THIN_NN; ++a)
        if (a < nn) {
            double t = x[a];
#pragma unroll
            for (int b = 0; b < THIN_NN; ++b)
                if (b < a) t = fma(-Lnn[a + b * THIN_NN], x[b], t);
            x[a] = t / Lnn[a + a * THIN_NN];
            if (lane == 0) bc[r0 + a] = x[a];
        }
    const double *Lan = blk + nn;
    for (int i = lane; i < na; i += 32) {
        double t = 0.0;
#pragma unroll
        for (int a = 0; a < THIN_NN; ++a)
            if (a < nn) t = fma(Lan[i + (long long)a * nj], x[a], t);
        bc[rows[i]] -= t;
    }
}

__global__ void __launch_bounds__(256) thin_trsm_bwd_kernel(int nn, int na, int nj, const double *__restrict__ blk, const int *__restrict__ rows,
                                                            int r0, double *__restrict__ B, long long ldb, long long nrhs) {
    __shared__ double Lnn[THIN_NN * THIN_NN];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid < nn * nn) Lnn[(tid % nn) + (tid / nn) * THIN_NN] = blk[(tid % nn) + (long long)(tid / nn) * nj];
    __syncthreads();
    const long long c = (long long)blockIdx.x * 8 + warp;
    if (c >= nrhs) return;
    double *bc = B + c * ldb;
    const double *Lan = blk + nn;
    double acc[THIN_NN];
#pragma unroll
    for (int a = 0; a < THIN_NN; ++a) acc[a] = 0.0;
    for (int i = lane; i < na; i += 32) {
        const double v = bc[rows[i]];
#pragma unroll
        for (int a = 0; a < THIN_NN; ++a)
            if (a < nn) acc[a] = fma(Lan[i + (long long)a * nj], v, acc[a]);
    }
#pragma unroll
    for (int a = 0; a < THIN_NN; ++a)
        if (a < nn)
            for (int o = 16; o > 0; o >>= 1) acc[a] += __shfl_down_sync(0xffffffffu, acc[a], o);
    if (lane == 0) {
        double x[THIN_NN];
        double *bn = bc + r0;
#pragma unroll
        for (int a = 0; a < THIN_NN; ++a) x[a] = (a < nn) ? bn[a] - acc[a] : 0.0;
#pragma unroll
        for (int a = THIN_NN - 1; a >= 0; --a)
            if (a < nn) {
                double t = x[a];
#pragma unroll
                for (int b = THIN_NN - 1; b >= 0; --b)
                    if (b > a && b < nn) t = fma(-Lnn[b + a * THIN_NN], x[b], t);
                x[a] = t / Lnn[a + a * THIN_NN];
                bn[a] = x[a];
            }
    }
}

int big_trsm_node(smcp_sym *s, const BigNode &q, const double *L, double *B, int64_t ldb, int64_t nrhs, int trans);
// A RUN of consecutive thin supernodes in ONE launch: a right-hand side never interacts with another one, so the warp that
// owns a column walks the whole run by itself (forward: in post-order, backward: reversed) -- no dependency between warps,
// no launch per supernode (rand_SDP: 75 launches of ~20 us per direction -> 3).  desc[i] = {nn, na, nj, r0} (int4),
// off[i] = {offset of the block in blkval, offset of the separator rows in rowidx}.
__global__ void __launch_bounds__(256) thin_trsm_run_kernel(const int4 *__restrict__ desc, const longlong2 *__restrict__ off, int i0, int i1, int trans,
                                                            const double *__restrict__ L, const int *__restrict__ rowidx, double *__restrict__ B,
                                                            long long ldb, long long nrhs) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long c = (long long)blockIdx.x * 8 + warp;
    if (c >= nrhs) return;
    double *bc = B + c * ldb;
    for (int q = 0; q < i1 - i0; ++q) {
        const int i = trans ? i1 - 1 - q : i0 + q;
        const int4 d = desc[i];
        const int nn = d.x, na = d.y, nj = d.z, r0 = d.w;
        const double *blk = L + off[i].x;
        const double *Lan = blk + nn;
        const int *rows = rowidx + off[i].y;
        double x[THIN_NN];
        if (!trans) {
            // every lane solves the nn x nn system of its column (same arithmetic), lane 0 stores it
#pragma unroll
            for (int a = 0; a < THIN_NN; ++a) x[a] = (a < nn) ? bc[r0 + a] : 0.0;
            __syncwarp();
#pragma unroll
            for (int a = 0; a < THIN_NN; ++a)
                if (a < nn) {
                    double t = x[a];
#pragma unroll
                    for (int b = 0; b < THIN_NN; ++b)
                        if (b < a) t = fma(-__ldg(blk + a + (long long)b * nj), x[b], t);
                    x[a] = t / __ldg(blk + a + (long long)a * nj);
                    if (lane == 0) bc[r0 + a] = x[a];
                }
            for (int r = lane; r < na; r += 32) {
                double t = 0.0;
#pragma unroll
                for (int a = 0; a < THIN_NN; ++a)
                    if (a < nn) t = fma(Lan[r + (long long)a * nj], x[a], t);
                bc[rows[r]] -= t;
            }
        } else {
            double acc[THIN_NN];
#pragma unroll
            for (int a = 0; a < THIN_NN; ++a) acc[a] = 0.0;
            for (int r = lane; r < na; r += 32) {
                const double v = bc[rows[r]];
#pragma unroll
                for (int a = 0; a < THIN_NN; ++a)
                    if (a < nn) acc[a] = fma(Lan[r + (long long)a * nj], v, acc[a]);
            }
#pragma unroll
            for (int a = 0; a < THIN_NN; ++a)
                if (a < nn)
                    for (int o = 16; o > 0; o >>= 1) acc[a] += __shfl_down_sync(0xffffffffu, acc[a], o);
            if (lane == 0) {
#pragma unroll
                for (int a = 0; a < THIN_NN; ++a) x[a] = (a < nn) ? bc[r0 + a] - acc[a] : 0.0;
#pragma unroll
                for (int a = THIN_NN - 1; a >= 0; --a)
                    if (a < nn) {
                        double t = x[a];
#pragma unroll
                        for (int b = THIN_NN - 1; b >= 0; --b)
                            if (b > a && b < nn) t = fma(-__ldg(blk + b + (long long)a * nj), x[b], t);
                        x[a] = t / __ldg(blk + a + (long long)a * nj);
                        bc[r0 + a] = x[a];
                    }
            }
        }
        // the next supernode of the run reads what this one wrote (other lanes' rows)
        __syncwarp();
    }
}

// the top set against many right-hand sides: runs of thin supernodes through thin_trsm_run_kernel, the others one by one
int big_trsm_all(smcp_sym *s, const double *L, double *B, int64_t ldb, int64_t nrhs, int trans) {
    smcp_ctx *ctx = s->ctx;
    const int nb = (int)s->big.size();
    if (!s->thin_desc) {
        std::vector<int4> d(nb);
        std::vector<longlong2> o(nb);
        for (int i = 0; i < nb; ++i) {
            const BigNode &q = s->big[i];
            d[i] = make_int4(q.nn, q.na, q.nj, q.r0);
            o[i] = make_longlong2(q.boff, q.rowoff + q.nn);
        }
        CUDA_TRY(cudaMalloc(&s->thin_desc, (size_t)nb * sizeof(int4)));
        CUDA_TRY(cudaMalloc(&s->thin_off, (size_t)nb * sizeof(longlong2)));
        CUDA_TRY(cudaMemcpy(s->thin_desc, d.data(), (size_t)nb * sizeof(int4), cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMemcpy(s->thin_off, o.data(), (size_t)nb * sizeof(longlong2), cudaMemcpyHostToDevice));
        s->allocs.push_back(s->thin_desc);
        s->allocs.push_back(s->thin_off);
    }
    auto thin = [&](int i) { return s->big[i].nn <= THIN_NN && s->big[i].na >= 1; };
    // maximal runs [a, b) of thin supernodes, in sweep order
    std::vector<std::pair<int, int>> segs;       // (begin, end); begin == end - 1 and not thin: a single generic node
    for (int i = 0; i < nb;) {
        int j = i + 1;
        if (thin(i)) while (j < nb && thin(j)) ++j;
        segs.push_back({i, j});
        i = j;
    }
    if (trans) std::reverse(segs.begin(), segs.end());
    for (auto &sg : segs) {
        if (thin(sg.first)) {
            LaunchScope ls_(ctx, "thin_trsm");
            thin_trsm_run_kernel<<<(unsigned)((nrhs + 7) / 8), 256, 0, ctx->stream>>>((const int4 *)s->thin_desc, (const longlong2 *)s->thin_off, sg.first,
                                                                                      sg.second, trans, L, s->d.rowidx, B, ldb, nrhs);
            CUDA_TRY(cudaGetLastError());
        } else if (big_trsm_node(s, s->big[sg.first], L, B, ldb, nrhs, trans)) return -1;
    }
    return 0;
}

int big_trsm_node(smcp_sym *s, const BigNode &q, const double *L, double *B, int64_t ldb, int64_t nrhs, int trans) {
    smcp_ctx *ctx = s->ctx;
    const int nn = q.nn, na = q.na, nj = q.nj;
    const double *blk = L + q.boff;
    const int r0 = q.r0;                                  // first row of the supernode (its columns are contiguous)
    const int *rows = s->d.rowidx + q.rowoff + nn;        // the separator rows
    if (nn <= THIN_NN && na >= 1) {
        LaunchScope ls_(ctx, "thin_trsm");
        if (!trans) thin_trsm_fwd_kernel<<<(unsigned)((nrhs + 7) / 8), 256, 0, ctx->stream>>>(nn, na, nj, blk, rows, r0, B, ldb, nrhs);
        else thin_trsm_bwd_kernel<<<(unsigned)((nrhs + 7) / 8), 256, 0, ctx->stream>>>(nn, na, nj, blk, rows, r0, B, ldb, nrhs);
        CUDA_TRY(cudaGetLastError());
        return 0;
    }
    if (na && grow((void **)&s->big_cat, &s->big_cat_cap, (size_t)na * nrhs * sizeof(double))) return -1;
    double *T = s->big_cat;
    if (!trans) {
        if (d_trsm_left_lower(ctx, false, blk, nj, nn, B + r0, ldb, nrhs)) return -1;
        if (na) {
            // T(i, c) = sum_k L_an(i, k) B_nu(k, c)
            if (launch_gemm(ctx, false, true, blk + nn, nj, B + r0, ldb, T, na, na, nrhs, nn, 1.0, 0, 0, 0, "front_gemm_dmma")) return -1;
            ELEM(big_rows_sub_kernel, (long long)na * nrhs, B, ldb, rows, na, nrhs, T);
        }
    } else {
        if (na) {
            ELEM(big_rows_gather_kernel, (long long)na * nrhs, B, ldb, rows, na, nrhs, T);
            // B_nu(i, c) -= sum_k L_an(k, i) B_alpha(k, c)
            if (launch_gemm(ctx, true, true, blk + nn, nj, T, na, B + r0, ldb, nn, nrhs, na, -1.0, 1, 0, 0, "front_gemm_dmma")) return -1;
        }
        if (d_trsm_left_lower(ctx, true, blk, nj, nn, B + r0, ldb, nrhs)) return -1;
    }
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// ---- Hessian factor: Lt block and Y_aa ----------------------------------------------------------
int big_hess_prep(smcp_sym *s, const BigNode &q, const double *L0, const double *Y0, double *Lt_out, double *Yaa_out) {
    smcp_ctx *ctx = s->ctx;
    const int nn = q.nn, na = q.na, nj = q.nj;
    const double *Lb = L0 + q.boff;
    double *Ob = Lt_out + q.boff;
    ELEM(big_store_cols_kernel, (long long)nj * nn, Lb, Ob, nn, nj);
    if (na) {
        double *T = WS(0);
        ELEM(big_gather_aa_kernel, (long long)na * na, s->d.aaidx + q.uoff, Y0, Yaa_out + q.uoff, (long long)na * na);
        big_transpose(s, Lb + nn, nj, na, nn, T, nn);
        if (d_trsm_left_lower(ctx, true, Ob, nj, nn, T, nn, na)) return -1;                          // (L_an L_nn^-1)^T
        big_transpose(s, T, nn, nn, na, Ob + nn, nj);
    }
    CUDA_TRY(cudaGetLastError());
    return 0;
}

int big_hess_prep_inv(smcp_sym *s, const BigNode &q, const double *Yaa_all, double *Raa_all) {
    smcp_ctx *ctx = s->ctx;
    const int na = q.na;
    if (!na) return 0;
    ELEM(big_copy_mat_kernel, (long long)na * na, Yaa_all + q.uoff, na, Raa_all + q.uoff, na, na, na, 0);
    if (front_potrf(ctx, Raa_all + q.uoff, na, na, na, BIG_INFO)) return -1;
    big_flag_kernel<<<1, 1, 0, ctx->stream>>>(BIG_INFO, s->fail);
    // strictly upper part <- 0 (the factorisation leaves Y's entries there; the half factors use R as a dense block)
    ELEM(big_copy_mat_kernel, (long long)na * na, Raa_all + q.uoff, na, Raa_all + q.uoff, na, na, na, 1);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// ---------------------------------------------------------------------------------------
// Batched forward Hessian over the top set (Schur assembly with dense constraints: hundreds of
// matrices at ONE scaling point).  L and Y are shared by the batch, so every triangular solve
// runs on the concatenated right-hand sides (nn x nn*B) and every product is a strided batched
// DMMA GEMM with a shared operand; the elementwise steps carry the matrix index in blockIdx.y.
// ---------------------------------------------------------------------------------------
__global__ void big_front_full_b_kernel(BigArgs r, long long nupd, const double *__restrict__ X, long long nblk, long long boff,
                                        double *__restrict__ F, long long sF) {
    const int nj = r.nj, nn = r.nn;
    const long long b = blockIdx.y;
    r.ub += b * nupd;
    const double *blk = X + b * nblk + boff;
    double *Fb = F + b * sF;
    BIG_LOOP((long long)nj * nj) {
        const int i = (int)(idx % nj), j = (int)(idx / nj);
        const int hi = max(i, j), lo = min(i, j);
        double v = (lo < nn) ? blk[hi + (long long)lo * nj] : 0.0;
        Fb[idx] = v + big_children(r, i, j, false);
    }
}

__global__ void big_copy_b_kernel(const double *__restrict__ S, long long lds, long long sS, double *__restrict__ U, long long ldu, long long sU,
                                  int rows, int cols) {
    const long long b = blockIdx.y;
    S += b * sS;
    U += b * sU;
    BIG_LOOP((long long)rows * cols) {
        const int i = (int)(idx % rows), j = (int)(idx / rows);
        U[i + (long long)j * ldu] = S[i + (long long)j * lds];
    }
}

__global__ void big_transpose_b_kernel(const double *__restrict__ A, long long lda, long long sA, int rows, int cols,
                                       double *__restrict__ Bt, long long ldb, long long sB) {
    __shared__ double tile[32][33];
    A += (long long)blockIdx.z * sA;
    Bt += (long long)blockIdx.z * sB;
    const int bx = blockIdx.x * 32, by = blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int i = bx + threadIdx.x, j = by + r;
        tile[r][threadIdx.x] = (i < rows && j < cols) ? A[i + (long long)j * lda] : 0.0;
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int i = by + threadIdx.x, j = bx + r;
        if (i < cols && j < rows) Bt[i + (long long)j * ldb] = tile[threadIdx.x][r];
    }
}

__global__ void big_sym_store_b_kernel(const double *__restrict__ T, long long ldt, long long sT, double *__restrict__ blk, long long ldb, long long sB,
                                       int n, double alpha, double beta) {
    const long long b = blockIdx.y;
    T += b * sT;
    blk += b * sB;
    BIG_LOOP((long long)n * n) {
        const int i = (int)(idx % n), j = (int)(idx / n);
        double *d = blk + i + (long long)j * ldb;
        if (i >= j) {
            const double t = 0.5 * (T[i + (long long)j * ldt] + T[j + (long long)i * ldt]);
            *d = (alpha != 0.0 ? alpha * *d : 0.0) + beta * t;
        } else *d = 0.0;
    }
}

__global__ void big_gather_aa_b_kernel(const int *__restrict__ aaidx, const double *__restrict__ X, long long nblk, double *__restrict__ dst,
                                       long long sD, long long total) {
    const long long b = blockIdx.y;
    const double *Xb = X + b * nblk;
    double *d = dst + b * sD;
    BIG_LOOP(total) d[idx] = Xb[aaidx[idx]];
}

static dim3 egrid_b(smcp_sym *s, long long total, int64_t nb) {
    long long g = (total + 255) / 256;
    g = std::max<long long>(1, std::min<long long>(g, (long long)s->ctx->num_sms * 4));
    return dim3((unsigned)g, (unsigned)nb);
}
#define ELEMB(name, total, nb, ...)                                                  \
    do {                                                                             \
        LaunchScope ls_(ctx, "front_elem_batch");                                    \
        name<<<egrid_b(s, (total), (nb)), 256, 0, ctx->stream>>>(__VA_ARGS__);       \
    } while (0)

static int big_transpose_b(smcp_sym *s, const double *A, int64_t lda, int64_t sA, int rows, int cols, double *Bt, int64_t ldb, int64_t sB, int64_t nb) {
    if (rows <= 0 || cols <= 0) return 0;
    smcp_ctx *ctx = s->ctx;
    for (int64_t z0 = 0; z0 < nb; z0 += 32768) {
        const int64_t nz = std::min<int64_t>(32768, nb - z0);
        dim3 grid((rows + 31) / 32, (cols + 31) / 32, (unsigned)nz), block(32, 8);
        LaunchScope ls(ctx, "front_elem_batch");
        big_transpose_b_kernel<<<grid, block, 0, ctx->stream>>>(A + z0 * sA, lda, sA, rows, cols, Bt + z0 * sB, ldb, sB);
    }
    return 0;
}

static int GB(smcp_sym *s, bool ta, bool tb, const double *A, int64_t lda, int64_t sA, const double *B, int64_t ldb, int64_t sB,
              double *C, int64_t ldc, int64_t sC, int64_t M, int64_t N, int64_t K, double alpha, int acc, int64_t nb) {
    return launch_gemm_batched(s->ctx, ta, tb, A, lda, sA, B, ldb, sB, C, ldc, sC, M, N, K, alpha, acc, nb, "front_gemm_dmma_batch");
}

// the elementwise kernels take the matrix index from blockIdx.y (<= 65535)
static const int64_t BIG_BATCH_MAX = 32768;

static int big_hess_up_batched(smcp_sym *s, const BigNode &q, const double *Lt, const double *Yaa_all, double *X, int64_t nb,
                               double *W, size_t sW) {
    smcp_ctx *ctx = s->ctx;
    const int nn = q.nn, na = q.na, nj = q.nj;
    const long long nblk = s->d.nblk, nupd = s->d.nupd;
    const double *Lb = Lt + q.boff, *Ltan = Lb + nn, *Yaa = Yaa_all + q.uoff;
    // per matrix: F (nj^2) | T1 (nn * max(nn, na)) | T2 (nn^2), stride sW
    double *F = W, *T1 = W + (size_t)nj * nj, *T2 = T1 + (size_t)nn * std::max(nn, na);
    double *Fan = F + nn, *Faa = F + nn + (size_t)nn * nj, *Fna = F + (size_t)nn * nj;
    ELEMB(big_front_full_b_kernel, (long long)nj * nj, nb, big_args(s, q, 0), nupd, X, nblk, q.boff, F, (long long)sW);
    if (na) {
        if (GB(s, false, true, Ltan, nj, 0, F, nj, sW, Fan, nj, sW, na, nn, nn, -1.0, 1, nb)) return -1;       // K_an = F_an - Lt F_nn
        if (GB(s, false, true, Ltan, nj, 0, Fna, nj, sW, Faa, nj, sW, na, na, nn, -1.0, 1, nb)) return -1;     // U' = F_aa - Lt F_an(old)^T
        if (GB(s, false, false, Fan, nj, sW, Ltan, nj, 0, Faa, nj, sW, na, na, nn, -1.0, 1, nb)) return -1;    //      - K_an Lt^T
        ELEMB(big_copy_b_kernel, (long long)na * na, nb, Faa, nj, (long long)sW, s->upd + q.uoff, na, nupd, na, na);
    }
    // M_nn = D^{-1} F_nn D^{-1} on the concatenated nn x (nn * nb) right-hand sides: compact copies first
    // (T2 blocks are contiguous only when sW == nn*nn, so the concatenation lives in its own buffer)
    double *C1 = s->big_cat, *C2 = s->big_cat + (size_t)nn * std::max(nn, na) * nb;
    ELEMB(big_copy_b_kernel, (long long)nn * nn, nb, F, nj, (long long)sW, C2, nn, (long long)nn * nn, nn, nn);
    if (d_trsm_left_lower(ctx, false, Lb, nj, nn, C2, nn, (int64_t)nn * nb)) return -1;          // L^-1 F
    big_transpose_b(s, C2, nn, (int64_t)nn * nn, nn, nn, C1, nn, (int64_t)nn * nn, nb);
    if (d_trsm_left_lower(ctx, false, Lb, nj, nn, C1, nn, (int64_t)nn * nb)) return -1;          // L^-1 F L^-T
    if (d_trsm_left_lower(ctx, true, Lb, nj, nn, C1, nn, (int64_t)nn * nb)) return -1;           // L^-T (.)
    big_transpose_b(s, C1, nn, (int64_t)nn * nn, nn, nn, C2, nn, (int64_t)nn * nn, nb);
    if (d_trsm_left_lower(ctx, true, Lb, nj, nn, C2, nn, (int64_t)nn * nb)) return -1;           // D^-1 F D^-1
    if (na) {
        // M_an = Y_aa K_an D^{-1}: W = D^{-1} K_an^T (nn x na per matrix, concatenated), M_an = Y_aa W^T
        big_transpose_b(s, Fan, nj, (int64_t)sW, na, nn, C1, nn, (int64_t)nn * na, nb);
        if (d_trsm_left_lower(ctx, false, Lb, nj, nn, C1, nn, (int64_t)na * nb)) return -1;
        if (d_trsm_left_lower(ctx, true, Lb, nj, nn, C1, nn, (int64_t)na * nb)) return -1;
        if (GB(s, false, false, Yaa, na, 0, C1, nn, (int64_t)nn * na, X + q.boff + nn, nj, nblk, na, nn, na, 1.0, 0, nb)) return -1;
    }
    ELEMB(big_sym_store_b_kernel, (long long)nn * nn, nb, C2, nn, (long long)nn * nn, X + q.boff, nj, nblk, nn, 0.0, 1.0);
    (void)T1; (void)T2;
    CUDA_TRY(cudaGetLastError());
    return 0;
}

static int big_hess_down_batched(smcp_sym *s, const BigNode &q, const double *Lt, double *X, int64_t nb, double *W, size_t sW) {
    smcp_ctx *ctx = s->ctx;
    const int nn = q.nn, na = q.na, nj = q.nj;
    if (!na) return 0;
    const long long nblk = s->d.nblk;
    const double *Ltan = Lt + q.boff + nn;
    // per matrix (stride sW): Zaa (na^2) | Mold (na*nn) | S (nn^2)  -- all within 3 nj^2
    double *Zaa = W, *Mold = W + (size_t)na * na, *S = Mold + (size_t)na * nn;
    double *blk = X + q.boff;
    ELEMB(big_gather_aa_b_kernel, (long long)na * na, nb, s->d.aaidx + q.uoff, X, nblk, Zaa, (long long)sW, (long long)na * na);
    ELEMB(big_copy_b_kernel, (long long)na * nn, nb, blk + nn, nj, nblk, Mold, na, (long long)sW, na, nn);
    if (GB(s, false, true, Zaa, na, sW, Ltan, nj, 0, blk + nn, nj, nblk, na, nn, na, -1.0, 1, nb)) return -1;        // Z_an = M_an - Z_aa Lt
    if (GB(s, true, true, Ltan, nj, 0, Mold, na, sW, S, nn, sW, nn, nn, na, 1.0, 0, nb)) return -1;                  // S = Lt^T M_an(old)
    if (GB(s, true, true, blk + nn, nj, nblk, Ltan, nj, 0, S, nn, sW, nn, nn, na, 1.0, 1, nb)) return -1;            //   + Z_an^T Lt
    ELEMB(big_sym_store_b_kernel, (long long)nn * nn, nb, S, nn, (long long)sW, blk, nj, nblk, nn, 1.0, -1.0);        // Z_nn = M_nn - sym(S)
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// top-set part of a batched forward Hessian: called between the two tree-kernel sweeps
int big_hess_fwd_batched(smcp_sym *s, const double *Lt, const double *Yaa_all, double *U, int64_t batch) {
    int max_nj = 1;
    for (const BigNode &q : s->big) max_nj = std::max(max_nj, q.nj);
    const size_t sW = (size_t)3 * max_nj * max_nj;
    int64_t chunk = (int64_t)std::max<size_t>(1, ((size_t)3 << 30) / (sW * sizeof(double)));
    chunk = std::min<int64_t>(std::min<int64_t>(chunk, batch), BIG_BATCH_MAX);
    if (grow((void **)&s->big_bws, &s->big_bws_cap, (size_t)chunk * sW * sizeof(double))) return -1;
    if (grow((void **)&s->big_cat, &s->big_cat_cap, (size_t)chunk * 2 * (size_t)max_nj * max_nj * sizeof(double))) return -1;
    for (int64_t b0 = 0; b0 < batch; b0 += chunk) {
        const int64_t nb = std::min(chunk, batch - b0);
        double *Ub = U + (size_t)b0 * s->d.nblk;
        // the children's update matrices of matrix b0 + b start at upd + (b0 + b) * nupd
        double *upd_saved = s->upd;
        s->upd = upd_saved + (size_t)b0 * s->d.nupd;
        int rc = 0;
        for (const BigNode &q : s->big)
            if ((rc = big_hess_up_batched(s, q, Lt, Yaa_all, Ub, nb, s->big_bws, sW))) break;
        if (!rc)
            for (auto it = s->big.rbegin(); it != s->big.rend(); ++it)
                if ((rc = big_hess_down_batched(s, *it, Lt, Ub, nb, s->big_bws, sW))) break;
        s->upd = upd_saved;
        if (rc) return rc;
    }
    return 0;
}
