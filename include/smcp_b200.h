/*
 * smcp_b200.h — C ABI of the B200-native Newton-system hot path of SMCP's chordal
 * interior-point solvers (kktsolver='chol').
 *
 * The reference (cvxopt/smcp) has no FFI registry: the boundary this library replaces is
 *   (1) the chompack operator API imported at src/python/solvers.py:82-97 and 1364-1379,
 *   (2) cvxopt.lapack.potrf/potrs, cvxopt.base.gemv on the dense Schur complement H and
 *       the sparse constraint matrix Av (src/python/solvers.py:486, 501, 526, 374, 382),
 *   (3) the per-iteration members of the C extension smcp.misc (src/C/misc.c:1057-1102):
 *       Av_to_spmatrix (475-521), scal_diag (542-557), SCMcolumn2 (620-663).
 * Each entry point below names the reference call it stands in for.  Plain pointers and
 * sizes only; indices are 64-bit signed like CVXOPT's int_t (src/C/cvxopt.h:46); all
 * floating-point data is FP64.  Handles are opaque.  Every function returns 0 on success,
 * a positive LAPACK-style `info` where documented, and a negative value on a CUDA / usage
 * error (text via smcp_last_error()).  No CPU fallback exists: without a CUDA device
 * smcp_ctx_create fails.
 *
 * Threading: one context per process / GPU, calls issued from one host thread; work is
 * enqueued on the context's stream and the call synchronises only when a value returns to
 * the host (info flags, dot products, vectors).
 */
#ifndef SMCP_B200_H
#define SMCP_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct smcp_ctx smcp_ctx;    /* device, stream, scratch                           */
typedef struct smcp_sym smcp_sym;    /* clique tree + storage layout (chompack.symbolic)  */
typedef struct smcp_hess smcp_hess;  /* scaling point (L, Y) prepared for hessian()       */
typedef struct smcp_op smcp_op;      /* constraint operator Av and Schur complement H     */

/* ---- context ------------------------------------------------------------------------ */
int smcp_ctx_create(int device, smcp_ctx **out);
int smcp_ctx_destroy(smcp_ctx *ctx);
int smcp_ctx_sync(smcp_ctx *ctx);
const char *smcp_last_error(void);
int smcp_version(void);
/* number of kernels this library has launched on the context since creation */
int64_t smcp_ctx_launch_count(smcp_ctx *ctx);
/* CUDA-event timer on the context's stream: start, then stop returns milliseconds */
int smcp_timer_start(smcp_ctx *ctx);
int smcp_timer_stop(smcp_ctx *ctx, double *ms_out);
/* named per-kernel-family accumulators (ms and launches) for bench.py's roofline leg */
int smcp_prof_enable(smcp_ctx *ctx, int on);
int smcp_prof_get(smcp_ctx *ctx, const char *name, double *ms_out, int64_t *launches_out);
/* accumulated work of a family: matrices processed (chordal kernels), algorithmic flops (GEMM) */
int smcp_prof_get_work(smcp_ctx *ctx, const char *name, double *work_out);
/* comma-separated names of the families that have accumulated time since the last reset */
int smcp_prof_list(smcp_ctx *ctx, char *buf, int64_t cap);
int smcp_prof_reset(smcp_ctx *ctx);
/* device time of whole API regions ("kkt_assemble", "kkt_factor", "kkt_solve", "kkt_allgather"): one
 * event pair per call on the context's stream, no synchronisation until read; ms and calls since reset */
int smcp_region_get(smcp_ctx *ctx, const char *name, double *ms_out, int64_t *calls_out);
int smcp_region_reset(smcp_ctx *ctx);
/* comma-separated names of all regions seen so far: the kkt_* ones and one per chordal operation
 * ("op_cholesky", "op_completion", "op_hessian", "op_hessian_inv", "op_hessian_batch", ...) */
int smcp_region_list(smcp_ctx *ctx, char *buf, int64_t cap);
/* write (flush) a buffer larger than L2 */
int smcp_flush_l2(smcp_ctx *ctx);

/* ---- symbolic object: chompack.symbolic(Vp) (solvers.py:314, 1555) --------------------
 * All arrays are host int64.  The layout is the one produced by
 * smcp_b200/symbolic.py:Symbolic (supernodes in post-order, contiguous columns). */
typedef struct smcp_sym_desc {
    int64_t n, nsn, nvp, nblk, nupd;
    const int64_t *snptr;    /* nsn+1: first column of each supernode                      */
    const int64_t *snpar;    /* nsn  : parent supernode or -1                              */
    const int64_t *rowptr;   /* nsn+1                                                       */
    const int64_t *rowidx;   /* row indices (own columns first, then separator)            */
    const int64_t *blkptr;   /* nsn+1: offset of each (nn+na) x nn block in blkval          */
    const int64_t *updptr;   /* nsn+1: offset of each na x na update matrix                 */
    const int64_t *chptr;    /* nsn+1                                                       */
    const int64_t *chidx;    /* children                                                    */
    const int64_t *relptr;   /* nsn+1                                                       */
    const int64_t *relidx;   /* positions of the separator inside the parent's row list    */
    const int64_t *aaidx;    /* nupd : blkval offsets of the alpha x alpha entries          */
    const int64_t *vec2blk;  /* nvp  : blkval offset of the q-th non-zero of Vp (CCS order) */
    const int64_t *diagblk;  /* n    : blkval offset of each diagonal entry                 */
    const double  *wdot;     /* nblk : trace weights (2 strict lower, 1 diagonal, 0 pad)    */
    /* task partition for the persistent dependency-driven kernels (bottom-up order)       */
    int64_t ntask;
    const int64_t *task_ptr; /* ntask+1 */
    const int64_t *task_sn;  /* nsn     */
    const int64_t *dep_ptr;  /* ntask+1 */
    const int64_t *dep_idx;
} smcp_sym_desc;

int smcp_sym_create(smcp_ctx *ctx, const smcp_sym_desc *desc, smcp_sym **out);
int smcp_sym_destroy(smcp_sym *sym);
/* size the per-pattern workspaces for batches of up to `batch` matrices now (otherwise they grow on
 * first use, e.g. at the first batched line search of a solve) */
int smcp_sym_reserve(smcp_sym *sym, int64_t batch);

/* ---- chordal matrices: chompack.cspmatrix -----------------------------------------------
 * A chordal matrix is `nblk` doubles in device memory (the `blkval` buffer of a cspmatrix).
 * `count` matrices are allocated contiguously (stride nblk). */
int smcp_csp_alloc(smcp_sym *sym, int64_t count, double **dev_out);     /* zero-filled     */
int smcp_csp_free(smcp_sym *sym, double *dev);
int smcp_csp_copy(smcp_sym *sym, double *dst, const double *src, int64_t count);
/* cspmatrix(symb) + spmatrix: scatter |Vp| host values (lower CCS order of Vp)           */
int smcp_csp_from_vec(smcp_sym *sym, double *dst, const double *host_vec);
/* X.spmatrix(reordered=False, symmetric=False).V                                          */
int smcp_csp_to_vec(smcp_sym *sym, const double *src, double *host_vec);
int smcp_csp_get(smcp_sym *sym, const double *src, double *host_blk);    /* raw blkval      */
int smcp_csp_set(smcp_sym *sym, double *dst, const double *host_blk);
/* y += a*x (cspmatrix +,-,+=), x *= a (blas.scal(a, X.blkval))                              */
int smcp_csp_axpy(smcp_sym *sym, double a, const double *x, double *y);
int smcp_csp_scal(smcp_sym *sym, double a, double *x);
/* chompack.dot(X, Y) */
int smcp_csp_dot(smcp_sym *sym, const double *x, const double *y, double *out);
/* sum(log(X.diag())) (solvers.py:395, 925) */
int smcp_csp_sumlogdiag(smcp_sym *sym, const double *x, double *out);

/* chompack.cholesky / completion: in place on `batch` matrices (stride nblk);
 * info_host[b] = 0 on success, 1 if matrix b is not positive definite / not completable
 * (the reference signals this with ArithmeticError, e.g. solvers.py:640-645).            */
int smcp_csp_cholesky(smcp_sym *sym, double *x, int64_t batch, int32_t *info_host);
int smcp_csp_completion(smcp_sym *sym, double *x, int64_t batch, int32_t *info_host);
/* chompack.projected_inverse / llt (solvers.py:891, 904) */
int smcp_csp_projected_inverse(smcp_sym *sym, double *x, int64_t batch);
int smcp_csp_llt(smcp_sym *sym, double *x, int64_t batch);
/* step-length probes (line searches, solvers.py:615-647, 2187-2207): for each gamma_k,
 * test X + gamma_k*dX with cholesky (kind=0) or completion (kind=1) as ONE device batch;
 * info_host[k] as above, sumlogdiag_host[k] = sum(log(diag(L_k))) when it succeeded.      */
int smcp_csp_probe(smcp_sym *sym, int kind, const double *x, const double *dx,
                   const double *gammas_host, int64_t count, int32_t *info_host,
                   double *sumlogdiag_host);
/* chompack.trsm(L, B[, trans='T']): B (n x nrhs, column-major, rows in Vp order, DEVICE) */
int smcp_csp_trsm(smcp_sym *sym, const double *L, double *B_dev, int64_t ldb, int64_t nrhs, int trans);

/* ---- randomized rounding (an extension: the reference has none) ------------------------------
 * Gaussian samples of the max-det completion: with L from smcp_csp_completion (P_V((L L^T)^-1) = X),
 * B[:, c] = L^-T g_{col0+c}, c = 0..k-1, g_j the standard normal vector of sample j under `seed`
 * (Philox4x64-10, Box-Muller; entry i of sample j depends only on (seed, j, i)).
 * B: n x k column-major on the device, rows in the internal order of sym. */
int smcp_csp_sample(smcp_sym *sym, const double *L, uint64_t seed, int64_t col0,
                    double *B_dev, int64_t ldb, int64_t k);
/* ±1 rounding: trials t = 0..trials-1 of s_t = sign(L^-T g_t); values_host[t] = sum over the nc
 * lower-triangular objective entries (internal coordinates, host arrays) of c s_r s_c (x2 off the diagonal);
 * x_host = s of the smallest value (lowest t on ties), *best_out = that t.  `chunk` trials per pass
 * (0: as many as fit in 1 GiB of n x chunk doubles), rounded up to whole solve blocks: the trials are solved in
 * blocks of equal width, at most 256 columns, so every output is independent of chunk.  The workspace is
 * allocated once per call; nothing of size n x trials leaves the device. */
int smcp_round_pm1(smcp_sym *sym, const double *L, uint64_t seed, int64_t trials, int64_t chunk,
                   int64_t nc, const int64_t *crow, const int64_t *ccol, const double *cval,
                   double *values_host, int8_t *x_host, int64_t *best_out);
/* One-flip local search of ±1 vectors against f(x) = sum_ij C_ij x_i x_j, C the symmetric matrix of the nc
 * objective entries (host arrays; entries off the diagonal count for both triangles, duplicates are summed in input
 * order).  With s_i = sum_{j != i} C_ij x_j, a_i = sum_{j != i} |C_ij| (both in increasing j) and the gain
 * g_i = x_i s_i, each step flips the vertex of largest g_i among those with g_i > tol a_i (lowest index on ties),
 * which lowers f by 4 g_i; the search stops when none qualifies or after max_flips flips.  Values are evaluated as
 * smcp_round_pm1 evaluates its trials.  Needs n <= 2^20 (-2 beyond), max_flips >= 0 and a finite tol >= 0.
 * smcp_round_pm1_ls: smcp_round_pm1 with the search run on every trial; values0_host[t] is the value of trial t
 * before the search, flips_host[t] its number of flips, and values_host, x_host and *best_out refer to the searched
 * trials.  The search reuses the pass's sample buffer for s.
 * smcp_pm1_local_search: the search on k caller-given vectors x_host (k x n int8, row t = vector t, every entry ±1),
 * replaced by the searched ones; values_host[t] and flips_host[t] as above.  Its workspace follows the pass rule of
 * smcp_round_pm1 (n x pass doubles within 1 GiB). */
int smcp_round_pm1_ls(smcp_sym *sym, const double *L, uint64_t seed, int64_t trials, int64_t chunk,
                      int64_t nc, const int64_t *crow, const int64_t *ccol, const double *cval,
                      int64_t max_flips, double tol, double *values0_host,
                      double *values_host, int8_t *x_host, int64_t *best_out, int64_t *flips_host);
int smcp_pm1_local_search(smcp_ctx *ctx, int64_t n, int64_t k, int8_t *x_host,
                          int64_t nc, const int64_t *crow, const int64_t *ccol, const double *cval,
                          int64_t max_flips, double tol, double *values_host, int64_t *flips_host);
/* Tabu search of ±1 vectors against the same f, rows, s_i and g_i.  D_0 = 0; move u flips the admissible vertex i of
 * largest g_i (lowest index on ties) and sets D_{u+1} = D_u - 4 g_i (in double, in that form); D_best is the smallest D
 * so far, updated on a strict decrease only.  A vertex flipped by move u is tabu during moves u+1 .. u+tenure; every
 * vertex that is not tabu is admissible whatever its gain, a tabu vertex only when D_u - 4 g_i < D_best (aspiration).
 * Then s is updated along row i as in the one-flip search.  The search stops after tabu_iters moves, or when no vertex
 * is admissible (possible only for tenure >= n), and returns the vector of the earliest move count at which D reached
 * D_best (the start if D never drops below 0).  Values are evaluated as smcp_round_pm1 evaluates its trials.  Needs
 * n <= 2^19, 0 <= tenure <= 8192 and tabu_iters >= 0 (-2 otherwise).
 * smcp_round_pm1_tabu: smcp_round_pm1_ls, with the tabu search run on every trial after the one-flip search (which runs
 * only when max_flips > 0; flips_host is 0 otherwise); values0_host[t] is the value of the rounded trial t,
 * values1_host[t] its value before the tabu search, moves_host[t] its number of moves and best_iter_host[t] the move
 * count of the returned vector; values_host, x_host and *best_out refer to the trials after the tabu search.
 * smcp_pm1_tabu_search: the tabu search (tabu_iters = iters) on k caller-given vectors x_host (k x n int8, every entry
 * ±1), replaced by the searched ones; values_host, moves_host and best_iter_host as above.  Its workspace follows the
 * pass rule of smcp_round_pm1 (n x pass doubles within 1 GiB). */
int smcp_round_pm1_tabu(smcp_sym *sym, const double *L, uint64_t seed, int64_t trials, int64_t chunk,
                        int64_t nc, const int64_t *crow, const int64_t *ccol, const double *cval,
                        int64_t max_flips, double tol, double *values0_host,
                        double *values_host, int8_t *x_host, int64_t *best_out, int64_t *flips_host,
                        int64_t tabu_iters, int64_t tenure, double *values1_host, int64_t *moves_host,
                        int64_t *best_iter_host);
int smcp_pm1_tabu_search(smcp_ctx *ctx, int64_t n, int64_t k, int8_t *x_host,
                         int64_t nc, const int64_t *crow, const int64_t *ccol, const double *cval,
                         int64_t iters, int64_t tenure, double *values_host, int64_t *moves_host,
                         int64_t *best_iter_host);
/* Low-rank (Burer-Monteiro) solve of  min C . X  s.t.  X_ii = b_i (b_i > 0 finite), X >= 0  with X = V V^T, V n x r
 * (1 <= r <= 512), by the mixing method: colours of a greedy colouring of C's off-diagonal pattern (vertex i takes the
 * smallest colour none of its lower-index neighbours has) are swept in order, and every vertex i of a colour gets
 * v_i <- -sqrt(b_i) w_i / ||w_i||, w_i = sum_{j != i} C_ij v_j (unchanged when w_i = 0).  C is given by nc objective
 * entries as in smcp_pm1_local_search.  Row i of the start is the standard normal sample i of smcp_csp_sample's
 * generator (length r) scaled to norm sqrt(b_i).  f_k = sum_i C_ii b_i + <v_i, w_i> after k sweeps goes to f_host[k];
 * the run stops after the first sweep k with f_{k-1} - f_k <= tol max(1, |f_k|), or after max_sweeps sweeps
 * (*sweeps_out; f_host holds max_sweeps + 1 doubles, of which sweeps + 1 are written).  V_host receives V (n x r,
 * row-major), y_host y_i = (C_ii b_i + <v_i, w_i>) / b_i at the final V, *colors_out the number of colours.  Every
 * result is bitwise reproducible (lowrank.cu states the summation orders).  -2: r outside 1..512, b_i <= 0 or not
 * finite, max_sweeps < 0, a negative or non-finite tol, or an entry outside 0..n-1. */
int smcp_lowrank_solve(smcp_ctx *ctx, int64_t n, int64_t r, int64_t nc, const int64_t *crow, const int64_t *ccol,
                       const double *cval, const double *b, uint64_t seed, int64_t max_sweeps, double tol,
                       double *V_host, double *f_host, double *y_host, int64_t *sweeps_out, int64_t *colors_out);
/* ±1 rounding from a low-rank factor: smcp_round_pm1 with the samples V g_t, V the n x r factor V_host (row-major,
 * original coordinates, as smcp_lowrank_solve returns it) and g_t the length-r normal sample t under seed, computed in
 * blocks of one width as one DMMA product each, so every output is independent of chunk.  The objective entries are in
 * the coordinates of V.  The one-flip search runs on every trial when max_flips > 0 (tol, values0_host, flips_host as
 * in smcp_round_pm1_ls), the tabu search when tabu_iters > 0 (tenure, values1_host, moves_host, best_iter_host as in
 * smcp_round_pm1_tabu); values0_host and flips_host are needed when either search runs, the other search outputs
 * when the tabu search runs, and may be null otherwise.  The limits on n and tenure are those of the searches. */
int smcp_round_pm1_factor(smcp_ctx *ctx, int64_t n, int64_t r, const double *V_host, uint64_t seed, int64_t trials,
                          int64_t chunk, int64_t nc, const int64_t *crow, const int64_t *ccol, const double *cval,
                          int64_t max_flips, double tol, int64_t tabu_iters, int64_t tenure,
                          double *values0_host, double *values1_host, double *values_host, int8_t *x_host,
                          int64_t *best_out, int64_t *flips_host, int64_t *moves_host, int64_t *best_iter_host);

/* ---- barrier Hessian: chompack.hessian(L, Y, U, adj=None, inv=...) ---------------------- */
int smcp_hess_create(smcp_sym *sym, const double *L, const double *Y, smcp_hess **out);
int smcp_hess_destroy(smcp_hess *h);
/* U <- P(S^-1 U S^-1) (inv=0) or its inverse map (inv=1) on `batch` matrices (stride nblk) */
int smcp_hess_apply(smcp_hess *h, double *U, int64_t batch, int inv);
/* chompack.hessian(L, Y, U, adj=False/True, inv=...) (solvers.py:917, 978, 1121, 1126): the half factors
 * G (adj=0, inv=0), G^adj (1, 0), G^-1 (0, 1), G^-adj (1, 1) with hessian = G^adj o G; in place on a batch */
int smcp_hess_apply_half(smcp_hess *h, double *U_dev, int64_t batch, int inv, int adj);

/* ---- constraint operator and Schur complement (kkt_chol, solvers.py:477-541) ------------
 * Av: |Vp| x m CCS, rows in vector-space order, columns already permuted so that the last
 * `Ns` are the "sparse" constraints (solvers.py:246-268).                                  */
int smcp_op_create(smcp_sym *sym, int64_t m, int64_t Ns, const int64_t *colptr,
                   const int64_t *rowind, const double *values, smcp_op **out);
int smcp_op_destroy(smcp_op *op);
/* (row, col) of every stored entry of Av in the internal order of the symbolic object;
 * needed by the sparse-constraint technique (the Ip/Jp/Kl arguments of misc.SCMcolumn2,
 * src/C/misc.c:620-663) */
int smcp_op_set_entry_coords(smcp_op *op, const int64_t *rows_int, const int64_t *cols_int);
/* rows of the dense weighted constraint copy built at smcp_op_create for the "dense" constraints:
 * 0 without one (no dense constraint), |blkval| for the full copy, the number of distinct rows of blkval
 * any constraint touches for the support copy (chosen when they are at most a quarter of |blkval|;
 * SMCP_B200_AVW_SUPPORT=0 / =1 forces the full / the support copy) */
int smcp_op_dense_rows(smcp_op *op, int64_t *rows_out);
/* Amap: v = 2*Av^T*vec_half(X) (solvers.py:369-378); col >= 0 evaluates one entry only    */
int smcp_op_amap(smcp_op *op, const double *X, int64_t col, double *host_out);
/* Aadj: X = mat(Av*y) (solvers.py:380-384) */
int smcp_op_aadj(smcp_op *op, const double *host_y, double *X);
/* assemble the lower triangle of H (H_ij = A_i . Hess(A_j)); columns [j0, j1) only when
 * sharding across GPUs (pass 0, m for everything)                                          */
int smcp_kkt_assemble(smcp_op *op, smcp_hess *h, int64_t j0, int64_t j1);
/* multi-GPU: assemble the column blocks q = rank (mod nranks) of `block` columns as one batch */
int smcp_kkt_assemble_cyclic(smcp_op *op, smcp_hess *h, int64_t block, int rank, int nranks);
/* kktsolver='qr' (solvers.py:413-475, 1843-1904) in SYRK form: Z = [G(A_1) ... G(A_m)] with the half factor
 * G of the Hessian, H = Z^T Z in the trace inner product by one triangular DMMA product (then smcp_kkt_factor /
 * smcp_kkt_solve as usual); z_tmul: out[j] = <G(A_j), X>; z_mul: X = sum_j y[j] G(A_j).  Needs Ns = 0.
 * h = NULL takes G = identity: H is then the Gram matrix <A_i, A_j> of the constraints, whose Cholesky solve
 * gives the least-norm start of SDP.solve_phase1 (base.py:383-396: syrk + CHOLMOD in the reference). */
int smcp_kkt_assemble_syrk(smcp_op *op, smcp_hess *h);
int smcp_kkt_z_tmul(smcp_op *op, const double *X_dev, double *host_out);
int smcp_kkt_z_mul(smcp_op *op, const double *host_y, double *X_dev);
/* kktsolver='qr' in Householder form (the reference's geqrf / ormqr / trtrs): forms Zw as
 * smcp_kkt_assemble_syrk does, factors Zw = Q1 R on the device, keeps Q1 (nblk x m) in place of Zw
 * and L = R^T with diag(L) >= 0 as the lower triangle of H (L L^T = the SYRK-form H).  info_host = k > 0
 * at the first k with R_kk <= 1e-14 max R_ii (Z rank deficient).  Needs Ns = 0.  Afterwards
 * smcp_kkt_z_tmul / smcp_kkt_z_mul refuse until the next smcp_kkt_assemble_syrk.               */
int smcp_kkt_factor_qr(smcp_op *op, smcp_hess *h, int32_t *info_host);
/* Newton solve of the Householder form: with g = G_dev (= G(b_x), a chordal matrix) and r = host_r
 * (= kk b_y), y = H^-1 (r + Z^T g) into host_y and X_dev = Z y - g (the argument of G^adj) through Q1 and
 * L only; refuses without a successful smcp_kkt_factor_qr                                      */
int smcp_kkt_qr_solve(smcp_op *op, const double *G_dev, const double *host_r, double *host_y, double *X_dev);
/* lapack.potrf(H): info_host = 0 ok, k > 0 if the leading minor of order k is not PD        */
int smcp_kkt_factor(smcp_op *op, int32_t *info_host);
/* lapack.potrs(H, y) in place on a host m-vector */
int smcp_kkt_solve(smcp_op *op, double *host_y);
/* raw access to H (m x m column-major, device) for tests, gathers and multi-GPU exchange  */
int smcp_kkt_get_H(smcp_op *op, double *host_H);
int smcp_kkt_set_H(smcp_op *op, const double *host_H);
int smcp_kkt_H_devptr(smcp_op *op, double **dev_out);

/* ---- multi-GPU (one process per GPU): NCCL communicator owned by the library ------------ */
int smcp_comm_unique_id(char *id_out_128);
int smcp_comm_init(smcp_ctx *ctx, int rank, int nranks, const char *id_128);
int smcp_comm_destroy(smcp_ctx *ctx);
/* distributed lapack.potrf (solvers.py:501, 1931) on the block-cyclic column blocks of 128 columns
 * assembled by smcp_kkt_assemble_cyclic(block = 128): owners factor and ncclBroadcast their panels,
 * every rank updates its own column tiles; on return every rank holds the complete factor */
int smcp_kkt_factor_dist(smcp_op *op, int rank, int nranks, int32_t *info_host);
/* the same with an explicit distribution block (a multiple of 128 columns; the `block` given to
 * smcp_kkt_assemble_cyclic).  256 keeps 8 ranks busy at m = 10 000 while each trailing update still
 * runs with K = 256 */
int smcp_kkt_factor_block(smcp_op *op, int64_t block, int rank, int nranks, int32_t *info_host);
/* all-gather the block-cyclic column blocks of H assembled by each rank */
int smcp_kkt_allgather(smcp_op *op, int64_t block, int rank, int nranks);

/* ---- host-side symbolic analysis in native code (no CUDA; SURVEY.md 8(f) rank 1) ---------
 * Native twins of smcp_b200/symbolic.py with identical tie-breaking (bit-identical results).
 * Patterns are lower-triangular CCS, int64 indices. */
/* cvxopt.amd.order stand-in (solvers.py:192-198, 278-279): exact minimum degree, ties by index */
int smcp_host_min_degree(int64_t n, const int64_t *colptr, const int64_t *rowind, int64_t *perm);
/* chompack.maxcardsearch (solvers.py:301, 1542): reverse maximum-cardinality-search order */
int smcp_host_maxcardsearch(int64_t n, const int64_t *colptr, const int64_t *rowind, int64_t *order);
/* embedding step of chompack.symbolic (solvers.py:305-308) for a pattern already in elimination
 * order: call with frowind = NULL to get fcolptr (sizes), then again to fill frowind; parent
 * (elimination tree) may be NULL */
int smcp_host_embed(int64_t n, const int64_t *colptr, const int64_t *rowind, int64_t *fcolptr,
                    int64_t *frowind, int64_t *parent);
/* the alpha x alpha gather map of chompack.symbolic's clique tree (smcp_sym_desc.aaidx) from the
 * supernode arrays of smcp_sym_desc; nn = columns and nj = rows of every supernode */
int smcp_host_aaidx(int64_t nsn, const int64_t *snpar, const int64_t *nn, const int64_t *nj, const int64_t *relptr,
                    const int64_t *relidx, const int64_t *blkptr, const int64_t *updptr, int64_t *aaidx);
/* supernode partition (maximal supernodes, first-qualifying-child rule), post-ordered relabelling, row lists and
 * relative indices of a filled pattern in a perfect elimination ordering: chompack.symbolic (solvers.py:314, 1555).
 * Caller-allocated outputs: perm[n], snptr[n+1], snpar[n], rowptr[n+1], rowidx[n + nnz], relptr[n+1], relidx[nnz]. */
int smcp_host_supernodes(int64_t n, const int64_t *colptr, const int64_t *rowind, int64_t *nsn_out, int64_t *perm,
                         int64_t *snptr, int64_t *snpar, int64_t *rowptr, int64_t *rowidx, int64_t *relptr, int64_t *relidx);

/* ---- the dense LAPACK/BLAS calls of the path on host buffers (column-major) -----------------
 * Parity tests and micro-benchmarks of the kernels behind smcp_kkt_factor / smcp_kkt_solve and the
 * frontal matrices of large supernodes; `ms_out` (may be NULL) receives the device time.
 * smcp_dense_potrf: cvxopt.lapack.potrf(A) (solvers.py:501, 1931); ncols < m factors the leading
 *   ncols columns and leaves the Schur complement in the trailing block (a frontal matrix of
 *   chompack.cholesky).  info as dpotrf.
 * smcp_dense_trsm: B <- L^{-1} B (trans = 0) or L^{-T} B (trans = 1), L lower triangular: the two
 *   halves of cvxopt.lapack.potrs (solvers.py:526) and chompack.trsm on a dense supernode (491-492).
 * smcp_dense_gemm: C = [C +] alpha op(A) op(B)^T on the FP64 tensor cores; ta / tb = 1: the operand
 *   is stored K-major (A[k + i*lda]); tri = 1: lower triangle only (the contraction of
 *   solvers.py:486 and every frontal update).
 * smcp_dense_geqrf / smcp_dense_orgqr: lapack.geqrf / lapack.orgqr of an M x N matrix, M >= N
 *   (Householder vectors below the diagonal with a unit diagonal, LAPACK's beta and tau; orgqr
 *   overwrites them with the M x N Q1), by the blocked Householder QR of kktsolver='qr'. */
int smcp_dense_potrf(smcp_ctx *ctx, double *A_host, int64_t lda, int64_t m, int64_t ncols, int32_t *info_host, double *ms_out);
int smcp_dense_trsm(smcp_ctx *ctx, int trans, const double *L_host, int64_t ldl, int64_t n, double *B_host, int64_t ldb,
                    int64_t nrhs, double *ms_out);
int smcp_dense_gemm(smcp_ctx *ctx, int ta, int tb, const double *A_host, int64_t lda, const double *B_host, int64_t ldb,
                    double *C_host, int64_t ldc, int64_t M, int64_t N, int64_t K, double alpha, int accumulate, int tri,
                    double *ms_out);
int smcp_dense_geqrf(smcp_ctx *ctx, double *A_host, int64_t lda, int64_t M, int64_t N, double *tau_host, double *ms_out);
int smcp_dense_orgqr(smcp_ctx *ctx, double *A_host, int64_t lda, int64_t M, int64_t N, const double *tau_host, double *ms_out);

#ifdef __cplusplus
}
#endif
#endif /* SMCP_B200_H */
