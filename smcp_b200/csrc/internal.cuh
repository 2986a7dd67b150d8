// Internal declarations shared by the translation units of libsmcp_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include <vector>
#include <map>
#include "../../include/smcp_b200.h"

void smcp_set_error(const char *fmt, ...);

#define CUDA_TRY(expr)                                                                   \
    do {                                                                                 \
        cudaError_t _e = (expr);                                                         \
        if (_e != cudaSuccess) {                                                         \
            smcp_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr,                 \
                           cudaGetErrorString(_e));                                      \
            return -1;                                                                   \
        }                                                                                \
    } while (0)

struct ProfEntry {
    double ms = 0.0;
    int64_t launches = 0;
    double work = 0.0;      // matrices processed (chordal kernels) or algorithmic flops (GEMM)
};

// Device time of a whole API region (assembly, factorisation, solve of the Schur complement) without
// synchronising: a pair of events per call, resolved when the accumulator is read.
struct RegionAcc {
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> pending;
    double ms = 0.0;
    int64_t calls = 0;
};

// Scratch of one concurrent LANE (lanes_fork / lane_select / lanes_join, capi.cu): supernodes of the top set whose
// work is independent (completion, chol(Y_aa), the local phase of the inverse Hessian) are issued round-robin
// on a few streams; every helper launches on ctx->stream with ctx's scratch buffers, so selecting a lane swaps
// these members with the lane's own copies.
struct CtxLane {
    cudaStream_t stream = nullptr;
    cudaEvent_t done = nullptr;
    double *gemm_ws = nullptr;
    size_t gemm_ws_cap = 0;
    double *trs_dinv = nullptr;
    size_t trs_dinv_cap = 0;
    unsigned *gridbar = nullptr;
    unsigned gridbar_next = 0;
};

struct smcp_ctx {
    std::map<std::string, RegionAcc> regions;
    std::vector<cudaEvent_t> region_pool;
    int device = 0;
    int num_sms = 148;
    cudaStream_t stream = nullptr;
    cudaStream_t stream2 = nullptr;                 // look-ahead stream of the dense Cholesky (panels + broadcasts)
    std::vector<cudaEvent_t> potrf_ev;              // fork/join events of the look-ahead pipeline
    void *wave_buf = nullptr;                       // potrs_wave_kernel: published block solutions + flags
    size_t wave_cap = 0;
    unsigned wave_epoch = 0;
    int64_t wave_nb = -1;                           // block count the flag layout of wave_buf belongs to
    double *potrf_pt = nullptr;                     // K-major copies of the Cholesky panels (single-GPU look-ahead path)
    size_t potrf_pt_cap = 0;
    int potrf_grid_cap = 0;                         // > 0: potrf_tile uses at most this many CTAs (look-ahead panel next to a GEMM)
    const char *potrf_family = nullptr;             // profile family of the next d_potrf (default "potrf_dmma")
    int prof_mute = 0;                              // > 0: nested LaunchScopes do not time (an outer scope does)
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;       // user timer
    cudaEvent_t pev0 = nullptr, pev1 = nullptr;     // profiling events
    int64_t launches = 0;
    bool prof = false;
    std::map<std::string, ProfEntry> prof_acc;
    double *flush_buf = nullptr;
    size_t flush_bytes = 0;
    double *gemm_ws = nullptr;          // split-K partial results
    size_t gemm_ws_cap = 0;
    void *nccl_comm = nullptr;
    int comm_rank = 0, comm_nranks = 1;   // set by smcp_comm_init
    double *trs_dinv = nullptr;         // inverted diagonal blocks for the few-right-hand-side triangular solves (front.cu)
    size_t trs_dinv_cap = 0;
    unsigned *gridbar = nullptr;        // counters of the hand-rolled grid barrier (potrf_tile_kernel)
    unsigned gridbar_next = 0;
    std::vector<CtxLane> lanes;         // lanes[i - 1] = lane i >= 1 (lane 0 is `stream` itself)
    int lane_cur = 0;                   // lane whose members are currently swapped in
    int lanes_active = 0;               // > 1 between lanes_fork and lanes_join
    cudaEvent_t lane_fork_ev = nullptr;
    double *qr_ws = nullptr;            // blocked Householder QR (qr.cu): V | Y | W | partial sums
    size_t qr_ws_cap = 0;
    // pinned staging for small host<->device transfers
    void *pinned = nullptr;
    size_t pinned_bytes = 0;
};

// RAII helper: counts a launch and (when profiling) times the enclosed kernel(s).
struct LaunchScope {
    smcp_ctx *ctx;
    const char *name;
    int n;
    double work;
    bool active;
    int64_t launches0;       // ctx->launches after this scope's own n: nested launches are credited to it too
    LaunchScope(smcp_ctx *c, const char *nm, int nlaunch = 1, double work = 0.0);
    ~LaunchScope();
};

struct RegionScope {
    smcp_ctx *ctx;
    RegionAcc *acc;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    RegionScope(smcp_ctx *c, const char *name);
    ~RegionScope();
};

// Device-side view of the symbolic object (int32 indices).
struct SymDev {
    int n, nsn, nvp, nblk, nupd;
    const int *snptr, *snpar, *rowptr, *rowidx, *chptr, *chidx, *relptr, *relidx;
    const int *nn, *na;
    const int *aaidx, *vec2blk, *diagblk;
    const long long *blkptr, *updptr;      // 64-bit: nblk*batch can exceed 2^31
    const double *wdot;
};

struct TaskSched {
    int ntask;
    const int *task_ptr, *task_sn, *dep_ptr, *dep_idx;
};

// Extra device tables of the warp-per-chain kernels for tiny cliques (chordal_small.cu).
// A "step" is one supernode visit of a sweep; its descriptor is two int4:
//   up  : {nn | na<<4 | flags<<8 | run<<16, blkptr[k], rowslot, slotpos}, {upd tile, och_beg, och_cnt, sqptr[k]}
//   down: {nn | na<<4 | flags<<8 | run<<16, blkptr[k], rowslot, slotpos}, {updptr[k], 0, 0, 0}
// run = number of consecutive "uniform" steps starting here (same clique shape as the previous step,
// separator = leading rows of the next clique), processed in the position layout.
// rowslot: nibble q = slot of the q-th row of the clique; slotpos: nibble s = position of the row
// that owns slot s (15 = slot unused).  A chunk is {p_begin, p_end, blk_lo, blk_hi}, {sq_lo, sq_hi, 0, 0}.
struct SmallDev {
    const int4 *up_steps, *down_steps;
    const int4 *up_chunks, *down_chunks, *add_chunks;            // add: also bounded by the local fronts
    const int *up_chunk_ptr, *down_chunk_ptr, *add_chunk_ptr;    // ntask+1 each
    const int *och;           // update-matrix tiles of the children that are not the previous step
    const long long *sqptr;   // nsn+1: offsets of the nj x nj local fronts in the F scratch
    long long nsq;
    int ntiles;               // supernodes whose update matrix goes through a global 8 x 8 tile
    const int *wide_sn;       // supernodes with more than one column
    int nwide;
};

// A supernode of the "top set" processed by the dense multi-CTA path (bigfront.cu)
struct BigNode {
    int k, nn, na, nj, nch;
    long long boff, uoff;        // offsets of its block in blkval and of its update matrix
    long long inv_off, ch_off;   // offsets into big_inv (nch x nj) and big_ch (nch)
    long long rowoff;            // offset of its row list in rowidx
    int r0;                      // its first row / column (the columns of a supernode are contiguous)
};
#define BIG_NWS 6                // nj x nj workspaces of the dense path

struct smcp_sym {
    smcp_ctx *ctx;
    SymDev d;
    TaskSched up, down, flat;    // bottom-up, top-down and dependency-free schedules
    int max_nj, max_nn, max_na;
    std::vector<void *> allocs;  // device allocations owned by the object
    // scheduler state
    unsigned *counter = nullptr;     // work-queue head
    unsigned *done = nullptr;        // per (task, batch) completion epoch
    size_t done_cap = 0;
    unsigned epoch = 0;
    int *fail = nullptr;             // per batch element failure flags (device)
    size_t fail_cap = 0;
    // workspaces (grown on demand)
    double *upd = nullptr;           // batch x nupd update matrices
    size_t upd_cap = 0;
    double *cta_ws = nullptr;        // per-CTA scratch
    size_t cta_ws_cap = 0;
    double *tmp = nullptr;           // batch x nblk temporary (out-of-place ops)
    size_t tmp_cap = 0;
    double *probe_buf = nullptr;     // candidates of the batched line-search probes (smcp_csp_probe)
    size_t probe_cap = 0;
    double *red = nullptr;           // reduction scratch
    size_t red_cap = 0;
    // tiny-clique path (max_nj <= 8): warp-per-chain sweeps, see chordal_small.cu
    bool small = false;
    SmallDev sm = {};
    double *fbuf = nullptr;          // batch x nsq local fronts (llt, inverse Hessian)
    size_t fbuf_cap = 0;
    // chain clique trees with single-column supernodes: segment-parallel sweeps (chordal_chain.cuh)
    bool chain = false;
    int chW = 0, chN = 0, chP = 0, ch_root_off = 0, ch_root_nj = 0;
    double *ch_state = nullptr;      // batch x P x D boundary states
    size_t ch_state_cap = 0;
    // top set of large supernodes (and their ancestors) processed by dense kernels for single matrices (bigfront.cu)
    std::vector<BigNode> big;    // ascending supernode index = post-order
    const int *big_flag = nullptr, *big_inv = nullptr, *big_ch = nullptr;
    double *big_ws = nullptr;      // BIG_NWS workspaces per lane
    size_t big_ws_stride = 0;
    int *big_info = nullptr;       // one flag per lane
    unsigned *thin_counters = nullptr;   // one arrival counter per lane (thin_down_kernel)
    double *thin_dinv = nullptr;         // inverted diagonal blocks of R = chol(Y_aa) per top-set supernode (thin inverse Hessian)
    std::vector<size_t> thin_dinv_off;
    std::vector<uint64_t> thin_dinv_gen; // scaling point (raa_gen) the cached blocks belong to
    uint64_t raa_gen_next = 0, raa_gen_cur = 0;
    cudaStream_t tree_side = nullptr;    // side stream of the tree kernels that overlap with the top-set lanes (chordal.cu)
    cudaEvent_t tree_ev[2] = {nullptr, nullptr};
    bool tree_pending = false;
    void *thin_desc = nullptr, *thin_off = nullptr;   // per top-set supernode {nn, na, nj, r0} / {block offset, separator rows offset}
    double *thin_w = nullptr;            // W = D^-1 K_an^T of every thin supernode (forward Hessian)
    std::vector<size_t> thin_w_off;
    std::vector<cudaStream_t> thin_side; // side streams of the M_an products
    std::vector<cudaEvent_t> thin_ev;    // 2 per top-set supernode: thin_up done / product done
    std::vector<int> thin_pending;
    double *big_dinv = nullptr;          // (L_nn L_nn^T)^-1 of the wide top-set supernodes (forward Hessian), per scaling point
    std::vector<size_t> big_dinv_off;
    std::vector<uint64_t> big_dinv_gen;
    uint64_t lt_gen_next = 0, lt_gen_cur = 0;
    std::vector<std::vector<int>> big_up, big_down;   // indices into `big` by height (leaves first) / by depth (root first)
    int big_nlanes = 1;            // lanes the top set may use (1 = everything on the main stream)
    int big_lane = 0;              // lane the next big_* call works in
    int max_nj_small = 0;        // largest frontal matrix left to the tree kernels when the top set is skipped
    double *big_hinv = nullptr;                         // inverse Hessian: K_nn | K_an of every top-set supernode (blkval layout)
    size_t big_hinv_cap = 0;
    double *big_bws = nullptr, *big_cat = nullptr;      // batched top-set workspaces (grown on demand)
    size_t big_bws_cap = 0, big_cat_cap = 0;
    // buffers of destroyed smcp_hess objects, reused by the next one (a new scaling point every IPM
    // iteration: cudaMalloc / cudaFree are synchronising driver calls and do not belong in the loop)
    struct HessBufs { double *Lt, *Yaa, *Raa, *phi; };
    std::vector<HessBufs> hess_pool;
    // host copies used by the operator setup
    std::vector<int> h_vec2blk;
    std::vector<int64_t> h_snptr;
};

struct smcp_hess {
    smcp_sym *sym;
    double *Lt = nullptr;      // nblk: nu-nu part = L_nn (lower), alpha-nu part = L_an L_nn^{-1}
    double *Yaa = nullptr;     // nupd: Y_{alpha alpha}, full symmetric
    double *Raa = nullptr;     // nupd: chol(Y_aa) (lazily, for the inverse map)
    bool have_Raa = false;
    uint64_t lt_gen = 0;           // generation of Lt (keys smcp_sym::big_dinv)
    uint64_t raa_gen = 0;          // generation of Raa (keys caches derived from it: smcp_sym::thin_dinv)
    double *phi_up = nullptr, *phi_dn = nullptr, *psi_up = nullptr, *psi_dn = nullptr;   // chain path: segment propagators of the two sweeps
    bool have_phi = false;
    bool chain_ok = true;      // the segment propagators of this scaling point are tame enough for the segment-parallel sweeps
    double chain_gamma = 0.0;  // largest |entry| of the propagators (growth of the boundary recurrence)
    const double *L = nullptr; // the factor it was built from (not owned)
};

int sym_ensure(smcp_sym *s, int64_t batch, bool need_tmp);
int grow(void **p, size_t *cap, size_t bytes);
// concurrent lanes (capi.cu): fork n lanes off ctx->stream, make lane i current, join them all back
int lanes_fork(smcp_ctx *ctx, int n);
void lane_select(smcp_ctx *ctx, int i);
int lanes_join(smcp_ctx *ctx);

// tiny-clique kernels (chordal_small.cu); same contracts as the k_* functions below
int small_setup(smcp_sym *s, const smcp_sym_desc *D, const std::vector<int> &tp, const std::vector<int> &ts,
                const std::vector<int> &tp2, const std::vector<int> &ts2);
int ks_cholesky(smcp_sym *s, double *x, int64_t batch, int32_t *info_host);
int ks_completion(smcp_sym *s, double *x, int64_t batch, int32_t *info_host);
int ks_projinv(smcp_sym *s, double *x, int64_t batch);
int ks_llt(smcp_sym *s, double *x, int64_t batch);
int ks_hess_prep(smcp_hess *h, const double *L, const double *Y);
int ks_hess_prep_inv(smcp_hess *h);
int ks_hess_apply(smcp_hess *h, double *U, int64_t batch, int inv);
int fetch_fail(smcp_sym *s, int64_t batch, int32_t *info_host);

// chordal kernels (chordal.cu)
int k_cholesky(smcp_sym *s, double *x, int64_t batch, int32_t *info_host);
int k_completion(smcp_sym *s, double *x, int64_t batch, int32_t *info_host);
int k_projinv(smcp_sym *s, double *x, int64_t batch);
int k_llt(smcp_sym *s, double *x, int64_t batch);
int k_hess_prep(smcp_hess *h, const double *L, const double *Y);
int k_hess_prep_inv(smcp_hess *h);
int k_hess_apply(smcp_hess *h, double *U, int64_t batch, int inv);
int k_hess_apply_half(smcp_hess *h, double *U, int64_t batch, int inv, int adj);
int k_trsm(smcp_sym *s, const double *L, double *B, int64_t ldb, int64_t nrhs, int trans);
int k_axpy(smcp_sym *s, double a, const double *x, double *y, int64_t len);
int k_scal(smcp_sym *s, double a, double *x, int64_t len);
int k_dot(smcp_sym *s, const double *x, const double *y, double *out_host);
int k_sumlogdiag(smcp_sym *s, const double *x, int64_t batch, double *out_host);
int k_scatter_vec(smcp_sym *s, double *dst, const double *dev_vec);
int k_gather_vec(smcp_sym *s, const double *src, double *dev_vec);
int k_axpy_batch(smcp_sym *s, const double *x, const double *dx, const double *gam_dev, double *out, int64_t count);

// randomized rounding (rounding.cu): Gaussian samples L^-T g of the max-det completion, +-1 trials against the objective
int k_sample(smcp_sym *s, const double *L, uint64_t seed, int64_t col0, double *B, int64_t ldb, int64_t k);
int k_round_pm1(smcp_sym *s, const double *L, uint64_t seed, int64_t trials, int64_t chunk, int64_t nc, const int64_t *crow,
                const int64_t *ccol, const double *cval, double *values_host, int8_t *x_host, int64_t *best_out);
// one-flip local search of the +-1 trials (rounding.cu): inside smcp_round_pm1's passes, and on caller-given vectors
int k_round_pm1_ls(smcp_sym *s, const double *L, uint64_t seed, int64_t trials, int64_t chunk, int64_t nc, const int64_t *crow,
                   const int64_t *ccol, const double *cval, int64_t max_flips, double tol, double *values0_host,
                   double *values_host, int8_t *x_host, int64_t *best_out, int64_t *flips_host);
int k_pm1_local_search(smcp_ctx *ctx, int64_t n, int64_t k, int8_t *x_host, int64_t nc, const int64_t *crow, const int64_t *ccol,
                       const double *cval, int64_t max_flips, double tol, double *values_host, int64_t *flips_host);
// tabu search of the +-1 trials (rounding.cu): after the one-flip search inside smcp_round_pm1's passes, and on
// caller-given vectors
int k_round_pm1_tabu(smcp_sym *s, const double *L, uint64_t seed, int64_t trials, int64_t chunk, int64_t nc,
                     const int64_t *crow, const int64_t *ccol, const double *cval, int64_t max_flips, double tol,
                     double *values0_host, double *values_host, int8_t *x_host, int64_t *best_out, int64_t *flips_host,
                     int64_t tabu_iters, int64_t tenure, double *values1_host, int64_t *moves_host, int64_t *best_iter_host);
int k_pm1_tabu_search(smcp_ctx *ctx, int64_t n, int64_t k, int8_t *x_host, int64_t nc, const int64_t *crow, const int64_t *ccol,
                      const double *cval, int64_t iters, int64_t tenure, double *values_host, int64_t *moves_host,
                      int64_t *best_iter_host);
// rounding of the +-1 trials sign(V g_t) from a low-rank factor V (n x r, row-major, host), with the searches of
// k_round_pm1_tabu (max_flips = 0 and tabu_iters = 0: plain rounding; the search outputs may then be null)
int k_round_pm1_factor(smcp_ctx *ctx, int64_t n, int64_t r, const double *V_host, uint64_t seed, int64_t trials, int64_t chunk,
                       int64_t nc, const int64_t *crow, const int64_t *ccol, const double *cval, int64_t max_flips, double tol,
                       int64_t tabu_iters, int64_t tenure, double *values0_host, double *values1_host, double *values_host,
                       int8_t *x_host, int64_t *best_out, int64_t *flips_host, int64_t *moves_host, int64_t *best_iter_host);
// B[i + c ldb] = entry i < n of the standard normal sample col0 + c < col0 + k under seed (round_normal_kernel)
int launch_round_normals(smcp_ctx *ctx, uint64_t seed, int64_t col0, int n, double *B, int64_t ldb, int64_t k);

// device workspace of one call, freed (after the stream drains) when it goes out of scope
struct RoundWs {
    smcp_ctx *ctx;
    const char *fn;
    std::vector<void *> p;
    ~RoundWs() {
        cudaStreamSynchronize(ctx->stream);
        for (void *q : p) cudaFree(q);
    }
    void *alloc(size_t bytes) {
        void *q = nullptr;
        if (cudaMalloc(&q, bytes < 16 ? 16 : bytes) != cudaSuccess) {
            cudaGetLastError();
            smcp_set_error("%s: cudaMalloc(%zu bytes) failed", fn, bytes);
            return nullptr;
        }
        p.push_back(q);
        return q;
    }
};

// the rows of the one-flip search on the device (see round_ls_kernel in rounding.cu): CSR of the off-diagonal entries of
// C from both triangles, increasing columns, duplicates summed in input order, and thr_i = tol sum_j |C_ij|
struct LsRows {
    long long *rp = nullptr;
    int *col = nullptr;
    double *val = nullptr, *thr = nullptr;
};
struct LsRowsHost {
    std::vector<long long> rp;
    std::vector<int> col;
};
// entries must lie in 0..n-1 (checked by the caller); with `host`, the host copy of rp and col is kept there
int ls_rows_upload(RoundWs &ws, int n, int64_t nc, const int64_t *crow, const int64_t *ccol, const double *cval, double tol,
                   LsRows &d, LsRowsHost *host);

// low-rank (Burer-Monteiro) solve of min C . X s.t. X_ii = b_i, X >= 0 by the mixing method (lowrank.cu)
int k_lowrank_solve(smcp_ctx *ctx, int64_t n, int64_t r, int64_t nc, const int64_t *crow, const int64_t *ccol, const double *cval,
                    const double *b, uint64_t seed, int64_t max_sweeps, double tol, double *V_host, double *f_host, double *y_host,
                    int64_t *sweeps_out, int64_t *colors_out);

// dense path for the top set of large supernodes (bigfront.cu)
int big_setup(smcp_sym *s, const smcp_sym_desc *D);
int big_cholesky(smcp_sym *s, const BigNode &q, double *X, int64_t b);
int big_llt(smcp_sym *s, const BigNode &q, double *X, int64_t b);
int big_hess_up(smcp_sym *s, const BigNode &q, const double *Lt, const double *Yaa_all, double *X, int64_t b);
int big_hess_down(smcp_sym *s, const BigNode &q, const double *Lt, double *X, int64_t b);
int big_thin_join(smcp_sym *s);
int big_hess_inv_local(smcp_sym *s, const BigNode &q, const double *Lt, const double *Raa_all, const double *X, int64_t b, double *KS);
int big_hess_inv_sweep(smcp_sym *s, const BigNode &q, const double *Lt, double *X, int64_t b, const double *KS);
int big_projinv(smcp_sym *s, const BigNode &q, double *X, int64_t b);
int big_completion(smcp_sym *s, const BigNode &q, double *X, const double *Xin, int64_t b);
int big_hess_prep(smcp_sym *s, const BigNode &q, const double *L0, const double *Y0, double *Lt_out, double *Yaa_out);
int big_hess_prep_inv(smcp_sym *s, const BigNode &q, const double *Yaa_all, double *Raa_all);
int big_lanes_begin(smcp_sym *s);          // returns the number of lanes (>= 1), -1 on error
void big_lane_pick(smcp_sym *s, int lane);
int big_lanes_end(smcp_sym *s);
int big_trsm_node(smcp_sym *s, const BigNode &q, const double *L, double *B, int64_t ldb, int64_t nrhs, int trans);
int big_trsm_all(smcp_sym *s, const double *L, double *B, int64_t ldb, int64_t nrhs, int trans);
int big_hess_fwd_batched(smcp_sym *s, const double *Lt, const double *Yaa_all, double *U, int64_t batch);

// blocked triangular solves (front.cu)
int d_trsm_left_lower(smcp_ctx *ctx, bool trans, const double *L, int64_t ldl, int64_t n, double *B, int64_t ldb, int64_t nrhs);

// dense kernels (dense.cu)
// factor the leading ncols columns of the m x m matrix H (leading dimension ld); ncols < m leaves the
// Schur complement in the trailing block; nranks > 1: block-cyclic columns with NCCL panel broadcasts
int d_potrf(smcp_ctx *ctx, double *H, int64_t ld, int64_t m, int64_t ncols, int32_t *info_dev, int rank, int nranks, int64_t block = 0);
int d_potrs(smcp_ctx *ctx, const double *H, int64_t m, double *y_dev);
bool potrs_wave_for(const smcp_ctx *ctx, int64_t m);
int d_potrs_wave(smcp_ctx *ctx, const double *H, int64_t m, const double *Dinv, double *y_dev);
// potrs as one thread-block-cluster launch on the inverted 64 x 64 diagonal blocks (potrs_cluster.cu)
bool potrs_cluster_for(int64_t m);
int d_potrs_prepare(smcp_ctx *ctx, const double *H, int64_t ld, int64_t m, double *Dinv);
int d_potrs_cluster(smcp_ctx *ctx, const double *H, int64_t m, const double *Dinv, double *y_dev);
int d_trs_cluster(smcp_ctx *ctx, const double *H, int64_t ld, int64_t m, const double *Dinv, double *y_dev, int64_t ldy, int64_t nrhs,
                  int do_fwd, int do_bwd, const char *name);
int launch_gemm_cyc(smcp_ctx *ctx, bool ta, bool tb, const double *A, int64_t lda, const double *B, int64_t ldb, double *C,
                    int64_t ldc, int64_t M, int64_t N, int64_t K, double alpha, int accumulate, int tri, int64_t tri_off,
                    const char *name, int jb0, int jbstride, int tpb = 1);
int launch_gemm_batched(smcp_ctx *ctx, bool ta, bool tb, const double *A, int64_t lda, int64_t sA, const double *B, int64_t ldb,
                        int64_t sB, double *C, int64_t ldc, int64_t sC, int64_t M, int64_t N, int64_t K, double alpha,
                        int accumulate, int64_t batch, const char *name);
// single-launch tile Cholesky and slab triangular solves for L2-resident matrices (dense_tile.cu)
bool potrf_tile_fits(const smcp_ctx *ctx, int64_t mm, int64_t npiv, bool panel_only);
int potrf_tile(smcp_ctx *ctx, double *H, int64_t ld, int64_t mm, int64_t npiv, bool panel_only, int32_t *info_dev, int col_off);
bool trsm_slab_fits(int64_t n);
int trsm_slab(smcp_ctx *ctx, bool trans, const double *L, int64_t ldl, int64_t n, double *B, int64_t ldb, int64_t nrhs);
// blocked Householder QR of an M x N matrix, M >= N (qr.cu): lapack.geqrf / lapack.orgqr semantics in place
int d_geqrf(smcp_ctx *ctx, double *A, int64_t lda, int64_t M, int64_t N, double *tau_dev);
int d_orgqr(smcp_ctx *ctx, double *A, int64_t lda, int64_t M, int64_t N, const double *tau_dev);
// L = R^T (lower, leading dimension ldl) with diag(L) >= 0 from the R of d_geqrf; sgn[i] = sign of R(i, i);
// info_dev = first k (1-based) with |R_kk| <= 1e-14 max |R_ii|, 0 if none
int qr_extract_lower(smcp_ctx *ctx, const double *A, int64_t lda, int64_t m, double *L, int64_t ldl, double *sgn, int *info_dev);
// column c of A (M x N) times sgn[c]
int qr_apply_colsign(smcp_ctx *ctx, double *A, int64_t lda, int64_t M, int64_t N, const double *sgn);
// TMA-fed DMMA GEMM for K-major operands (gemm_tma.cu)
bool gemm_tma_eligible(const double *A, int64_t lda, const double *B, int64_t ldb, int64_t M, int64_t N, int64_t K);
int launch_gemm_tma_tn(smcp_ctx *ctx, const double *A, int64_t lda, const double *B, int64_t ldb, double *C, int64_t ldc,
                       int64_t M, int64_t N, int64_t K, double alpha, int accumulate, int tri, int64_t tri_off, const char *name);
// NCCL helpers on the library's communicator (capi.cu): grouped broadcasts, max-reduction of an int32 flag,
// in-place all-gather of equal chunks of doubles
int comm_group_start();
int comm_group_end();
int comm_allreduce_max_i32(smcp_ctx *ctx, int *ptr, size_t count, cudaStream_t s);
int comm_allgather(smcp_ctx *ctx, double *base, size_t chunk, cudaStream_t s);
// ncclBroadcast of `count` doubles in place on stream s (capi.cu)
int comm_bcast(smcp_ctx *ctx, double *ptr, size_t count, int root, cudaStream_t s);
int launch_gemm(smcp_ctx *ctx, bool ta, bool tb, const double *A, int64_t lda, const double *B, int64_t ldb, double *C,
                int64_t ldc, int64_t M, int64_t N, int64_t K, double alpha, int accumulate, int tri, int64_t tri_off,
                const char *name);
// C(lower blocks, rows i0.. ) = A^T * B : A is K x M (col-major, ld K), B is K x N
int d_gemm_tn(smcp_ctx *ctx, const double *A, int64_t lda, const double *B, int64_t ldb, double *C,
              int64_t ldc, int64_t M, int64_t N, int64_t K, int64_t row_lo_of_col0);
