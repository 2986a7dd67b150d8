// Supernodal chordal-matrix kernels for sm_100a: cholesky, completion, projected inverse,
// llt, barrier Hessian (forward and inverse), chordal trsm and the level-1 reductions.
//
// These replace the chompack routines SMCP calls once or many times per interior-point
// iteration (reference call sites: src/python/solvers.py:82-97 imports; cholesky e.g. 884,
// 2354; completion 874, 2344; projected_inverse 891, 2361; llt 904, 1721; hessian 483, 524,
// 531, 1913, 1952, 1959 and the inverse map 405, 1735, 2021; trsm 491-492; dot: 52 sites).
//
// Execution model (B200-first, not a translation of chompack's Python recursion):
//  * every routine works on a BATCH of chordal matrices that share one clique tree (the m
//    constraint matrices of the Schur complement, or the candidates of a line search);
//  * one persistent kernel per routine.  Work items are (task, batch element) pairs where a
//    task is a connected piece of the clique tree (a chain or a small subtree) that one CTA
//    walks sequentially; items are handed out through an atomic queue in a topological
//    order and cross-task dependencies are resolved with release/acquire epoch flags in
//    global memory, so there is no host round trip and no launch per tree level.  Because
//    every CTA of the grid is co-resident and items are claimed in topological order, the
//    lowest unfinished item can always run: the scheme cannot deadlock;
//  * frontal matrices are staged in shared memory when they fit (tiny cliques: band and
//    max-cut patterns) and in a per-CTA global scratch otherwise;
//  * extend-add is done by the parent, child after child, so sums are formed in a fixed
//    order (bitwise reproducible; no floating-point atomics anywhere).
#include "internal.cuh"
#include <cstdio>
#include <algorithm>

#include "chordal_ops.cuh"

#define TID ((int)threadIdx.x)
#define NT ((int)blockDim.x)

// ---------------------------------------------------------------------------------------
// persistent dependency-driven kernel
// ---------------------------------------------------------------------------------------
template <int OP>
__global__ void tree_kernel(TreeArgs a) {
    extern __shared__ double smem_ws[];
    __shared__ int s_item;
    double *ws = a.use_smem ? smem_ws : a.cta_ws + (long long)blockIdx.x * a.ws_stride;
    const int total = a.T.ntask * a.B;
    for (;;) {
        if (TID == 0) s_item = (int)atomicAdd(a.counter, 1u);
        __syncthreads();
        int item = s_item;
        __syncthreads();
        if (item >= total) break;
        int t = item / a.B, b = item % a.B;
        if (TID == 0) {
            for (int d = a.T.dep_ptr[t]; d < a.T.dep_ptr[t + 1]; ++d) {
                const unsigned *flag = a.done + (long long)a.T.dep_idx[d] * a.B + b;
                while (ld_acquire(flag) != a.epoch) __nanosleep(32);
            }
        }
        __syncthreads();
        __threadfence();
        for (int p = a.T.task_ptr[t]; p < a.T.task_ptr[t + 1]; ++p) {
            if (a.skipflag && a.skipflag[a.T.task_sn[p]]) continue;   // dense top-set path (bigfront.cu)
            Node q = node_of(a.S, a.T.task_sn[p]);
            if (OP == OP_CHOL) op_chol<false>(a, q, b);
            else if (OP == OP_LLT) op_llt<false>(a, q, b, ws);
            else if (OP == OP_PROJINV) op_projinv<false>(a, q, b, ws);
            else if (OP == OP_COMPL) op_compl<false>(a, q, b, ws);
            else if (OP == OP_HPREP) op_hprep<false>(a, q);
            else if (OP == OP_HPREP_INV) op_hprep_inv<false>(a, q);
            else if (OP == OP_HFWD_UP) op_hfwd_up<false>(a, q, b, ws);
            else if (OP == OP_HFWD_DOWN) op_hfwd_down<false>(a, q, b, ws);
            else if (OP == OP_HINV) op_hinv<false>(a, q, b, ws);
            __syncthreads();
        }
        __threadfence();
        __syncthreads();
        if (TID == 0) st_release(a.done + (long long)t * a.B + b, a.epoch);
    }
}

// ---------------------------------------------------------------------------------------
// host launchers
// ---------------------------------------------------------------------------------------
static const size_t SMEM_WS_LIMIT = 200 * 1024;     // fronts up to nj = 79 stay in shared memory (227 KB per CTA on sm_100)

static size_t ws_doubles(const smcp_sym *s, bool skip_big) {
    size_t nj = (size_t)(skip_big ? s->max_nj_small : s->max_nj);
    return 4 * nj * nj + 8;
}

int sym_ensure(smcp_sym *s, int64_t batch, bool need_tmp) {
    smcp_ctx *ctx = s->ctx;
    size_t need_done = (size_t)(s->d.nsn) * (size_t)batch * sizeof(unsigned);
    if (need_done > s->done_cap) {
        if (s->done) cudaFree(s->done);
        CUDA_TRY(cudaMalloc(&s->done, need_done));
        CUDA_TRY(cudaMemsetAsync(s->done, 0, need_done, ctx->stream));
        s->done_cap = need_done;
    }
    if (grow((void **)&s->fail, &s->fail_cap, (size_t)batch * sizeof(int))) return -1;
    const size_t upd_per = s->small ? (size_t)s->sm.ntiles * 64 : (size_t)s->d.nupd;
    if (grow((void **)&s->upd, &s->upd_cap, ((size_t)batch * upd_per + 1) * sizeof(double))) return -1;
    if (need_tmp && grow((void **)&s->tmp, &s->tmp_cap, (size_t)batch * (size_t)s->d.nblk * sizeof(double))) return -1;
    return 0;
}

template <int OP>
static int launch_tree(smcp_sym *s, TreeArgs &a, const TaskSched &T, int64_t batch, int threads, const char *name) {
    smcp_ctx *ctx = s->ctx;
    a.S = s->d;
    a.T = T;
    a.B = (int)batch;
    a.counter = s->counter;
    a.done = s->done;
    a.epoch = ++s->epoch;
    a.fail = s->fail;
    size_t wsd = ws_doubles(s, a.skipflag != nullptr);
    size_t smem = wsd * sizeof(double);
    a.use_smem = smem <= SMEM_WS_LIMIT;
    auto kern = tree_kernel<OP>;
    if (a.use_smem) {
        CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    } else {
        smem = 0;
    }
    int per_sm = 0;
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, smem));
    if (per_sm < 1) { smcp_set_error("tree kernel does not fit on an SM"); return -1; }
    long long items = (long long)T.ntask * batch;
    long long grid = (long long)per_sm * ctx->num_sms;
    if (grid > items) grid = items;
    if (grid < 1) grid = 1;
    if (!a.use_smem) {
        if (grow((void **)&s->cta_ws, &s->cta_ws_cap, (size_t)grid * wsd * sizeof(double))) return -1;
        a.cta_ws = s->cta_ws;
        a.ws_stride = (long long)wsd;
    }
    CUDA_TRY(cudaMemsetAsync(s->counter, 0, sizeof(unsigned), ctx->stream));
    {
        LaunchScope ls(ctx, name, 1, (double)batch);
        kern<<<(unsigned)grid, threads, smem, ctx->stream>>>(a);
    }
    CUDA_TRY(cudaGetLastError());
    return 0;
}

static int pick_threads_nj(int nj) {
    if (nj <= 8) return 32;
    if (nj <= 16) return 64;
    if (nj <= 48) return 128;
    return 256;
}
static int pick_threads(const smcp_sym *s, bool skip_big = false) { return pick_threads_nj(skip_big ? s->max_nj_small : s->max_nj); }

int fetch_fail(smcp_sym *s, int64_t batch, int32_t *info_host) {
    smcp_ctx *ctx = s->ctx;
    CUDA_TRY(cudaMemcpyAsync(info_host, s->fail, (size_t)batch * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return 0;
}

// single matrices (or a handful): the top set of large supernodes goes to the dense kernels of
// bigfront.cu (after the tree kernel in leaves-to-root sweeps, before it in root-to-leaves sweeps)
static bool use_big(const smcp_sym *s, int64_t batch) { return !s->big.empty() && batch <= 4; }

// Number of ranks that share the per-supernode-independent operations on the top set (completion, the
// Cholesky factors of Y_aa): all ranks of the communicator when the library runs as N replicas of one
// solve (bench / drivers under torchrun); 1 otherwise.
static int dist_ops(const smcp_sym *s, int64_t batch) {
    const smcp_ctx *ctx = s->ctx;
    if (!ctx->nccl_comm || ctx->comm_nranks < 2 || batch != 1 || s->big.size() < 2) return 1;
    return ctx->comm_nranks;
}

// One sweep over the top set, level by level; the supernodes of a level go round-robin to the concurrent lanes.
template <class F>
static int big_sweep(smcp_sym *s, const std::vector<std::vector<int>> &levels, F f) {
    for (const std::vector<int> &lev : levels) {
        const int nl = lev.size() > 1 ? big_lanes_begin(s) : 1;
        if (nl < 0) return -1;
        int j = 0, rc = 0;
        for (int i : lev) {
            if (nl > 1) big_lane_pick(s, j++ % nl);
            if (f(s->big[i])) { rc = -1; break; }
        }
        if ((nl > 1 && big_lanes_end(s)) || rc) return -1;
    }
    return 0;
}

// The tree kernel of an operation whose top-set part does not depend on it (completion, chol(Y_aa), the local phase of
// the inverse Hessian: all per-supernode independent) runs on a side stream next to the concurrent lanes of the top set;
// side_join() makes the main stream wait for it.  Off while profiling (per-launch events).
struct SideScope {
    smcp_sym *s;
    cudaStream_t saved = nullptr;
    bool on = false;
    SideScope(smcp_sym *sym, bool enable) : s(sym) {
        smcp_ctx *ctx = s->ctx;
        if (!enable || ctx->prof || ctx->lanes_active) return;
        if (!s->tree_side) {
            if (cudaStreamCreateWithFlags(&s->tree_side, cudaStreamNonBlocking) != cudaSuccess) { s->tree_side = nullptr; return; }
            cudaEventCreateWithFlags(&s->tree_ev[0], cudaEventDisableTiming);
            cudaEventCreateWithFlags(&s->tree_ev[1], cudaEventDisableTiming);
        }
        cudaEventRecord(s->tree_ev[0], ctx->stream);
        cudaStreamWaitEvent(s->tree_side, s->tree_ev[0], 0);
        saved = ctx->stream;
        ctx->stream = s->tree_side;
        on = true;
    }
    ~SideScope() {
        if (!on) return;
        cudaEventRecord(s->tree_ev[1], s->tree_side);
        s->ctx->stream = saved;
        s->tree_pending = true;
    }
};
static int side_join(smcp_sym *s) {
    if (s->tree_pending) {
        CUDA_TRY(cudaStreamWaitEvent(s->ctx->stream, s->tree_ev[1], 0));
        s->tree_pending = false;
    }
    return 0;
}

int k_cholesky(smcp_sym *s, double *x, int64_t batch, int32_t *info_host) {
    RegionScope rs(s->ctx, batch > 1 ? "op_cholesky_batch" : "op_cholesky");
    if (s->small) return ks_cholesky(s, x, batch, info_host);
    if (sym_ensure(s, batch, false)) return -1;
    CUDA_TRY(cudaMemsetAsync(s->fail, 0, (size_t)batch * sizeof(int), s->ctx->stream));
    TreeArgs a = {};
    a.X = x;
    a.upd = s->upd;
    const bool big = use_big(s, batch);
    if (big) a.skipflag = s->big_flag;
    if (launch_tree<OP_CHOL>(s, a, s->up, batch, pick_threads(s, big), batch > 1 ? "cholesky_batch" : "cholesky")) return -1;
    if (big)
        for (int64_t b = 0; b < batch; ++b)
            if (big_sweep(s, s->big_up, [&](const BigNode &q) { return big_cholesky(s, q, x, b); })) return -1;
    if (info_host) return fetch_fail(s, batch, info_host);
    return 0;
}

int k_llt(smcp_sym *s, double *x, int64_t batch) {
    RegionScope rs(s->ctx, "op_llt");
    if (s->small) return ks_llt(s, x, batch);
    if (sym_ensure(s, batch, false)) return -1;
    TreeArgs a = {};
    a.X = x;
    a.upd = s->upd;
    const bool big = use_big(s, batch);
    if (big) a.skipflag = s->big_flag;
    if (launch_tree<OP_LLT>(s, a, s->up, batch, pick_threads(s, big), "llt")) return -1;
    if (big)
        for (int64_t b = 0; b < batch; ++b)
            if (big_sweep(s, s->big_up, [&](const BigNode &q) { return big_llt(s, q, x, b); })) return -1;
    return 0;
}

int k_projinv(smcp_sym *s, double *x, int64_t batch) {
    RegionScope rs(s->ctx, "op_projected_inverse");
    if (s->small) return ks_projinv(s, x, batch);
    if (sym_ensure(s, batch, false)) return -1;
    TreeArgs a = {};
    a.X = x;
    const bool big = use_big(s, batch);
    if (big) {
        a.skipflag = s->big_flag;
        for (int64_t b = 0; b < batch; ++b)
            if (big_sweep(s, s->big_down, [&](const BigNode &q) { return big_projinv(s, q, x, b); })) return -1;
    }
    return launch_tree<OP_PROJINV>(s, a, s->down, batch, pick_threads(s, big), "projected_inverse");
}

static TaskSched flat_sched(const smcp_sym *s) { return s->flat; }

int k_completion(smcp_sym *s, double *x, int64_t batch, int32_t *info_host) {
    RegionScope rs(s->ctx, batch > 1 ? "op_completion_batch" : "op_completion");
    if (s->small) return ks_completion(s, x, batch, info_host);
    if (sym_ensure(s, batch, true)) return -1;
    smcp_ctx *ctx = s->ctx;
    CUDA_TRY(cudaMemsetAsync(s->fail, 0, (size_t)batch * sizeof(int), ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(s->tmp, x, (size_t)batch * s->d.nblk * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
    TreeArgs a = {};
    a.X = x;
    a.Xin = s->tmp;
    const bool big = use_big(s, batch);
    if (big) a.skipflag = s->big_flag;
    {
        SideScope side(s, big);
        if (launch_tree<OP_COMPL>(s, a, flat_sched(s), batch, pick_threads(s, big), batch > 1 ? "completion_batch" : "completion")) return -1;
    }
    if (big) {
        // The completion of a supernode depends on the INPUT matrix only (SURVEY App. A.3), so with several
        // ranks (replicas of the same solve) the supernodes of the top set are shared out round-robin and
        // every owner broadcasts its block of L: the 27 factorisations of ~1100-row separators of the
        // rand_SDP pattern run 27/N per rank.  All ranks end with bitwise identical data and verdicts.
        const int nr = dist_ops(s, batch), rk = ctx->comm_rank;
        // ... and on one GPU the supernodes a rank owns are issued round-robin on a few concurrent lanes
        const int nl = big_lanes_begin(s);
        if (nl < 0) return -1;
        int rc = 0, mine = 0;
        for (int64_t b = 0; b < batch && !rc; ++b) {
            int idx = 0;
            for (const BigNode &q : s->big) {
                if (nr == 1 || idx % nr == rk) {
                    big_lane_pick(s, mine++ % nl);
                    if (big_completion(s, q, x, s->tmp, b)) { rc = -1; break; }
                }
                ++idx;
            }
        }
        if (big_lanes_end(s) || rc) return -1;
        if (side_join(s)) return -1;
        if (nr > 1) {
            if (comm_group_start()) return -1;
            int idx = 0;
            for (const BigNode &q : s->big) {
                if (comm_bcast(ctx, x + q.boff, (size_t)q.nj * q.nn, idx % nr, ctx->stream)) { comm_group_end(); return -1; }
                ++idx;
            }
            if (comm_group_end()) return -1;
            if (comm_allreduce_max_i32(ctx, s->fail, 1, ctx->stream)) return -1;
        }
    }
    if (info_host) return fetch_fail(s, batch, info_host);
    return 0;
}

int k_hess_prep(smcp_hess *h, const double *L, const double *Y) {
    RegionScope rs(h->sym->ctx, "op_hessian_prep");
    if (h->sym->small) return ks_hess_prep(h, L, Y);
    smcp_sym *s = h->sym;
    if (sym_ensure(s, 1, false)) return -1;
    h->lt_gen = ++s->lt_gen_next;
    TreeArgs a = {};
    a.L0 = L;
    a.Y0 = Y;
    a.Lt_out = h->Lt;
    a.Yaa_out = h->Yaa;
    const bool big = use_big(s, 1);
    if (big) a.skipflag = s->big_flag;
    {
        SideScope side(s, big);
        if (launch_tree<OP_HPREP>(s, a, flat_sched(s), 1, pick_threads(s, big), "hessian_prep")) return -1;
    }
    if (big)
        {
            // independent per supernode
            std::vector<std::vector<int>> all(1);
            for (int i = 0; i < (int)s->big.size(); ++i) all[0].push_back(i);
            if (big_sweep(s, all, [&](const BigNode &q) { return big_hess_prep(s, q, L, Y, h->Lt, h->Yaa); })) return -1;
            if (side_join(s)) return -1;
        }
    return 0;
}

int k_hess_prep_inv(smcp_hess *h) {
    RegionScope rs(h->sym->ctx, "op_hessian_prep_inv");
    if (h->sym->small) return ks_hess_prep_inv(h);
    smcp_sym *s = h->sym;
    if (sym_ensure(s, 1, false)) return -1;
    CUDA_TRY(cudaMemsetAsync(s->fail, 0, sizeof(int), s->ctx->stream));
    h->raa_gen = ++s->raa_gen_next;
    TreeArgs a = {};
    a.Yaa = h->Yaa;
    a.Raa = h->Raa;
    const bool big = use_big(s, 1);
    if (big) a.skipflag = s->big_flag;
    {
        SideScope side(s, big);
        if (launch_tree<OP_HPREP_INV>(s, a, flat_sched(s), 1, pick_threads(s, big), "hessian_prep_inv")) return -1;
    }
    if (big) {
        // independent per supernode as well: chol(Y_aa) of the top set shared out over the ranks
        smcp_ctx *ctx = s->ctx;
        const int nr = dist_ops(s, 1), rk = ctx->comm_rank;
        const int nl = big_lanes_begin(s);
        if (nl < 0) return -1;
        int idx = 0, rc = 0, mine = 0;
        for (const BigNode &q : s->big) {
            if (nr == 1 || idx % nr == rk) {
                big_lane_pick(s, mine++ % nl);
                if (big_hess_prep_inv(s, q, h->Yaa, h->Raa)) { rc = -1; break; }
            }
            ++idx;
        }
        if (big_lanes_end(s) || rc) return -1;
        if (side_join(s)) return -1;
        if (nr > 1) {
            if (comm_group_start()) return -1;
            idx = 0;
            for (const BigNode &q : s->big) {
                if (q.na && comm_bcast(ctx, h->Raa + q.uoff, (size_t)q.na * q.na, idx % nr, ctx->stream)) { comm_group_end(); return -1; }
                ++idx;
            }
            if (comm_group_end()) return -1;
            if (comm_allreduce_max_i32(ctx, s->fail, 1, ctx->stream)) return -1;
        }
    }
    return 0;
}

int k_hess_apply(smcp_hess *h, double *U, int64_t batch, int inv) {
    RegionScope rs(h->sym->ctx, inv ? (batch > 4 ? "op_hessian_inv_batch" : "op_hessian_inv") : (batch > 4 ? "op_hessian_batch" : "op_hessian"));
    if (h->sym->small) return ks_hess_apply(h, U, batch, inv);
    smcp_sym *s = h->sym;
    if (sym_ensure(s, batch, false)) return -1;
    TreeArgs a = {};
    a.X = U;
    a.upd = s->upd;
    a.Lt = h->Lt;
    a.Yaa = h->Yaa;
    a.Raa = h->Raa;
    // forward map on a batch (Schur assembly): the top set goes to the batched dense path
    const bool bigb = !inv && !s->big.empty() && batch > 4;
    const bool big = use_big(s, batch);
    if (big || bigb) a.skipflag = s->big_flag;
    int threads = pick_threads(s, big || bigb);
    s->lt_gen_cur = h->lt_gen;
    if (!inv) {
        const bool many = batch >= 32;
        if (launch_tree<OP_HFWD_UP>(s, a, s->up, batch, threads, many ? "hessian_up_batch" : "hessian_up")) return -1;
        if (bigb && big_hess_fwd_batched(s, h->Lt, h->Yaa, U, batch)) return -1;
        if (big)
            for (int64_t b = 0; b < batch; ++b) {
                if (big_sweep(s, s->big_up, [&](const BigNode &q) { return big_hess_up(s, q, h->Lt, h->Yaa, U, b); })) return -1;
                if (big_thin_join(s)) return -1;
                if (big_sweep(s, s->big_down, [&](const BigNode &q) { return big_hess_down(s, q, h->Lt, U, b); })) return -1;
            }
        return launch_tree<OP_HFWD_DOWN>(s, a, s->down, batch, threads, many ? "hessian_down_batch" : "hessian_down");
    }
    if (!h->have_Raa) {
        if (k_hess_prep_inv(h)) return -1;
        h->have_Raa = true;
    }
    {
        // the small supernodes' sweep and the top set's local phase touch disjoint data (the top set is closed under ancestors)
        SideScope side(s, big && batch == 1);
        if (launch_tree<OP_HINV>(s, a, s->up, batch, threads, batch >= 32 ? "hessian_inv_batch" : "hessian_inv")) return -1;
    }
    if (big) {
        // top set: the per-supernode part first (independent: shared out over the ranks of a replicated solve,
        // results exchanged by grouped broadcasts of nj x nn doubles per supernode), then the leaves-to-root sweep
        smcp_ctx *ctx = s->ctx;
        if (grow((void **)&s->big_hinv, &s->big_hinv_cap, (size_t)s->d.nblk * sizeof(double))) return -1;
        const int nr = dist_ops(s, batch), rk = ctx->comm_rank;
        s->raa_gen_cur = h->raa_gen;
        for (int64_t b = 0; b < batch; ++b) {
            const int nl = big_lanes_begin(s);
            if (nl < 0) return -1;
            int idx = 0, rc = 0, mine = 0;
            for (const BigNode &q : s->big) {
                if (nr == 1 || idx % nr == rk) {
                    big_lane_pick(s, mine++ % nl);
                    if (big_hess_inv_local(s, q, h->Lt, h->Raa, U, b, s->big_hinv)) { rc = -1; break; }
                }
                ++idx;
            }
            if (big_lanes_end(s) || rc) return -1;
            if (side_join(s)) return -1;
            if (nr > 1) {
                if (comm_group_start()) return -1;
                idx = 0;
                for (const BigNode &q : s->big) {
                    if (comm_bcast(ctx, s->big_hinv + q.boff, (size_t)q.nj * q.nn, idx % nr, ctx->stream)) { comm_group_end(); return -1; }
                    ++idx;
                }
                if (comm_group_end()) return -1;
            }
            if (big_sweep(s, s->big_up, [&](const BigNode &q) { return big_hess_inv_sweep(s, q, h->Lt, U, b, s->big_hinv); })) return -1;
        }
    }
    return 0;
}

// Half factors of the Hessian (chompack.hessian(L, Y, U, adj=False/True, inv=...), reference call sites
// src/python/solvers.py:917, 978, 1121, 1126): G, G^adj, G^-1, G^-adj with hessian = G^adj G.  The
// drivers only need ||G(u)|| (smcp_b200.chordal.hessian_norm), so these run through the generic
// CTA-per-supernode sweeps on every pattern (no chain / tiny-clique / dense top-set variants).
int k_hess_apply_half(smcp_hess *h, double *U, int64_t batch, int inv, int adj) {
    smcp_sym *s = h->sym;
    RegionScope rs(s->ctx, "op_hessian_half");
    if (sym_ensure(s, batch, false)) return -1;
    if (grow((void **)&s->upd, &s->upd_cap, ((size_t)batch * (size_t)s->d.nupd + 1) * sizeof(double))) return -1;
    if (!h->have_Raa) {
        if (k_hess_prep_inv(h)) return -1;
        h->have_Raa = true;
    }
    TreeArgs a = {};
    a.X = U;
    a.upd = s->upd;
    a.Lt = h->Lt;
    a.Yaa = h->Yaa;
    a.Raa = h->Raa;
    const int threads = pick_threads(s, false);
    if (!inv) {
        a.half = 1;
        if (!adj) return launch_tree<OP_HFWD_UP>(s, a, s->up, batch, threads, "hessian_half");
        return launch_tree<OP_HFWD_DOWN>(s, a, s->down, batch, threads, "hessian_half");
    }
    a.half = adj ? 1 : 2;
    return launch_tree<OP_HINV>(s, a, s->up, batch, threads, "hessian_half");
}

// ---------------------------------------------------------------------------------------
// chordal trsm: B <- L^{-1} B / L^{-T} B, B dense n x nrhs (rows in internal order)
// One CTA per block of right-hand sides walks the whole tree (columns are independent).
// ---------------------------------------------------------------------------------------
__global__ void trsm_kernel(SymDev S, const double *L, double *B, long long ldb, int nrhs, int trans, int cols_per_cta, const int *skipflag,
                            int use_smem) {
    int c0 = blockIdx.x * cols_per_cta;
    int nc = min(cols_per_cta, nrhs - c0);
    if (nc <= 0) return;
    // the block of right-hand sides lives in shared memory for the whole sweep when it fits: the
    // separator rows of a supernode are scattered, and read-modify-write round trips to L2 per supernode
    // made this kernel a latency chain (14 ms per sweep on the n = 2000 rand_SDP pattern)
    extern __shared__ double trsm_sm[];
    double *Bg = B + (long long)c0 * ldb;
    double *Bc = Bg;
    const long long ldg = ldb;
    if (use_smem) {
        for (long long idx = TID; idx < (long long)S.n * nc; idx += NT) trsm_sm[idx] = Bg[idx % S.n + (idx / S.n) * ldg];
        __syncthreads();
        Bc = trsm_sm;
        ldb = S.n;
    }
    if (!trans) {
        for (int k = 0; k < S.nsn; ++k) {
            if (skipflag && skipflag[k]) continue;       // top set: dense kernels (big_trsm_node)
            int nn = S.nn[k], na = S.na[k], nj = nn + na;
            const double *blk = L + S.blkptr[k];
            const int *rows = S.rowidx + S.rowptr[k];
            int r0 = rows[0];
            // solve with L_nn on rows r0..r0+nn-1 (contiguous)
            for (int j = 0; j < nn; ++j) {
                double d = blk[j + (long long)j * nj];
                for (int c = TID; c < nc; c += NT) Bc[r0 + j + (long long)c * ldb] /= d;
                __syncthreads();
                int nr = nn - j - 1, tot = nr * nc;
                for (int idx = TID; idx < tot; idx += NT) {
                    int r = idx % nr, c = idx / nr;
                    Bc[r0 + j + 1 + r + (long long)c * ldb] -= blk[j + 1 + r + (long long)j * nj] * Bc[r0 + j + (long long)c * ldb];
                }
                __syncthreads();
            }
            // B_alpha -= L_an B_nu
            for (int idx = TID; idx < na * nc; idx += NT) {
                int i = idx % na, c = idx / na;
                double s = 0.0;
                for (int r = 0; r < nn; ++r) s = fma(blk[nn + i + (long long)r * nj], Bc[r0 + r + (long long)c * ldb], s);
                Bc[rows[nn + i] + (long long)c * ldb] -= s;
            }
            __syncthreads();
        }
    } else {
        for (int k = S.nsn - 1; k >= 0; --k) {
            if (skipflag && skipflag[k]) continue;
            int nn = S.nn[k], na = S.na[k], nj = nn + na;
            const double *blk = L + S.blkptr[k];
            const int *rows = S.rowidx + S.rowptr[k];
            int r0 = rows[0];
            for (int idx = TID; idx < nn * nc; idx += NT) {
                int r = idx % nn, c = idx / nn;
                double s = 0.0;
                for (int i = 0; i < na; ++i) s = fma(blk[nn + i + (long long)r * nj], Bc[rows[nn + i] + (long long)c * ldb], s);
                Bc[r0 + r + (long long)c * ldb] -= s;
            }
            __syncthreads();
            for (int j = nn - 1; j >= 0; --j) {
                double d = blk[j + (long long)j * nj];
                for (int c = TID; c < nc; c += NT) Bc[r0 + j + (long long)c * ldb] /= d;
                __syncthreads();
                int tot = j * nc;
                for (int idx = TID; idx < tot; idx += NT) {
                    int i = idx % j, c = idx / j;
                    Bc[r0 + i + (long long)c * ldb] -= blk[j + (long long)i * nj] * Bc[r0 + j + (long long)c * ldb];
                }
                __syncthreads();
            }
        }
    }
    if (use_smem) {
        __syncthreads();
        for (long long idx = TID; idx < (long long)S.n * nc; idx += NT) Bg[idx % S.n + (idx / S.n) * ldg] = trsm_sm[idx];
    }
}

// Many right-hand sides: a column never interacts with another one, so a WARP owns a column for the whole sweep (its n
// entries in shared memory) and needs no block barrier at all -- trsm_kernel above walks the supernodes with 2 nn + 1
// __syncthreads each (2.5 ms per sweep over the 731 small supernodes of the rand_SDP n = 2000 pattern, a latency chain).
#define TW_WARPS 4
__global__ void __launch_bounds__(32 * TW_WARPS) trsm_warp_kernel(SymDev S, const double *__restrict__ L, double *__restrict__ B, long long ldb,
                                                                  long long nrhs, int trans, const int *__restrict__ skipflag) {
    extern __shared__ double tw_sm[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long c = (long long)blockIdx.x * TW_WARPS + warp;
    if (c >= nrhs) return;
    double *b = tw_sm + (size_t)warp * S.n;
    double *Bg = B + c * ldb;
    for (int r = lane; r < S.n; r += 32) b[r] = Bg[r];
    __syncwarp();
    if (!trans) {
        for (int k = 0; k < S.nsn; ++k) {
            if (skipflag && skipflag[k]) continue;
            const int nn = S.nn[k], na = S.na[k], nj = nn + na;
            const double *blk = L + S.blkptr[k];
            const int *rows = S.rowidx + S.rowptr[k];
            const int r0 = rows[0];
            for (int j = 0; j < nn; ++j) {
                const double xj = b[r0 + j] / blk[j + (long long)j * nj];
                __syncwarp();
                if (lane == 0) b[r0 + j] = xj;
                for (int r = j + 1 + lane; r < nn; r += 32) b[r0 + r] = fma(-blk[r + (long long)j * nj], xj, b[r0 + r]);
                __syncwarp();
            }
            for (int i = lane; i < na; i += 32) {
                double t = 0.0;
                for (int r = 0; r < nn; ++r) t = fma(blk[nn + i + (long long)r * nj], b[r0 + r], t);
                b[rows[nn + i]] -= t;
            }
            __syncwarp();
        }
    } else {
        for (int k = S.nsn - 1; k >= 0; --k) {
            if (skipflag && skipflag[k]) continue;
            const int nn = S.nn[k], na = S.na[k], nj = nn + na;
            const double *blk = L + S.blkptr[k];
            const int *rows = S.rowidx + S.rowptr[k];
            const int r0 = rows[0];
            for (int r = 0; r < nn; ++r) {
                double t = 0.0;
                for (int i = lane; i < na; i += 32) t = fma(blk[nn + i + (long long)r * nj], b[rows[nn + i]], t);
                for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
                if (lane == 0) b[r0 + r] -= t;
            }
            __syncwarp();
            for (int j = nn - 1; j >= 0; --j) {
                const double xj = b[r0 + j] / blk[j + (long long)j * nj];
                __syncwarp();
                if (lane == 0) b[r0 + j] = xj;
                for (int i = lane; i < j; i += 32) b[r0 + i] = fma(-blk[j + (long long)i * nj], xj, b[r0 + i]);
                __syncwarp();
            }
        }
    }
    for (int r = lane; r < S.n; r += 32) Bg[r] = b[r];
}

int k_trsm(smcp_sym *s, const double *L, double *B, int64_t ldb, int64_t nrhs, int trans) {
    RegionScope rs(s->ctx, "op_trsm");
    smcp_ctx *ctx = s->ctx;
    int cols = 8;
    // right-hand sides staged in shared memory (up to 200 KB per CTA): n x cols doubles
    const size_t smem_cap = 200 * 1024;
    int use_smem = 0;
    size_t smem = 0;
    {
        int fit = (int)(smem_cap / ((size_t)s->d.n * sizeof(double)));
        if (fit >= 1) {
            cols = std::min(cols, fit);
            // keep enough CTAs in flight: at least ~2 per SM when there are that many right-hand sides
            while (cols > 1 && (nrhs + cols - 1) / cols < 2 * ctx->num_sms && nrhs >= 2 * ctx->num_sms) --cols;
            use_smem = 1;
            smem = (size_t)s->d.n * cols * sizeof(double);
            static size_t attr = 0;
            if (smem > attr) {
                CUDA_TRY(cudaFuncSetAttribute(trsm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_cap));
                attr = smem_cap;
            }
        }
    }
    int grid = (int)((nrhs + cols - 1) / cols);
    if (grid < 1) return 0;
    // many right-hand sides (the dense inverse of the sparse-constraint technique: n of them) on a
    // pattern with a dense top set: the top supernodes -- where the flops are -- go through the slab
    // solves and DMMA products of bigfront.cu; the top set is closed under ancestors, so in the forward
    // sweep it comes after everything else and in the backward sweep before
    const bool big = !s->big.empty() && nrhs >= 32;
    if (big && trans && big_trsm_all(s, L, B, ldb, nrhs, 1)) return -1;
    const size_t tw_smem = (size_t)TW_WARPS * s->d.n * sizeof(double);
    if (nrhs >= 64 && tw_smem <= 96 * 1024) {
        static size_t tw_attr = 0;
        if (tw_smem > tw_attr) {
            CUDA_TRY(cudaFuncSetAttribute(trsm_warp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
            tw_attr = 96 * 1024;
        }
        LaunchScope ls(ctx, "chordal_trsm");
        trsm_warp_kernel<<<(unsigned)((nrhs + TW_WARPS - 1) / TW_WARPS), 32 * TW_WARPS, tw_smem, ctx->stream>>>(s->d, L, B, ldb, nrhs, trans,
                                                                                                         big ? s->big_flag : nullptr);
    } else {
        LaunchScope ls(ctx, "chordal_trsm");
        trsm_kernel<<<grid, 128, smem, ctx->stream>>>(s->d, L, B, ldb, (int)nrhs, trans, cols, big ? s->big_flag : nullptr, use_smem);
    }
    if (big && !trans && big_trsm_all(s, L, B, ldb, nrhs, 0)) return -1;
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// ---------------------------------------------------------------------------------------
// level-1 kernels
// ---------------------------------------------------------------------------------------
__global__ void axpy_kernel(double a, const double *__restrict__ x, double *__restrict__ y, long long n) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < n; i += stride) y[i] = __dadd_rn(y[i], __dmul_rn(a, x[i]));   // no FMA: matches y += a*x
}
__global__ void scal_kernel(double a, double *x, long long n) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < n; i += stride) x[i] *= a;
}
// out[k*n + i] = x[i] + gam[k]*dx[i]
__global__ void axpy_batch_kernel(const double *__restrict__ x, const double *__restrict__ dx,
                                  const double *__restrict__ gam, double *__restrict__ out, long long n, int count) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        double xv = x[i], dv = dx[i];
        for (int k = 0; k < count; ++k) out[(long long)k * n + i] = __dadd_rn(xv, __dmul_rn(gam[k], dv));
    }
}

static int grid_for(smcp_ctx *ctx, long long n, int threads) {
    long long g = (n + threads - 1) / threads;
    long long cap = (long long)ctx->num_sms * 8;
    if (g > cap) g = cap;
    if (g < 1) g = 1;
    return (int)g;
}

int k_axpy(smcp_sym *s, double a, const double *x, double *y, int64_t len) {
    smcp_ctx *ctx = s->ctx;
    {
        LaunchScope ls(ctx, "level1");
        axpy_kernel<<<grid_for(ctx, len, 256), 256, 0, ctx->stream>>>(a, x, y, len);
    }
    CUDA_TRY(cudaGetLastError());
    return 0;
}
int k_scal(smcp_sym *s, double a, double *x, int64_t len) {
    smcp_ctx *ctx = s->ctx;
    {
        LaunchScope ls(ctx, "level1");
        scal_kernel<<<grid_for(ctx, len, 256), 256, 0, ctx->stream>>>(a, x, len);
    }
    CUDA_TRY(cudaGetLastError());
    return 0;
}
int k_axpy_batch(smcp_sym *s, const double *x, const double *dx, const double *gam_dev, double *out, int64_t count) {
    smcp_ctx *ctx = s->ctx;
    {
        LaunchScope ls(ctx, "level1");
        axpy_batch_kernel<<<grid_for(ctx, s->d.nblk, 256), 256, 0, ctx->stream>>>(x, dx, gam_dev, out, s->d.nblk, (int)count);
    }
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// deterministic two-stage weighted dot: fixed grid, fixed per-thread ranges, tree reduce
#define RED_BLOCKS 256
#define RED_THREADS 256
__device__ double block_reduce_sum(double v) {
    __shared__ double sh[RED_THREADS / 32];
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    double r = 0.0;
    if (threadIdx.x < 32) {
        r = (threadIdx.x < blockDim.x / 32) ? sh[threadIdx.x] : 0.0;
        for (int o = 16; o > 0; o >>= 1) r += __shfl_down_sync(0xffffffffu, r, o);
    }
    __syncthreads();
    return r;
}
__global__ void dot_stage1(const double *__restrict__ x, const double *__restrict__ y,
                           const double *__restrict__ w, long long n, double *part) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    long long stride = (long long)gridDim.x * blockDim.x;
    double s = 0.0;
    for (; i < n; i += stride) s = fma(x[i] * w[i], y[i], s);
    s = block_reduce_sum(s);
    if (threadIdx.x == 0) part[blockIdx.x] = s;
}
__global__ void sum_stage2(const double *part, int n, double *out) {
    double s = 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) s += part[i];
    s = block_reduce_sum(s);
    if (threadIdx.x == 0) *out = s;
}
__global__ void logdiag_stage1(const double *__restrict__ x, const int *__restrict__ diag, int n, long long stride_b, double *part) {
    // blockIdx.y = batch element
    const double *xb = x + (long long)blockIdx.y * stride_b;
    double s = 0.0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) s += log(xb[diag[i]]);
    s = block_reduce_sum(s);
    if (threadIdx.x == 0) part[blockIdx.y * gridDim.x + blockIdx.x] = s;
}
__global__ void sum_stage2_batch(const double *part, int n, double *out) {
    double s = 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) s += part[blockIdx.x * n + i];
    s = block_reduce_sum(s);
    if (threadIdx.x == 0) out[blockIdx.x] = s;
}

int k_dot(smcp_sym *s, const double *x, const double *y, double *out_host) {
    smcp_ctx *ctx = s->ctx;
    if (grow((void **)&s->red, &s->red_cap, (RED_BLOCKS + 8) * sizeof(double))) return -1;
    {
        LaunchScope ls(ctx, "reduce", 2);
        dot_stage1<<<RED_BLOCKS, RED_THREADS, 0, ctx->stream>>>(x, y, s->d.wdot, s->d.nblk, s->red);
        sum_stage2<<<1, RED_THREADS, 0, ctx->stream>>>(s->red, RED_BLOCKS, s->red + RED_BLOCKS);
    }
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(out_host, s->red + RED_BLOCKS, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int k_sumlogdiag(smcp_sym *s, const double *x, int64_t batch, double *out_host) {
    smcp_ctx *ctx = s->ctx;
    const int nb = 32;
    if (grow((void **)&s->red, &s->red_cap, ((size_t)batch * (nb + 1) + RED_BLOCKS + 8) * sizeof(double))) return -1;
    double *part = s->red;
    double *outd = s->red + (size_t)batch * nb;
    {
        LaunchScope ls(ctx, "reduce", 2);
        logdiag_stage1<<<dim3(nb, (unsigned)batch), RED_THREADS, 0, ctx->stream>>>(x, s->d.diagblk, s->d.n, s->d.nblk, part);
        sum_stage2_batch<<<(unsigned)batch, RED_THREADS, 0, ctx->stream>>>(part, nb, outd);
    }
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(out_host, outd, (size_t)batch * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return 0;
}

__global__ void scatter_vec_kernel(double *dst, const double *vec, const int *map, int n) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) dst[map[i]] = vec[i];
}
__global__ void gather_vec_kernel(const double *src, double *vec, const int *map, int n) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) vec[i] = src[map[i]];
}
int k_scatter_vec(smcp_sym *s, double *dst, const double *dev_vec) {
    smcp_ctx *ctx = s->ctx;
    CUDA_TRY(cudaMemsetAsync(dst, 0, (size_t)s->d.nblk * sizeof(double), ctx->stream));
    {
        LaunchScope ls(ctx, "level1");
        scatter_vec_kernel<<<grid_for(ctx, s->d.nvp, 256), 256, 0, ctx->stream>>>(dst, dev_vec, s->d.vec2blk, s->d.nvp);
    }
    CUDA_TRY(cudaGetLastError());
    return 0;
}
int k_gather_vec(smcp_sym *s, const double *src, double *dev_vec) {
    smcp_ctx *ctx = s->ctx;
    {
        LaunchScope ls(ctx, "level1");
        gather_vec_kernel<<<grid_for(ctx, s->d.nvp, 256), 256, 0, ctx->stream>>>(src, dev_vec, s->d.vec2blk, s->d.nvp);
    }
    CUDA_TRY(cudaGetLastError());
    return 0;
}
