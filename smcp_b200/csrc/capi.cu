// C ABI of libsmcp_b200.so (see include/smcp_b200.h): context, symbolic object, chordal
// matrix buffers, constraint operator, Schur complement assembly / factorisation / solve.
#include "internal.cuh"
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <cmath>
#include <algorithm>
#include <utility>
#include <dlfcn.h>

static thread_local char g_err[1024] = "";

void smcp_set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

extern "C" const char *smcp_last_error(void) { return g_err; }
extern "C" int smcp_version(void) { return 100; }

int grow(void **p, size_t *cap, size_t bytes) {
    if (bytes <= *cap) return 0;
    if (*p) cudaFree(*p);
    *p = nullptr;
    *cap = 0;
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(p, want);
    if (e != cudaSuccess) {
        smcp_set_error("cudaMalloc(%zu bytes) failed: %s", want, cudaGetErrorString(e));
        return -1;
    }
    *cap = want;
    return 0;
}

LaunchScope::LaunchScope(smcp_ctx *c, const char *nm, int nlaunch, double w) : ctx(c), name(nm), n(nlaunch), work(w) {
    ctx->launches += n;
    active = ctx->prof && ctx->prof_mute == 0;
    launches0 = ctx->launches;
    if (active) cudaEventRecord(ctx->pev0, ctx->stream);
}
LaunchScope::~LaunchScope() {
    if (active) {
        cudaEventRecord(ctx->pev1, ctx->stream);
        cudaEventSynchronize(ctx->pev1);
        float ms = 0.f;
        cudaEventElapsedTime(&ms, ctx->pev0, ctx->pev1);
        ProfEntry &e = ctx->prof_acc[name];
        e.ms += ms;
        e.launches += n + (ctx->launches - launches0);
        e.work += work;
    }
}

static cudaEvent_t region_event(smcp_ctx *ctx) {
    if (!ctx->region_pool.empty()) {
        cudaEvent_t e = ctx->region_pool.back();
        ctx->region_pool.pop_back();
        return e;
    }
    cudaEvent_t e = nullptr;
    cudaEventCreate(&e);
    return e;
}
static void region_resolve(smcp_ctx *ctx, RegionAcc &a) {
    for (auto &pr : a.pending) {
        float ms = 0.f;
        cudaEventSynchronize(pr.second);
        if (cudaEventElapsedTime(&ms, pr.first, pr.second) == cudaSuccess) a.ms += ms;
        ctx->region_pool.push_back(pr.first);
        ctx->region_pool.push_back(pr.second);
    }
    a.pending.clear();
}
RegionScope::RegionScope(smcp_ctx *c, const char *name) : ctx(c), acc(&c->regions[name]) {
    if (acc->pending.size() >= 4096) region_resolve(ctx, *acc);
    e0 = region_event(ctx);
    e1 = region_event(ctx);
    cudaEventRecord(e0, ctx->stream);
}
RegionScope::~RegionScope() {
    cudaEventRecord(e1, ctx->stream);
    acc->pending.push_back({e0, e1});
    acc->calls += 1;
}
extern "C" int smcp_region_get(smcp_ctx *ctx, const char *name, double *ms_out, int64_t *calls_out) {
    auto it = ctx->regions.find(name);
    if (it == ctx->regions.end()) { *ms_out = 0.0; *calls_out = 0; return 0; }
    region_resolve(ctx, it->second);
    *ms_out = it->second.ms;
    *calls_out = it->second.calls;
    return 0;
}
extern "C" int smcp_region_list(smcp_ctx *ctx, char *buf, int64_t cap) {
    std::string out;
    for (auto &kv : ctx->regions) {
        if (!out.empty()) out += ",";
        out += kv.first;
    }
    if ((int64_t)out.size() + 1 > cap) { smcp_set_error("smcp_region_list: buffer too small"); return -2; }
    memcpy(buf, out.c_str(), out.size() + 1);
    return 0;
}
extern "C" int smcp_region_reset(smcp_ctx *ctx) {
    for (auto &kv : ctx->regions) {
        region_resolve(ctx, kv.second);
        kv.second.ms = 0.0;
        kv.second.calls = 0;
    }
    return 0;
}

// ---------------------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------------------
extern "C" int smcp_ctx_create(int device, smcp_ctx **out) {
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        smcp_set_error("no CUDA device available (%s); this library has no CPU fallback",
                       e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
        return -1;
    }
    CUDA_TRY(cudaSetDevice(device));
    smcp_ctx *ctx = new smcp_ctx();
    ctx->device = device;
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    ctx->num_sms = prop.multiProcessorCount;
    CUDA_TRY(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    {
        // the look-ahead stream carries the critical path of the blocked Cholesky (next panel + its broadcast): its CTAs go first
        int prio_lo = 0, prio_hi = 0;
        CUDA_TRY(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
        CUDA_TRY(cudaStreamCreateWithPriority(&ctx->stream2, cudaStreamNonBlocking, prio_hi));
    }
    CUDA_TRY(cudaEventCreate(&ctx->ev0));
    CUDA_TRY(cudaEventCreate(&ctx->ev1));
    CUDA_TRY(cudaEventCreate(&ctx->pev0));
    CUDA_TRY(cudaEventCreate(&ctx->pev1));
    ctx->pinned_bytes = 1 << 20;
    CUDA_TRY(cudaMallocHost(&ctx->pinned, ctx->pinned_bytes));
    *out = ctx;
    return 0;
}

// ---- concurrent lanes ---------------------------------------------------------------------------
// lanes_fork(n): lanes 1 .. n-1 wait for everything issued on the main stream so far; lane_select(i): the
// helpers (launch_gemm, d_potrf, d_trsm_left_lower, the elementwise kernels) now launch on lane i's stream
// with lane i's scratch; lanes_join(): the main stream waits for every lane.  Host code between fork and
// join must not synchronise on ctx->stream expecting the lanes to be covered.
static void lane_swap(smcp_ctx *ctx, CtxLane &L) {
    std::swap(ctx->stream, L.stream);
    std::swap(ctx->gemm_ws, L.gemm_ws);
    std::swap(ctx->gemm_ws_cap, L.gemm_ws_cap);
    std::swap(ctx->trs_dinv, L.trs_dinv);
    std::swap(ctx->trs_dinv_cap, L.trs_dinv_cap);
    std::swap(ctx->gridbar, L.gridbar);
    std::swap(ctx->gridbar_next, L.gridbar_next);
}
void lane_select(smcp_ctx *ctx, int i) {
    if (i == ctx->lane_cur) return;
    if (ctx->lane_cur > 0) lane_swap(ctx, ctx->lanes[ctx->lane_cur - 1]);
    ctx->lane_cur = 0;
    if (i > 0) {
        lane_swap(ctx, ctx->lanes[i - 1]);
        ctx->lane_cur = i;
    }
}
int lanes_fork(smcp_ctx *ctx, int n) {
    if (n <= 1 || ctx->lanes_active) return 0;
    while ((int)ctx->lanes.size() < n - 1) {
        CtxLane L;
        CUDA_TRY(cudaStreamCreateWithFlags(&L.stream, cudaStreamNonBlocking));
        CUDA_TRY(cudaEventCreateWithFlags(&L.done, cudaEventDisableTiming));
        ctx->lanes.push_back(L);
    }
    if (!ctx->lane_fork_ev) CUDA_TRY(cudaEventCreateWithFlags(&ctx->lane_fork_ev, cudaEventDisableTiming));
    CUDA_TRY(cudaEventRecord(ctx->lane_fork_ev, ctx->stream));
    for (int i = 0; i < n - 1; ++i) CUDA_TRY(cudaStreamWaitEvent(ctx->lanes[i].stream, ctx->lane_fork_ev, 0));
    ctx->lanes_active = n;
    return 0;
}
int lanes_join(smcp_ctx *ctx) {
    if (!ctx->lanes_active) return 0;
    lane_select(ctx, 0);
    for (int i = 0; i < ctx->lanes_active - 1; ++i) {
        CUDA_TRY(cudaEventRecord(ctx->lanes[i].done, ctx->lanes[i].stream));
        CUDA_TRY(cudaStreamWaitEvent(ctx->stream, ctx->lanes[i].done, 0));
    }
    ctx->lanes_active = 0;
    return 0;
}

extern "C" int smcp_ctx_destroy(smcp_ctx *ctx) {
    if (!ctx) return 0;
    cudaSetDevice(ctx->device);
    lanes_join(ctx);
    cudaStreamSynchronize(ctx->stream);
    for (CtxLane &L : ctx->lanes) {
        if (L.gemm_ws) cudaFree(L.gemm_ws);
        if (L.trs_dinv) cudaFree(L.trs_dinv);
        if (L.gridbar) cudaFree(L.gridbar);
        cudaEventDestroy(L.done);
        cudaStreamDestroy(L.stream);
    }
    if (ctx->lane_fork_ev) cudaEventDestroy(ctx->lane_fork_ev);
    if (ctx->flush_buf) cudaFree(ctx->flush_buf);
    if (ctx->gemm_ws) cudaFree(ctx->gemm_ws);
    if (ctx->gridbar) cudaFree(ctx->gridbar);
    if (ctx->wave_buf) cudaFree(ctx->wave_buf);
    if (ctx->potrf_pt) cudaFree(ctx->potrf_pt);
    if (ctx->trs_dinv) cudaFree(ctx->trs_dinv);
    if (ctx->qr_ws) cudaFree(ctx->qr_ws);
    if (ctx->pinned) cudaFreeHost(ctx->pinned);
    cudaEventDestroy(ctx->ev0);
    cudaEventDestroy(ctx->ev1);
    cudaEventDestroy(ctx->pev0);
    cudaEventDestroy(ctx->pev1);
    for (cudaEvent_t e : ctx->potrf_ev) cudaEventDestroy(e);
    for (auto &kv : ctx->regions) region_resolve(ctx, kv.second);
    for (cudaEvent_t e : ctx->region_pool) cudaEventDestroy(e);
    cudaStreamDestroy(ctx->stream2);
    cudaStreamDestroy(ctx->stream);
    delete ctx;
    return 0;
}

extern "C" int smcp_ctx_sync(smcp_ctx *ctx) {
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return 0;
}
extern "C" int64_t smcp_ctx_launch_count(smcp_ctx *ctx) { return ctx->launches; }
extern "C" int smcp_timer_start(smcp_ctx *ctx) {
    CUDA_TRY(cudaEventRecord(ctx->ev0, ctx->stream));
    return 0;
}
extern "C" int smcp_timer_stop(smcp_ctx *ctx, double *ms_out) {
    CUDA_TRY(cudaEventRecord(ctx->ev1, ctx->stream));
    CUDA_TRY(cudaEventSynchronize(ctx->ev1));
    float ms = 0.f;
    CUDA_TRY(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    *ms_out = ms;
    return 0;
}
extern "C" int smcp_prof_enable(smcp_ctx *ctx, int on) {
    ctx->prof = on != 0;
    return 0;
}
extern "C" int smcp_prof_get(smcp_ctx *ctx, const char *name, double *ms_out, int64_t *launches_out) {
    auto it = ctx->prof_acc.find(name);
    if (it == ctx->prof_acc.end()) {
        *ms_out = 0.0;
        *launches_out = 0;
        return 0;
    }
    *ms_out = it->second.ms;
    *launches_out = it->second.launches;
    return 0;
}
extern "C" int smcp_prof_get_work(smcp_ctx *ctx, const char *name, double *work_out) {
    auto it = ctx->prof_acc.find(name);
    *work_out = it == ctx->prof_acc.end() ? 0.0 : it->second.work;
    return 0;
}
extern "C" int smcp_prof_list(smcp_ctx *ctx, char *buf, int64_t cap) {
    std::string out;
    for (auto &kv : ctx->prof_acc) {
        if (!out.empty()) out += ",";
        out += kv.first;
    }
    if ((int64_t)out.size() + 1 > cap) { smcp_set_error("smcp_prof_list: buffer too small"); return -2; }
    memcpy(buf, out.c_str(), out.size() + 1);
    return 0;
}
extern "C" int smcp_prof_reset(smcp_ctx *ctx) {
    ctx->prof_acc.clear();
    return 0;
}
extern "C" int smcp_flush_l2(smcp_ctx *ctx) {
    size_t bytes = (size_t)256 << 20;
    if (!ctx->flush_buf) {
        CUDA_TRY(cudaMalloc(&ctx->flush_buf, bytes));
        ctx->flush_bytes = bytes;
    }
    CUDA_TRY(cudaMemsetAsync(ctx->flush_buf, 1, ctx->flush_bytes, ctx->stream));
    return 0;
}

// ---------------------------------------------------------------------------------------
// symbolic object
// ---------------------------------------------------------------------------------------
template <class T, class S>
static int upload(smcp_sym *s, const S *src, size_t n, const T **dst) {
    std::vector<T> tmp(n ? n : 1);
    for (size_t i = 0; i < n; ++i) tmp[i] = (T)src[i];
    void *d = nullptr;
    CUDA_TRY(cudaMalloc(&d, (n ? n : 1) * sizeof(T)));
    CUDA_TRY(cudaMemcpy(d, tmp.data(), (n ? n : 1) * sizeof(T), cudaMemcpyHostToDevice));
    s->allocs.push_back(d);
    *dst = (const T *)d;
    return 0;
}

static int upload_sched(smcp_sym *s, int ntask, const std::vector<int> &tp, const std::vector<int> &ts,
                        const std::vector<int> &dp, const std::vector<int> &di, TaskSched *out) {
    out->ntask = ntask;
    if (upload<int, int>(s, tp.data(), tp.size(), &out->task_ptr)) return -1;
    if (upload<int, int>(s, ts.data(), ts.size(), &out->task_sn)) return -1;
    if (upload<int, int>(s, dp.data(), dp.size(), &out->dep_ptr)) return -1;
    if (upload<int, int>(s, di.data(), di.size(), &out->dep_idx)) return -1;
    return 0;
}

extern "C" int smcp_sym_create(smcp_ctx *ctx, const smcp_sym_desc *D, smcp_sym **out) {
    CUDA_TRY(cudaSetDevice(ctx->device));
    if (D->nblk >= (1LL << 31) || D->nupd >= (1LL << 31)) {
        smcp_set_error("pattern too large for 32-bit block offsets");
        return -2;
    }
    smcp_sym *s = new smcp_sym();
    s->ctx = ctx;
    SymDev &d = s->d;
    d.n = (int)D->n; d.nsn = (int)D->nsn; d.nvp = (int)D->nvp; d.nblk = (int)D->nblk; d.nupd = (int)D->nupd;
    const int nsn = d.nsn;
    std::vector<int> nn(nsn), na(nsn);
    s->max_nj = s->max_nn = s->max_na = 0;
    for (int k = 0; k < nsn; ++k) {
        nn[k] = (int)(D->snptr[k + 1] - D->snptr[k]);
        na[k] = (int)(D->rowptr[k + 1] - D->rowptr[k]) - nn[k];
        s->max_nn = std::max(s->max_nn, nn[k]);
        s->max_na = std::max(s->max_na, na[k]);
        s->max_nj = std::max(s->max_nj, nn[k] + na[k]);
    }
    int rc = 0;
    rc |= upload<int, int64_t>(s, D->snptr, nsn + 1, &d.snptr);
    rc |= upload<int, int64_t>(s, D->snpar, nsn, &d.snpar);
    rc |= upload<int, int64_t>(s, D->rowptr, nsn + 1, &d.rowptr);
    rc |= upload<int, int64_t>(s, D->rowidx, D->rowptr[nsn], &d.rowidx);
    rc |= upload<int, int64_t>(s, D->chptr, nsn + 1, &d.chptr);
    rc |= upload<int, int64_t>(s, D->chidx, D->chptr[nsn], &d.chidx);
    rc |= upload<int, int64_t>(s, D->relptr, nsn + 1, &d.relptr);
    rc |= upload<int, int64_t>(s, D->relidx, D->relptr[nsn], &d.relidx);
    rc |= upload<int, int>(s, nn.data(), nsn, &d.nn);
    rc |= upload<int, int>(s, na.data(), nsn, &d.na);
    rc |= upload<int, int64_t>(s, D->aaidx, D->nupd, &d.aaidx);
    rc |= upload<int, int64_t>(s, D->vec2blk, D->nvp, &d.vec2blk);
    rc |= upload<int, int64_t>(s, D->diagblk, D->n, &d.diagblk);
    rc |= upload<long long, int64_t>(s, D->blkptr, nsn + 1, &d.blkptr);
    rc |= upload<long long, int64_t>(s, D->updptr, nsn + 1, &d.updptr);
    rc |= upload<double, double>(s, D->wdot, D->nblk, &d.wdot);
    if (rc) return -1;
    s->h_vec2blk.assign(D->nvp, 0);
    for (int64_t i = 0; i < D->nvp; ++i) s->h_vec2blk[i] = (int)D->vec2blk[i];

    // schedules
    const int nt = (int)D->ntask;
    std::vector<int> tp(nt + 1), ts(nsn), dp(nt + 1), di(D->dep_ptr[nt]);
    for (int i = 0; i <= nt; ++i) { tp[i] = (int)D->task_ptr[i]; dp[i] = (int)D->dep_ptr[i]; }
    for (int i = 0; i < nsn; ++i) ts[i] = (int)D->task_sn[i];
    for (size_t i = 0; i < di.size(); ++i) di[i] = (int)D->dep_idx[i];
    if (upload_sched(s, nt, tp, ts, dp, di, &s->up)) return -1;
    // top-down: reversed task order, reversed supernode order, dependency = parent's task
    std::vector<int> task_of(nsn);
    for (int t = 0; t < nt; ++t)
        for (int p = tp[t]; p < tp[t + 1]; ++p) task_of[ts[p]] = t;
    std::vector<int> tp2(nt + 1), ts2(nsn), dp2(nt + 1), di2;
    tp2[0] = 0; dp2[0] = 0;
    for (int t2 = 0; t2 < nt; ++t2) {
        int t = nt - 1 - t2;
        int len = tp[t + 1] - tp[t];
        for (int p = 0; p < len; ++p) ts2[tp2[t2] + p] = ts[tp[t + 1] - 1 - p];
        tp2[t2 + 1] = tp2[t2] + len;
        int top = ts[tp[t + 1] - 1];
        int64_t par = D->snpar[top];
        if (par >= 0) di2.push_back(nt - 1 - task_of[par]);
        dp2[t2 + 1] = (int)di2.size();
    }
    if (upload_sched(s, nt, tp2, ts2, dp2, di2, &s->down)) return -1;
    std::vector<int> tp3(nsn + 1), ts3(nsn), dp3(nsn + 1, 0), di3;
    for (int i = 0; i <= nsn; ++i) tp3[i] = i;
    for (int i = 0; i < nsn; ++i) ts3[i] = i;
    if (upload_sched(s, nsn, tp3, ts3, dp3, di3, &s->flat)) return -1;
    s->max_nj_small = s->max_nj;
    // large frontal matrices: dense multi-CTA path; an explicit SMCP_B200_BIG_NJ also applies to
    // tiny-clique patterns (tests), which then stay on the CTA-per-supernode kernels
    if ((s->max_nj > 8 || getenv("SMCP_B200_BIG_NJ")) && big_setup(s, D)) return -1;
    // tiny cliques: warp-per-chain kernels (SMCP_B200_NO_SMALL=1 forces the CTA kernels)
    if (s->max_nj <= 8 && s->big.empty() && !getenv("SMCP_B200_NO_SMALL") && small_setup(s, D, tp, ts, tp2, ts2)) return -1;

    CUDA_TRY(cudaMalloc(&s->counter, 64));
    CUDA_TRY(cudaMemset(s->counter, 0, 64));
    if (sym_ensure(s, 1, true)) return -1;
    *out = s;
    return 0;
}

extern "C" int smcp_sym_destroy(smcp_sym *s) {
    if (!s) return 0;
    cudaStreamSynchronize(s->ctx->stream);
    for (cudaStream_t st : s->thin_side) { cudaStreamSynchronize(st); cudaStreamDestroy(st); }
    for (cudaEvent_t e : s->thin_ev) cudaEventDestroy(e);
    if (s->tree_side) { cudaStreamSynchronize(s->tree_side); cudaStreamDestroy(s->tree_side); cudaEventDestroy(s->tree_ev[0]); cudaEventDestroy(s->tree_ev[1]); }
    for (void *p : s->allocs) cudaFree(p);
    if (s->counter) cudaFree(s->counter);
    if (s->done) cudaFree(s->done);
    if (s->fail) cudaFree(s->fail);
    if (s->upd) cudaFree(s->upd);
    if (s->cta_ws) cudaFree(s->cta_ws);
    if (s->tmp) cudaFree(s->tmp);
    if (s->red) cudaFree(s->red);
    if (s->fbuf) cudaFree(s->fbuf);
    if (s->ch_state) cudaFree(s->ch_state);
    if (s->probe_buf) cudaFree(s->probe_buf);
    if (s->big_bws) cudaFree(s->big_bws);
    if (s->big_hinv) cudaFree(s->big_hinv);
    if (s->big_cat) cudaFree(s->big_cat);
    for (auto &b : s->hess_pool) {
        cudaFree(b.Lt); cudaFree(b.Yaa); cudaFree(b.Raa);
        if (b.phi) cudaFree(b.phi);
    }
    delete s;
    return 0;
}

// ---------------------------------------------------------------------------------------
// chordal matrices
// ---------------------------------------------------------------------------------------
extern "C" int smcp_csp_alloc(smcp_sym *s, int64_t count, double **dev_out) {
    size_t bytes = (size_t)count * s->d.nblk * sizeof(double);
    CUDA_TRY(cudaMalloc((void **)dev_out, bytes ? bytes : 8));
    CUDA_TRY(cudaMemsetAsync(*dev_out, 0, bytes, s->ctx->stream));
    return 0;
}
extern "C" int smcp_csp_free(smcp_sym *s, double *dev) {
    (void)s;
    if (dev) CUDA_TRY(cudaFree(dev));
    return 0;
}
extern "C" int smcp_csp_copy(smcp_sym *s, double *dst, const double *src, int64_t count) {
    CUDA_TRY(cudaMemcpyAsync(dst, src, (size_t)count * s->d.nblk * sizeof(double), cudaMemcpyDeviceToDevice, s->ctx->stream));
    return 0;
}

static int stage_buf(smcp_sym *s, size_t bytes, double **out) {
    // device staging area for host vectors (reuses the reduction scratch)
    if (grow((void **)&s->red, &s->red_cap, bytes + 4096)) return -1;
    *out = s->red;
    return 0;
}

extern "C" int smcp_csp_from_vec(smcp_sym *s, double *dst, const double *host_vec) {
    double *dv;
    if (stage_buf(s, (size_t)s->d.nvp * sizeof(double), &dv)) return -1;
    CUDA_TRY(cudaMemcpyAsync(dv, host_vec, (size_t)s->d.nvp * sizeof(double), cudaMemcpyHostToDevice, s->ctx->stream));
    if (k_scatter_vec(s, dst, dv)) return -1;
    CUDA_TRY(cudaStreamSynchronize(s->ctx->stream));   // host_vec may be pageable / reused
    return 0;
}
extern "C" int smcp_csp_to_vec(smcp_sym *s, const double *src, double *host_vec) {
    double *dv;
    if (stage_buf(s, (size_t)s->d.nvp * sizeof(double), &dv)) return -1;
    if (k_gather_vec(s, src, dv)) return -1;
    CUDA_TRY(cudaMemcpyAsync(host_vec, dv, (size_t)s->d.nvp * sizeof(double), cudaMemcpyDeviceToHost, s->ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(s->ctx->stream));
    return 0;
}
extern "C" int smcp_csp_get(smcp_sym *s, const double *src, double *host_blk) {
    CUDA_TRY(cudaMemcpyAsync(host_blk, src, (size_t)s->d.nblk * sizeof(double), cudaMemcpyDeviceToHost, s->ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(s->ctx->stream));
    return 0;
}
extern "C" int smcp_csp_set(smcp_sym *s, double *dst, const double *host_blk) {
    CUDA_TRY(cudaMemcpyAsync(dst, host_blk, (size_t)s->d.nblk * sizeof(double), cudaMemcpyHostToDevice, s->ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(s->ctx->stream));
    return 0;
}
extern "C" int smcp_csp_axpy(smcp_sym *s, double a, const double *x, double *y) { return k_axpy(s, a, x, y, s->d.nblk); }
extern "C" int smcp_csp_scal(smcp_sym *s, double a, double *x) { return k_scal(s, a, x, s->d.nblk); }
extern "C" int smcp_csp_dot(smcp_sym *s, const double *x, const double *y, double *out) { return k_dot(s, x, y, out); }
extern "C" int smcp_csp_sumlogdiag(smcp_sym *s, const double *x, double *out) { return k_sumlogdiag(s, x, 1, out); }
extern "C" int smcp_csp_cholesky(smcp_sym *s, double *x, int64_t batch, int32_t *info) { return k_cholesky(s, x, batch, info); }
extern "C" int smcp_csp_completion(smcp_sym *s, double *x, int64_t batch, int32_t *info) { return k_completion(s, x, batch, info); }
extern "C" int smcp_csp_projected_inverse(smcp_sym *s, double *x, int64_t batch) { return k_projinv(s, x, batch); }
extern "C" int smcp_csp_llt(smcp_sym *s, double *x, int64_t batch) { return k_llt(s, x, batch); }


extern "C" int smcp_sym_reserve(smcp_sym *s, int64_t batch) {
    if (batch < 1) return 0;
    if (sym_ensure(s, batch, true)) return -1;
    if (grow((void **)&s->probe_buf, &s->probe_cap, ((size_t)batch * s->d.nblk + batch + 16) * sizeof(double))) return -1;
    if (grow((void **)&s->red, &s->red_cap, ((size_t)batch * 40 + 1024) * sizeof(double) + (size_t)s->d.nvp * sizeof(double) + 4096)) return -1;
    return 0;
}

extern "C" int smcp_csp_probe(smcp_sym *s, int kind, const double *x, const double *dx, const double *gammas_host,
                              int64_t count, int32_t *info_host, double *sumlogdiag_host) {
    smcp_ctx *ctx = s->ctx;
    if (count <= 0) return 0;
    if (grow((void **)&s->probe_buf, &s->probe_cap, ((size_t)count * s->d.nblk + count + 16) * sizeof(double))) return -1;
    double *gam = s->probe_buf + (size_t)count * s->d.nblk;
    CUDA_TRY(cudaMemcpyAsync(gam, gammas_host, (size_t)count * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    if (k_axpy_batch(s, x, dx, gam, s->probe_buf, count)) return -1;
    int rc = kind == 0 ? k_cholesky(s, s->probe_buf, count, info_host) : k_completion(s, s->probe_buf, count, info_host);
    if (rc) return rc;
    if (sumlogdiag_host) return k_sumlogdiag(s, s->probe_buf, count, sumlogdiag_host);
    return 0;
}

extern "C" int smcp_csp_trsm(smcp_sym *s, const double *L, double *B_dev, int64_t ldb, int64_t nrhs, int trans) {
    return k_trsm(s, L, B_dev, ldb, nrhs, trans);
}
extern "C" int smcp_csp_sample(smcp_sym *s, const double *L, uint64_t seed, int64_t col0, double *B_dev, int64_t ldb, int64_t k) {
    return k_sample(s, L, seed, col0, B_dev, ldb, k);
}
extern "C" int smcp_round_pm1(smcp_sym *s, const double *L, uint64_t seed, int64_t trials, int64_t chunk, int64_t nc,
                              const int64_t *crow, const int64_t *ccol, const double *cval, double *values_host, int8_t *x_host,
                              int64_t *best_out) {
    return k_round_pm1(s, L, seed, trials, chunk, nc, crow, ccol, cval, values_host, x_host, best_out);
}
extern "C" int smcp_round_pm1_ls(smcp_sym *s, const double *L, uint64_t seed, int64_t trials, int64_t chunk, int64_t nc,
                                 const int64_t *crow, const int64_t *ccol, const double *cval, int64_t max_flips, double tol,
                                 double *values0_host, double *values_host, int8_t *x_host, int64_t *best_out, int64_t *flips_host) {
    return k_round_pm1_ls(s, L, seed, trials, chunk, nc, crow, ccol, cval, max_flips, tol, values0_host, values_host, x_host,
                          best_out, flips_host);
}
extern "C" int smcp_pm1_local_search(smcp_ctx *ctx, int64_t n, int64_t k, int8_t *x_host, int64_t nc, const int64_t *crow,
                                     const int64_t *ccol, const double *cval, int64_t max_flips, double tol, double *values_host,
                                     int64_t *flips_host) {
    return k_pm1_local_search(ctx, n, k, x_host, nc, crow, ccol, cval, max_flips, tol, values_host, flips_host);
}
extern "C" int smcp_round_pm1_tabu(smcp_sym *s, const double *L, uint64_t seed, int64_t trials, int64_t chunk, int64_t nc,
                                   const int64_t *crow, const int64_t *ccol, const double *cval, int64_t max_flips, double tol,
                                   double *values0_host, double *values_host, int8_t *x_host, int64_t *best_out, int64_t *flips_host,
                                   int64_t tabu_iters, int64_t tenure, double *values1_host, int64_t *moves_host,
                                   int64_t *best_iter_host) {
    return k_round_pm1_tabu(s, L, seed, trials, chunk, nc, crow, ccol, cval, max_flips, tol, values0_host, values_host, x_host,
                            best_out, flips_host, tabu_iters, tenure, values1_host, moves_host, best_iter_host);
}
extern "C" int smcp_pm1_tabu_search(smcp_ctx *ctx, int64_t n, int64_t k, int8_t *x_host, int64_t nc, const int64_t *crow,
                                    const int64_t *ccol, const double *cval, int64_t iters, int64_t tenure, double *values_host,
                                    int64_t *moves_host, int64_t *best_iter_host) {
    return k_pm1_tabu_search(ctx, n, k, x_host, nc, crow, ccol, cval, iters, tenure, values_host, moves_host, best_iter_host);
}
extern "C" int smcp_lowrank_solve(smcp_ctx *ctx, int64_t n, int64_t r, int64_t nc, const int64_t *crow, const int64_t *ccol,
                                  const double *cval, const double *b, uint64_t seed, int64_t max_sweeps, double tol,
                                  double *V_host, double *f_host, double *y_host, int64_t *sweeps_out, int64_t *colors_out) {
    return k_lowrank_solve(ctx, n, r, nc, crow, ccol, cval, b, seed, max_sweeps, tol, V_host, f_host, y_host, sweeps_out,
                           colors_out);
}
extern "C" int smcp_round_pm1_factor(smcp_ctx *ctx, int64_t n, int64_t r, const double *V_host, uint64_t seed, int64_t trials,
                                     int64_t chunk, int64_t nc, const int64_t *crow, const int64_t *ccol, const double *cval,
                                     int64_t max_flips, double tol, int64_t tabu_iters, int64_t tenure, double *values0_host,
                                     double *values1_host, double *values_host, int8_t *x_host, int64_t *best_out,
                                     int64_t *flips_host, int64_t *moves_host, int64_t *best_iter_host) {
    return k_round_pm1_factor(ctx, n, r, V_host, seed, trials, chunk, nc, crow, ccol, cval, max_flips, tol, tabu_iters, tenure,
                              values0_host, values1_host, values_host, x_host, best_out, flips_host, moves_host, best_iter_host);
}

// ---------------------------------------------------------------------------------------
// Hessian factor
// ---------------------------------------------------------------------------------------
extern "C" int smcp_hess_create(smcp_sym *s, const double *L, const double *Y, smcp_hess **out) {
    smcp_hess *h = new smcp_hess();
    h->sym = s;
    h->L = L;
    if (!s->hess_pool.empty()) {
        const smcp_sym::HessBufs b = s->hess_pool.back();
        s->hess_pool.pop_back();
        h->Lt = b.Lt; h->Yaa = b.Yaa; h->Raa = b.Raa; h->phi_up = b.phi;      // phi is refilled by chain_prepare
    } else {
        CUDA_TRY(cudaMalloc(&h->Lt, (size_t)(s->d.nblk + 1) * sizeof(double)));
        CUDA_TRY(cudaMalloc(&h->Yaa, (size_t)(s->d.nupd + 1) * sizeof(double)));
        CUDA_TRY(cudaMalloc(&h->Raa, (size_t)(s->d.nupd + 1) * sizeof(double)));
    }
    if (k_hess_prep(h, L, Y)) return -1;
    *out = h;
    return 0;
}
extern "C" int smcp_hess_destroy(smcp_hess *h) {
    if (!h) return 0;
    smcp_sym *s = h->sym;
    if (s->hess_pool.size() < 4) {
        // work still queued on the stream may read these buffers; the next owner writes them in stream order
        s->hess_pool.push_back({h->Lt, h->Yaa, h->Raa, h->phi_up});
    } else {
        cudaStreamSynchronize(s->ctx->stream);
        cudaFree(h->Lt);
        cudaFree(h->Yaa);
        cudaFree(h->Raa);
        if (h->phi_up) cudaFree(h->phi_up);      // one allocation: phi_up | phi_dn | psi_up | psi_dn
    }
    delete h;
    return 0;
}
extern "C" int smcp_hess_apply(smcp_hess *h, double *U, int64_t batch, int inv) { return k_hess_apply(h, U, batch, inv); }
extern "C" int smcp_hess_apply_half(smcp_hess *h, double *U, int64_t batch, int inv, int adj) { return k_hess_apply_half(h, U, batch, inv, adj); }

// ---------------------------------------------------------------------------------------
// constraint operator, Schur complement
// ---------------------------------------------------------------------------------------
struct smcp_op {
    smcp_sym *sym = nullptr;
    int64_t m = 0, Ns = 0, md = 0, nnz = 0;
    // CSC (rows = blkval offsets)
    long long *colptr = nullptr;
    int *rowblk = nullptr;
    double *vals = nullptr, *valsw = nullptr;
    int *ent_r = nullptr, *ent_c = nullptr;      // internal (row, col) of each entry
    // sparse-constraint technique, position form: the distinct (row, col) positions touched by the
    // sparse columns, and for every entry of a sparse column the index of its position
    int *pos_r = nullptr, *pos_c = nullptr, *sp_pid = nullptr;
    int npos = 0;
    long long sp_base = 0;        // first entry of the first sparse column
    double sp_avg_nnz = 0.0;
    double *ell_val = nullptr;       // sparse constraints in column-major ELL form (entry q of constraint md + i at [q * ms + i]):
    int *ell_pid = nullptr;          //   coalesced row walk of the position kernels; null when the row lengths are too uneven
    int ell_w = 0;                   // entries per row (max nnz)
    double *Kpos = nullptr;          // materialised position kernel matrix (scm_kmat_kernel), ldk x npos
    size_t Kpos_cap = 0;
    bool Kpos_valid = false;         // built from the current Zinv
    // CSR over blkval rows
    long long *r_ptr = nullptr;
    int *r_col = nullptr;
    double *r_val = nullptr;
    // dense weighted copy w.Av (nblk x m) for the DMMA assembly (only if md > 0)
    double *AvW = nullptr;
    // ... or, when few rows of blkval are touched by any constraint (filled patterns), the same copy on
    // those rows only: AvWs (lds x m, lds = nsup rounded up to even) on the sorted support rows sup[0..nsup),
    // srow[p] = position of rowblk[p] in sup.  Exactly one of AvW / AvWs is set when md > 0.
    double *AvWs = nullptr;
    int *sup = nullptr, *srow = nullptr;
    long long nsup = 0, lds = 0;
    double *Ubs = nullptr;        // Hessian batch gathered onto the support rows (lds x ncols)
    size_t Ubs_cap = 0;
    double *H = nullptr;
    int *info_dev = nullptr;
    double *yv = nullptr;
    double *Ub = nullptr;
    size_t Ub_cap = 0;
    double *Zinv = nullptr;       // n x n dense inverse for the sparse-constraint technique
    double *Zq = nullptr;         // kktsolver='qr': Z = [G(A_1) ... G(A_m)] weighted by sqrt(wdot), nblk x m
    int zq_state = 0;             // what Zq holds: 0 nothing, 1 Zw (SYRK form), 2 Q1 of Zw = Q1 R (Householder form)
    double *qr_tau = nullptr;     // Householder form: tau (m), signs of diag(R) (m), right-hand side r (m)
    double *sqrtw = nullptr;      // sqrt of the trace inner-product weights (nblk)
    double *Dinv = nullptr;       // inverses of the 64 x 64 diagonal blocks of chol(H) (potrs)
    std::vector<long long> h_colptr;
    void *allocs[16] = {0};
};

__global__ void amap_kernel(const long long *__restrict__ colptr, const int *__restrict__ rowblk,
                            const double *__restrict__ valsw, const double *__restrict__ X, double *out,
                            long long col0, int ncols) {
    int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    int lane = threadIdx.x & 31;
    if (w >= ncols) return;
    long long c = col0 + w;
    double s = 0.0;
    for (long long p = colptr[c] + lane; p < colptr[c + 1]; p += 32) s = fma(valsw[p], X[rowblk[p]], s);
    for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
    if (lane == 0) out[w] = s;
}

// dense variant for (nearly) dense Av: column c of the weighted dense copy AvW is contiguous, one CTA
// per column streams it once (coalesced 8-byte loads, 4 independent accumulators per thread) against
// X, which stays in L2; fixed reduction tree -> deterministic.  SUP: the copy holds the support rows
// only (AvWs, column stride lda), row r of it multiplies X[sup[r]].
template <bool SUP>
__global__ void __launch_bounds__(256) amap_dense_kernel(const double *__restrict__ AvW, long long lda, long long nblk,
                                                         const int *__restrict__ sup, const double *__restrict__ X,
                                                         double *out, long long col0) {
    const double *a = AvW + (col0 + blockIdx.x) * lda;
    auto x = [&](long long r) { return SUP ? X[sup[r]] : X[r]; };
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    long long r = threadIdx.x;
    for (; r + 768 < nblk; r += 1024) {
        s0 = fma(a[r], x(r), s0);
        s1 = fma(a[r + 256], x(r + 256), s1);
        s2 = fma(a[r + 512], x(r + 512), s2);
        s3 = fma(a[r + 768], x(r + 768), s3);
    }
    for (; r < nblk; r += 256) s0 = fma(a[r], x(r), s0);
    double s = (s0 + s1) + (s2 + s3);
    __shared__ double sh[8];
    for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x < 32) {
        double v = threadIdx.x < 8 ? sh[threadIdx.x] : 0.0;
        for (int o = 4; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
        if (threadIdx.x == 0) out[blockIdx.x] = v;
    }
}

__global__ void aadj_kernel(const long long *__restrict__ r_ptr, const int *__restrict__ r_col,
                            const double *__restrict__ r_val, const double *__restrict__ y, double *X, int nrows) {
    int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    int lane = threadIdx.x & 31;
    if (w >= nrows) return;
    double s = 0.0;
    for (long long p = r_ptr[w] + lane; p < r_ptr[w + 1]; p += 32) s = fma(r_val[p], y[r_col[p]], s);
    for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
    if (lane == 0) X[w] = s;
}

__global__ void scatter_cols_kernel(const long long *__restrict__ colptr, const int *__restrict__ rowblk,
                                    const double *__restrict__ vals, double *U, long long ldu, long long c0, int ncols) {
    // one CTA per column
    int c = blockIdx.x;
    if (c >= ncols) return;
    double *u = U + (long long)c * ldu;
    for (long long p = colptr[c0 + c] + threadIdx.x; p < colptr[c0 + c + 1]; p += blockDim.x) u[rowblk[p]] = vals[p];
}

// as scatter_cols_kernel onto the support rows (compact row srow[p]), each value times scale[rowblk[p]] if scale is set
__global__ void scatter_support_kernel(const long long *__restrict__ colptr, const int *__restrict__ srow,
                                       const int *__restrict__ rowblk, const double *__restrict__ vals,
                                       const double *__restrict__ scale, double *U, long long ldu, long long c0, int ncols) {
    int c = blockIdx.x;
    if (c >= ncols) return;
    double *u = U + (long long)c * ldu;
    for (long long p = colptr[c0 + c] + threadIdx.x; p < colptr[c0 + c + 1]; p += blockDim.x)
        u[srow[p]] = scale ? vals[p] * scale[rowblk[p]] : vals[p];
}

// Ubs[k + j lds] = Ub[sup[k] + j nblk] for k < nsup, 0 on the padding rows k in [nsup, lds)
__global__ void support_gather_kernel(const double *__restrict__ Ub, long long nblk, const int *__restrict__ sup, long long nsup,
                                      long long lds, double *__restrict__ Ubs, long long ncols) {
    const long long total = lds * ncols;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const long long k = idx % lds, j = idx / lds;
        Ubs[idx] = k < nsup ? Ub[sup[k] + j * nblk] : 0.0;
    }
}

template <class T>
static int dev_upload(const std::vector<T> &v, T **out) {
    size_t n = v.size() ? v.size() : 1;
    CUDA_TRY(cudaMalloc((void **)out, n * sizeof(T)));
    if (v.size()) CUDA_TRY(cudaMemcpy(*out, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
    return 0;
}

extern "C" int smcp_op_create(smcp_sym *s, int64_t m, int64_t Ns, const int64_t *colptr, const int64_t *rowind,
                              const double *values, smcp_op **out) {
    smcp_ctx *ctx = s->ctx;
    CUDA_TRY(cudaSetDevice(ctx->device));
    smcp_op *op = new smcp_op();
    op->sym = s;
    op->m = m;
    op->Ns = Ns;
    op->md = m - Ns;
    const int64_t nnz = colptr[m];
    op->nnz = nnz;
    const int nblk = s->d.nblk;
    std::vector<long long> cp(m + 1);
    for (int64_t i = 0; i <= m; ++i) cp[i] = colptr[i];
    op->h_colptr = cp;
    std::vector<int> rb(nnz);
    std::vector<double> wd(nblk);
    CUDA_TRY(cudaMemcpy(wd.data(), s->d.wdot, (size_t)nblk * sizeof(double), cudaMemcpyDeviceToHost));
    std::vector<double> vw(nnz);
    for (int64_t p = 0; p < nnz; ++p) {
        rb[p] = s->h_vec2blk[rowind[p]];
        vw[p] = values[p] * wd[rb[p]];
    }
    // CSR over blkval rows (deterministic: columns ascending inside each row)
    std::vector<long long> rp(nblk + 1, 0);
    for (int64_t p = 0; p < nnz; ++p) rp[rb[p] + 1]++;
    for (int i = 0; i < nblk; ++i) rp[i + 1] += rp[i];
    std::vector<int> rc(nnz);
    std::vector<double> rv(nnz);
    {
        std::vector<long long> fill(rp.begin(), rp.end() - 1);
        for (int64_t c = 0; c < m; ++c)
            for (int64_t p = colptr[c]; p < colptr[c + 1]; ++p) {
                long long q = fill[rb[p]]++;
                rc[q] = (int)c;
                rv[q] = values[p];
            }
    }
    std::vector<double> vals(values, values + nnz);
    if (dev_upload(cp, &op->colptr) || dev_upload(rb, &op->rowblk) || dev_upload(vals, &op->vals) ||
        dev_upload(vw, &op->valsw) || dev_upload(rp, &op->r_ptr) || dev_upload(rc, &op->r_col) ||
        dev_upload(rv, &op->r_val))
        return -1;
    CUDA_TRY(cudaMalloc(&op->H, (size_t)std::max<int64_t>(m * m, 1) * sizeof(double)));
    CUDA_TRY(cudaMemset(op->H, 0, (size_t)std::max<int64_t>(m * m, 1) * sizeof(double)));
    CUDA_TRY(cudaMalloc(&op->info_dev, 64));
    CUDA_TRY(cudaMalloc(&op->yv, (size_t)(m + 1) * sizeof(double)));
    CUDA_TRY(cudaMalloc(&op->Dinv, (size_t)((m + 63) / 64 + 1) * 64 * 64 * sizeof(double)));
    // rows of blkval that some constraint touches (all m columns: the rows of H below the dense block come from
    // the same product); the dense copy keeps only those when they are at most a quarter of blkval.
    // SMCP_B200_AVW_SUPPORT=0 / =1 forces the full / the support copy.
    bool support = false;
    std::vector<int> sup, srow;
    if (op->md > 0) {
        std::vector<int> cidx(nblk, -1);
        for (int64_t p = 0; p < nnz; ++p) cidx[rb[p]] = 0;
        for (int r = 0; r < nblk; ++r)
            if (cidx[r] == 0) { cidx[r] = (int)sup.size(); sup.push_back(r); }
        const char *env = getenv("SMCP_B200_AVW_SUPPORT");
        const int mode = env && !strcmp(env, "0") ? 0 : env && !strcmp(env, "1") ? 1 : -1;
        support = !sup.empty() && (mode == 1 || (mode == -1 && (double)sup.size() <= 0.25 * (double)nblk));
        if (support) {
            srow.resize(nnz);
            for (int64_t p = 0; p < nnz; ++p) srow[p] = cidx[rb[p]];
        }
    }
    if (support) {
        op->nsup = (long long)sup.size();
        op->lds = (op->nsup + 1) & ~1LL;          // even: 16-byte aligned columns for the TMA operand path
        if (dev_upload(sup, &op->sup) || dev_upload(srow, &op->srow)) return -1;
        size_t bytes = (size_t)op->lds * (size_t)m * sizeof(double);
        CUDA_TRY(cudaMalloc(&op->AvWs, bytes));
        CUDA_TRY(cudaMemsetAsync(op->AvWs, 0, bytes, ctx->stream));
        LaunchScope ls(ctx, "setup");
        scatter_support_kernel<<<(unsigned)m, 128, 0, ctx->stream>>>(op->colptr, op->srow, op->rowblk, op->valsw, nullptr, op->AvWs,
                                                                     op->lds, 0, (int)m);
    } else if (op->md > 0) {
        // dense weighted copy of all m columns (rows of H below the dense block included)
        size_t bytes = (size_t)nblk * (size_t)m * sizeof(double);
        CUDA_TRY(cudaMalloc(&op->AvW, bytes));
        CUDA_TRY(cudaMemsetAsync(op->AvW, 0, bytes, ctx->stream));
        LaunchScope ls(ctx, "setup");
        scatter_cols_kernel<<<(unsigned)m, 128, 0, ctx->stream>>>(op->colptr, op->rowblk, op->valsw, op->AvW, nblk, 0, (int)m);
    }
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    *out = op;
    return 0;
}

__global__ void scm_ell_build_kernel(const long long *__restrict__ colptr, const double *__restrict__ vals, const int *__restrict__ sp_pid,
                                     long long sp_base, long long md, long long ms, int ell_w, double *__restrict__ ell_val,
                                     int *__restrict__ ell_pid);
// (row, col) in the internal order of every entry of Av, needed by the sparse technique
extern "C" int smcp_op_set_entry_coords(smcp_op *op, const int64_t *rows_int, const int64_t *cols_int) {
    std::vector<int> r(op->nnz), c(op->nnz);
    for (int64_t p = 0; p < op->nnz; ++p) { r[p] = (int)rows_int[p]; c[p] = (int)cols_int[p]; }
    if (dev_upload(r, &op->ent_r) || dev_upload(c, &op->ent_c)) return -1;
    // positions touched by the sparse columns [md, m), sorted by (col, row) so that consecutive
    // positions share their column (shared-memory broadcasts in scm_position_kernel)
    const int64_t p0 = op->h_colptr[op->md], p1 = op->h_colptr[op->m];
    op->sp_base = p0;
    if (p1 > p0) {
        const int64_t n = op->sym->d.n;
        std::vector<std::pair<int64_t, int64_t>> key((size_t)(p1 - p0));
        for (int64_t p = p0; p < p1; ++p) key[(size_t)(p - p0)] = {(int64_t)c[p] * n + r[p], p - p0};
        std::sort(key.begin(), key.end());
        std::vector<int> pid((size_t)(p1 - p0)), pr, pc;
        int64_t last = -1;
        for (auto &kv : key) {
            if (kv.first != last) {
                last = kv.first;
                pr.push_back((int)(kv.first % n));
                pc.push_back((int)(kv.first / n));
            }
            pid[(size_t)kv.second] = (int)pr.size() - 1;
        }
        op->npos = (int)pr.size();
        op->sp_avg_nnz = (double)(p1 - p0) / (double)std::max<int64_t>(1, op->m - op->md);
        if (dev_upload(pid, &op->sp_pid) || dev_upload(pr, &op->pos_r) || dev_upload(pc, &op->pos_c)) return -1;
        // ELL copy of the sparse constraints for the coalesced row walk, unless the row lengths are too uneven
        const int64_t ms = op->m - op->md;
        int64_t w = 0;
        for (int64_t i = op->md; i < op->m; ++i) w = std::max<int64_t>(w, op->h_colptr[i + 1] - op->h_colptr[i]);
        if (w > 0 && (double)w <= 2.0 * op->sp_avg_nnz + 8.0 && (size_t)w * ms * 12 <= ((size_t)2 << 30)) {
            smcp_ctx *ctx = op->sym->ctx;
            CUDA_TRY(cudaMalloc(&op->ell_val, (size_t)w * ms * sizeof(double)));
            CUDA_TRY(cudaMalloc(&op->ell_pid, (size_t)w * ms * sizeof(int)));
            op->ell_w = (int)w;
            LaunchScope ls(ctx, "setup");
            scm_ell_build_kernel<<<(unsigned)std::min<int64_t>((w * ms + 255) / 256, 4096), 256, 0, ctx->stream>>>(
                op->colptr, op->vals, op->sp_pid, op->sp_base, op->md, ms, (int)w, op->ell_val, op->ell_pid);
            CUDA_TRY(cudaGetLastError());
            CUDA_TRY(cudaStreamSynchronize(ctx->stream));
        }
    }
    return 0;
}

extern "C" int smcp_op_destroy(smcp_op *op) {
    if (!op) return 0;
    cudaStreamSynchronize(op->sym->ctx->stream);
    cudaFree(op->colptr); cudaFree(op->rowblk); cudaFree(op->vals); cudaFree(op->valsw);
    cudaFree(op->r_ptr); cudaFree(op->r_col); cudaFree(op->r_val);
    if (op->ent_r) cudaFree(op->ent_r);
    if (op->sp_pid) { cudaFree(op->sp_pid); cudaFree(op->pos_r); cudaFree(op->pos_c); }
    if (op->ent_c) cudaFree(op->ent_c);
    if (op->AvW) cudaFree(op->AvW);
    if (op->AvWs) { cudaFree(op->AvWs); cudaFree(op->sup); cudaFree(op->srow); }
    if (op->Ubs) cudaFree(op->Ubs);
    if (op->Ub) cudaFree(op->Ub);
    if (op->Zinv) cudaFree(op->Zinv);
    if (op->Kpos) cudaFree(op->Kpos);
    if (op->ell_val) { cudaFree(op->ell_val); cudaFree(op->ell_pid); }
    if (op->Zq) cudaFree(op->Zq);
    if (op->qr_tau) cudaFree(op->qr_tau);
    if (op->sqrtw) cudaFree(op->sqrtw);
    if (op->Dinv) cudaFree(op->Dinv);
    cudaFree(op->H); cudaFree(op->info_dev); cudaFree(op->yv);
    delete op;
    return 0;
}

extern "C" int smcp_op_amap(smcp_op *op, const double *X, int64_t col, double *host_out) {
    smcp_ctx *ctx = op->sym->ctx;
    int64_t c0 = col >= 0 ? col : 0;
    int ncols = col >= 0 ? 1 : (int)op->m;
    if (ncols == 0) return 0;
    if (op->AvW && op->nnz * 4 >= (int64_t)op->sym->d.nblk * op->m) {
        LaunchScope ls(ctx, "amap_dense", 1, 8.0 * (double)op->sym->d.nblk * ncols);
        amap_dense_kernel<false><<<ncols, 256, 0, ctx->stream>>>(op->AvW, op->sym->d.nblk, op->sym->d.nblk, nullptr, X, op->yv, c0);
    } else if (op->AvWs && op->nnz * 4 >= op->nsup * op->m) {
        LaunchScope ls(ctx, "amap_dense", 1, 12.0 * (double)op->nsup * ncols);
        amap_dense_kernel<true><<<ncols, 256, 0, ctx->stream>>>(op->AvWs, op->lds, op->nsup, op->sup, X, op->yv, c0);
    } else {
        LaunchScope ls(ctx, "amap", 1, 12.0 * (double)(op->h_colptr[c0 + ncols] - op->h_colptr[c0]));
        amap_kernel<<<(ncols * 32 + 255) / 256, 256, 0, ctx->stream>>>(op->colptr, op->rowblk, op->valsw, X, op->yv, c0, ncols);
    }
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(host_out, op->yv, (size_t)ncols * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return 0;
}

extern "C" int smcp_op_dense_rows(smcp_op *op, int64_t *rows_out) {
    *rows_out = op->AvWs ? op->nsup : op->AvW ? op->sym->d.nblk : 0;
    return 0;
}

extern "C" int smcp_op_aadj(smcp_op *op, const double *host_y, double *X) {
    smcp_ctx *ctx = op->sym->ctx;
    CUDA_TRY(cudaMemcpyAsync(op->yv, host_y, (size_t)op->m * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    int nrows = op->sym->d.nblk;
    {
        LaunchScope ls(ctx, "aadj", 1, 12.0 * (double)op->nnz);
        aadj_kernel<<<(unsigned)(((long long)nrows * 32 + 255) / 256), 256, 0, ctx->stream>>>(op->r_ptr, op->r_col, op->r_val, op->yv, X, nrows);
    }
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));   // host_y may be reused by the caller
    return 0;
}

// sparse-constraint technique (solvers.py:489-497 + misc.c:620-663) on the dense inverse
// Z = S^{-1} (internal order): H[i, j] = sum_{(r,c) in A_j} sum_{(r1,c1) in A_i}
//   alpha beta [Z(r1,r) Z(c1,c) + (r1 != c1) Z(c1,r) Z(r1,c)],  alpha doubled off the diagonal.
__global__ void scm_sparse_kernel(const long long *__restrict__ colptr, const double *__restrict__ vals,
                                  const int *__restrict__ er, const int *__restrict__ ec,
                                  const double *__restrict__ Z, long long n, double *H, long long m,
                                  long long j0) {
    long long j = j0 + blockIdx.x;
    long long pj0 = colptr[j], pj1 = colptr[j + 1];
    for (long long i = j + threadIdx.x; i < m; i += blockDim.x) {
        double acc = 0.0;
        for (long long p = pj0; p < pj1; ++p) {
            int r = er[p], c = ec[p];
            double alpha = vals[p] * (r != c ? 2.0 : 1.0);
            const double *Zr = Z + (long long)r * n, *Zc = Z + (long long)c * n;
            double t = 0.0;
            for (long long q = colptr[i]; q < colptr[i + 1]; ++q) {
                int r1 = er[q], c1 = ec[q];
                double beta = vals[q];
                double v = Zr[r1] * Zc[c1];
                if (r1 != c1) v = fma(Zr[c1], Zc[r1], v);
                t = fma(beta, v, t);
            }
            acc = fma(alpha, t, acc);
        }
        H[i + j * m] = acc;
    }
}


// Sparse-constraint technique in POSITION form (same sums as misc.SCMcolumn2, src/C/misc.c:620-663,
// regrouped).  With Z = S^{-1} and the entries (r, c, alpha') of A_j (alpha' doubled off the
// diagonal) define on every position (p, q) that any sparse constraint touches
//     G_j(p, q) = sum_e alpha'_e [ Z(p, r_e) Z(q, c_e) + (p != q) Z(q, r_e) Z(p, c_e) ],
// then H[i, j] = sum_{(p, q, beta) in A_i} beta G_j(p, q).  The pairwise loop of the reference
// costs nnz(A_j) * sum_i nnz(A_i) gathers per column; this form costs npos * nnz(A_j) for G_j plus
// sum_i nnz(A_i) for the products: at m = 10^4, 80 non-zeros per constraint that is 12x fewer
// operations, and all gathers hit shared memory.
// One CTA per column j: the columns r_e, c_e of Z are staged E entries at a time in shared memory,
// every thread keeps KPOS positions in registers; afterwards G_j replaces the staged columns in
// shared memory and the threads walk the rows i >= j.
#define SCM_T 512
// H[i, j] = sum_{(pid, beta) in A_i} beta G_j(pid) for the rows i >= j, G_j in shared memory; one thread per row,
// entries in storage order (the same sums in CSR and ELL form: the ELL padding adds beta = 0 terms)
__device__ __noinline__ void scm_rows(const double *G, const long long *__restrict__ colptr, const double *__restrict__ vals,
                                         const int *__restrict__ sp_pid, long long sp_base, const double *__restrict__ ell_val,
                                         const int *__restrict__ ell_pid, int ell_w, long long md, double *H, long long m, long long j) {
    const long long ms = m - md;
    for (long long i = j + threadIdx.x; i < m; i += SCM_T) {
        double t = 0.0;
        if (ell_val) {
            const double *ev = ell_val + (i - md);
            const int *ep = ell_pid + (i - md);
#pragma unroll 4
            for (int q = 0; q < ell_w; ++q) t = fma(ev[q * ms], G[ep[q * ms]], t);
        } else {
            for (long long q = colptr[i]; q < colptr[i + 1]; ++q) t = fma(vals[q], G[sp_pid[q - sp_base]], t);
        }
        H[i + j * m] = t;
    }
}
__global__ void scm_ell_build_kernel(const long long *__restrict__ colptr, const double *__restrict__ vals, const int *__restrict__ sp_pid,
                                     long long sp_base, long long md, long long ms, int ell_w, double *__restrict__ ell_val,
                                     int *__restrict__ ell_pid) {
    const long long total = ms * ell_w;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const long long i = idx % ms;
        const int q = (int)(idx / ms);
        const long long p = colptr[md + i] + q;
        const bool live = p < colptr[md + i + 1];
        ell_val[idx] = live ? vals[p] : 0.0;
        ell_pid[idx] = live ? sp_pid[p - sp_base] : 0;
    }
}

template <int KPOS>
__global__ void __launch_bounds__(SCM_T, 1)
scm_position_kernel(const long long *__restrict__ colptr, const double *__restrict__ vals, const int *__restrict__ er,
                    const int *__restrict__ ec, const int *__restrict__ sp_pid, long long sp_base,
                    const int *__restrict__ pos_r, const int *__restrict__ pos_c, int npos, const double *__restrict__ Z,
                    int n, double *H, long long m, long long j0, int E, const double *__restrict__ ell_val,
                    const int *__restrict__ ell_pid, int ell_w, long long md) {
    extern __shared__ double scm_sm[];      // max(2 E n, npos) doubles
    __shared__ double alpha_s[64];
    __shared__ int col_s[128];
    const int tid = threadIdx.x;
    const long long j = j0 + blockIdx.x;
    const long long pj0 = colptr[j], pj1 = colptr[j + 1];
    unsigned prq[KPOS];          // row | col << 16 (n < 65536 is checked on the host)
    double acc[KPOS];
#pragma unroll
    for (int k = 0; k < KPOS; ++k) {
        const int pid = k * SCM_T + tid;
        prq[k] = pid < npos ? ((unsigned)pos_r[pid] | ((unsigned)pos_c[pid] << 16)) : 0u;
        acc[k] = 0.0;
    }
    for (long long e0 = pj0; e0 < pj1; e0 += E) {
        const int ne = (int)min((long long)E, pj1 - e0);
        __syncthreads();
        if (tid < ne) {
            const int r = er[e0 + tid], c = ec[e0 + tid];
            alpha_s[tid] = vals[e0 + tid] * (r != c ? 2.0 : 1.0);
            col_s[2 * tid] = r;
            col_s[2 * tid + 1] = c;
        }
        __syncthreads();
        for (int q = 0; q < 2 * ne; ++q) {
            const double *Zc = Z + (long long)col_s[q] * n;
            for (int i = tid; i < n; i += SCM_T) scm_sm[q * n + i] = Zc[i];
        }
        __syncthreads();
        for (int e = 0; e < ne; ++e) {
            const double al = alpha_s[e];
            const double *zr = scm_sm + 2 * e * n, *zc = zr + n;
#pragma unroll
            for (int k = 0; k < KPOS; ++k) {
                const int p_ = (int)(prq[k] & 0xffffu), q_ = (int)(prq[k] >> 16);
                double v = zr[p_] * zc[q_];
                if (p_ != q_) v = fma(zr[q_], zc[p_], v);
                acc[k] = fma(al, v, acc[k]);
            }
        }
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < KPOS; ++k) {
        const int pid = k * SCM_T + tid;
        if (pid < npos) scm_sm[pid] = acc[k];
    }
    __syncthreads();
    scm_rows(scm_sm, colptr, vals, sp_pid, sp_base, ell_val, ell_pid, ell_w, md, H, m, j);
}


// POSITION form with a materialised kernel matrix.  G_j(p, q) = sum_e alpha'_e K[(p, q), (r_e, c_e)] with
//     K[(p, q), (r, c)] = Z(p, r) Z(q, c) + (p != q) Z(q, r) Z(p, c)
// over the npos positions the sparse constraints touch.  scm_position_kernel recomputes K's entries for
// every constraint entry (4 shared-memory gathers with bank conflicts each: npos * nnz(A) of them, the
// bound of that kernel); here K is built ONCE per scaling point (npos^2 entries, same expressions, so the
// same bits) and column j streams the nnz(A_j) columns of K it needs: coalesced 8-byte loads, HBM bound at
// 8 * npos * nnz(A) bytes in total (rand_SDP n = 2000, m = 10^4: 2 GB for K, 100 GB streamed).
__global__ void __launch_bounds__(SCM_T)
scm_kmat_kernel(const int *__restrict__ pos_r, const int *__restrict__ pos_c, int npos, const double *__restrict__ Z, int n,
                double *__restrict__ K, long long ldk) {
    extern __shared__ double km_sm[];       // Z(:, r) | Z(:, c)
    const int tid = threadIdx.x;
    const int e = blockIdx.x;
    const int r = pos_r[e], c = pos_c[e];
    const double *Zr = Z + (long long)r * n, *Zc = Z + (long long)c * n;
    for (int i = tid; i < n; i += SCM_T) {
        km_sm[i] = Zr[i];
        km_sm[n + i] = Zc[i];
    }
    __syncthreads();
    const double *zr = km_sm, *zc = km_sm + n;
    double *Ke = K + (long long)e * ldk;
    for (int pid = tid; pid < ldk; pid += SCM_T) {
        double v = 0.0;
        if (pid < npos) {
            const int p_ = pos_r[pid], q_ = pos_c[pid];
            v = zr[p_] * zc[q_];
            if (p_ != q_) v = fma(zr[q_], zc[p_], v);
        }
        Ke[pid] = v;
    }
}

template <int KPOS>
__global__ void __launch_bounds__(SCM_T, 1)
scm_kstream_kernel(const long long *__restrict__ colptr, const double *__restrict__ vals, const int *__restrict__ er,
                   const int *__restrict__ ec, const int *__restrict__ sp_pid, long long sp_base, int npos, long long ldk,
                   const double *__restrict__ K, double *H, long long m, long long j0, const double *__restrict__ ell_val,
                   const int *__restrict__ ell_pid, int ell_w, long long md) {
    extern __shared__ double scm_sm[];      // ldk doubles: G_j
    const int tid = threadIdx.x;
    const long long j = j0 + blockIdx.x;
    const long long pj0 = colptr[j], pj1 = colptr[j + 1];
    // thread tid accumulates the positions 2 (k SCM_T + tid) and + 1, k < KPOS / 2 (16-byte loads; ldk is even)
    double2 acc[KPOS / 2];
#pragma unroll
    for (int k = 0; k < KPOS / 2; ++k) acc[k] = make_double2(0.0, 0.0);
    for (long long e = pj0; e < pj1; ++e) {
        const double al = vals[e] * (er[e] != ec[e] ? 2.0 : 1.0);
        const double2 *Ke = reinterpret_cast<const double2 *>(K + (long long)sp_pid[e - sp_base] * ldk) + tid;
        double2 v[KPOS / 2];
#pragma unroll
        for (int k = 0; k < KPOS / 2; ++k) v[k] = (2 * (k * SCM_T + tid) < npos) ? __ldcs(Ke + k * SCM_T) : make_double2(0.0, 0.0);
#pragma unroll
        for (int k = 0; k < KPOS / 2; ++k) {
            acc[k].x = fma(al, v[k].x, acc[k].x);
            acc[k].y = fma(al, v[k].y, acc[k].y);
        }
    }
#pragma unroll
    for (int k = 0; k < KPOS / 2; ++k) {
        const int pid = 2 * (k * SCM_T + tid);
        if (pid < npos) reinterpret_cast<double2 *>(scm_sm)[k * SCM_T + tid] = acc[k];
    }
    __syncthreads();
    scm_rows(scm_sm, colptr, vals, sp_pid, sp_base, ell_val, ell_pid, ell_w, md, H, m, j);
}

// technique 1 on a set of column ranges: ONE batched Hessian over all of them (the chordal kernels
// are latency/issue bound, small batches waste the machine), then one DMMA contraction per range
static int assemble_dense_ranges(smcp_op *op, smcp_hess *h, const std::vector<std::pair<int64_t, int64_t>> &ranges) {
    smcp_sym *s = op->sym;
    smcp_ctx *ctx = s->ctx;
    const int64_t m = op->m;
    const long long nblk = s->d.nblk;
    if (ranges.empty()) return 0;
    // support copy: the Hessian batch is gathered onto the support rows and contracted over K = nsup of them
    const bool support = op->AvWs != nullptr;
    size_t per_col = ((size_t)nblk + (size_t)s->d.nupd + (support ? (size_t)op->lds : 0)) * sizeof(double);
    int64_t cap = (int64_t)std::max<size_t>(1, ((size_t)6 << 30) / per_col);
    cap = std::min<int64_t>(cap, 2048);
    // split ranges that exceed the capacity, then group consecutive pieces up to `cap` columns
    std::vector<std::pair<int64_t, int64_t>> pieces;
    for (auto r : ranges)
        for (int64_t c0 = r.first; c0 < r.second; c0 += cap) pieces.push_back({c0, std::min(r.second, c0 + cap)});
    size_t gi = 0;
    while (gi < pieces.size()) {
        size_t ge = gi;
        int64_t ncols = 0;
        while (ge < pieces.size() && ncols + (pieces[ge].second - pieces[ge].first) <= cap) {
            ncols += pieces[ge].second - pieces[ge].first;
            ++ge;
        }
        if (grow((void **)&op->Ub, &op->Ub_cap, (size_t)ncols * nblk * sizeof(double))) return -1;
        CUDA_TRY(cudaMemsetAsync(op->Ub, 0, (size_t)ncols * nblk * sizeof(double), ctx->stream));
        int64_t off = 0;
        for (size_t q = gi; q < ge; ++q) {
            const int64_t c0 = pieces[q].first, nc = pieces[q].second - c0;
            LaunchScope ls(ctx, "scatter_cols");
            scatter_cols_kernel<<<(unsigned)nc, 128, 0, ctx->stream>>>(op->colptr, op->rowblk, op->vals, op->Ub + (size_t)off * nblk, nblk, c0, (int)nc);
            off += nc;
        }
        if (k_hess_apply(h, op->Ub, ncols, 0)) return -1;
        if (support) {
            if (grow((void **)&op->Ubs, &op->Ubs_cap, (size_t)ncols * op->lds * sizeof(double))) return -1;
            const long long total = (long long)ncols * op->lds;
            LaunchScope ls(ctx, "support_gather", 1, 20.0 * (double)op->nsup * (double)ncols);
            support_gather_kernel<<<(unsigned)std::min<long long>((total + 255) / 256, (long long)ctx->num_sms * 16), 256, 0, ctx->stream>>>(
                op->Ub, nblk, op->sup, op->nsup, op->lds, op->Ubs, ncols);
        }
        off = 0;
        for (size_t q = gi; q < ge; ++q) {
            const int64_t c0 = pieces[q].first, nc = pieces[q].second - c0;
            // H[c0:m, c0:c0+nc] = (w.Av[:, c0:m])^T W
            if (support) {
                if (d_gemm_tn(ctx, op->AvWs + (size_t)c0 * op->lds, op->lds, op->Ubs + (size_t)off * op->lds, op->lds, op->H + c0 + c0 * m, m,
                              m - c0, nc, op->nsup, 0)) return -1;
            } else if (d_gemm_tn(ctx, op->AvW + (size_t)c0 * nblk, nblk, op->Ub + (size_t)off * nblk, nblk, op->H + c0 + c0 * m, m, m - c0, nc, nblk, 0)) return -1;
            off += nc;
        }
        gi = ge;
    }
    return 0;
}

// technique 2: sparse constraints through the dense inverse of S (columns [s0, s1))
__global__ void set_identity_cols_kernel(double *Z, long long n, long long c0, long long c1) {
    long long i = c0 + (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < c1) Z[i + i * n] = 1.0;
}
__global__ void set_identity_kernel(double *Z, long long n) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) Z[i + i * n] = 1.0;
}

// dense inverse of S (internal order) for the sparse-constraint technique.  Several ranks: every rank solves
// for its slice of the columns (equal chunks; the buffer is padded to nranks * chunk columns) and the slices
// are all-gathered over NVLink -- a collective: every rank of the communicator must call it.
static int build_zinv(smcp_op *op, smcp_hess *h, bool sharded) {
    smcp_sym *s = op->sym;
    smcp_ctx *ctx = s->ctx;
    const long long n = s->d.n;
    const int nr = sharded ? ctx->comm_nranks : 1, rk = sharded ? ctx->comm_rank : 0;
    const long long chunk = (n + nr - 1) / nr;
    if (!op->Zinv) CUDA_TRY(cudaMalloc(&op->Zinv, (size_t)n * (size_t)std::max<long long>(chunk * ctx->comm_nranks + 1, n) * sizeof(double)));
    const long long c0 = std::min<long long>(n, rk * chunk), c1 = std::min<long long>(n, c0 + chunk);
    CUDA_TRY(cudaMemsetAsync(op->Zinv + (size_t)rk * chunk * n, 0, (size_t)chunk * n * sizeof(double), ctx->stream));
    if (c1 > c0) {
        {
            LaunchScope ls(ctx, "setup");
            set_identity_cols_kernel<<<(unsigned)((c1 - c0 + 255) / 256), 256, 0, ctx->stream>>>(op->Zinv, n, c0, c1);
        }
        if (k_trsm(s, h->L, op->Zinv + (size_t)c0 * n, n, c1 - c0, 0)) return -1;
        if (k_trsm(s, h->L, op->Zinv + (size_t)c0 * n, n, c1 - c0, 1)) return -1;
    }
    if (nr > 1 && comm_allgather(ctx, op->Zinv, (size_t)chunk * n, ctx->stream)) return -1;
    op->Kpos_valid = false;
    return 0;
}

static int assemble_sparse_range(smcp_op *op, smcp_hess *h, int64_t s0, int64_t s1, bool fresh_inverse) {
    smcp_sym *s = op->sym;
    smcp_ctx *ctx = s->ctx;
    const int64_t m = op->m;
    if (s1 <= s0) return 0;
    if (!op->ent_r) { smcp_set_error("entry coordinates not set (smcp_op_set_entry_coords)"); return -2; }
    const long long n = s->d.n;
    if (fresh_inverse && build_zinv(op, h, false)) return -1;
    // position form when the staged columns of Z fit in shared memory and the constraints are not
    // (almost) single entries; otherwise the pairwise form of the reference
    const long long cap = 25600;                 // doubles of dynamic shared memory (200 KB)
    const int E = (int)std::min<long long>(64, cap / (2 * n));
    if (op->sp_pid && E >= 2 && n < 65536 && op->npos <= 32 * SCM_T && op->npos + 1 <= cap && op->sp_avg_nnz >= 3.0) {
        const int kpos = (op->npos + SCM_T - 1) / SCM_T;
        // materialised kernel matrix when it fits (SMCP_B200_SCM_KMAT_GB, default 4 GB) and pays: building it
        // costs npos^2 entries, the direct form npos * nnz per column
        const double kmat_gb = getenv("SMCP_B200_SCM_KMAT_GB") ? atof(getenv("SMCP_B200_SCM_KMAT_GB")) : 4.0;
        const long long ldk = (op->npos + 1) & ~1LL;
        const double kbytes = (double)ldk * (double)op->npos * 8.0;
        // counted, not avg * (m - md): that product can round below an exact 2 npos
        const int64_t nnz_sp = op->h_colptr[m] - op->h_colptr[op->md];
        if (kbytes <= kmat_gb * 1073741824.0 && 2 * n <= cap && nnz_sp >= 2 * (int64_t)op->npos) {
            if (!op->Kpos_valid) {
                if (grow((void **)&op->Kpos, &op->Kpos_cap, (size_t)kbytes)) return -1;
                LaunchScope ls(ctx, "scm_kmat");
                CUDA_TRY(cudaFuncSetAttribute(scm_kmat_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(cap * 8)));
                scm_kmat_kernel<<<(unsigned)op->npos, SCM_T, (size_t)2 * n * sizeof(double), ctx->stream>>>(op->pos_r, op->pos_c, op->npos, op->Zinv, (int)n, op->Kpos, ldk);
                op->Kpos_valid = true;
            }
            // algorithmic bytes: the nnz(A_j) columns of K each column j streams + the lower triangle of H written
            const double kbytes_streamed = 8.0 * (double)ldk * (double)(op->h_colptr[s1] - op->h_colptr[s0])
                                           + 8.0 * ((double)(m - s0) * (m - s0 + 1) - (double)(m - s1) * (m - s1 + 1)) / 2.0;
            LaunchScope ls(ctx, "scm_kstream", 1, kbytes_streamed);
#define SCM_KLAUNCH(K_)                                                                                                      \
    do {                                                                                                                    \
        CUDA_TRY(cudaFuncSetAttribute(scm_kstream_kernel<K_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(cap * 8))); \
        scm_kstream_kernel<K_><<<(unsigned)(s1 - s0), SCM_T, (size_t)ldk * sizeof(double), ctx->stream>>>(op->colptr, op->vals,     \
            op->ent_r, op->ent_c, op->sp_pid, op->sp_base, op->npos, ldk, op->Kpos, op->H, m, s0, op->ell_val, op->ell_pid,  \
            op->ell_w, op->md);                                                                                              \
    } while (0)
            if (kpos <= 8) SCM_KLAUNCH(8);
            else if (kpos <= 16) SCM_KLAUNCH(16);
            else SCM_KLAUNCH(32);
#undef SCM_KLAUNCH
            CUDA_TRY(cudaGetLastError());
            return 0;
        }
        const size_t smem = (size_t)std::max<long long>(2LL * E * n, op->npos) * sizeof(double);
        LaunchScope ls(ctx, "scm_position");
#define SCM_LAUNCH(K_)                                                                                                      \
    do {                                                                                                                    \
        CUDA_TRY(cudaFuncSetAttribute(scm_position_kernel<K_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(cap * 8))); \
        scm_position_kernel<K_><<<(unsigned)(s1 - s0), SCM_T, smem, ctx->stream>>>(op->colptr, op->vals, op->ent_r, op->ent_c, \
            op->sp_pid, op->sp_base, op->pos_r, op->pos_c, op->npos, op->Zinv, (int)n, op->H, m, s0, E, op->ell_val,         \
            op->ell_pid, op->ell_w, op->md);                                                                                 \
    } while (0)
        if (kpos <= 8) SCM_LAUNCH(8);
        else if (kpos <= 16) SCM_LAUNCH(16);
        else SCM_LAUNCH(32);
#undef SCM_LAUNCH
    } else {
        LaunchScope ls(ctx, "scm_sparse");
        scm_sparse_kernel<<<(unsigned)(s1 - s0), 128, 0, ctx->stream>>>(op->colptr, op->vals, op->ent_r, op->ent_c, op->Zinv, n, op->H, m, s0);
    }
    CUDA_TRY(cudaGetLastError());
    return 0;
}

extern "C" int smcp_kkt_assemble(smcp_op *op, smcp_hess *h, int64_t j0, int64_t j1) {
    RegionScope rs(op->sym->ctx, "kkt_assemble");
    const int64_t m = op->m, md = op->md;
    if (j1 > m) j1 = m;
    int64_t d0 = std::max<int64_t>(j0, 0), d1 = std::min<int64_t>(j1, md);
    if (d1 > d0 && assemble_dense_ranges(op, h, {{d0, d1}})) return -1;
    if (assemble_sparse_range(op, h, std::max<int64_t>(j0, md), j1, true)) return -1;
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// the column blocks q = rank (mod nranks) of `block` columns each, as ONE batch
extern "C" int smcp_kkt_assemble_cyclic(smcp_op *op, smcp_hess *h, int64_t block, int rank, int nranks) {
    RegionScope rs(op->sym->ctx, "kkt_assemble");
    const int64_t m = op->m, md = op->md;
    if (block < 1 || nranks < 1 || rank < 0 || rank >= nranks) { smcp_set_error("smcp_kkt_assemble_cyclic: bad arguments"); return -2; }
    std::vector<std::pair<int64_t, int64_t>> dense;
    bool fresh = true;
    for (int64_t c0 = (int64_t)rank * block; c0 < m; c0 += (int64_t)nranks * block) {
        const int64_t c1 = std::min(m, c0 + block);
        if (c0 < md) dense.push_back({c0, std::min(c1, md)});
    }
    if (assemble_dense_ranges(op, h, dense)) return -1;
    if (op->Ns > 0) {
        // the dense inverse is shared by all sparse columns: built once, collectively when the communicator spans the ranks
        smcp_ctx *ctx = op->sym->ctx;
        if (build_zinv(op, h, nranks > 1 && ctx->nccl_comm && ctx->comm_nranks == nranks && ctx->comm_rank == rank)) return -1;
        fresh = false;
    }
    for (int64_t c0 = (int64_t)rank * block; c0 < m; c0 += (int64_t)nranks * block) {
        const int64_t c1 = std::min(m, c0 + block);
        if (c1 > md && assemble_sparse_range(op, h, std::max(c0, md), c1, fresh)) return -1;
    }
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// ---------------------------------------------------------------------------------------
// kktsolver='qr' in SYRK form (solvers.py:413-475; SURVEY 8f rank 3): Z = [G(A_1) ... G(A_m)] with the
// half factor G of the Hessian, H = Z^T Z (trace inner product) by one triangular DMMA product.
// ---------------------------------------------------------------------------------------
__global__ void sqrtw_kernel(const double *__restrict__ w, double *__restrict__ out, long long n) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = sqrt(w[i]);
}
// Z[r + j*nblk] *= sw[r]  (mode 0);  x[r] = sw[r] > 0 ? x[r] / sw[r] : 0 (mode 1, one column);  x[r] *= sw[r] (mode 2)
__global__ void rowscale_kernel(double *__restrict__ Z, const double *__restrict__ sw, long long nblk, long long ncols, int mode) {
    const long long total = nblk * ncols;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const double s = sw[idx % nblk];
        if (mode == 1) Z[idx] = s > 0.0 ? Z[idx] / s : 0.0;
        else Z[idx] *= s;
    }
}
// x[r] = sum_j Z[r + j*nblk] y[j]: thread per row, coalesced over rows, y staged in shared memory
__global__ void __launch_bounds__(256) zmul_kernel(const double *__restrict__ Z, long long nblk, long long m, const double *__restrict__ y,
                                                   double *__restrict__ x) {
    __shared__ double ys[256];
    const long long r = (long long)blockIdx.x * 256 + threadIdx.x;
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    for (long long j0 = 0; j0 < m; j0 += 256) {
        __syncthreads();
        if (j0 + threadIdx.x < m) ys[threadIdx.x] = y[j0 + threadIdx.x];
        __syncthreads();
        const int nj = (int)min((long long)256, m - j0);
        if (r < nblk) {
            const double *z = Z + r + j0 * nblk;
            int j = 0;
            for (; j + 3 < nj; j += 4) {
                s0 = fma(z[(long long)j * nblk], ys[j], s0);
                s1 = fma(z[(long long)(j + 1) * nblk], ys[j + 1], s1);
                s2 = fma(z[(long long)(j + 2) * nblk], ys[j + 2], s2);
                s3 = fma(z[(long long)(j + 3) * nblk], ys[j + 3], s3);
            }
            for (; j < nj; ++j) s0 = fma(z[(long long)j * nblk], ys[j], s0);
        }
    }
    if (r < nblk) x[r] = (s0 + s1) + (s2 + s3);
}

static int ensure_sqrtw(smcp_op *op) {
    smcp_sym *s = op->sym;
    if (!op->sqrtw) {
        const long long nblk = s->d.nblk;
        CUDA_TRY(cudaMalloc(&op->sqrtw, (size_t)nblk * sizeof(double)));
        sqrtw_kernel<<<(unsigned)((nblk + 255) / 256), 256, 0, s->ctx->stream>>>(s->d.wdot, op->sqrtw, nblk);
    }
    return 0;
}

// Zw = diag(sqrt(wdot)) [G(A_1) ... G(A_m)] in op->Zq (G = identity when h is NULL)
static int form_zw(smcp_op *op, smcp_hess *h, const char *who) {
    smcp_sym *s = op->sym;
    smcp_ctx *ctx = s->ctx;
    const int64_t m = op->m;
    const long long nblk = s->d.nblk;
    if (op->Ns) { smcp_set_error("%s: the sparse-constraint technique does not apply (Ns must be 0)", who); return -2; }
    const size_t bytes = (size_t)nblk * (size_t)m * sizeof(double);
    if (bytes > ((size_t)96 << 30)) { smcp_set_error("kktsolver='qr' needs m*|blkval| doubles (%.1f GB)", bytes / 1073741824.0); return -2; }
    op->zq_state = 0;
    if (!op->Zq) CUDA_TRY(cudaMalloc(&op->Zq, bytes ? bytes : 8));
    if (ensure_sqrtw(op)) return -1;
    CUDA_TRY(cudaMemsetAsync(op->Zq, 0, bytes, ctx->stream));
    {
        LaunchScope ls(ctx, "scatter_cols");
        scatter_cols_kernel<<<(unsigned)m, 128, 0, ctx->stream>>>(op->colptr, op->rowblk, op->vals, op->Zq, nblk, 0, (int)m);
    }
    if (h) {
        // G on all columns, in chunks that keep the update-matrix workspace (chunk x nupd doubles) below 4 GB
        const size_t per = ((size_t)s->d.nupd + 1) * sizeof(double);
        const int64_t chunk = std::max<int64_t>(1, std::min<int64_t>(m, (int64_t)(((size_t)4 << 30) / per)));
        for (int64_t c0 = 0; c0 < m; c0 += chunk)
            if (k_hess_apply_half(h, op->Zq + (size_t)c0 * nblk, std::min(chunk, m - c0), 0, 0)) return -1;
    }
    {
        LaunchScope ls(ctx, "level1");
        rowscale_kernel<<<ctx->num_sms * 8, 256, 0, ctx->stream>>>(op->Zq, op->sqrtw, nblk, m, 0);
    }
    op->zq_state = 1;
    CUDA_TRY(cudaGetLastError());
    return 0;
}

extern "C" int smcp_kkt_assemble_syrk(smcp_op *op, smcp_hess *h) {
    smcp_ctx *ctx = op->sym->ctx;
    RegionScope rs(ctx, "kkt_assemble");
    const int64_t m = op->m;
    const long long nblk = op->sym->d.nblk;
    if (!h && op->AvWs) {
        // Gram matrix sum_p w_p A_pi A_pj of the constraints over the support rows: one triangular product with
        // K = nsup of the sqrt(w)-weighted support copy (in the Ubs workspace; Zq is not formed and stays refused
        // by smcp_kkt_z_tmul / z_mul)
        if (op->Ns) { smcp_set_error("smcp_kkt_assemble_syrk: the sparse-constraint technique does not apply (Ns must be 0)"); return -2; }
        op->zq_state = 0;
        if (ensure_sqrtw(op)) return -1;
        const size_t bytes = (size_t)op->lds * (size_t)m * sizeof(double);
        if (grow((void **)&op->Ubs, &op->Ubs_cap, bytes)) return -1;
        CUDA_TRY(cudaMemsetAsync(op->Ubs, 0, bytes, ctx->stream));
        {
            LaunchScope ls(ctx, "scatter_cols");
            scatter_support_kernel<<<(unsigned)m, 128, 0, ctx->stream>>>(op->colptr, op->srow, op->rowblk, op->vals, op->sqrtw, op->Ubs,
                                                                         op->lds, 0, (int)m);
        }
        if (launch_gemm(ctx, true, true, op->Ubs, op->lds, op->Ubs, op->lds, op->H, m, m, m, op->nsup, 1.0, 0, 1, 0, "schur_syrk_dmma")) return -1;
        CUDA_TRY(cudaGetLastError());
        return 0;
    }
    if (int rc = form_zw(op, h, "smcp_kkt_assemble_syrk")) return rc;
    if (launch_gemm(ctx, true, true, op->Zq, nblk, op->Zq, nblk, op->H, m, m, m, nblk, 1.0, 0, 1, 0, "schur_syrk_dmma")) return -1;
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// out[j] = <G(A_j), X> in the trace inner product  (X: a chordal matrix on the device)
extern "C" int smcp_kkt_z_tmul(smcp_op *op, const double *X, double *host_out) {
    smcp_sym *s = op->sym;
    smcp_ctx *ctx = s->ctx;
    if (op->zq_state != 1) { smcp_set_error("smcp_kkt_z_tmul: no SYRK-form assembly (Zq holds %s)", op->zq_state ? "Q1 of the Householder form" : "nothing"); return -2; }
    const long long nblk = s->d.nblk;
    if (grow((void **)&s->tmp, &s->tmp_cap, (size_t)nblk * sizeof(double))) return -1;
    CUDA_TRY(cudaMemcpyAsync(s->tmp, X, (size_t)nblk * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
    {
        LaunchScope ls(ctx, "level1");
        rowscale_kernel<<<ctx->num_sms * 2, 256, 0, ctx->stream>>>(s->tmp, op->sqrtw, nblk, 1, 2);
    }
    {
        LaunchScope ls(ctx, "amap_dense", 1, 8.0 * (double)nblk * (double)op->m);
        amap_dense_kernel<false><<<(unsigned)op->m, 256, 0, ctx->stream>>>(op->Zq, nblk, nblk, nullptr, s->tmp, op->yv, 0);
    }
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(host_out, op->yv, (size_t)op->m * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return 0;
}

// X = sum_j y_j G(A_j)
extern "C" int smcp_kkt_z_mul(smcp_op *op, const double *host_y, double *X) {
    smcp_sym *s = op->sym;
    smcp_ctx *ctx = s->ctx;
    if (op->zq_state != 1) { smcp_set_error("smcp_kkt_z_mul: no SYRK-form assembly (Zq holds %s)", op->zq_state ? "Q1 of the Householder form" : "nothing"); return -2; }
    const long long nblk = s->d.nblk;
    CUDA_TRY(cudaMemcpyAsync(op->yv, host_y, (size_t)op->m * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    {
        LaunchScope ls(ctx, "aadj", 1, 8.0 * (double)nblk * (double)op->m);
        zmul_kernel<<<(unsigned)((nblk + 255) / 256), 256, 0, ctx->stream>>>(op->Zq, nblk, op->m, op->yv, X);
    }
    {
        LaunchScope ls(ctx, "level1");
        rowscale_kernel<<<ctx->num_sms * 2, 256, 0, ctx->stream>>>(X, op->sqrtw, nblk, 1, 1);
    }
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));       // host_y may be reused by the caller
    return 0;
}

// ---------------------------------------------------------------------------------------
// kktsolver='qr' in Householder form, the reference's kkt_qr (solvers.py:413-475: geqrf / ormqr / trtrs):
// Zw = Q1 R with Q1 (nblk x m) formed explicitly in Zq and L = R^T (diag >= 0) in H, so that L L^T is the
// SYRK-form H and the solves never multiply by R and undo it:
//   gw = sqrt(w) g,  c = Q1^T gw,  a = L^-1 r,  v = a + c,  y = L^-T v,  x = (Q1 v - gw) / sqrt(w)
// ---------------------------------------------------------------------------------------
// x[r] = (q[r] - gw[r]) / sw[r], and -g[r] where the weight is 0 (entries outside the vector space: the
// SYRK form's z_mul(y) - g there)
__global__ void qr_xout_kernel(const double *__restrict__ q, const double *__restrict__ gw, const double *g,
                               const double *__restrict__ sw, double *x, long long n) {
    for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (long long)gridDim.x * blockDim.x) {
        const double s = sw[r];
        x[r] = s > 0.0 ? (q[r] - gw[r]) / s : -g[r];
    }
}
__global__ void qr_vadd_kernel(double *__restrict__ v, const double *__restrict__ a, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) v[i] = a[i] + v[i];
}

extern "C" int smcp_kkt_factor_qr(smcp_op *op, smcp_hess *h, int32_t *info_host) {
    smcp_sym *s = op->sym;
    smcp_ctx *ctx = s->ctx;
    const int64_t m = op->m;
    const long long nblk = s->d.nblk;
    if (m > nblk) { smcp_set_error("smcp_kkt_factor_qr: more constraints (%lld) than rows of Z (%lld)", (long long)m, nblk); return -2; }
    {
        RegionScope rs(ctx, "kkt_assemble");
        if (int rc = form_zw(op, h, "smcp_kkt_factor_qr")) return rc;
        op->zq_state = 0;           // Zq is overwritten with Q1 below
    }
    if (!op->qr_tau) CUDA_TRY(cudaMalloc(&op->qr_tau, (size_t)3 * std::max<int64_t>(m, 1) * sizeof(double)));
    {
        RegionScope rs(ctx, "kkt_factor");
        if (d_geqrf(ctx, op->Zq, nblk, nblk, m, op->qr_tau)) return -1;
        if (qr_extract_lower(ctx, op->Zq, nblk, m, op->H, m, op->qr_tau + m, op->info_dev)) return -1;
        if (d_orgqr(ctx, op->Zq, nblk, nblk, m, op->qr_tau)) return -1;
        if (qr_apply_colsign(ctx, op->Zq, nblk, nblk, m, op->qr_tau + m)) return -1;
        if (d_potrs_prepare(ctx, op->H, m, m, op->Dinv)) return -1;
    }
    CUDA_TRY(cudaMemcpyAsync(info_host, op->info_dev, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    op->zq_state = *info_host ? 0 : 2;
    return 0;
}

extern "C" int smcp_kkt_qr_solve(smcp_op *op, const double *G_dev, const double *host_r, double *host_y, double *X_dev) {
    smcp_sym *s = op->sym;
    smcp_ctx *ctx = s->ctx;
    if (op->zq_state != 2) { smcp_set_error("smcp_kkt_qr_solve: no Householder-form factorisation (smcp_kkt_factor_qr)"); return -2; }
    const int64_t m = op->m;
    const long long nblk = s->d.nblk;
    double *rv = op->qr_tau + 2 * m;
    if (grow((void **)&s->tmp, &s->tmp_cap, (size_t)2 * nblk * sizeof(double))) return -1;
    double *gw = s->tmp, *q = s->tmp + nblk;
    CUDA_TRY(cudaMemcpyAsync(rv, host_r, (size_t)m * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    {
        RegionScope rs(ctx, "kkt_solve");
        CUDA_TRY(cudaMemcpyAsync(gw, G_dev, (size_t)nblk * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
        {
            LaunchScope ls(ctx, "level1");
            rowscale_kernel<<<ctx->num_sms * 2, 256, 0, ctx->stream>>>(gw, op->sqrtw, nblk, 1, 2);
        }
        if (d_trs_cluster(ctx, op->H, m, m, op->Dinv, rv, m, 1, 1, 0, "potrs")) return -1;        // a = L^-1 r
        {
            LaunchScope ls(ctx, "qr_qmul", 1, 8.0 * (double)nblk * (double)m);
            amap_dense_kernel<false><<<(unsigned)m, 256, 0, ctx->stream>>>(op->Zq, nblk, nblk, nullptr, gw, op->yv, 0);      // c = Q1^T gw
        }
        {
            LaunchScope ls(ctx, "level1");
            qr_vadd_kernel<<<(unsigned)((m + 255) / 256), 256, 0, ctx->stream>>>(op->yv, rv, m);          // v = a + c
        }
        {
            LaunchScope ls(ctx, "qr_qmul", 1, 8.0 * (double)nblk * (double)m);
            zmul_kernel<<<(unsigned)((nblk + 255) / 256), 256, 0, ctx->stream>>>(op->Zq, nblk, m, op->yv, q);   // Q1 v
        }
        {
            LaunchScope ls(ctx, "level1");
            qr_xout_kernel<<<ctx->num_sms * 2, 256, 0, ctx->stream>>>(q, gw, G_dev, op->sqrtw, X_dev, nblk);
        }
        if (d_trs_cluster(ctx, op->H, m, m, op->Dinv, op->yv, m, 1, 0, 1, "potrs")) return -1;    // y = L^-T v
    }
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(host_y, op->yv, (size_t)m * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return 0;
}

extern "C" int smcp_kkt_factor(smcp_op *op, int32_t *info_host) {
    smcp_ctx *ctx = op->sym->ctx;
    {
        RegionScope rs(ctx, "kkt_factor");
        if (d_potrf(ctx, op->H, op->m, op->m, op->m, op->info_dev, 0, 1)) return -1;
        if ((potrs_cluster_for(op->m) || potrs_wave_for(ctx, op->m)) && d_potrs_prepare(ctx, op->H, op->m, op->m, op->Dinv)) return -1;
    }
    CUDA_TRY(cudaMemcpyAsync(info_host, op->info_dev, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return 0;
}

// Distributed lapack.potrf (north star (3), SURVEY 8e): H holds, on every rank, the column blocks
// of 128 columns it owns (block q belongs to rank q mod nranks; smcp_kkt_assemble_cyclic with
// block = 128).  Owners factor their blocks and broadcast them; on return every rank has the
// complete factor.  nranks = 1 is smcp_kkt_factor.
extern "C" int smcp_kkt_factor_dist(smcp_op *op, int rank, int nranks, int32_t *info_host) {
    smcp_ctx *ctx = op->sym->ctx;
    if (nranks < 1 || rank < 0 || rank >= nranks) { smcp_set_error("smcp_kkt_factor_dist: bad arguments"); return -2; }
    if (nranks > 1 && !ctx->nccl_comm) { smcp_set_error("NCCL communicator not initialised"); return -2; }
    {
        RegionScope rs(ctx, "kkt_factor");
        if (d_potrf(ctx, op->H, op->m, op->m, op->m, op->info_dev, rank, nranks)) return -1;
        if ((potrs_cluster_for(op->m) || potrs_wave_for(ctx, op->m)) && d_potrs_prepare(ctx, op->H, op->m, op->m, op->Dinv)) return -1;
    }
    CUDA_TRY(cudaMemcpyAsync(info_host, op->info_dev, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return 0;
}

// as smcp_kkt_factor_dist with an explicit distribution block (a multiple of 128 columns; the block
// smcp_kkt_assemble_cyclic was called with)
extern "C" int smcp_kkt_factor_block(smcp_op *op, int64_t block, int rank, int nranks, int32_t *info_host) {
    smcp_ctx *ctx = op->sym->ctx;
    if (nranks < 1 || rank < 0 || rank >= nranks || block < 128 || block % 128) { smcp_set_error("smcp_kkt_factor_block: bad arguments"); return -2; }
    if (nranks > 1 && !ctx->nccl_comm) { smcp_set_error("NCCL communicator not initialised"); return -2; }
    {
        RegionScope rs(ctx, "kkt_factor");
        if (d_potrf(ctx, op->H, op->m, op->m, op->m, op->info_dev, rank, nranks, block)) return -1;
        if ((potrs_cluster_for(op->m) || potrs_wave_for(ctx, op->m)) && d_potrs_prepare(ctx, op->H, op->m, op->m, op->Dinv)) return -1;
    }
    CUDA_TRY(cudaMemcpyAsync(info_host, op->info_dev, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return 0;
}

// ---------------------------------------------------------------------------------------
// dense kernels on host buffers (column-major), the LAPACK/BLAS calls of the path on their own:
// lapack.potrf (solvers.py:501), the triangular solves behind lapack.potrs (solvers.py:526) and
// chompack.trsm on a dense root supernode (solvers.py:491-492), blas.gemm-shaped frontal updates.
// Used by the parity tests and scripts/bench_dense.py; `ms_out` (optional) is the device time.
// ---------------------------------------------------------------------------------------
struct DevBuf {
    double *p = nullptr;
    ~DevBuf() { if (p) cudaFree(p); }
};

extern "C" int smcp_dense_potrf(smcp_ctx *ctx, double *A_host, int64_t lda, int64_t m, int64_t ncols, int32_t *info_host, double *ms_out) {
    CUDA_TRY(cudaSetDevice(ctx->device));
    if (m <= 0 || lda < m) { smcp_set_error("smcp_dense_potrf: bad arguments"); return -2; }
    DevBuf A, I;
    CUDA_TRY(cudaMalloc(&A.p, (size_t)lda * m * sizeof(double)));
    CUDA_TRY(cudaMalloc(&I.p, 64));
    CUDA_TRY(cudaMemcpyAsync(A.p, A_host, (size_t)lda * m * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(cudaEventRecord(ctx->ev0, ctx->stream));
    if (d_potrf(ctx, A.p, lda, m, ncols, (int32_t *)I.p, 0, 1)) return -1;
    CUDA_TRY(cudaEventRecord(ctx->ev1, ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(A_host, A.p, (size_t)lda * m * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(info_host, I.p, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    if (ms_out) {
        float ms = 0.f;
        CUDA_TRY(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
        *ms_out = ms;
    }
    return 0;
}

extern "C" int smcp_dense_trsm(smcp_ctx *ctx, int trans, const double *L_host, int64_t ldl, int64_t n, double *B_host, int64_t ldb,
                               int64_t nrhs, double *ms_out) {
    CUDA_TRY(cudaSetDevice(ctx->device));
    if (n <= 0 || nrhs <= 0 || ldl < n || ldb < n) { smcp_set_error("smcp_dense_trsm: bad arguments"); return -2; }
    DevBuf L, B;
    CUDA_TRY(cudaMalloc(&L.p, (size_t)ldl * n * sizeof(double)));
    CUDA_TRY(cudaMalloc(&B.p, (size_t)ldb * nrhs * sizeof(double)));
    CUDA_TRY(cudaMemcpyAsync(L.p, L_host, (size_t)ldl * n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(B.p, B_host, (size_t)ldb * nrhs * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(cudaEventRecord(ctx->ev0, ctx->stream));
    if (d_trsm_left_lower(ctx, trans != 0, L.p, ldl, n, B.p, ldb, nrhs)) return -1;
    CUDA_TRY(cudaEventRecord(ctx->ev1, ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(B_host, B.p, (size_t)ldb * nrhs * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    if (ms_out) {
        float ms = 0.f;
        CUDA_TRY(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
        *ms_out = ms;
    }
    return 0;
}

// C = [C +] alpha op(A) op(B)^T in the convention of launch_gemm (dense.cu): ta/tb = 1 reads the
// operand K-major (A[k + i*lda]); tri = 1 computes the lower triangle only
extern "C" int smcp_dense_gemm(smcp_ctx *ctx, int ta, int tb, const double *A_host, int64_t lda, const double *B_host, int64_t ldb,
                               double *C_host, int64_t ldc, int64_t M, int64_t N, int64_t K, double alpha, int accumulate, int tri,
                               double *ms_out) {
    CUDA_TRY(cudaSetDevice(ctx->device));
    const size_t na = (size_t)lda * (ta ? M : K), nb = (size_t)ldb * (tb ? N : K), nc = (size_t)ldc * N;
    DevBuf A, B, Cd;
    CUDA_TRY(cudaMalloc(&A.p, na * sizeof(double)));
    CUDA_TRY(cudaMalloc(&B.p, nb * sizeof(double)));
    CUDA_TRY(cudaMalloc(&Cd.p, nc * sizeof(double)));
    CUDA_TRY(cudaMemcpyAsync(A.p, A_host, na * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(B.p, B_host, nb * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(Cd.p, C_host, nc * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(cudaEventRecord(ctx->ev0, ctx->stream));
    if (launch_gemm(ctx, ta != 0, tb != 0, A.p, lda, B.p, ldb, Cd.p, ldc, M, N, K, alpha, accumulate, tri, 0, "dense_gemm_dmma")) return -1;
    CUDA_TRY(cudaEventRecord(ctx->ev1, ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(C_host, Cd.p, nc * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    if (ms_out) {
        float ms = 0.f;
        CUDA_TRY(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
        *ms_out = ms;
    }
    return 0;
}

extern "C" int smcp_dense_geqrf(smcp_ctx *ctx, double *A_host, int64_t lda, int64_t M, int64_t N, double *tau_host, double *ms_out) {
    CUDA_TRY(cudaSetDevice(ctx->device));
    if (N < 1 || M < N || lda < M) { smcp_set_error("smcp_dense_geqrf: bad arguments (needs 1 <= N <= M <= lda)"); return -2; }
    DevBuf A, T;
    CUDA_TRY(cudaMalloc(&A.p, (size_t)lda * N * sizeof(double)));
    CUDA_TRY(cudaMalloc(&T.p, (size_t)N * sizeof(double)));
    CUDA_TRY(cudaMemcpyAsync(A.p, A_host, (size_t)lda * N * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(cudaEventRecord(ctx->ev0, ctx->stream));
    if (d_geqrf(ctx, A.p, lda, M, N, T.p)) return -1;
    CUDA_TRY(cudaEventRecord(ctx->ev1, ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(A_host, A.p, (size_t)lda * N * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(tau_host, T.p, (size_t)N * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    if (ms_out) {
        float ms = 0.f;
        CUDA_TRY(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
        *ms_out = ms;
    }
    return 0;
}

extern "C" int smcp_dense_orgqr(smcp_ctx *ctx, double *A_host, int64_t lda, int64_t M, int64_t N, const double *tau_host, double *ms_out) {
    CUDA_TRY(cudaSetDevice(ctx->device));
    if (N < 1 || M < N || lda < M) { smcp_set_error("smcp_dense_orgqr: bad arguments (needs 1 <= N <= M <= lda)"); return -2; }
    DevBuf A, T;
    CUDA_TRY(cudaMalloc(&A.p, (size_t)lda * N * sizeof(double)));
    CUDA_TRY(cudaMalloc(&T.p, (size_t)N * sizeof(double)));
    CUDA_TRY(cudaMemcpyAsync(A.p, A_host, (size_t)lda * N * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(T.p, tau_host, (size_t)N * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(cudaEventRecord(ctx->ev0, ctx->stream));
    if (d_orgqr(ctx, A.p, lda, M, N, T.p)) return -1;
    CUDA_TRY(cudaEventRecord(ctx->ev1, ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(A_host, A.p, (size_t)lda * N * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    if (ms_out) {
        float ms = 0.f;
        CUDA_TRY(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
        *ms_out = ms;
    }
    return 0;
}

extern "C" int smcp_kkt_solve(smcp_op *op, double *host_y) {
    smcp_ctx *ctx = op->sym->ctx;
    CUDA_TRY(cudaMemcpyAsync(op->yv, host_y, (size_t)op->m * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    {
        RegionScope rs(ctx, "kkt_solve");
        if (potrs_wave_for(ctx, op->m) ? d_potrs_wave(ctx, op->H, op->m, op->Dinv, op->yv)
                                       : potrs_cluster_for(op->m) ? d_potrs_cluster(ctx, op->H, op->m, op->Dinv, op->yv)
                                                                  : d_potrs(ctx, op->H, op->m, op->yv)) return -1;
    }
    CUDA_TRY(cudaMemcpyAsync(host_y, op->yv, (size_t)op->m * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return 0;
}

extern "C" int smcp_kkt_get_H(smcp_op *op, double *host_H) {
    smcp_ctx *ctx = op->sym->ctx;
    CUDA_TRY(cudaMemcpyAsync(host_H, op->H, (size_t)op->m * op->m * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return 0;
}
extern "C" int smcp_kkt_set_H(smcp_op *op, const double *host_H) {
    smcp_ctx *ctx = op->sym->ctx;
    CUDA_TRY(cudaMemcpyAsync(op->H, host_H, (size_t)op->m * op->m * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return 0;
}
extern "C" int smcp_kkt_H_devptr(smcp_op *op, double **dev_out) {
    *dev_out = op->H;
    return 0;
}

// ---------------------------------------------------------------------------------------
// NCCL (loaded lazily so that the library works without it on a single GPU)
// ---------------------------------------------------------------------------------------
typedef struct { char internal[128]; } nccl_uid;
typedef int (*fn_getuid)(nccl_uid *);
typedef int (*fn_init)(void **, int, nccl_uid, int);
typedef int (*fn_destroy)(void *);
typedef int (*fn_bcast)(const void *, void *, size_t, int, int, void *, cudaStream_t);
typedef int (*fn_group)(void);
typedef int (*fn_allreduce)(const void *, void *, size_t, int, int, void *, cudaStream_t);
typedef int (*fn_allgather)(const void *, void *, size_t, int, void *, cudaStream_t);
static fn_allreduce p_allreduce;
static fn_allgather p_allgather;
static void *g_nccl = nullptr;
static fn_getuid p_getuid;
static fn_init p_init;
static fn_destroy p_destroy;
static fn_bcast p_bcast;
static fn_group p_gstart, p_gend;

static int load_nccl() {
    if (g_nccl) return 0;
    g_nccl = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!g_nccl) g_nccl = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!g_nccl) { smcp_set_error("cannot load libnccl.so.2: %s", dlerror()); return -1; }
    p_getuid = (fn_getuid)dlsym(g_nccl, "ncclGetUniqueId");
    p_init = (fn_init)dlsym(g_nccl, "ncclCommInitRank");
    p_destroy = (fn_destroy)dlsym(g_nccl, "ncclCommDestroy");
    p_bcast = (fn_bcast)dlsym(g_nccl, "ncclBroadcast");
    p_gstart = (fn_group)dlsym(g_nccl, "ncclGroupStart");
    p_gend = (fn_group)dlsym(g_nccl, "ncclGroupEnd");
    p_allreduce = (fn_allreduce)dlsym(g_nccl, "ncclAllReduce");
    p_allgather = (fn_allgather)dlsym(g_nccl, "ncclAllGather");
    if (!p_getuid || !p_init || !p_destroy || !p_bcast || !p_gstart || !p_gend || !p_allreduce || !p_allgather) {
        smcp_set_error("libnccl is missing required symbols");
        return -1;
    }
    return 0;
}

extern "C" int smcp_comm_unique_id(char *id_out_128) {
    if (load_nccl()) return -1;
    nccl_uid id;
    int rc = p_getuid(&id);
    if (rc) { smcp_set_error("ncclGetUniqueId failed (%d)", rc); return -1; }
    memcpy(id_out_128, id.internal, 128);
    return 0;
}
extern "C" int smcp_comm_init(smcp_ctx *ctx, int rank, int nranks, const char *id_128) {
    if (load_nccl()) return -1;
    CUDA_TRY(cudaSetDevice(ctx->device));
    nccl_uid id;
    memcpy(id.internal, id_128, 128);
    int rc = p_init(&ctx->nccl_comm, nranks, id, rank);
    if (rc) { smcp_set_error("ncclCommInitRank failed (%d)", rc); return -1; }
    ctx->comm_rank = rank;
    ctx->comm_nranks = nranks;
    return 0;
}
extern "C" int smcp_comm_destroy(smcp_ctx *ctx) {
    if (ctx->nccl_comm) p_destroy(ctx->nccl_comm);
    ctx->nccl_comm = nullptr;
    ctx->comm_rank = 0;
    ctx->comm_nranks = 1;
    return 0;
}

int comm_group_start() { return p_gstart ? p_gstart() : -1; }
int comm_group_end() { return p_gend ? p_gend() : -1; }
int comm_allreduce_max_i32(smcp_ctx *ctx, int *ptr, size_t count, cudaStream_t s) {
    if (!ctx->nccl_comm) { smcp_set_error("NCCL communicator not initialised"); return -2; }
    int rc = p_allreduce(ptr, ptr, count, 2 /* ncclInt32 */, 2 /* ncclMax */, ctx->nccl_comm, s);
    if (rc) { smcp_set_error("ncclAllReduce failed (%d)", rc); return -1; }
    ctx->launches += 1;
    return 0;
}
// every rank contributes `chunk` doubles at base + rank*chunk; all ranks end with nranks*chunk doubles
int comm_allgather(smcp_ctx *ctx, double *base, size_t chunk, cudaStream_t s) {
    if (!ctx->nccl_comm) { smcp_set_error("NCCL communicator not initialised"); return -2; }
    int rc = p_allgather(base + (size_t)ctx->comm_rank * chunk, base, chunk, 8 /* ncclFloat64 */, ctx->nccl_comm, s);
    if (rc) { smcp_set_error("ncclAllGather failed (%d)", rc); return -1; }
    ctx->launches += 1;
    return 0;
}

int comm_bcast(smcp_ctx *ctx, double *ptr, size_t count, int root, cudaStream_t s) {
    if (!ctx->nccl_comm) { smcp_set_error("NCCL communicator not initialised"); return -2; }
    int rc = p_bcast(ptr, ptr, count, 8 /* ncclFloat64 */, root, ctx->nccl_comm, s);
    if (rc) { smcp_set_error("ncclBroadcast failed (%d)", rc); return -1; }
    ctx->launches += 1;
    return 0;
}

// Column blocks of H are owned block-cyclically: block q (columns [q*block, (q+1)*block))
// belongs to rank q % nranks.  Every owner broadcasts its blocks (rows j.. of each column
// block, i.e. the lower trapezoid) so that all ranks end up with the full lower triangle.
extern "C" int smcp_kkt_allgather(smcp_op *op, int64_t block, int rank, int nranks) {
    smcp_ctx *ctx = op->sym->ctx;
    RegionScope rs(ctx, "kkt_allgather");
    (void)rank;
    if (!ctx->nccl_comm) { smcp_set_error("NCCL communicator not initialised"); return -2; }
    const int64_t m = op->m;
    p_gstart();
    for (int64_t q = 0, c0 = 0; c0 < m; ++q, c0 += block) {
        int64_t nc = std::min(block, m - c0);
        double *ptr = op->H + c0 * m;       // whole columns (contiguous)
        int rc = p_bcast(ptr, ptr, (size_t)nc * m, 8 /* ncclFloat64 */, (int)(q % nranks), ctx->nccl_comm, ctx->stream);
        if (rc) { p_gend(); smcp_set_error("ncclBroadcast failed (%d)", rc); return -1; }
    }
    p_gend();
    ctx->launches += 1;
    return 0;
}
