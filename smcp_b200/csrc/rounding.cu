// Randomized rounding of a chordal SDP solution (an extension: the reference has no rounding).
//
// With L from smcp_csp_completion, the max-det completion is X_hat = (L L^T)^-1 = L^-T L^-1, so L^-T g has
// covariance X_hat for a standard normal g: one chordal trsm (k_trsm, trans = 1) per block of samples, and no
// dense n x n matrix anywhere.
//  * round_normal: counter-based standard normals.  Entry i of sample j is a function of (seed, j, i) only:
//    Philox4x64-10 with key (seed, 0) and counter (i / 4, j, 0, 0) (Random123's constants, as NumPy's
//    np.random.Philox, which increments its counter before it generates), two 53-bit uniforms
//    u = ((w >> 11) + 0.5) 2^-53 per pair of words, Box-Muller.  Results do not depend on the launch shape.
//  * round_eval: Goemans-Williamson +-1 trials s_t = sign(v_t) (sign(0) = +1) against the objective, given as
//    nc lower-triangular entries (r, c, coef) with the factor 2 off the diagonal folded into coef:
//    value_t = sum_q coef_q s_t[r_q] s_t[c_q].  The signs of 64 trials are packed into one word per row
//    (each sample entry is read once), a warp owns one 64-trial word group and a fixed slice of entries, and
//    the per-slice partial sums are added in a fixed order: the values are bitwise reproducible and do not
//    depend on how many trials a pass holds.  The best trial (smallest value, lowest t on ties) is tracked on
//    the device and only its sign vector returns to the host.
#include "internal.cuh"
#include <algorithm>
#include <cmath>

__device__ __forceinline__ void philox4x64_10(unsigned long long c[4], unsigned long long k0, unsigned long long k1) {
    const unsigned long long M0 = 0xD2E7470EE14C6C93ULL, M1 = 0xCA5A826395121157ULL;
    const unsigned long long W0 = 0x9E3779B97F4A7C15ULL, W1 = 0xBB67AE8584CAA73BULL;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        if (r) { k0 += W0; k1 += W1; }
        const unsigned long long hi0 = __umul64hi(M0, c[0]), lo0 = M0 * c[0];
        const unsigned long long hi1 = __umul64hi(M1, c[2]), lo1 = M1 * c[2];
        const unsigned long long o0 = hi1 ^ c[1] ^ k0, o2 = hi0 ^ c[3] ^ k1;
        c[0] = o0;
        c[1] = lo1;
        c[2] = o2;
        c[3] = lo0;
    }
}

// a uniform in (0, 1) from the top 53 bits of a word (exact in FP64)
__device__ __forceinline__ double u53(unsigned long long w) { return ((double)(w >> 11) + 0.5) * 0x1.0p-53; }

// B[i + c * ldb] = entry i of sample col0 + c, i < n, c < k; one thread per four rows of one sample
__global__ void round_normal_kernel(unsigned long long seed, long long col0, int n, long long k, double *__restrict__ B, long long ldb) {
    const long long nr = (n + 3) / 4;
    const long long total = nr * k;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const long long r = idx % nr, c = idx / nr;
        unsigned long long w[4] = {(unsigned long long)r, (unsigned long long)(col0 + c), 0ULL, 0ULL};
        philox4x64_10(w, seed, 0ULL);
        double z[4];
#pragma unroll
        for (int q = 0; q < 4; q += 2) {
            const double rad = sqrt(-2.0 * log(u53(w[q])));
            double sn, cs;
            sincospi(2.0 * u53(w[q + 1]), &sn, &cs);
            z[q] = rad * cs;
            z[q + 1] = rad * sn;
        }
        double *b = B + c * ldb + 4 * r;
        const int m = (int)min(4LL, (long long)n - 4 * r);
#pragma unroll
        for (int q = 0; q < 4; ++q)
            if (q < m) b[q] = z[q];
    }
}

// bits[g * n + i], bit b = (V[i + (64 g + b) ldv] < 0) for the T trials of the pass; blockIdx.y = word group g
__global__ void round_pack_kernel(const double *__restrict__ V, long long ldv, int n, int T, unsigned long long *__restrict__ bits) {
    const int g = blockIdx.y;
    const int t0 = 64 * g, nb = min(64, T - t0);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        unsigned long long w = 0ULL;
        for (int b = 0; b < nb; ++b) w |= (unsigned long long)(V[i + (long long)(t0 + b) * ldv] < 0.0) << b;
        bits[(long long)g * n + i] = w;
    }
}

// part[(g * S + s) * 64 + t] = sum over the entries of slice s = blockIdx.x of +-coef for trial 64 g + t.  Warp w of the
// block takes the 32-entry tiles w, w + EV_WARPS, ... of the slice; lane l keeps trials 2l and 2l + 1.  The lanes
// gather the words of a tile together and then walk it in order through shuffles (fixed summation order).
#define EV_WARPS 8
__global__ void __launch_bounds__(32 * EV_WARPS) round_eval_kernel(const int *__restrict__ er, const int *__restrict__ ec,
                                                                  const double *__restrict__ ev, long long nc, long long per,
                                                                  const unsigned long long *__restrict__ bits, int n,
                                                                  double *__restrict__ part) {
    __shared__ double sh[EV_WARPS][64];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int S = gridDim.x, s = blockIdx.x, g = blockIdx.y;
    const unsigned long long *wg = bits + (long long)g * n;
    const long long e0 = (long long)s * per, e1 = min(nc, e0 + per);
    double a0 = 0.0, a1 = 0.0;
    for (long long base = e0 + 32LL * warp; base < e1; base += 32LL * EV_WARPS) {
        const long long e = base + lane;
        unsigned long long x = 0ULL;
        double c = 0.0;
        if (e < e1) {
            x = wg[er[e]] ^ wg[ec[e]];
            c = ev[e];
        }
        const int cnt = (int)min(32LL, e1 - base);
        for (int j = 0; j < cnt; ++j) {
            const unsigned long long xj = __shfl_sync(0xffffffffu, x, j);
            const double cj = __shfl_sync(0xffffffffu, c, j);
            a0 += ((xj >> (2 * lane)) & 1ULL) ? -cj : cj;
            a1 += ((xj >> (2 * lane + 1)) & 1ULL) ? -cj : cj;
        }
    }
    sh[warp][2 * lane] = a0;
    sh[warp][2 * lane + 1] = a1;
    __syncthreads();
    if (threadIdx.x < 64) {
        double v = 0.0;
        for (int w = 0; w < EV_WARPS; ++w) v += sh[w][threadIdx.x];
        part[((long long)g * S + s) * 64 + threadIdx.x] = v;
    }
}

// values[t0 + t] = sum of the S slice partial sums of trial t, in slice order
__global__ void round_sum_kernel(const double *__restrict__ part, int S, int T, long long t0, double *__restrict__ values) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= T) return;
    const int g = t >> 6, b = t & 63;
    double v = 0.0;
    for (int s = 0; s < S; ++s) v += part[((long long)g * S + s) * 64 + b];
    values[t0 + t] = v;
}

struct RoundBest {
    double v;
    long long t;     // -1: none yet
};

// smallest value of the pass (lowest t on ties); when it beats the best of the earlier passes (which hold lower t),
// it becomes the best and its sign vector is written to x.  One block of BEST_THREADS threads.
#define BEST_THREADS 1024
__global__ void __launch_bounds__(BEST_THREADS) round_best_kernel(const double *__restrict__ values, long long t0, int T,
                                                                  const unsigned long long *__restrict__ bits, int n,
                                                                  RoundBest *best, signed char *__restrict__ x) {
    __shared__ double sv[BEST_THREADS];
    __shared__ long long st[BEST_THREADS];
    __shared__ int upd;
    const int tid = threadIdx.x;
    double bv = INFINITY;
    long long bt = -1;
    for (int t = tid; t < T; t += BEST_THREADS) {
        const double v = values[t0 + t];
        if (v < bv) { bv = v; bt = t0 + t; }      // ascending t: the first of equal values stays
    }
    sv[tid] = bv;
    st[tid] = bt;
    __syncthreads();
    for (int o = BEST_THREADS / 2; o > 0; o >>= 1) {
        if (tid < o) {
            const long long tb = st[tid + o], ta = st[tid];
            if (tb >= 0 && (ta < 0 || sv[tid + o] < sv[tid] || (sv[tid + o] == sv[tid] && tb < ta))) {
                sv[tid] = sv[tid + o];
                st[tid] = tb;
            }
        }
        __syncthreads();
    }
    if (tid == 0) {
        upd = st[0] >= 0 && (best->t < 0 || sv[0] < best->v);
        if (upd) {
            best->v = sv[0];
            best->t = st[0];
        }
    }
    __syncthreads();
    if (!upd) return;
    const long long tl = st[0] - t0;
    const unsigned long long *wg = bits + (tl >> 6) * n;
    const int b = (int)(tl & 63);
    for (int i = tid; i < n; i += BEST_THREADS) x[i] = ((wg[i] >> b) & 1ULL) ? -1 : 1;
}

static int launch_normals(smcp_sym *s, uint64_t seed, int64_t col0, double *B, int64_t ldb, int64_t k) {
    smcp_ctx *ctx = s->ctx;
    const long long total = (long long)((s->d.n + 3) / 4) * k;
    const long long grid = std::max(1LL, std::min((total + 255) / 256, (long long)ctx->num_sms * 16));
    {
        LaunchScope ls(ctx, "round_normal");
        round_normal_kernel<<<(unsigned)grid, 256, 0, ctx->stream>>>(seed, col0, s->d.n, k, B, ldb);
    }
    CUDA_TRY(cudaGetLastError());
    return 0;
}

int k_sample(smcp_sym *s, const double *L, uint64_t seed, int64_t col0, double *B, int64_t ldb, int64_t k) {
    if (k < 0 || col0 < 0 || ldb < s->d.n || (k > 0 && !B) || !L) {
        smcp_set_error("smcp_csp_sample: need k >= 0, col0 >= 0, ldb >= n and device buffers");
        return -2;
    }
    if (k == 0) return 0;
    if (launch_normals(s, seed, col0, B, ldb, k)) return -1;
    return k_trsm(s, L, B, ldb, k, 1);
}

// largest number of trials a pass holds: bounds the word groups (grid.y) and the slice partial sums
#define ROUND_MAX_PASS 65536
// columns of one trsm call; every call of a smcp_round_pm1 has the same width, so the samples of a trial are the
// same bits whatever the pass size (k_trsm picks its kernels from the number of right-hand sides)
#define ROUND_BLOCK 256

int k_round_pm1(smcp_sym *s, const double *L, uint64_t seed, int64_t trials, int64_t chunk, int64_t nc, const int64_t *crow,
                const int64_t *ccol, const double *cval, double *values_host, int8_t *x_host, int64_t *best_out) {
    smcp_ctx *ctx = s->ctx;
    const int n = s->d.n;
    if (trials < 1 || chunk < 0 || nc < 0) {
        smcp_set_error("smcp_round_pm1: need trials >= 1, chunk >= 0, nc >= 0 (got %lld, %lld, %lld)", (long long)trials,
                       (long long)chunk, (long long)nc);
        return -2;
    }
    if (!L || !values_host || !x_host || !best_out || (nc > 0 && (!crow || !ccol || !cval))) {
        smcp_set_error("smcp_round_pm1: null argument");
        return -2;
    }
    std::vector<int> hr((size_t)nc), hc((size_t)nc);
    std::vector<double> hv((size_t)nc);
    for (int64_t q = 0; q < nc; ++q) {
        if (crow[q] < 0 || crow[q] >= n || ccol[q] < 0 || ccol[q] >= n) {
            smcp_set_error("smcp_round_pm1: objective entry %lld at (%lld, %lld) is outside 0..%d", (long long)q, (long long)crow[q],
                           (long long)ccol[q], n - 1);
            return -2;
        }
        hr[q] = (int)crow[q];
        hc[q] = (int)ccol[q];
        hv[q] = crow[q] == ccol[q] ? cval[q] : 2.0 * cval[q];
    }
    // solve blocks: as few as hold ROUND_BLOCK columns each, all of the same width tb (within 1 GiB)
    const int64_t fit = std::max<int64_t>(1, (int64_t(1) << 30) / (8 * (int64_t)n));
    const int64_t bmax = std::min<int64_t>(ROUND_BLOCK, fit);
    const int64_t nblocks = (trials + bmax - 1) / bmax;
    const int64_t tb = (trials + nblocks - 1) / nblocks;
    // blocks per pass: chunk trials rounded up to whole blocks; 0 = as many as fit in 1 GiB
    const int64_t cap = std::max<int64_t>(1, std::min<int64_t>(fit, ROUND_MAX_PASS) / tb);
    int64_t bp = chunk == 0 ? cap : std::min<int64_t>((chunk + tb - 1) / tb, cap);
    bp = std::min(bp, nblocks);
    const int64_t pw = bp * tb;                    // trials per pass
    const int64_t nwmax = (pw + 63) / 64;
    // entry slices: a fixed partition of the entry list, independent of the trials
    const int S = (int)std::min<int64_t>(256, std::max<int64_t>(1, (nc + 511) / 512));
    const long long per = std::max<long long>(1, (nc + S - 1) / S);

    struct Ws {
        smcp_ctx *ctx;
        std::vector<void *> p;
        ~Ws() {
            cudaStreamSynchronize(ctx->stream);
            for (void *q : p) cudaFree(q);
        }
    } ws{ctx, {}};
    auto alloc = [&](size_t bytes) -> void * {
        void *q = nullptr;
        if (cudaMalloc(&q, std::max<size_t>(bytes, 16)) != cudaSuccess) {
            cudaGetLastError();
            smcp_set_error("smcp_round_pm1: cudaMalloc(%zu bytes) failed", bytes);
            return nullptr;
        }
        ws.p.push_back(q);
        return q;
    };
    double *V = (double *)alloc((size_t)n * pw * sizeof(double));
    unsigned long long *bits = (unsigned long long *)alloc((size_t)n * nwmax * sizeof(unsigned long long));
    double *part = (double *)alloc((size_t)nwmax * S * 64 * sizeof(double));
    double *values = (double *)alloc((size_t)trials * sizeof(double));
    RoundBest *best = (RoundBest *)alloc(sizeof(RoundBest));
    signed char *x = (signed char *)alloc((size_t)n);
    int *er = (int *)alloc((size_t)nc * sizeof(int));
    int *ec = (int *)alloc((size_t)nc * sizeof(int));
    double *ev = (double *)alloc((size_t)nc * sizeof(double));
    if (!V || !bits || !part || !values || !best || !x || !er || !ec || !ev) return -1;
    const RoundBest none{0.0, -1};
    CUDA_TRY(cudaMemcpyAsync(best, &none, sizeof(none), cudaMemcpyHostToDevice, ctx->stream));
    if (nc) {
        CUDA_TRY(cudaMemcpyAsync(er, hr.data(), (size_t)nc * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
        CUDA_TRY(cudaMemcpyAsync(ec, hc.data(), (size_t)nc * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
        CUDA_TRY(cudaMemcpyAsync(ev, hv.data(), (size_t)nc * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    }
    for (int64_t b0 = 0; b0 < nblocks; b0 += bp) {
        const int64_t b1 = std::min(nblocks, b0 + bp);
        const int64_t t0 = b0 * tb;
        for (int64_t b = b0; b < b1; ++b) {
            double *Vb = V + (size_t)(b - b0) * tb * n;
            if (launch_normals(s, seed, b * tb, Vb, n, tb)) return -1;
            if (k_trsm(s, L, Vb, n, tb, 1)) return -1;
        }
        const int T = (int)std::min<int64_t>(trials - t0, (b1 - b0) * tb);
        const int nw = (T + 63) / 64;
        {
            LaunchScope ls(ctx, "round_eval", 4);
            round_pack_kernel<<<dim3((unsigned)((n + 255) / 256), (unsigned)nw), 256, 0, ctx->stream>>>(V, n, n, T, bits);
            round_eval_kernel<<<dim3((unsigned)S, (unsigned)nw), 32 * EV_WARPS, 0, ctx->stream>>>(er, ec, ev, nc, per, bits, n, part);
            round_sum_kernel<<<(unsigned)((T + 255) / 256), 256, 0, ctx->stream>>>(part, S, T, t0, values);
            round_best_kernel<<<1, BEST_THREADS, 0, ctx->stream>>>(values, t0, T, bits, n, best, x);
        }
        CUDA_TRY(cudaGetLastError());
    }
    RoundBest hb;
    CUDA_TRY(cudaMemcpyAsync(values_host, values, (size_t)trials * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(x_host, x, (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(&hb, best, sizeof(hb), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    if (hb.t < 0) {
        smcp_set_error("smcp_round_pm1: no trial has a finite value");
        return -1;
    }
    *best_out = hb.t;
    return 0;
}
