// lapack.potrs (src/python/solvers.py:526, 1954: y <- H^{-1} y with the Cholesky factor of the m x m Schur
// complement) as ONE launch of a thread-block CLUSTER.
//
// A triangular solve with one right-hand side is m dependent steps, and a single CTA can only pull the
// factor out of L2 at ~100 GB/s (the round-1 kernel: 0.24 ms per solve at m = 1000, 3.5 ms at m = 10^4).
// Here the 64-row blocks of the vector are owned cyclically by the R CTAs of a cluster (R = 8 or 16):
//   step b:  the owner of block b applies the INVERSE of the 64 x 64 diagonal block (computed once per
//            factorisation by trtri64_kernel, like the triangular solves of MAGMA / cuBLAS) to its fully
//            updated y_b and writes x_b into the shared memory of every CTA of the cluster (DSMEM);
//            cluster barrier;
//            every CTA subtracts L(blk, b) x_b from the blocks blk > b it owns (the block the next step
//            needs first), reading each tile of the factor exactly once, 16 loads in flight per thread.
// The backward sweep with L^T mirrors it.  All sums have a fixed order: bitwise reproducible.
// Inverting only the 64 x 64 DIAGONAL blocks keeps the solve as accurate as substitution up to the
// condition of those blocks (the iterative refinement of the Newton systems, solvers.py:907-913, absorbs
// it).  Orders whose blocks outnumber what the wavefront kernel can own go to the substitution kernel
// of dense.cu.
#include "internal.cuh"
#include <cooperative_groups.h>
#include <algorithm>

namespace cg = cooperative_groups;

#define PC_T 256

// Dinv[b] = L(b, b)^{-1} for every 64 x 64 diagonal block b (lower triangular, column-major 64 x 64,
// zero above the diagonal; rows/columns beyond m: identity).  One CTA per block, one column per thread.
__global__ void __launch_bounds__(64) trtri64_kernel(const double *__restrict__ H, long long ld, long long m, double *__restrict__ Dinv) {
    __shared__ double Ls[64 * 65];
    const int b = blockIdx.x, tid = threadIdx.x;
    const long long k0 = 64LL * b;
    for (int idx = tid; idx < 64 * 64; idx += 64) {
        const int r = idx & 63, c = idx >> 6;
        double v = (r == c) ? 1.0 : 0.0;
        if (r >= c && k0 + r < m && k0 + c < m) v = H[(k0 + r) + (k0 + c) * ld];
        Ls[c * 65 + r] = v;
    }
    __syncthreads();
    // column tid of the inverse: solve L x = e_tid (x_r = 0 for r < tid)
    double x[64];
#pragma unroll
    for (int r = 0; r < 64; ++r) x[r] = 0.0;
    const int c = tid;
#pragma unroll
    for (int r = 0; r < 64; ++r) {
        if (r >= c) {
            double s = (r == c) ? 1.0 : 0.0;
#pragma unroll
            for (int p = 0; p < 64; ++p)
                if (p < r && p >= c) s = fma(-Ls[p * 65 + r], x[p], s);
            x[r] = s / Ls[r * 65 + r];
        }
    }
    double *D = Dinv + (long long)b * 4096;
#pragma unroll
    for (int r = 0; r < 64; ++r) D[r + c * 64] = x[r];
}

struct PotrsArgs {
    const double *L;
    long long ld;
    int m;
    const double *Dinv;
    double *y;
    long long ldy;      // right-hand sides are columns of y, solved one after the other
    int nrhs;
    int do_fwd, do_bwd; // L^-1 and / or L^-T
};

// 64 x 64 tile times a 64-vector: out[r] (-)= sum_c T(r, c) x[c]; the 256 threads split each row's sum in 4
// column groups (16 independent loads per thread), partial sums combined in a fixed order through `part`.
// TRANS: T(r, c) = A[c + r*lda] (the tile of L read transposed).
template <bool TRANS>
__device__ __forceinline__ void tile_gemv(const double *__restrict__ A, long long lda, int rows, int cols, const double *x, double *part, int tid) {
    const int r = tid & 63, g = tid >> 6;
    double s0 = 0.0, s1 = 0.0;
    if (r < rows) {
        double v[16];
#pragma unroll
        for (int q = 0; q < 16; ++q) {
            const int c = 16 * g + q;
            v[q] = (c < cols) ? (TRANS ? A[c + (long long)r * lda] : A[r + (long long)c * lda]) : 0.0;
        }
#pragma unroll
        for (int q = 0; q < 16; q += 2) {
            s0 = fma(v[q], x[16 * g + q], s0);
            s1 = fma(v[q + 1], x[16 * g + q + 1], s1);
        }
    }
    part[g * 64 + r] = s0 + s1;
}

template <bool BWD>
__device__ __forceinline__ void cluster_sweep(const PotrsArgs &a, cg::cluster_group &cluster, double *ys, double *xb, double *part, double *Ds,
                                              int tid) {
    const int R = (int)cluster.num_blocks(), rk = (int)cluster.block_rank();
    const int nb = (a.m + 63) / 64;
    for (int q = 0; q < nb; ++q) {
        const int b = BWD ? nb - 1 - q : q;
        const int kb = min(64, a.m - 64 * b);
        double *xcur = xb + (q & 1) * 64;
        if (b % R == rk) {
            // x_b = Dinv_b y_b (backward: Dinv_b^T y_b)
            const double *D = a.Dinv + (long long)b * 4096;
            tile_gemv<BWD>(D, 64, 64, 64, ys + (b / R) * 64, part, tid);
            __syncthreads();
            if (tid < 64) {
                const double xv = (tid < kb) ? (part[tid] + part[64 + tid]) + (part[128 + tid] + part[192 + tid]) : 0.0;
                ys[(b / R) * 64 + tid] = xv;
                for (int t = 0; t < R; ++t) cluster.map_shared_rank(xcur, t)[tid] = xv;
            }
        }
        cluster.sync();
        // blocks this CTA owns on the far side of b, nearest first (the next step needs that one), four
        // tiles of the factor per round: 64 loads in flight per thread, one pair of barriers per round
        int o = 1;
        for (;;) {
            int tb[4], nt = 0;
            for (; nt < 4; ++o) {
                const int blk = BWD ? b - o : b + o;
                if (blk < 0 || blk >= nb) break;
                if (blk % R == rk) tb[nt++] = blk;
            }
            if (!nt) break;
            const int r = tid & 63, g = tid >> 6;
            double v[4][16];
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                if (t < nt) {
                    const int blk = tb[t];
                    const int rows = min(64, a.m - 64 * blk);
                    // forward : y_blk -= L(blk, b) x_b       tile entry (r, c) at L[64 blk + r, 64 b + c]
                    // backward: y_blk -= L(b, blk)^T x_b     tile entry (r, c) at L[64 b + c, 64 blk + r]
                    const double *T = BWD ? a.L + 64LL * b + 64LL * blk * a.ld : a.L + 64LL * blk + 64LL * b * a.ld;
#pragma unroll
                    for (int e = 0; e < 16; ++e) {
                        const int c = 16 * g + e;
                        v[t][e] = (r < rows && c < kb) ? (BWD ? T[c + (long long)r * a.ld] : T[r + (long long)c * a.ld]) : 0.0;
                    }
                }
            }
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                if (t < nt) {
                    double s0 = 0.0, s1 = 0.0;
#pragma unroll
                    for (int e = 0; e < 16; e += 2) {
                        s0 = fma(v[t][e], xcur[16 * g + e], s0);
                        s1 = fma(v[t][e + 1], xcur[16 * g + e + 1], s1);
                    }
                    part[t * 256 + g * 64 + r] = s0 + s1;
                }
            }
            __syncthreads();
            {
                const int t = tid >> 6, rr = tid & 63;
                if (t < nt) {
                    const double *pp = part + t * 256;
                    ys[(tb[t] / R) * 64 + rr] -= (pp[rr] + pp[64 + rr]) + (pp[128 + rr] + pp[192 + rr]);
                }
            }
            __syncthreads();
        }
    }
    (void)Ds;
}

__global__ void __launch_bounds__(PC_T, 1) potrs_cluster_kernel(PotrsArgs a) {
    extern __shared__ double pcsm[];
    cg::cluster_group cluster = cg::this_cluster();
    const int R = (int)cluster.num_blocks(), rk = (int)cluster.block_rank();
    const int tid = threadIdx.x;
    const int nb = (a.m + 63) / 64;
    const int nloc = (nb + R - 1) / R;
    double *ys = pcsm;                  // nloc x 64: the blocks of y this CTA owns
    double *xb = ys + nloc * 64;        // 2 x 64: x of the current step (written by its owner through DSMEM)
    double *part = xb + 128;            // 4 tiles x 4 x 64 partial sums
    cluster.sync();
    for (int rhs = 0; rhs < a.nrhs; ++rhs) {
        double *y = a.y + (long long)rhs * a.ldy;
        for (int idx = tid; idx < nloc * 64; idx += PC_T) {
            const int b = (idx >> 6) * R + rk;
            const long long i = 64LL * b + (idx & 63);
            ys[idx] = (b < nb && i < a.m) ? y[i] : 0.0;
        }
        __syncthreads();
        if (a.do_fwd) cluster_sweep<false>(a, cluster, ys, xb, part, nullptr, tid);
        cluster.sync();
        if (a.do_bwd) cluster_sweep<true>(a, cluster, ys, xb, part, nullptr, tid);
        __syncthreads();
        for (int idx = tid; idx < nloc * 64; idx += PC_T) {
            const int b = (idx >> 6) * R + rk;
            const long long i = 64LL * b + (idx & 63);
            if (b < nb && i < a.m) y[i] = ys[idx];
        }
        cluster.sync();                 // no CTA may run ahead (or exit) while others still write into its shared memory
    }
}

// ---------------------------------------------------------------------------------------
// potrs from m = 512 on (and the only sensible form once the factor does not fit in L2: m = 10^4 is 400 MB per sweep): the
// whole grid as a flag-driven wavefront.
// Block rows (64 rows) are owned cyclically by the CTAs of a co-resident grid (cooperative launch, one CTA per SM).
// Step b of the forward sweep: every CTA has ALREADY loaded its tiles L(blk, b), blk > b, into registers; it then waits
// for the flag of x_b (written to global memory by the owner of block b), subtracts L(blk, b) x_b from the blocks it
// owns, and the owner of block b + 1 applies the inverted diagonal block (trtri64_kernel) and publishes x_{b+1}.  The
// dependent chain per step is flag -> 64 x 64 product -> 64 x 64 product -> flag (~3 us); the factor is streamed once
// per sweep by all SMs (the cluster kernel above streams it through 16 SMs: 5.1 ms at m = 10^4; the launch chain of
// dense.cu: 3.6 ms in 160 launches).  The backward sweep mirrors it by block columns; forward and backward results
// use different flag values and buffers, so no grid barrier separates the sweeps.  Fixed summation order.
// ---------------------------------------------------------------------------------------
struct WaveArgs {
    const double *L;
    long long ld;
    int m;
    const double *Dinv;
    double *y;
    double *xf, *xb;        // nb x 64 each: published forward / backward block solutions
    unsigned *flag;         // nb: 1 = forward x ready, 2 = backward x ready
    unsigned base;          // flag values of this launch are base + 1, base + 2 (the array is never cleared)
};
#define PW_T 256
#define PW_MAXOWN 4

__device__ __forceinline__ unsigned pw_ld_acquire(const unsigned *p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void pw_st_release(unsigned *p, unsigned v) {
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

template <bool BWD>
__device__ __forceinline__ void wave_sweep(const WaveArgs &a, double *ys, double *xs, double *part, int tid) {
    const int G = (int)gridDim.x, rk = (int)blockIdx.x;
    const int nb = (a.m + 63) / 64;
    const int r = tid & 63, g = tid >> 6;
    double *xg = BWD ? a.xb : a.xf;
    const unsigned ready = a.base + (BWD ? 2u : 1u);
    // the first block of the sweep has no predecessor: its owner publishes it straight away
    {
        const int b0 = BWD ? nb - 1 : 0;
        if (b0 % G == rk) {
            const double *D = a.Dinv + (long long)b0 * 4096;
            tile_gemv<BWD>(D, 64, 64, 64, ys + (b0 / G) * 64, part, tid);
            __syncthreads();
            if (tid < 64) {
                const int kb0 = min(64, a.m - 64 * b0);
                const double xv = (tid < kb0) ? (part[tid] + part[64 + tid]) + (part[128 + tid] + part[192 + tid]) : 0.0;
                ys[(b0 / G) * 64 + tid] = xv;
                xg[(long long)b0 * 64 + tid] = xv;
            }
            __syncthreads();
            if (tid == 0) { __threadfence(); pw_st_release(a.flag + b0, ready); }
        }
    }
    for (int q = 0; q + 1 < nb; ++q) {
        const int b = BWD ? nb - 1 - q : q;
        const int kb = min(64, a.m - 64 * b);
        const int nxt = BWD ? b - 1 : b + 1;
        // owned blocks on the far side of b, nearest first
        int tb[PW_MAXOWN], nt = 0;
        if (BWD) {
            // largest owned block below b, then steps of G
            int blk = (b - 1) - (((b - 1) - rk) % G + G) % G;
            for (; blk >= 0 && nt < PW_MAXOWN; blk -= G) tb[nt++] = blk;
        } else {
            int blk = (b + 1) + ((rk - (b + 1)) % G + G) % G;
            for (; blk < nb && nt < PW_MAXOWN; blk += G) tb[nt++] = blk;
        }
        if (!nt) continue;                                   // uniform per CTA; this CTA has nothing left in this sweep
        double v[PW_MAXOWN][16];
#pragma unroll
        for (int t = 0; t < PW_MAXOWN; ++t) {
            if (t < nt) {
                const int blk = tb[t];
                const int rows = min(64, a.m - 64 * blk);
                const double *T = BWD ? a.L + 64LL * b + 64LL * blk * a.ld : a.L + 64LL * blk + 64LL * b * a.ld;
#pragma unroll
                for (int e = 0; e < 16; ++e) {
                    const int c = 16 * g + e;
                    v[t][e] = (r < rows && c < kb) ? (BWD ? T[c + (long long)r * a.ld] : T[r + (long long)c * a.ld]) : 0.0;
                }
            }
        }
        // (a forward flag may already carry the backward value: the backward x_b exists only after every consumer of the
        // forward x_b has finished its forward sweep, but accept both to be safe -- the forward buffer is never reused)
        if (tid == 0) {
            for (;;) {
                const unsigned f = pw_ld_acquire(a.flag + b);
                if (f == ready || (!BWD && f == a.base + 2u)) break;
            }
        }
        __syncthreads();
        if (tid < 64) xs[tid] = __ldcg(xg + (long long)b * 64 + tid);
        __syncthreads();
#pragma unroll
        for (int t = 0; t < PW_MAXOWN; ++t) {
            if (t < nt) {
                double s0 = 0.0, s1 = 0.0;
#pragma unroll
                for (int e = 0; e < 16; e += 2) {
                    s0 = fma(v[t][e], xs[16 * g + e], s0);
                    s1 = fma(v[t][e + 1], xs[16 * g + e + 1], s1);
                }
                part[t * 256 + g * 64 + r] = s0 + s1;
            }
        }
        __syncthreads();
        {
            const int t = tid >> 6, rr = tid & 63;
            if (t < nt) {
                const double *pp = part + t * 256;
                ys[(tb[t] / G) * 64 + rr] -= (pp[rr] + pp[64 + rr]) + (pp[128 + rr] + pp[192 + rr]);
            }
        }
        __syncthreads();
        if (nxt % G == rk) {
            // the next block is complete: x = Dinv y (backward: Dinv^T y), publish
            const double *D = a.Dinv + (long long)nxt * 4096;
            tile_gemv<BWD>(D, 64, 64, 64, ys + (nxt / G) * 64, part, tid);
            __syncthreads();
            if (tid < 64) {
                const int kbn = min(64, a.m - 64 * nxt);
                const double xv = (tid < kbn) ? (part[tid] + part[64 + tid]) + (part[128 + tid] + part[192 + tid]) : 0.0;
                ys[(nxt / G) * 64 + tid] = xv;
                xg[(long long)nxt * 64 + tid] = xv;
            }
            __syncthreads();
            if (tid == 0) { __threadfence(); pw_st_release(a.flag + nxt, ready); }
        }
    }
}

__global__ void __launch_bounds__(PW_T, 1) potrs_wave_kernel(WaveArgs a) {
    extern __shared__ double pwsm[];
    const int G = (int)gridDim.x, rk = (int)blockIdx.x, tid = threadIdx.x;
    const int nb = (a.m + 63) / 64;
    const int nloc = (nb + G - 1) / G;
    double *ys = pwsm;                    // nloc x 64: the blocks of y this CTA owns
    double *xs = ys + nloc * 64;          // 64: x of the current step
    double *part = xs + 64;               // PW_MAXOWN x 4 x 64 partial sums
    for (int idx = tid; idx < nloc * 64; idx += PW_T) {
        const int b = (idx >> 6) * G + rk;
        const long long i = 64LL * b + (idx & 63);
        ys[idx] = (b < nb && i < a.m) ? a.y[i] : 0.0;
    }
    __syncthreads();
    wave_sweep<false>(a, ys, xs, part, tid);
    __syncthreads();
    wave_sweep<true>(a, ys, xs, part, tid);
    __syncthreads();
    for (int idx = tid; idx < nloc * 64; idx += PW_T) {
        const int b = (idx >> 6) * G + rk;
        const long long i = 64LL * b + (idx & 63);
        if (b < nb && i < a.m) a.y[i] = ys[idx];
    }
}

// from m = 512 on the wavefront beats the 16-CTA cluster kernel as well (m = 1000: 0.22 -> 0.13 ms, m = 4000: 1.75 -> 0.43 ms,
// profiles/r02_v39_potrs_wave_min.log)
static const int64_t POTRS_WAVE_MIN = 512;
bool potrs_wave_for(const smcp_ctx *ctx, int64_t m) {
    const int64_t nb = (m + 63) / 64;
    return m >= POTRS_WAVE_MIN && nb <= (int64_t)PW_MAXOWN * ctx->num_sms;
}

int d_potrs_wave(smcp_ctx *ctx, const double *H, int64_t m, const double *Dinv, double *y_dev) {
    if (m <= 0) return 0;
    const int64_t nb = (m + 63) / 64;
    const int G = (int)std::min<int64_t>(nb, ctx->num_sms);
    const int nloc = (int)((nb + G - 1) / G);
    const size_t need = (size_t)nb * 128 * sizeof(double) + (size_t)nb * sizeof(unsigned) + 64;
    if (need > ctx->wave_cap) {
        if (ctx->wave_buf) cudaFree(ctx->wave_buf);
        ctx->wave_buf = nullptr;
        ctx->wave_cap = 0;
        CUDA_TRY(cudaMalloc(&ctx->wave_buf, need));
        CUDA_TRY(cudaMemsetAsync(ctx->wave_buf, 0, need, ctx->stream));
        ctx->wave_cap = need;
        ctx->wave_epoch = 0;
    }
    WaveArgs a;
    a.L = H; a.ld = m; a.m = (int)m; a.Dinv = Dinv; a.y = y_dev;
    a.xf = (double *)ctx->wave_buf;
    a.xb = a.xf + nb * 64;
    a.flag = (unsigned *)(a.xb + nb * 64);
    // the flag array sits behind the two solution buffers, so its place depends on the order of the matrix: start from
    // clean flags whenever the order changes (and before the epoch counter wraps)
    if (ctx->wave_epoch > 0xfffffff0u || ctx->wave_nb != nb) {
        CUDA_TRY(cudaMemsetAsync(ctx->wave_buf, 0, need, ctx->stream));
        ctx->wave_epoch = 0;
        ctx->wave_nb = nb;
    }
    a.base = ctx->wave_epoch;
    ctx->wave_epoch += 2;
    const size_t smem = (size_t)(nloc * 64 + 64 + PW_MAXOWN * 256) * sizeof(double);
    void *args[] = {&a};
    LaunchScope ls(ctx, "potrs", 1, 8.0 * (double)m * (double)m);
    CUDA_TRY(cudaLaunchCooperativeKernel((void *)potrs_wave_kernel, dim3((unsigned)G), dim3(PW_T), args, smem, ctx->stream));
    return 0;
}

int d_potrs_prepare(smcp_ctx *ctx, const double *H, int64_t ld, int64_t m, double *Dinv) {
    if (m <= 0) return 0;
    LaunchScope ls(ctx, "potrs_trtri");
    trtri64_kernel<<<(unsigned)((m + 63) / 64), 64, 0, ctx->stream>>>(H, ld, m, Dinv);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// One cluster (16 SMs at most) streams the whole factor: fine while it sits in L2 and the solve is a
// latency chain (m = 1000: 0.09 ms against 0.24), slower than the many-SM streamed updates of dense.cu
// once the factor is hundreds of MB (m = 10^4: 5.1 ms against 3.6)
bool potrs_cluster_for(int64_t m) { return m <= 4096; }

int d_potrs_cluster(smcp_ctx *ctx, const double *H, int64_t m, const double *Dinv, double *y_dev) {
    return d_trs_cluster(ctx, H, m, m, Dinv, y_dev, m, 1, 1, 1, "potrs");
}

// L^-1 and / or L^-T applied to a few right-hand sides (columns of y); L lower triangular n x n (leading
// dimension ld) whose inverted 64 x 64 diagonal blocks are in Dinv (d_potrs_prepare)
int d_trs_cluster(smcp_ctx *ctx, const double *H, int64_t ld, int64_t m, const double *Dinv, double *y_dev, int64_t ldy, int64_t nrhs,
                  int do_fwd, int do_bwd, const char *name) {
    if (m <= 0 || nrhs <= 0) return 0;
    const int nb = (int)((m + 63) / 64);
    int R = nb >= 64 ? 16 : 8;
    if (R > nb) R = std::max(1, nb);
    // cluster sizes must divide the grid; powers of two up to 16
    int Rp = 1;
    while (Rp * 2 <= R) Rp *= 2;
    R = Rp;
    const int nloc = (nb + R - 1) / R;
    const size_t smem = (size_t)(nloc * 64 + 128 + 1024) * sizeof(double);
    static bool attr = false;
    if (!attr) {
        CUDA_TRY(cudaFuncSetAttribute(potrs_cluster_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
        CUDA_TRY(cudaFuncSetAttribute(potrs_cluster_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        attr = true;
    }
    if (smem > 200 * 1024) { smcp_set_error("d_potrs_cluster: m too large"); return -2; }
    PotrsArgs a;
    a.L = H; a.ld = ld; a.m = (int)m; a.Dinv = Dinv; a.y = y_dev;
    a.ldy = ldy; a.nrhs = (int)nrhs; a.do_fwd = do_fwd; a.do_bwd = do_bwd;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)R);
    cfg.blockDim = dim3(PC_T);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = ctx->stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = (unsigned)R;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    LaunchScope ls(ctx, name, 1, 4.0 * (double)m * (double)m * (double)nrhs * (do_fwd + do_bwd));
    CUDA_TRY(cudaLaunchKernelEx(&cfg, potrs_cluster_kernel, a));
    return 0;
}
