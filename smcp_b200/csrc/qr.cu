// Blocked Householder QR of a tall-skinny FP64 matrix (lapack.geqrf / lapack.orgqr, the factorisation behind
// the reference's kkt_qr, src/python/solvers.py:413-475, 1843-1904) with LAPACK's conventions: the Householder
// vectors below the diagonal with an implicit unit diagonal, beta = -sign(alpha) * ||(alpha, x)||, and tau.
//
//  * panel (qr_panel_kernel, cooperative launch): nb = 32 columns, each CTA owns a contiguous slab of rows,
//    kept in shared memory when it fits and read from global memory otherwise.  Every column takes two
//    grid-wide reductions (the norm, then v^T A for the rest of the panel): per-CTA partial sums, a grid
//    barrier, and the same fixed-order sum in every CTA, so all CTAs hold the same bits and no floating-point
//    atomics are needed.  The kernel also forms the triangular factor T of the block reflector (dlarft,
//    forward / columnwise) from a third reduction, the Gram matrix V^T V, and writes V with its explicit
//    ones and zeros and Y = V T^T (geqrf) or Y = V T (orgqr) to a workspace.
//  * trailing update (qr_wy_dmma): Q_p^T C = C - V T^T V^T C = C - Y (V^T C) with the FP64 tensor-core
//    GEMM of dense.cu / gemm_tma.cu (K = the remaining rows for V^T C, K = nb for the update).
//  * orgqr: the same block reflectors applied backwards to [I; 0], in place of the Householder vectors
//    (the panel kernel rebuilds T and Y from V and tau before the panel's columns are overwritten).
#include "internal.cuh"
#include <algorithm>

#define QR_NB 32
#define QR_T 256
#define QR_SLAB_BYTES (160 * 1024)                 // shared-memory slab budget of the panel kernel
#define QR_PART (1 + QR_NB + QR_NB * QR_NB + 1)    // per-CTA partial sums: norm | v^T A | Gram | alpha

struct QrPanelArgs {
    double *A;            // the panel: A[r + c*lda], r in [0, mp), c in [0, jb) (row / column j0 of the matrix)
    long long lda, mp;
    int jb;
    int factor;           // 1: factor the panel (geqrf); 0: V and tau given (orgqr), only T, V, Y are formed
    int ytrans;           // 1: Y = V T^T (geqrf update, Q^T C); 0: Y = V T (orgqr, Q C)
    double *tau;          // jb entries: written (factor) or read
    double *V, *Y;        // mp x jb explicit V and Y, leading dimension ldw
    long long ldw;
    double *part;         // gridDim.x x QR_PART partial sums
    unsigned *bar;        // grid-barrier counter, zero at launch
    long long S;          // rows per CTA (>= jb: CTA 0 owns the rows of R)
    int use_smem;         // the slab lives in shared memory (leading dimension S | 1)
};

__device__ __forceinline__ unsigned qr_ld_acquire(const unsigned *p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
// barrier over the co-resident grid (cooperative launch): one arrival per CTA on a monotone counter
__device__ __forceinline__ void qr_grid_barrier(unsigned *ctr, unsigned &target) {
    __syncthreads();
    if (threadIdx.x == 0) {
        target += gridDim.x;
        __threadfence();
        atomicAdd(ctr, 1u);
        while (qr_ld_acquire(ctr) < target) { }
    }
    __syncthreads();
}

// sum over the CTA in a fixed order; the result is returned to every thread
__device__ __forceinline__ double qr_block_sum(double s, double *red) {
    for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    double t = 0.0;
    for (int w = 0; w < QR_T / 32; ++w) t += red[w];
    return t;
}

__global__ void __launch_bounds__(QR_T, 1) qr_panel_kernel(QrPanelArgs a) {
    extern __shared__ double qr_slab[];
    __shared__ double red[QR_T / 32][QR_NB];
    __shared__ double wk[QR_NB];
    __shared__ double T[QR_NB][QR_NB + 1];
    __shared__ double gram[QR_NB][QR_NB + 1];
    __shared__ double sc[4];
    __shared__ double taus[QR_NB];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int jb = a.jb;
    const long long r0 = (long long)blockIdx.x * a.S;
    const long long nloc = max(0LL, min(a.mp, r0 + a.S) - r0);
    double *part = a.part + (size_t)blockIdx.x * QR_PART;
    unsigned target = 0;
    double *P;
    long long ld;
    if (a.use_smem) {
        P = qr_slab;
        ld = a.S | 1;
        for (int c = 0; c < jb; ++c)
            for (long long i = tid; i < nloc; i += QR_T) P[i + c * ld] = a.A[r0 + i + c * a.lda];
    } else {
        P = a.A + r0;
        ld = a.lda;
    }
    __syncthreads();

    if (!a.factor && tid < jb) taus[tid] = a.tau[tid];
    if (a.factor) {
        for (int c = 0; c < jb; ++c) {
            // (a) squared norm of the part of column c below the diagonal; CTA 0 also publishes alpha = A(c, c)
            double s = 0.0;
            for (long long i = tid; i < nloc; i += QR_T)
                if (r0 + i > c) { const double x = P[i + c * ld]; s = fma(x, x, s); }
            s = qr_block_sum(s, &red[0][0]);
            if (tid == 0) {
                __stcg(part, s);
                if (blockIdx.x == 0) __stcg(part + QR_PART - 1, P[c + c * ld]);
            }
            qr_grid_barrier(a.bar, target);
            if (tid == 0) {
                double sigma = 0.0;
                for (unsigned b = 0; b < gridDim.x; ++b) sigma += __ldcg(a.part + (size_t)b * QR_PART);
                const double alpha = __ldcg(a.part + QR_PART - 1);
                double beta = alpha, tau = 0.0, scal = 1.0;
                if (sigma > 0.0) {
                    beta = -copysign(sqrt(fma(alpha, alpha, sigma)), alpha);
                    tau = (beta - alpha) / beta;
                    scal = 1.0 / (alpha - beta);
                }
                sc[0] = beta; sc[1] = tau; sc[2] = scal;
                if (blockIdx.x == 0) a.tau[c] = tau;
                taus[c] = tau;
            }
            __syncthreads();
            const double beta = sc[0], tau = sc[1], scal = sc[2];
            // (b) v = x / (alpha - beta) below the diagonal, R(c, c) = beta
            for (long long i = tid; i < nloc; i += QR_T) {
                const long long r = r0 + i;
                if (r == c) P[i + c * ld] = beta;
                else if (r > c) P[i + c * ld] *= scal;
            }
            __syncthreads();
            // (c) partial sums of v^T A(:, k) for the columns k > c of the panel (v_c = 1): thread (row group
            // warp, column lane) walks the rows warp, warp + 8, ... of its column
            {
                double t = 0.0;
                if (lane > c && lane < jb)
                    for (long long i = warp; i < nloc; i += QR_T / 32) {
                        const long long r = r0 + i;
                        if (r < c) continue;
                        t = fma(r == c ? 1.0 : P[i + c * ld], P[i + lane * ld], t);
                    }
                red[warp][lane] = t;
            }
            __syncthreads();
            if (tid < jb) {
                double t = 0.0;
                for (int w = 0; w < QR_T / 32; ++w) t += red[w][tid];
                __stcg(part + 1 + tid, t);
            }
            qr_grid_barrier(a.bar, target);
            if (tid < jb) {
                double t = 0.0;
                for (unsigned b = 0; b < gridDim.x; ++b) t += __ldcg(a.part + (size_t)b * QR_PART + 1 + tid);
                wk[tid] = t;
            }
            __syncthreads();
            // (d) A(:, k) -= tau v (v^T A(:, k)), k > c, in the layout of (c)
            if (tau != 0.0 && lane > c && lane < jb) {
                const double tw = tau * wk[lane];
                for (long long i = warp; i < nloc; i += QR_T / 32) {
                    const long long r = r0 + i;
                    if (r < c) continue;
                    P[i + lane * ld] = fma(-tw, r == c ? 1.0 : P[i + c * ld], P[i + lane * ld]);
                }
            }
            __syncthreads();
        }
    }

    // Gram matrix V^T V of the explicit V (unit diagonal, zeros above): partial sums of the entries (i, k), i < k
    {
        double g4[QR_NB * QR_NB / QR_T];
#pragma unroll
        for (int q = 0; q < QR_NB * QR_NB / QR_T; ++q) g4[q] = 0.0;
        for (long long i = 0; i < nloc; ++i) {
            const long long r = r0 + i;
#pragma unroll
            for (int q = 0; q < QR_NB * QR_NB / QR_T; ++q) {
                const int e = tid + q * QR_T, ii = e % QR_NB, kk = e / QR_NB;
                if (ii < kk && kk < jb && r >= kk) {
                    const double vi = r == ii ? 1.0 : P[i + ii * ld];
                    const double vk = r == kk ? 1.0 : P[i + kk * ld];
                    g4[q] = fma(vi, vk, g4[q]);
                }
            }
        }
#pragma unroll
        for (int q = 0; q < QR_NB * QR_NB / QR_T; ++q) __stcg(part + 1 + QR_NB + tid + q * QR_T, g4[q]);
    }
    qr_grid_barrier(a.bar, target);
#pragma unroll
    for (int q = 0; q < QR_NB * QR_NB / QR_T; ++q) {
        const int e = tid + q * QR_T, ii = e % QR_NB, kk = e / QR_NB;
        double t = 0.0;
        if (ii < kk && kk < jb)
            for (unsigned b = 0; b < gridDim.x; ++b) t += __ldcg(a.part + (size_t)b * QR_PART + 1 + QR_NB + e);
        gram[ii][kk] = t;
    }
    // T (dlarft, forward, columnwise): T(i, i) = tau_i, T(0:i, i) = -tau_i T(0:i, 0:i) V(:, 0:i)^T v_i
    for (int e = tid; e < QR_NB * QR_NB; e += QR_T) T[e % QR_NB][e / QR_NB] = 0.0;
    __syncthreads();
    for (int i = 0; i < jb; ++i) {
        const double ti = taus[i];
        if (tid < i) {
            double t = 0.0;
            for (int l = tid; l < i; ++l) t = fma(T[tid][l], gram[l][i], t);
            T[tid][i] = -ti * t;
        }
        if (tid == i) T[i][i] = ti;
        __syncthreads();
    }
    // the matrix Y is multiplied by: Tm[k][l] = T(k, l) (Y = V T^T) or T(l, k) (Y = V T)
    for (int e = tid; e < QR_NB * QR_NB; e += QR_T) {
        const int k = e / QR_NB, l = e % QR_NB;
        gram[k][l] = a.ytrans ? T[k][l] : T[l][k];
    }
    __syncthreads();
    // explicit V and Y = V T^T (ytrans) or V T, row by row
    for (long long i = tid; i < nloc; i += QR_T) {
        const long long r = r0 + i;
        double v[QR_NB];
#pragma unroll
        for (int l = 0; l < QR_NB; ++l) v[l] = (l >= jb || r < l) ? 0.0 : (r == l ? 1.0 : P[i + l * ld]);
        for (int k = 0; k < jb; ++k) {
            double y = 0.0;
#pragma unroll
            for (int l = 0; l < QR_NB; ++l) y = fma(v[l], gram[k][l], y);
            a.Y[r + k * a.ldw] = y;
        }
#pragma unroll
        for (int k = 0; k < QR_NB; ++k)
            if (k < jb) a.V[r + k * a.ldw] = v[k];
    }
    if (a.factor && a.use_smem) {
        __syncthreads();
        for (int c = 0; c < jb; ++c)
            for (long long i = tid; i < nloc; i += QR_T) a.A[r0 + i + c * a.lda] = P[i + c * ld];
    }
    if (!a.factor) {
        // orgqr: the panel's columns become the columns of [I; 0] the block reflector is applied to
        __syncthreads();
        for (int c = 0; c < jb; ++c)
            for (long long i = tid; i < nloc; i += QR_T) a.A[r0 + i + c * a.lda] = (r0 + i == c) ? 1.0 : 0.0;
    }
}

static int qr_panel(smcp_ctx *ctx, double *A, int64_t lda, int64_t mp, int jb, int factor, double *tau, double *V, double *Y,
                    int64_t ldw, double *part, int gmax) {
    // CTAs own at least 64 rows (>= jb: the rows of R stay in CTA 0)
    int G = (int)std::max<int64_t>(1, std::min<int64_t>(gmax, mp / 64));
    long long S = (mp + G - 1) / G;
    const bool use_smem = (size_t)((S | 1) * jb) * sizeof(double) <= QR_SLAB_BYTES;
    const size_t smem = use_smem ? (size_t)((S | 1) * jb) * sizeof(double) : 0;
    QrPanelArgs a;
    a.A = A; a.lda = lda; a.mp = mp; a.jb = jb; a.factor = factor; a.ytrans = factor;
    a.tau = tau; a.V = V; a.Y = Y; a.ldw = ldw; a.part = part; a.S = S; a.use_smem = use_smem ? 1 : 0;
    if (!ctx->gridbar) {
        CUDA_TRY(cudaMalloc(&ctx->gridbar, 64 * 64));
        CUDA_TRY(cudaMemset(ctx->gridbar, 0, 64 * 64));
    }
    a.bar = ctx->gridbar + 16 * (ctx->gridbar_next++ & 63);
    CUDA_TRY(cudaMemsetAsync(a.bar, 0, sizeof(unsigned), ctx->stream));
    void *args[] = {&a};
    LaunchScope ls(ctx, "qr_panel", 1, factor ? 4.0 * (double)mp * jb * jb : 2.0 * (double)mp * jb * jb);
    CUDA_TRY(cudaLaunchCooperativeKernel((void *)qr_panel_kernel, dim3((unsigned)G), dim3(QR_T), args, smem, ctx->stream));
    return 0;
}

// workspace of one factorisation: V | Y (ldw x nb each) | W (nb x N) | partial sums (gmax x QR_PART); returns gmax
static int qr_workspace(smcp_ctx *ctx, int64_t M, int64_t N, int64_t *ldw, double **V, double **Y, double **W, double **part) {
    static bool attr = false;
    if (!attr) {
        CUDA_TRY(cudaFuncSetAttribute(qr_panel_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, QR_SLAB_BYTES));
        attr = true;
    }
    // every CTA of the cooperative panel kernel must be resident: the grid never exceeds what the occupancy
    // query reports for the largest slab (one CTA per SM)
    int per_sm = 0;
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, qr_panel_kernel, QR_T, QR_SLAB_BYTES));
    if (per_sm < 1) { smcp_set_error("qr_panel_kernel: no CTA fits on an SM"); return -1; }
    const int gmax = std::min(ctx->num_sms, ctx->num_sms * per_sm);
    *ldw = (M + 1) & ~1LL;
    const size_t need = (size_t)(2 * *ldw * QR_NB + QR_NB * N + (int64_t)gmax * QR_PART) * sizeof(double);
    if (grow((void **)&ctx->qr_ws, &ctx->qr_ws_cap, need)) return -1;
    *V = ctx->qr_ws;
    *Y = *V + *ldw * QR_NB;
    *W = *Y + *ldw * QR_NB;
    *part = *W + QR_NB * N;
    return gmax;
}

int d_geqrf(smcp_ctx *ctx, double *A, int64_t lda, int64_t M, int64_t N, double *tau) {
    if (N <= 0) return 0;
    if (M < N || lda < M) { smcp_set_error("d_geqrf: needs M >= N and lda >= M"); return -2; }
    int64_t ldw;
    double *V, *Y, *W, *part;
    const int gmax = qr_workspace(ctx, M, N, &ldw, &V, &Y, &W, &part);
    if (gmax < 0) return -1;
    for (int64_t j0 = 0; j0 < N; j0 += QR_NB) {
        const int jb = (int)std::min<int64_t>(QR_NB, N - j0);
        const int64_t mp = M - j0, nc = N - j0 - jb;
        double *Ap = A + j0 + j0 * lda;
        if (qr_panel(ctx, Ap, lda, mp, jb, 1, tau + j0, V, Y, ldw, part, gmax)) return -1;
        if (nc > 0) {
            double *C = Ap + jb * lda;
            // W = V^T C (jb x nc), then C -= Y W with Y = V T^T
            if (launch_gemm(ctx, true, true, V, ldw, C, lda, W, jb, jb, nc, mp, 1.0, 0, 0, 0, "qr_wy_dmma")) return -1;
            if (launch_gemm(ctx, false, true, Y, ldw, W, jb, C, lda, mp, nc, jb, -1.0, 1, 0, 0, "qr_wy_dmma")) return -1;
        }
    }
    CUDA_TRY(cudaGetLastError());
    return 0;
}

int d_orgqr(smcp_ctx *ctx, double *A, int64_t lda, int64_t M, int64_t N, const double *tau) {
    if (N <= 0) return 0;
    if (M < N || lda < M) { smcp_set_error("d_orgqr: needs M >= N and lda >= M"); return -2; }
    int64_t ldw;
    double *V, *Y, *W, *part;
    const int gmax = qr_workspace(ctx, M, N, &ldw, &V, &Y, &W, &part);
    if (gmax < 0) return -1;
    const int64_t np = (N + QR_NB - 1) / QR_NB;
    for (int64_t p = np - 1; p >= 0; --p) {
        const int64_t j0 = p * QR_NB;
        const int jb = (int)std::min<int64_t>(QR_NB, N - j0);
        const int64_t mp = M - j0, nc = N - j0;
        double *Ap = A + j0 + j0 * lda;
        // rows above the panel: the R entries become the zeros of [I; 0]
        if (j0 > 0) CUDA_TRY(cudaMemset2DAsync(A + j0 * lda, (size_t)lda * sizeof(double), 0, (size_t)j0 * sizeof(double), (size_t)jb, ctx->stream));
        // V and T of panel p, then its columns set to [I; 0]
        if (qr_panel(ctx, Ap, lda, mp, jb, 0, const_cast<double *>(tau) + j0, V, Y, ldw, part, gmax)) return -1;
        // Q(j0:, j0:) = (I - V T V^T) Q(j0:, j0:):  W = V^T Q, Q -= Y W with Y = V T
        if (launch_gemm(ctx, true, true, V, ldw, Ap, lda, W, jb, jb, nc, mp, 1.0, 0, 0, 0, "qr_wy_dmma")) return -1;
        if (launch_gemm(ctx, false, true, Y, ldw, W, jb, Ap, lda, mp, nc, jb, -1.0, 1, 0, 0, "qr_wy_dmma")) return -1;
    }
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// ---------------------------------------------------------------------------------------
// R of Z = Q1 R to the lower factor L = R^T with diag(L) >= 0 (rows of R with a negative diagonal entry and
// the matching columns of Q1 change sign), and the rank test of the QR form of kktsolver='qr'
// ---------------------------------------------------------------------------------------
__global__ void qr_rank_kernel(const double *__restrict__ A, long long lda, long long m, double *__restrict__ sgn, int *info) {
    __shared__ double red[QR_T / 32];
    double mx = 0.0;
    for (long long i = threadIdx.x; i < m; i += QR_T) {
        const double d = A[i + i * lda];
        sgn[i] = d < 0.0 ? -1.0 : 1.0;
        mx = fmax(mx, fabs(d));
    }
    for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_down_sync(0xffffffffu, mx, o));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = mx;
    __syncthreads();
    if (threadIdx.x == 0) {
        double g = 0.0;
        for (int w = 0; w < QR_T / 32; ++w) g = fmax(g, red[w]);
        int k = 0;
        for (long long i = 0; i < m && !k; ++i) {
            const double d = fabs(A[i + i * lda]);
            if (!(d > 1e-14 * g) || !isfinite(d)) k = (int)(i + 1);      // NaN fails too
        }
        *info = k;
    }
}
// L[j + i*ldl] = sgn[i] R(i, j), j >= i
__global__ void qr_lower_kernel(const double *__restrict__ A, long long lda, long long m, const double *__restrict__ sgn,
                                double *__restrict__ L, long long ldl) {
    const long long total = m * m;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const long long j = idx % m, i = idx / m;
        if (j >= i) L[j + i * ldl] = sgn[i] * A[i + j * lda];
    }
}
__global__ void qr_colsign_kernel(double *__restrict__ A, long long lda, long long M, long long N, const double *__restrict__ sgn) {
    const long long total = M * N;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const long long r = idx % M, c = idx / M;
        if (sgn[c] < 0.0) A[r + c * lda] = -A[r + c * lda];
    }
}

int qr_extract_lower(smcp_ctx *ctx, const double *A, int64_t lda, int64_t m, double *L, int64_t ldl, double *sgn, int *info_dev) {
    if (m <= 0) return 0;
    LaunchScope ls(ctx, "qr_qmul", 2);
    qr_rank_kernel<<<1, QR_T, 0, ctx->stream>>>(A, lda, m, sgn, info_dev);
    qr_lower_kernel<<<ctx->num_sms * 4, 256, 0, ctx->stream>>>(A, lda, m, sgn, L, ldl);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

int qr_apply_colsign(smcp_ctx *ctx, double *A, int64_t lda, int64_t M, int64_t N, const double *sgn) {
    if (M <= 0 || N <= 0) return 0;
    LaunchScope ls(ctx, "qr_qmul");
    qr_colsign_kernel<<<ctx->num_sms * 8, 256, 0, ctx->stream>>>(A, lda, M, N, sgn);
    CUDA_TRY(cudaGetLastError());
    return 0;
}
