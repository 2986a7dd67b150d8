// Dense FP64 kernels for the m x m Schur complement H: tensor-core GEMM (DMMA), blocked
// Cholesky (lapack.potrf, src/python/solvers.py:501, 1931) and the two triangular solves of
// lapack.potrs (solvers.py:526, 1954).
//
// FP64 has no tcgen05/UMMA kind on sm_100a; the FP64 tensor path is mma.sync.m8n8k4.f64
// (SASS: DMMA.8x8x4).  The GEMM below stages K-major operand tiles in shared memory with a
// 3-stage cp.async pipeline, pads the tile rows so the per-thread 8-byte fragment loads
// are bank-conflict free, and keeps a 32x32 accumulator tile per warp in registers (16 warps per CTA).
#include "internal.cuh"
#include <algorithm>

// ---------------------------------------------------------------------------------------
// DMMA GEMM:  C(i, j) = [C(i, j) +] alpha * sum_k A'(i, k) B'(j, k)
//   TA = true : A'(i, k) = A[k + i*lda] (K contiguous)     TA = false: A'(i, k) = A[i + k*lda]
//   TB = true : B'(j, k) = B[k + j*ldb] (K contiguous)     TB = false: B'(j, k) = B[j + k*ldb]
//   (true, true) = A^T B: Schur assembly; (false, false) = A B^T: SYRK-like updates;
//   (false, true) = A B and (true, false) = A^T B^T: frontal updates of large supernodes
// tri: only tiles that intersect {i + tri_off >= j} are computed (lower triangle).
// ---------------------------------------------------------------------------------------
#define BM 128
#define BN 128
#define BK 16
#define LDK (BK + 4)       // 20 doubles: rows shifted by 4 banks -> conflict-free fragments
#define STAGES 3
#define GEMM_THREADS 512       // 16 warps: 4 x 4 warp tiles of 32 x 32 (4 warps per scheduler keep the DMMA pipe fed)

__device__ __forceinline__ void cp_async8(void *smem, const void *gmem) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N)); }

__device__ __forceinline__ void dmma(double &c0, double &c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

// m16n8k8 FP64 tensor-core MMA (sm_90+; SASS DMMA.16x8x8).  Fragments (PTX ISA / CuTe
// SM90_16x8x8_F64F64F64F64_TN): g = lane >> 2, t = lane & 3;
//   a[v]: row g + 8*(v & 1), k = t + 4*(v >> 1);  b[v]: col g, k = t + 4*v;
//   c[v]: row g + 8*(v >> 1), col 2*t + (v & 1).
__device__ __forceinline__ void dmma16x8x8(double (&c)[4], const double (&a)[4], const double (&b)[2]) {
    asm volatile("mma.sync.aligned.m16n8k8.row.col.f64.f64.f64.f64 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+d"(c[0]), "+d"(c[1]), "+d"(c[2]), "+d"(c[3])
                 : "d"(a[0]), "d"(a[1]), "d"(a[2]), "d"(a[3]), "d"(b[0]), "d"(b[1]));
}

template <bool TN>
__device__ __forceinline__ void load_tile(double *sm, const double *G, long long ld, long long row0,
                                          long long nrows, long long k0, long long K, int tid) {
    // fills sm[r*LDK + k] for r in [0,128), k in [0,BK) with op(G)(row0+r, k0+k) or 0
    if (TN) {
        // G(k, r) at G[k + r*ld]; consecutive threads walk k (contiguous)
        for (int idx = tid; idx < 128 * BK; idx += GEMM_THREADS) {
            int k = idx % BK, r = idx / BK;
            double *dst = sm + r * LDK + k;
            if (row0 + r < nrows && k0 + k < K) cp_async8(dst, G + (k0 + k) + (row0 + r) * ld);
            else *dst = 0.0;
        }
    } else {
        // G(r, k) at G[r + k*ld]; consecutive threads walk r (contiguous)
        for (int idx = tid; idx < 128 * BK; idx += GEMM_THREADS) {
            int r = idx % 128, k = idx / 128;
            double *dst = sm + r * LDK + k;
            if (row0 + r < nrows && k0 + k < K) cp_async8(dst, G + (row0 + r) + (k0 + k) * ld);
            else *dst = 0.0;
        }
    }
}

template <bool TA, bool TB>
__global__ void __launch_bounds__(GEMM_THREADS)
gemm_dmma_kernel(const double *__restrict__ A, long long lda, const double *__restrict__ B, long long ldb,
                 double *__restrict__ C, long long ldc, long long M, long long N, long long K, double alpha,
                 int accumulate, int tri, long long tri_off, long long kchunk, long long split_stride,
                 int jt0, int jtstride, int jtb, long long bsA, long long bsB, int batched) {
    extern __shared__ double smem[];
    double *As = smem;                              // STAGES x 128 x LDK
    double *Bs = smem + STAGES * 128 * LDK;
    const long long i0 = (long long)blockIdx.x * BM;
    // column blocks jt0, jt0 + jtstride, ... of jtb tiles each: the block-cyclic owner of a column block
    // updates only its own tiles
    const long long j0 = (((long long)jt0 + (long long)(blockIdx.y / jtb) * jtstride) * jtb + (blockIdx.y % jtb)) * BN;
    if (j0 >= N) return;
    if (tri && (i0 + BM - 1 + tri_off < j0)) return;        // tile entirely above the diagonal
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wm = (warp & 3) * 32;       // 4 warps along M
    const int wn = (warp >> 2) * 32;      // 4 warps along N
    const int g = lane >> 2, t = lane & 3;
    // diagonal tiles of a triangular product: warp tiles entirely above the diagonal only help with the loads
    const bool wskip = tri && (i0 + wm + 31 + tri_off < j0 + wn);

    double acc[2][4][4];           // 2 x 4 tiles of 16 x 8 per warp (32 x 32)
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b)
#pragma unroll
            for (int v = 0; v < 4; ++v) acc[a][b][v] = 0.0;

    // split-K: slice blockIdx.z works on k in [kbeg, kend) and writes its own partial result;
    // batched: blockIdx.z is the matrix index and split_stride the stride of C
    const long long kbeg = batched ? 0 : (long long)blockIdx.z * kchunk;
    const long long kend = (kbeg + kchunk < K) ? kbeg + kchunk : K;
    C += (long long)blockIdx.z * split_stride;
    if (batched) {
        A += (long long)blockIdx.z * bsA;
        B += (long long)blockIdx.z * bsB;
    }
    const long long nk = (kend - kbeg + BK - 1) / BK;
    for (int s = 0; s < STAGES - 1; ++s) {
        if (s < nk) {
            load_tile<TA>(As + s * 128 * LDK, A, lda, i0, M, kbeg + (long long)s * BK, kend, tid);
            load_tile<TB>(Bs + s * 128 * LDK, B, ldb, j0, N, kbeg + (long long)s * BK, kend, tid);
        }
        cp_async_commit();
    }
    for (long long kt = 0; kt < nk; ++kt) {
        cp_async_wait<STAGES - 2>();
        __syncthreads();
        {
            long long nx = kt + STAGES - 1;
            if (nx < nk) {
                int s = (int)(nx % STAGES);
                load_tile<TA>(As + s * 128 * LDK, A, lda, i0, M, kbeg + nx * BK, kend, tid);
                load_tile<TB>(Bs + s * 128 * LDK, B, ldb, j0, N, kbeg + nx * BK, kend, tid);
            }
            cp_async_commit();
        }
        const double *as = As + (kt % STAGES) * 128 * LDK;
        const double *bs = Bs + (kt % STAGES) * 128 * LDK;
        if (wskip) continue;
#pragma unroll
        for (int kk = 0; kk < BK; kk += 8) {
            double af[2][4], bf[4][2];
#pragma unroll
            for (int a = 0; a < 2; ++a)
#pragma unroll
                for (int v = 0; v < 4; ++v) af[a][v] = as[(wm + a * 16 + g + 8 * (v & 1)) * LDK + kk + t + 4 * (v >> 1)];
#pragma unroll
            for (int b = 0; b < 4; ++b)
#pragma unroll
                for (int v = 0; v < 2; ++v) bf[b][v] = bs[(wn + b * 8 + g) * LDK + kk + t + 4 * v];
#pragma unroll
            for (int a = 0; a < 2; ++a)
#pragma unroll
                for (int b = 0; b < 4; ++b) dmma16x8x8(acc[a][b], af[a], bf[b]);
        }
    }
    cp_async_wait<0>();
    if (wskip) return;
    // epilogue: C(i, j), i = i0 + wm + a*16 + g + 8*(v>>1), j = j0 + wn + b*8 + 2t + (v&1)
#pragma unroll
    for (int a = 0; a < 2; ++a) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            long long i = i0 + wm + a * 16 + g + 8 * h;
            if (i >= M) continue;
#pragma unroll
            for (int b = 0; b < 4; ++b) {
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    long long j = j0 + wn + b * 8 + 2 * t + e;
                    if (j >= N) continue;
                    if (tri && i + tri_off < j) continue;
                    double *c = C + i + j * ldc;
                    double v = alpha * acc[a][b][2 * h + e];
                    *c = accumulate ? (*c + v) : v;
                }
            }
        }
    }
}

// sum of the split-K partial results in a fixed order (deterministic), lower part only when tri
__global__ void splitk_reduce_kernel(const double *__restrict__ P, long long split_stride, int splits, double *__restrict__ C,
                                     long long ldc, long long M, long long N, int tri, long long tri_off) {
    const long long total = M * N;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const long long i = idx % M, j = idx / M;
        if (tri && i + tri_off < j) continue;
        double s = 0.0;
        for (int z = 0; z < splits; ++z) s += P[(long long)z * split_stride + idx];
        C[i + j * ldc] = s;
    }
}

// K <= 16 (rank-k updates of the thin supernodes of a top set: nn = 1 .. 9 columns over a ~1100-row
// separator): the product is bound by reading and writing C, a 128 x 128 DMMA tile with a 3-stage
// pipeline is all overhead.  32 x 32 outputs per CTA, operands staged in shared memory once.
#define SK_MAX 16
template <bool TA, bool TB>
__global__ void __launch_bounds__(256) gemm_smallk_kernel(const double *__restrict__ A, long long lda, const double *__restrict__ B, long long ldb,
                                                          double *__restrict__ C, long long ldc, long long M, long long N, int K, double alpha,
                                                          int accumulate, int tri, long long tri_off) {
    __shared__ double As[SK_MAX][33], Bs[SK_MAX][33];
    const long long i0 = (long long)blockIdx.x * 32, j0 = (long long)blockIdx.y * 32;
    if (tri && i0 + 31 + tri_off < j0) return;
    const int tid = threadIdx.x;
    for (int idx = tid; idx < 32 * K; idx += 256) {
        // TA: A'(i, k) = A[k + i*lda] (k contiguous); else A[i + k*lda] (i contiguous)
        const int r = TA ? idx / K : idx % 32, k = TA ? idx % K : idx / 32;
        As[k][r] = (i0 + r < M) ? (TA ? A[k + (i0 + r) * lda] : A[(i0 + r) + (long long)k * lda]) : 0.0;
    }
    for (int idx = tid; idx < 32 * K; idx += 256) {
        const int r = TB ? idx / K : idx % 32, k = TB ? idx % K : idx / 32;
        Bs[k][r] = (j0 + r < N) ? (TB ? B[k + (j0 + r) * ldb] : B[(j0 + r) + (long long)k * ldb]) : 0.0;
    }
    __syncthreads();
    const int tx = tid & 31, ty = tid >> 5;
    const long long i = i0 + tx;
    if (i >= M) return;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const int jj = ty + 8 * q;
        const long long j = j0 + jj;
        if (j >= N || (tri && i + tri_off < j)) continue;
        double s = 0.0;
        for (int k = 0; k < K; ++k) s = fma(As[k][tx], Bs[k][jj], s);
        double *c = C + i + j * ldc;
        const double v = alpha * s;
        *c = accumulate ? (*c + v) : v;
    }
}

// N <= 16 with a long K (a thin supernode against its ~1100-row separator: M_an = Y_aa K_an D^-1,
// Z_an = M_an - Z_aa Lt, ...): a matrix times a few vectors.  The product is bound by streaming A
// once; a 128 x 128 DMMA tile would use 1/128 of its columns and a single wave of 9 CTAs.
//   TA = false (A[i + k*lda]): a CTA owns 32 rows, its 8 warps split K, lane = row (coalesced);
//   TA = true  (A[k + i*lda]): a warp owns a row, lanes stride over K (coalesced).
// Partial sums are combined in a fixed order (bitwise reproducible).
#define TN_MAX 16
#define TN_KC 128      // k-chunk of B staged in shared memory
template <bool TA, bool TB>
__global__ void __launch_bounds__(256) gemm_thin_kernel(const double *__restrict__ A, long long lda, const double *__restrict__ B, long long ldb,
                                                        double *__restrict__ C, long long ldc, long long M, int N, long long K, double alpha,
                                                        int accumulate) {
    __shared__ double tnsm[8 * 32 * TN_MAX];                                   // the B chunk, then the partial sums
    double (*Bs)[TN_MAX + 1] = reinterpret_cast<double (*)[TN_MAX + 1]>(tnsm);   // TN_KC x (TN_MAX + 1)
    double (*red)[32][TN_MAX] = reinterpret_cast<double (*)[32][TN_MAX]>(tnsm);  // 8 x 32 x TN_MAX
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    double acc[TN_MAX];
#pragma unroll
    for (int n = 0; n < TN_MAX; ++n) acc[n] = 0.0;
    const long long i0 = (long long)blockIdx.x * (TA ? 8 : 32);
    for (long long k0 = 0; k0 < K; k0 += TN_KC) {
        const int kc = (int)min((long long)TN_KC, K - k0);
        __syncthreads();
        for (int idx = tid; idx < TN_KC * N; idx += 256) {
            // TB: B'(n, k) = B[k + n*ldb] (k contiguous); else B[n + k*ldb] (n contiguous)
            const int n = TB ? idx / TN_KC : idx % N, k = TB ? idx % TN_KC : idx / N;
            Bs[k][n] = (k < kc) ? (TB ? B[(k0 + k) + (long long)n * ldb] : B[n + (k0 + k) * ldb]) : 0.0;
        }
        __syncthreads();
        if (!TA) {
            // warp w takes k = w, w + 8, ... of the chunk; lane = row
            const long long i = i0 + lane;
            double a8[TN_KC / 8];          // all loads of the chunk in flight before the first fma
#pragma unroll
            for (int q = 0; q < TN_KC / 8; ++q) {
                const int k = warp + 8 * q;
                a8[q] = (i < M && k < kc) ? A[i + (k0 + k) * lda] : 0.0;
            }
#pragma unroll
            for (int q = 0; q < TN_KC / 8; ++q)
#pragma unroll
                for (int n = 0; n < TN_MAX; ++n)
                    if (n < N) acc[n] = fma(a8[q], Bs[warp + 8 * q][n], acc[n]);
        } else {
            const long long i = i0 + warp;
            double a2[TN_KC / 32];
#pragma unroll
            for (int q = 0; q < TN_KC / 32; ++q) {
                const int k = lane + 32 * q;
                a2[q] = (i < M && k < kc) ? A[(k0 + k) + i * lda] : 0.0;
            }
#pragma unroll
            for (int q = 0; q < TN_KC / 32; ++q)
#pragma unroll
                for (int n = 0; n < TN_MAX; ++n)
                    if (n < N) acc[n] = fma(a2[q], Bs[lane + 32 * q][n], acc[n]);
        }
    }
    if (!TA) {
        __syncthreads();
#pragma unroll
        for (int n = 0; n < TN_MAX; ++n)
            if (n < N) red[warp][lane][n] = acc[n];
        __syncthreads();
        for (int idx = tid; idx < 32 * N; idx += 256) {
            const int r = idx % 32, n = idx / 32;
            const long long i = i0 + r;
            if (i >= M) continue;
            double s = 0.0;
            for (int w = 0; w < 8; ++w) s += red[w][r][n];
            double *c = C + i + (long long)n * ldc;
            *c = accumulate ? (*c + alpha * s) : alpha * s;
        }
    } else {
        const long long i = i0 + warp;
#pragma unroll
        for (int n = 0; n < TN_MAX; ++n)
            if (n < N) {
                double s = acc[n];
                for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
                if (lane == 0 && i < M) {
                    double *c = C + i + (long long)n * ldc;
                    *c = accumulate ? (*c + alpha * s) : alpha * s;
                }
            }
    }
}

int launch_gemm(smcp_ctx *ctx, bool ta, bool tb, const double *A, int64_t lda, const double *B, int64_t ldb,
                       double *C, int64_t ldc, int64_t M, int64_t N, int64_t K, double alpha, int accumulate,
                       int tri, int64_t tri_off, const char *name) {
    if (M > 0 && N > 0 && N <= TN_MAX && K > SK_MAX && !tri) {
        const unsigned grid = (unsigned)((M + (ta ? 8 : 32) - 1) / (ta ? 8 : 32));
        LaunchScope ls(ctx, "gemm_thin", 1, 8.0 * (double)K * (double)M);
#define TNL(TA_, TB_) gemm_thin_kernel<TA_, TB_><<<grid, 256, 0, ctx->stream>>>(A, lda, B, ldb, C, ldc, M, (int)N, K, alpha, accumulate)
        if (ta && tb) TNL(true, true);
        else if (!ta && !tb) TNL(false, false);
        else if (ta) TNL(true, false);
        else TNL(false, true);
#undef TNL
        CUDA_TRY(cudaGetLastError());
        return 0;
    }
    if (M > 0 && N > 0 && K > 0 && K <= SK_MAX) {
        dim3 grid((unsigned)((M + 31) / 32), (unsigned)((N + 31) / 32));
        LaunchScope ls(ctx, "gemm_smallk", 1, 2.0 * (double)K * (double)M * (double)N * (tri ? 0.5 : 1.0));
#define SK_LAUNCH(TA_, TB_) gemm_smallk_kernel<TA_, TB_><<<grid, 256, 0, ctx->stream>>>(A, lda, B, ldb, C, ldc, M, N, (int)K, alpha, accumulate, tri, tri_off)
        if (ta && tb) SK_LAUNCH(true, true);
        else if (!ta && !tb) SK_LAUNCH(false, false);
        else if (ta) SK_LAUNCH(true, false);
        else SK_LAUNCH(false, true);
#undef SK_LAUNCH
        CUDA_TRY(cudaGetLastError());
        return 0;
    }
    // K-major operands with 16-byte aligned columns: operand tiles fetched by TMA (gemm_tma.cu)
    if (ta && tb && gemm_tma_eligible(A, lda, B, ldb, M, N, K))
        return launch_gemm_tma_tn(ctx, A, lda, B, ldb, C, ldc, M, N, K, alpha, accumulate, tri, tri_off, name);
    return launch_gemm_cyc(ctx, ta, tb, A, lda, B, ldb, C, ldc, M, N, K, alpha, accumulate, tri, tri_off, name, 0, 1, 1);
}

// as launch_gemm, restricted to the column tiles jt0, jt0 + jtstride, ... (128 columns each)
int launch_gemm_cyc(smcp_ctx *ctx, bool ta, bool tb, const double *A, int64_t lda, const double *B, int64_t ldb,
                    double *C, int64_t ldc, int64_t M, int64_t N, int64_t K, double alpha, int accumulate,
                    int tri, int64_t tri_off, const char *name, int jt0, int jtstride, int jtb) {
    if (M <= 0 || N <= 0) return 0;
    if (jtb < 1) jtb = 1;
    const long long ntile_n = (N + BN - 1) / BN;
    const long long nblock_n = (ntile_n + jtb - 1) / jtb;          // column blocks of jtb tiles
    if (jt0 >= nblock_n) return 0;
    dim3 grid((unsigned)((M + BM - 1) / BM), (unsigned)(((nblock_n - jt0 + jtstride - 1) / jtstride) * jtb));
    auto tile_of = [&](unsigned bj) { return ((long long)jt0 + (long long)(bj / jtb) * jtstride) * jtb + (bj % jtb); };
    // split-K when the (lower-triangular) tile grid cannot fill the GPU and K is long: the Schur
    // assembly contracts over |blkval| ~ 10^4..10^6 rows into an m x m block
    long long ntiles = 0;
    for (unsigned bj = 0; bj < grid.y; ++bj)
        for (unsigned bi = 0; bi < grid.x; ++bi)
            if (tile_of(bj) < ntile_n && (!tri || (long long)bi * BM + BM - 1 + tri_off >= tile_of(bj) * BN)) ++ntiles;
    int splits = 1;
    if (!accumulate && alpha == 1.0 && K >= 2048 && ntiles > 0 && ntiles < ctx->num_sms) {
        splits = (int)(ctx->num_sms / ntiles);
        if (splits > 16) splits = 16;
        if ((long long)splits * 512 > K) splits = (int)(K / 512);
        if (splits < 1) splits = 1;
    }
    long long kchunk = K, split_stride = 0;
    double *Cout = C;
    int64_t ldout = ldc;
    if (splits > 1) {
        kchunk = ((K + splits - 1) / splits + BK - 1) / BK * BK;
        split_stride = M * N;
        if (grow((void **)&ctx->gemm_ws, &ctx->gemm_ws_cap, (size_t)splits * M * N * sizeof(double))) return -1;
        Cout = ctx->gemm_ws;
        ldout = M;
        grid.z = splits;
    }
    size_t smem = (size_t)2 * STAGES * 128 * LDK * sizeof(double);
    static bool attr_set = false;
    if (!attr_set) {
        CUDA_TRY(cudaFuncSetAttribute(gemm_dmma_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CUDA_TRY(cudaFuncSetAttribute(gemm_dmma_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CUDA_TRY(cudaFuncSetAttribute(gemm_dmma_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CUDA_TRY(cudaFuncSetAttribute(gemm_dmma_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_set = true;
    }
    // algorithmic flops: 2*K per computed entry of the (lower-triangular) result
    double pairs = 0.0;
    for (int64_t j = 0; j < N; ++j) {
        const int64_t jb = j / BN / jtb;
        if (jb < jt0 || (jb - jt0) % jtstride) continue;
        int64_t lo = tri ? j - tri_off : 0;            // rows i >= lo
        if (lo < 0) lo = 0;
        if (lo < M) pairs += (double)(M - lo);
    }
    {
        LaunchScope ls(ctx, name, 1, 2.0 * (double)K * pairs);
#define GEMM_LAUNCH(TA_, TB_) gemm_dmma_kernel<TA_, TB_><<<grid, GEMM_THREADS, smem, ctx->stream>>>(A, lda, B, ldb, Cout, ldout, M, N, K, alpha, accumulate, tri, tri_off, kchunk, split_stride, jt0, jtstride, jtb, 0LL, 0LL, 0)
        if (ta && tb) GEMM_LAUNCH(true, true);
        else if (!ta && !tb) GEMM_LAUNCH(false, false);
        else if (ta) GEMM_LAUNCH(true, false);
        else GEMM_LAUNCH(false, true);
#undef GEMM_LAUNCH
        if (splits > 1) {
            ctx->launches += 1;
            long long g = (M * N + 255) / 256;
            if (g > (long long)ctx->num_sms * 8) g = (long long)ctx->num_sms * 8;
            splitk_reduce_kernel<<<(unsigned)g, 256, 0, ctx->stream>>>(ctx->gemm_ws, split_stride, splits, C, ldc, M, N, tri, tri_off);
        }
    }
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// `batch` independent products with strides between consecutive A / B / C (0 = shared operand)
int launch_gemm_batched(smcp_ctx *ctx, bool ta, bool tb, const double *A, int64_t lda, int64_t sA, const double *B, int64_t ldb,
                        int64_t sB, double *C, int64_t ldc, int64_t sC, int64_t M, int64_t N, int64_t K, double alpha,
                        int accumulate, int64_t batch, const char *name) {
    if (M <= 0 || N <= 0 || batch <= 0) return 0;
    if (K <= 0) {
        if (accumulate) return 0;
        smcp_set_error("launch_gemm_batched: K = 0 without accumulation");
        return -2;
    }
    size_t smem = (size_t)2 * STAGES * 128 * LDK * sizeof(double);
    static bool attr_set = false;
    if (!attr_set) {
        CUDA_TRY(cudaFuncSetAttribute(gemm_dmma_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CUDA_TRY(cudaFuncSetAttribute(gemm_dmma_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CUDA_TRY(cudaFuncSetAttribute(gemm_dmma_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CUDA_TRY(cudaFuncSetAttribute(gemm_dmma_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_set = true;
    }
    for (int64_t z0 = 0; z0 < batch; z0 += 32768) {
        const int64_t nz = std::min<int64_t>(32768, batch - z0);
        dim3 grid((unsigned)((M + BM - 1) / BM), (unsigned)((N + BN - 1) / BN), (unsigned)nz);
        const double *Az = A + z0 * sA, *Bz = B + z0 * sB;
        double *Cz = C + z0 * sC;
        LaunchScope ls(ctx, name, 1, 2.0 * (double)K * (double)M * (double)N * (double)nz);
#define GEMM_LAUNCH(TA_, TB_) gemm_dmma_kernel<TA_, TB_><<<grid, GEMM_THREADS, smem, ctx->stream>>>(Az, lda, Bz, ldb, Cz, ldc, M, N, K, alpha, accumulate, 0, 0, K, sC, 0, 1, 1, sA, sB, 1)
        if (ta && tb) GEMM_LAUNCH(true, true);
        else if (!ta && !tb) GEMM_LAUNCH(false, false);
        else if (ta) GEMM_LAUNCH(true, false);
        else GEMM_LAUNCH(false, true);
#undef GEMM_LAUNCH
    }
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// C(i, j) = sum_k A(k, i) B(k, j) for i + row_lo_of_col0 >= j  (lower part of a column block of H)
int d_gemm_tn(smcp_ctx *ctx, const double *A, int64_t lda, const double *B, int64_t ldb, double *C,
              int64_t ldc, int64_t M, int64_t N, int64_t K, int64_t row_lo_of_col0) {
    return launch_gemm(ctx, true, true, A, lda, B, ldb, C, ldc, M, N, K, 1.0, 0, 1, row_lo_of_col0, "schur_gemm_dmma");
}

// ---------------------------------------------------------------------------------------
// blocked right-looking Cholesky (lower), column-major, in place (lapack.potrf, solvers.py:501)
// `ncols` < m gives the partial factorisation of a frontal matrix: the leading ncols columns
// hold L, the trailing (m - ncols)^2 block its Schur complement (the update matrix).
// ---------------------------------------------------------------------------------------
#define NB 64
namespace {
struct StreamSwap {      // run the launch helpers (which use ctx->stream) on another stream
    smcp_ctx *ctx;
    cudaStream_t saved;
    StreamSwap(smcp_ctx *c, cudaStream_t s) : ctx(c), saved(c->stream) { c->stream = s; }
    ~StreamSwap() { ctx->stream = saved; }
};
}  // namespace

// Pt(k, i) = P(i, k): the factored panel (rows x w, rows contiguous) as a K-major operand, so that its trailing update
// C -= P P^T runs through the TMA-fed GEMM (26.6 instead of ~21 TFLOP/s); 2 x 8 x rows x w bytes per panel, ~15 us
__global__ void panel_transpose_kernel(const double *__restrict__ P, long long ldp, long long rows, int w, double *__restrict__ Pt, long long ldt) {
    __shared__ double tile[32][33];
    const long long i0 = (long long)blockIdx.x * 32;
    const int k0 = blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const long long i = i0 + threadIdx.x;
        const int k = k0 + r;
        tile[r][threadIdx.x] = (i < rows && k < w) ? P[i + (long long)k * ldp] : 0.0;
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int k = k0 + threadIdx.x;
        const long long i = i0 + r;
        if (i < rows && k < w) Pt[k + i * ldt] = tile[threadIdx.x][r];
    }
}

// lapack.potrf (solvers.py:501, 1931) / partial factorisation of a frontal matrix.
//  * L2-resident matrices (m <= POTRF_TILE_MAX) on one GPU: ONE cooperative launch
//    (potrf_tile_kernel, dense_tile.cu).
//  * larger m: right-looking over column blocks of `block` columns (512 on one GPU, the distribution
//    block on several).  A block is factored by potrf_tile_kernel in panel mode (all rows of the
//    block column, updates confined to the block) and applied to the trailing matrix by ONE DMMA
//    GEMM with K = block, so C is re-read once per 512 columns instead of once per 64.
//  * several GPUs (north star (3), SURVEY 8e): 1-D block-cyclic columns, owner(q) = q mod nranks.
//    The owner of block q+1 applies panel q to it, factors it and broadcasts it (NCCL) on the
//    look-ahead stream while every rank applies panel q to the other blocks it owns.  Every rank ends
//    with the full factor, and the arithmetic per entry does not depend on the number of ranks.
static const int64_t POTRF_TILE_MAX = 2560;
static const int POTRF_LA_CTAS = 48;
int d_potrf(smcp_ctx *ctx, double *H, int64_t ld, int64_t m, int64_t ncols, int32_t *info_dev, int rank, int nranks, int64_t block) {
    if (ncols > m) ncols = m;
    if (nranks < 1) nranks = 1;
    if (m <= 0 || ncols <= 0) return 0;
    if (nranks > 1 && (ld != m || ncols != m)) { smcp_set_error("d_potrf: the distributed factorisation needs a full square matrix"); return -2; }
    LaunchScope outer(ctx, ctx->potrf_family ? ctx->potrf_family : "potrf_dmma", 0, (double)ncols * ncols * ncols / 3.0 + (double)(m - ncols) * ncols * (double)m);
    ctx->prof_mute++;
    struct Unmute { smcp_ctx *c; ~Unmute() { c->prof_mute--; } } unmute{ctx};
    CUDA_TRY(cudaMemsetAsync(info_dev, 0, sizeof(int), ctx->stream));
    if (nranks == 1 && m <= POTRF_TILE_MAX && potrf_tile_fits(ctx, m, ncols, false))
        return potrf_tile(ctx, H, ld, m, ncols, false, info_dev, 0);
    if (block <= 0) block = nranks > 1 ? 256 : 512;
    if (block % BN) { smcp_set_error("d_potrf: the column block must be a multiple of %d", BN); return -2; }
    const int tpb = (int)(block / BN);
    const int64_t nblocks = (ncols + block - 1) / block;
    auto blk_w = [&](int64_t q) { return std::min<int64_t>(block, ncols - q * block); };
    // panel q: all rows of block column q.  The last block of a PARTIAL factorisation whose width is
    // not a multiple of the tile size is factored together with its trailing update (tile mode).
    bool trailing_done = false;
    auto factor_block = [&](int64_t q) -> int {
        const int64_t c0 = q * block, w = blk_w(q);
        const bool last = c0 + w >= ncols;
        const bool full_mode = last && ncols < m && (w % 64) != 0;
        if (full_mode) trailing_done = true;
        if (!potrf_tile_fits(ctx, m - c0, w, !full_mode)) { smcp_set_error("d_potrf: panel too tall for the tile kernel"); return -2; }
        return potrf_tile(ctx, H + c0 + c0 * ld, ld, m - c0, w, !full_mode, info_dev, (int)c0);
    };
    // one GPU: the look-ahead schedule of the block-cyclic path -- panel q+1 on the second (high-priority) stream, on at most
    // POTRF_LA_CTAS SMs, while the main stream applies panel q to the rest.  m = 10^4: 25.6 -> 23.5 ms
    // (profiles/r02_v31_potrf_la.log).  The plain loop below serves ld != m, partial factorisations and
    // contexts without a second stream.
    if (nranks == 1 && !(ld == m && ncols == m && ctx->stream2)) {
        for (int64_t q = 0; q < nblocks; ++q) {
            const int64_t c0 = q * block, w = blk_w(q), c1 = c0 + w;
            if (factor_block(q)) return -1;
            if (c1 < m && !trailing_done) {
                const double *P1 = H + c1 + c0 * ld;
                if (launch_gemm(ctx, false, false, P1, ld, P1, ld, H + c1 + c1 * ld, ld, m - c1, m - c1, w, -1.0, 1, 1, 0, "potrf_syrk_dmma")) return -1;
            }
        }
        CUDA_TRY(cudaGetLastError());
        return 0;
    }
    // ---- block-cyclic over the ranks, look-ahead on the second stream
    cudaStream_t sB = ctx->stream, sA = ctx->stream2 ? ctx->stream2 : ctx->stream;
    const bool two = sA != sB;
    while ((int64_t)ctx->potrf_ev.size() < 2 * nblocks + 2) {
        cudaEvent_t e;
        CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        ctx->potrf_ev.push_back(e);
    }
    cudaEvent_t *E = ctx->potrf_ev.data(), *F = ctx->potrf_ev.data() + nblocks;
    cudaEvent_t fork = ctx->potrf_ev[2 * nblocks], join = ctx->potrf_ev[2 * nblocks + 1];
    if (two) {
        CUDA_TRY(cudaEventRecord(fork, sB));
        CUDA_TRY(cudaStreamWaitEvent(sA, fork, 0));
    }
    // one GPU: K-major copies of the panels (two buffers: panel q+1 is transposed while panel q is still being applied)
    const bool use_pt = nranks == 1 && (block % 2) == 0;
    double *PT[2] = {nullptr, nullptr};
    if (use_pt) {
        if (grow((void **)&ctx->potrf_pt, &ctx->potrf_pt_cap, (size_t)2 * block * m * sizeof(double))) return -1;
        PT[0] = ctx->potrf_pt;
        PT[1] = ctx->potrf_pt + (size_t)block * m;
    }
    auto transpose_panel = [&](int64_t q) -> int {
        const int64_t c0 = q * block, w = blk_w(q), c1 = c0 + w;
        if (c1 >= m) return 0;
        LaunchScope ls(ctx, "potrf_panel_t");
        panel_transpose_kernel<<<dim3((unsigned)((m - c1 + 31) / 32), (unsigned)((w + 31) / 32)), dim3(32, 8), 0, ctx->stream>>>(
            H + c1 + c0 * ld, ld, m - c1, (int)w, PT[q & 1], w);
        CUDA_TRY(cudaGetLastError());
        return 0;
    };
    {
        StreamSwap sw(ctx, sA);
        if (rank == 0 && factor_block(0)) return -1;
        if (nranks > 1 && comm_bcast(ctx, H, (size_t)blk_w(0) * ld, 0, sA)) return -1;
        if (use_pt && transpose_panel(0)) return -1;
        if (two) CUDA_TRY(cudaEventRecord(E[0], sA));
    }
    for (int64_t q = 0; q < nblocks; ++q) {
        const int64_t c0 = q * block, w = blk_w(q), c1 = c0 + w;
        if (c1 >= m) break;
        const double *P1 = H + c1 + c0 * ld;          // panel q, rows c1..
        if (two) CUDA_TRY(cudaStreamWaitEvent(sB, E[q], 0));
        int64_t c2 = c1;
        if (q + 1 < nblocks) {
            const int64_t w1 = blk_w(q + 1);
            c2 = c1 + w1;
            StreamSwap sw(ctx, sA);
            if (two && q >= 1) CUDA_TRY(cudaStreamWaitEvent(sA, F[q - 1], 0));
            if ((q + 1) % nranks == rank) {
                if (use_pt) {
                    if (launch_gemm(ctx, true, true, PT[q & 1], w, PT[q & 1], w, H + c1 + c1 * ld, ld, m - c1, w1, w, -1.0, 1, 1, 0, "potrf_syrk_dmma")) return -1;
                } else {
                    if (launch_gemm(ctx, false, false, P1, ld, P1, ld, H + c1 + c1 * ld, ld, m - c1, w1, w, -1.0, 1, 1, 0, "potrf_syrk_dmma")) return -1;
                }
                if (nranks == 1) ctx->potrf_grid_cap = POTRF_LA_CTAS;
                const int rcf = factor_block(q + 1);
                ctx->potrf_grid_cap = 0;
                if (rcf) return -1;
                if (use_pt && transpose_panel(q + 1)) return -1;
            }
            if (nranks > 1 && comm_bcast(ctx, H + c1 * ld, (size_t)w1 * ld, (int)((q + 1) % nranks), sA)) return -1;
            if (two) CUDA_TRY(cudaEventRecord(E[q + 1], sA));
        }
        if (c2 < m) {
            // panel q applied to the blocks >= q+2 this rank owns
            const double *P2 = H + c2 + c0 * ld;
            const int64_t qb = c2 / block;
            const int jb0 = (int)(((rank - qb) % nranks + nranks) % nranks);
            if (use_pt) {
                const double *T2 = PT[q & 1] + (size_t)(c2 - c1) * w;
                if (launch_gemm(ctx, true, true, T2, w, T2, w, H + c2 + c2 * ld, ld, m - c2, m - c2, w, -1.0, 1, 1, 0, "potrf_syrk_dmma")) return -1;
            } else if (launch_gemm_cyc(ctx, false, false, P2, ld, P2, ld, H + c2 + c2 * ld, ld, m - c2, m - c2, w, -1.0, 1, 1, 0,
                                "potrf_syrk_dmma", jb0, nranks, tpb)) return -1;
        }
        if (two) CUDA_TRY(cudaEventRecord(F[q], sB));
    }
    if (two) {
        CUDA_TRY(cudaEventRecord(join, sA));
        CUDA_TRY(cudaStreamWaitEvent(sB, join, 0));
    }
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// ---------------------------------------------------------------------------------------
// potrs: y <- L^{-T} L^{-1} y (lapack.potrs, solvers.py:526), single right-hand side.
// A triangular solve is m dependent steps whatever the hardware, so this is a latency kernel.
// potrs_kernel: one CTA of 1024 threads solves with the diagonal block [i0, i0+mm): the
// right-hand side lives in shared memory, each 64 x 64 diagonal block is staged in shared memory,
// substitution inside a block is done by one warp (row values in registers, pivot broadcast by
// shuffle, multiplication by the reciprocal pivots computed off the critical path), and the
// off-diagonal part of every block column is a GEMV spread over all 32 warps with independent
// partial sums.  Plain substitution, no explicit inverses: backward stable like the LAPACK
// routine it replaces.  m <= 1536: one launch does everything.  Larger m: blocks of 256 rows
// go through potrs_kernel and the rest of the matrix is streamed by multi-CTA GEMV kernels
// (fixed summation order, no atomics).
// ---------------------------------------------------------------------------------------
#define PS_THREADS 1024
// y[i] -= sum_{j < 64} A(i, j) x[j] for i < rows.  TR = false: A(i, j) = A[i + j*ld] (rows of a
// column panel); TR = true: A(i, j) = A[j + i*ld] (columns of a row panel).  tpr threads share
// an output when there are few of them; every thread keeps 8 loads in flight.
template <bool TR>
__device__ __forceinline__ void potrs_gemv(const double *__restrict__ A, long long ld, long long rows, const double *x, double *y, int t, int nt) {
    int tpr = 1;
    while (tpr < 16 && rows * (tpr * 2) <= nt) tpr *= 2;
    const int per = NB / tpr;                       // columns per thread: 64 .. 4
    const int part = t & (tpr - 1);
    const int j0 = part * per;
    for (long long base = 0; base < rows; base += nt / tpr) {
        const long long i = base + (t / tpr);
        double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
        if (i < rows && t < (nt / tpr) * tpr) {
            const double *Ar = TR ? A + i * ld + j0 : A + i + (long long)j0 * ld;
            const long long st = TR ? 1 : ld;
            if (per >= 8) {
                for (int j = 0; j < per; j += 8) {
                    double v[8];
#pragma unroll
                    for (int q = 0; q < 8; ++q) v[q] = Ar[(long long)(j + q) * st];
                    s0 = fma(v[0], x[j0 + j], s0);
                    s1 = fma(v[1], x[j0 + j + 1], s1);
                    s2 = fma(v[2], x[j0 + j + 2], s2);
                    s3 = fma(v[3], x[j0 + j + 3], s3);
                    s0 = fma(v[4], x[j0 + j + 4], s0);
                    s1 = fma(v[5], x[j0 + j + 5], s1);
                    s2 = fma(v[6], x[j0 + j + 6], s2);
                    s3 = fma(v[7], x[j0 + j + 7], s3);
                }
            } else {
                double v[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) v[q] = Ar[(long long)q * st];
                s0 = fma(v[0], x[j0], s0);
                s1 = fma(v[1], x[j0 + 1], s1);
                s2 = fma(v[2], x[j0 + 2], s2);
                s3 = fma(v[3], x[j0 + 3], s3);
            }
        }
        double sacc = (s0 + s1) + (s2 + s3);
        // the tpr partial sums of an output sit in consecutive lanes of one warp: fixed-order tree
        for (int o = 1; o < tpr; o <<= 1) sacc += __shfl_xor_sync(0xffffffffu, sacc, o);
        if (part == 0 && i < rows && t < (nt / tpr) * tpr) y[i] -= sacc;
    }
}

__global__ void __launch_bounds__(PS_THREADS) potrs_kernel(const double *__restrict__ Hfull, long long ld, long long i0, long long m,
                                                           double *__restrict__ yfull, int do_fwd, int do_bwd) {
    extern __shared__ double psm[];
    double *Lk = psm;                    // NB x (NB+1)
    double *rinv = Lk + NB * (NB + 1);   // NB
    double *tb = rinv + NB;              // NB
    double *ys = tb + NB;                // m
    const double *H = Hfull + i0 + i0 * ld;
    double *y = yfull + i0;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const long long nblkc = (m + NB - 1) / NB;
    for (long long i = tid; i < m; i += PS_THREADS) ys[i] = y[i];
    // forward: L x = y
    if (do_fwd)
    for (long long bi = 0; bi < nblkc; ++bi) {
        const long long k0 = bi * NB;
        const int kb = (int)min((long long)NB, m - k0);
        for (int idx = tid; idx < kb * kb; idx += PS_THREADS) {
            const int i = idx % kb, j = idx / kb;
            Lk[i * (NB + 1) + j] = H[(k0 + i) + (k0 + j) * ld];
        }
        __syncthreads();
        if (tid < kb) rinv[tid] = 1.0 / Lk[tid * (NB + 1) + tid];
        __syncthreads();
        if (warp == 0) {
            double x0 = (lane < kb) ? ys[k0 + lane] : 0.0;
            double x1 = (lane + 32 < kb) ? ys[k0 + lane + 32] : 0.0;
            for (int j = 0; j < kb; ++j) {
                const double xj = __shfl_sync(0xffffffffu, (j < 32) ? x0 : x1, j & 31) * rinv[j];
                if (lane == (j & 31)) { if (j < 32) x0 = xj; else x1 = xj; }
                if (lane > j) x0 = fma(-Lk[lane * (NB + 1) + j], xj, x0);
                if (lane + 32 > j && lane + 32 < kb) x1 = fma(-Lk[(lane + 32) * (NB + 1) + j], xj, x1);
            }
            if (lane < kb) ys[k0 + lane] = x0;
            if (lane + 32 < kb) ys[k0 + lane + 32] = x1;
        }
        __syncthreads();
        // rows below the block (then kb == NB): 8 loads in flight per thread, several threads per row
        // when few rows are left -- the loads are L2 round trips, four at a time left them exposed
        if (m - k0 - kb > 0) potrs_gemv<false>(H + (k0 + kb) + k0 * ld, ld, m - k0 - kb, ys + k0, ys + k0 + kb, tid, PS_THREADS);
        __syncthreads();
    }
    // backward: L^T x = y
    if (do_bwd)
    for (long long bi = nblkc - 1; bi >= 0; --bi) {
        const long long k0 = bi * NB;
        const int kb = (int)min((long long)NB, m - k0);
        for (int idx = tid; idx < kb * kb; idx += PS_THREADS) {
            const int i = idx % kb, j = idx / kb;
            Lk[i * (NB + 1) + j] = H[(k0 + i) + (k0 + j) * ld];
        }
        // t_c = y[k0+c] - sum_{i >= k0+kb} L(i, k0+c) y[i]: warp w takes columns w and w + 32
        for (int c = warp; c < kb; c += PS_THREADS / 32) {
            const double *Lc = H + (k0 + c) * ld;
            double s0 = 0.0, s1 = 0.0;
            long long i = k0 + kb + lane;
            for (; i + 224 < m; i += 256) {          // 8 loads in flight
                double v[8];
#pragma unroll
                for (int q = 0; q < 8; ++q) v[q] = Lc[i + 32 * q];
#pragma unroll
                for (int q = 0; q < 8; q += 2) {
                    s0 = fma(v[q], ys[i + 32 * q], s0);
                    s1 = fma(v[q + 1], ys[i + 32 * (q + 1)], s1);
                }
            }
            for (; i + 32 < m; i += 64) {
                s0 = fma(Lc[i], ys[i], s0);
                s1 = fma(Lc[i + 32], ys[i + 32], s1);
            }
            if (i < m) s0 = fma(Lc[i], ys[i], s0);
            double sacc = s0 + s1;
            for (int o = 16; o > 0; o >>= 1) sacc += __shfl_down_sync(0xffffffffu, sacc, o);
            if (lane == 0) tb[c] = ys[k0 + c] - sacc;
        }
        __syncthreads();
        if (tid < kb) rinv[tid] = 1.0 / Lk[tid * (NB + 1) + tid];
        __syncthreads();
        if (warp == 0) {
            double x0 = (lane < kb) ? tb[lane] : 0.0;
            double x1 = (lane + 32 < kb) ? tb[lane + 32] : 0.0;
            for (int j = kb - 1; j >= 0; --j) {
                const double xj = __shfl_sync(0xffffffffu, (j < 32) ? x0 : x1, j & 31) * rinv[j];
                if (lane == (j & 31)) { if (j < 32) x0 = xj; else x1 = xj; }
                if (lane < j) x0 = fma(-Lk[j * (NB + 1) + lane], xj, x0);
                if (lane + 32 < j) x1 = fma(-Lk[j * (NB + 1) + lane + 32], xj, x1);
            }
            if (lane < kb) ys[k0 + lane] = x0;
            if (lane + 32 < kb) ys[k0 + lane + 32] = x1;
        }
        __syncthreads();
    }
    for (long long i = tid; i < m; i += PS_THREADS) y[i] = ys[i];
}

#define PSB 256          // diagonal block of the multi-kernel solve
// forward update: y[i] -= sum_{j < kb} L(i, i0+j) x[i0+j] for i >= i0+kb.  64 rows per CTA, four
// column groups of threads, partial sums combined in a fixed order.
__global__ void __launch_bounds__(256) potrs_fwd_update_kernel(const double *__restrict__ H, long long ld, long long m, long long i0, int kb,
                                                               double *__restrict__ y) {
    __shared__ double xs[PSB];
    __shared__ double part[4][64];
    const int tid = threadIdx.x, r = tid & 63, cg = tid >> 6;
    for (int j = tid; j < kb; j += 256) xs[j] = y[i0 + j];
    __syncthreads();
    const long long row = i0 + kb + (long long)blockIdx.x * 64 + r;
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    if (row < m) {
        const int per = (kb + 3) / 4, j0 = cg * per, j1 = min(kb, j0 + per);
        const double *Lr = H + row + (i0 + j0) * ld;
        int j = j0;
        for (; j + 3 < j1; j += 4, Lr += 4 * ld) {
            s0 = fma(Lr[0], xs[j], s0);
            s1 = fma(Lr[ld], xs[j + 1], s1);
            s2 = fma(Lr[2 * ld], xs[j + 2], s2);
            s3 = fma(Lr[3 * ld], xs[j + 3], s3);
        }
        for (; j < j1; ++j, Lr += ld) s0 = fma(Lr[0], xs[j], s0);
    }
    part[cg][r] = (s0 + s1) + (s2 + s3);
    __syncthreads();
    if (cg == 0 && row < m) y[row] -= (part[0][r] + part[1][r]) + (part[2][r] + part[3][r]);
}

// backward update: y[c] -= sum_{i < kb} L(i0+i, c) x[i0+i] for c < i0: one warp per column
__global__ void __launch_bounds__(256) potrs_bwd_update_kernel(const double *__restrict__ H, long long ld, long long i0, int kb,
                                                               double *__restrict__ y) {
    __shared__ double xs[PSB];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int j = tid; j < kb; j += 256) xs[j] = y[i0 + j];
    __syncthreads();
    const long long c = (long long)blockIdx.x * 8 + warp;
    if (c >= i0) return;
    const double *Lc = H + i0 + c * ld;
    double s = 0.0;
    for (int i = lane; i < kb; i += 32) s = fma(Lc[i], xs[i], s);
    for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
    if (lane == 0) y[c] -= s;
}

// The factor is read by ONE CTA and between two solves the Hessian kernels stream hundreds of MB
// through L2, so every load of the solve would be a DRAM round trip: all SMs pull the lower
// triangle into L2 first (4 MB at m = 1000, a few microseconds at HBM speed).
__global__ void potrs_prefetch_kernel(const double *__restrict__ H, long long ld, long long m) {
    const long long lines_per_col = (m + 15) / 16;
    const long long total = m * lines_per_col;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const long long j = idx / lines_per_col, r = (idx % lines_per_col) * 16;
        if (r + 15 >= j) asm volatile("prefetch.global.L2 [%0];" ::"l"(H + r + j * ld));
    }
}

int d_potrs(smcp_ctx *ctx, const double *H, int64_t m, double *y_dev) {
    const int64_t single_max = 1536;
    const int64_t mm = (m <= single_max) ? m : PSB;
    const size_t smem = (size_t)(NB * (NB + 1) + 2 * NB + mm + 8) * sizeof(double);
    static size_t attr = 0;
    if (smem > attr) {
        CUDA_TRY(cudaFuncSetAttribute(potrs_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr = smem;
    }
    LaunchScope ls(ctx, "potrs", 0, 8.0 * (double)m * (double)m);
    ctx->prof_mute++;
    struct Unmute { smcp_ctx *c; ~Unmute() { c->prof_mute--; } } unmute{ctx};
    if (m <= single_max) {
        ctx->launches += 2;
        potrs_prefetch_kernel<<<ctx->num_sms, 256, 0, ctx->stream>>>(H, m, m);
        potrs_kernel<<<1, PS_THREADS, smem, ctx->stream>>>(H, m, 0, m, y_dev, 1, 1);
    } else {
        const int64_t nb = (m + PSB - 1) / PSB;
        for (int64_t b = 0; b < nb; ++b) {
            const int64_t i0 = b * PSB;
            const int kb = (int)std::min<int64_t>(PSB, m - i0);
            potrs_kernel<<<1, PS_THREADS, smem, ctx->stream>>>(H, m, i0, kb, y_dev, 1, 0);
            const int64_t below = m - i0 - kb;
            if (below > 0) potrs_fwd_update_kernel<<<(unsigned)((below + 63) / 64), 256, 0, ctx->stream>>>(H, m, m, i0, kb, y_dev);
            ctx->launches += 2;
        }
        for (int64_t b = nb - 1; b >= 0; --b) {
            const int64_t i0 = b * PSB;
            const int kb = (int)std::min<int64_t>(PSB, m - i0);
            potrs_kernel<<<1, PS_THREADS, smem, ctx->stream>>>(H, m, i0, kb, y_dev, 0, 1);
            if (i0 > 0) potrs_bwd_update_kernel<<<(unsigned)((i0 + 7) / 8), 256, 0, ctx->stream>>>(H, m, i0, kb, y_dev);
            ctx->launches += 2;
        }
    }
    CUDA_TRY(cudaGetLastError());
    return 0;
}
