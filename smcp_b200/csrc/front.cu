// Blocked triangular solves with a dense lower-triangular factor, on the whole GPU: a building
// block of the dense path for large frontal matrices (bigfront.cu).
//   X = L^{-1} B  /  X = L^{-T} B,  L lower n x n (leading dimension ldl), B n x nrhs.
// Right-looking over 64-row blocks: the 64 x 64 diagonal block is solved by trsm_diag_kernel
// (block in shared memory, one right-hand side per thread, 8-row register blocks), then ONE DMMA
// GEMM (dense.cu) with K = 64 updates all remaining rows.  Reference call sites of the routines
// built on it: src/python/solvers.py:884 (cholesky), 874 (completion), 891 (projected_inverse),
// 904 (llt), 483/524/531 (hessian), 405 (inverse hessian).
#include "internal.cuh"
#include <algorithm>

#define FNB 64
#define FLDT 66

// ---------------------------------------------------------------------------------------
// blocked triangular solves  X = L^{-1} B  /  X = L^{-T} B   (L lower, n x n, B n x nrhs)
// ---------------------------------------------------------------------------------------
// diagonal block: one right-hand side per thread, its kb values in shared memory (column-major
// over threads, conflict free), 8-row register blocks
template <bool TRANS>
__global__ void __launch_bounds__(128) trsm_diag_kernel(const double *__restrict__ L, long long ldl, int kb, double *B, long long ldb, long long nrhs) {
    extern __shared__ __align__(16) double tsm[];
    double *LT = tsm;                 // LT[c*FLDT + r] = L(r, c)
    double *xs = tsm + FNB * FLDT;    // kb x 128
    const int tid = threadIdx.x;
    for (int idx = tid; idx < FNB * FLDT; idx += 128) LT[idx] = 0.0;
    __syncthreads();
    for (int idx = tid; idx < kb * kb; idx += 128) {
        const int r = idx % kb, c = idx / kb;
        // forward solve reads columns of L (LT[c][r]); the transposed solve reads rows (LT[r][c])
        if (r >= c) LT[TRANS ? r * FLDT + c : c * FLDT + r] = L[r + (long long)c * ldl];
    }
    __syncthreads();
    const long long col = (long long)blockIdx.x * 128 + tid;
    if (col >= nrhs) return;
    double *P = B + col * ldb;
    for (int r = 0; r < kb; ++r) xs[r * 128 + tid] = P[r];
    if (!TRANS) {
        for (int c8 = 0; c8 < kb; c8 += 8) {
            double x8[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) x8[k] = (c8 + k < kb) ? xs[(c8 + k) * 128 + tid] : 0.0;
            for (int p = 0; p < c8; ++p) {
                const double xp = xs[p * 128 + tid];
                const double2 *lp = reinterpret_cast<const double2 *>(LT + p * FLDT + c8);
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const double2 lv = lp[k];
                    x8[2 * k] = fma(-xp, lv.x, x8[2 * k]);
                    x8[2 * k + 1] = fma(-xp, lv.y, x8[2 * k + 1]);
                }
            }
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                if (c8 + k < kb) {
                    const double xk = x8[k] / LT[(c8 + k) * FLDT + c8 + k];
                    x8[k] = xk;
#pragma unroll
                    for (int k2 = k + 1; k2 < 8; ++k2) x8[k2] = fma(-xk, LT[(c8 + k) * FLDT + c8 + k2], x8[k2]);
                }
            }
#pragma unroll
            for (int k = 0; k < 8; ++k)
                if (c8 + k < kb) {
                    xs[(c8 + k) * 128 + tid] = x8[k];
                    P[c8 + k] = x8[k];
                }
        }
    } else {
        // L^T x = b: backward over 8-row register blocks; LT[p*FLDT + c] = L(p, c)
        const int nb8 = (kb + 7) / 8;
        for (int b8 = nb8 - 1; b8 >= 0; --b8) {
            const int r8 = b8 * 8;
            double x8[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) x8[k] = (r8 + k < kb) ? xs[(r8 + k) * 128 + tid] : 0.0;
            for (int p = r8 + 8; p < kb; ++p) {
                const double xp = xs[p * 128 + tid];
                const double2 *lp = reinterpret_cast<const double2 *>(LT + p * FLDT + r8);
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const double2 lv = lp[k];
                    x8[2 * k] = fma(-xp, lv.x, x8[2 * k]);
                    x8[2 * k + 1] = fma(-xp, lv.y, x8[2 * k + 1]);
                }
            }
#pragma unroll
            for (int k = 7; k >= 0; --k) {
                if (r8 + k < kb) {
                    const double xk = x8[k] / LT[(r8 + k) * FLDT + r8 + k];
                    x8[k] = xk;
#pragma unroll
                    for (int k2 = 0; k2 < k; ++k2) x8[k2] = fma(-xk, LT[(r8 + k) * FLDT + r8 + k2], x8[k2]);
                }
            }
#pragma unroll
            for (int k = 0; k < 8; ++k)
                if (r8 + k < kb) {
                    xs[(r8 + k) * 128 + tid] = x8[k];
                    P[r8 + k] = x8[k];
                }
        }
    }
}

// n <= 32 (the nn x nn pivot blocks of thin supernodes, nn = 1 .. 9): one right-hand side per thread, the factor
// in shared memory, the column in registers -- a few microseconds instead of a slab launch with 200 KB of
// shared memory for a 1 x 1 solve.
template <bool TRANS>
__global__ void __launch_bounds__(128) trsm_tiny_kernel(const double *__restrict__ L, long long ldl, int n, double *__restrict__ B, long long ldb,
                                                        long long nrhs) {
    __shared__ double Ls[32 * 33];
    for (int idx = threadIdx.x; idx < n * n; idx += 128) {
        const int r = idx % n, c = idx / n;
        Ls[c * 33 + r] = (r >= c) ? L[r + (long long)c * ldl] : 0.0;
    }
    __syncthreads();
    const long long col = (long long)blockIdx.x * 128 + threadIdx.x;
    if (col >= nrhs) return;
    double *b = B + col * ldb;
    double x[32];
#pragma unroll
    for (int r = 0; r < 32; ++r) x[r] = (r < n) ? b[r] : 0.0;
    if (!TRANS) {
#pragma unroll
        for (int c = 0; c < 32; ++c)
            if (c < n) {
                const double xc = x[c] / Ls[c * 33 + c];
                x[c] = xc;
#pragma unroll
                for (int r = c + 1; r < 32; ++r)
                    if (r < n) x[r] = fma(-Ls[c * 33 + r], xc, x[r]);
            }
    } else {
#pragma unroll
        for (int c = 31; c >= 0; --c)
            if (c < n) {
                const double xc = x[c] / Ls[c * 33 + c];
                x[c] = xc;
#pragma unroll
                for (int r = 0; r < c; ++r) x[r] = fma(-Ls[r * 33 + c], xc, x[r]);
            }
    }
#pragma unroll
    for (int r = 0; r < 32; ++r)
        if (r < n) b[r] = x[r];
}

int d_trsm_left_lower(smcp_ctx *ctx, bool trans, const double *L, int64_t ldl, int64_t n, double *B, int64_t ldb, int64_t nrhs) {
    if (n <= 0 || nrhs <= 0) return 0;
    if (n <= 32) {
        LaunchScope ls(ctx, "trsm_tiny");
        const unsigned grid = (unsigned)((nrhs + 127) / 128);
        if (trans) trsm_tiny_kernel<true><<<grid, 128, 0, ctx->stream>>>(L, ldl, (int)n, B, ldb, nrhs);
        else trsm_tiny_kernel<false><<<grid, 128, 0, ctx->stream>>>(L, ldl, (int)n, B, ldb, nrhs);
        CUDA_TRY(cudaGetLastError());
        return 0;
    }
    // one or two right-hand sides against a large factor (the ~1100-row separators of thin supernodes):
    // a single CTA is bound by what one SM pulls out of L2; a cluster of 8-16 CTAs on the inverted
    // diagonal blocks (potrs_cluster.cu) takes ~0.07 ms instead of 0.25
    if (nrhs <= 2 && n >= 256 && n <= 16384) {
        const size_t need = (size_t)((n + 63) / 64) * 4096 * sizeof(double);
        if (grow((void **)&ctx->trs_dinv, &ctx->trs_dinv_cap, need)) return -1;
        if (d_potrs_prepare(ctx, L, ldl, n, ctx->trs_dinv)) return -1;
        return d_trs_cluster(ctx, L, ldl, n, ctx->trs_dinv, B, ldb, nrhs, trans ? 0 : 1, trans ? 1 : 0, "trsm_cluster");
    }
    // L2-resident factors: one launch, every CTA keeps 8 right-hand sides in shared memory for the whole
    // solve (dense_tile.cu); larger ones take the launch chain below
    if (trsm_slab_fits(n)) return trsm_slab(ctx, trans, L, ldl, n, B, ldb, nrhs);
    const size_t smem = (size_t)(FNB * FLDT + FNB * 128) * sizeof(double);
    static bool attr = false;
    if (!attr) {
        CUDA_TRY(cudaFuncSetAttribute(trsm_diag_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CUDA_TRY(cudaFuncSetAttribute(trsm_diag_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr = true;
    }
    const unsigned grid = (unsigned)((nrhs + 127) / 128);
    const int64_t nb = (n + FNB - 1) / FNB;
    // right-looking: after a 64-row block is solved the whole remainder is updated by ONE GEMM
    // with K = 64 and (rows left) x nrhs outputs, which fills the GPU; the left-looking form
    // (K growing, 64 output rows) runs on nrhs/128 CTAs and was 10x slower at n = 1186
    if (!trans) {
        for (int64_t bi = 0; bi < nb; ++bi) {
            const int64_t i0 = bi * FNB;
            const int kb = (int)std::min<int64_t>(FNB, n - i0);
            {
                LaunchScope ls(ctx, "front_trsm_diag");
                trsm_diag_kernel<false><<<grid, 128, smem, ctx->stream>>>(L + i0 + i0 * ldl, ldl, kb, B + i0, ldb, nrhs);
            }
            const int64_t below = n - i0 - kb;
            if (below > 0) {
                // B(i0+kb:n, :) -= L(i0+kb:n, i0:i0+kb) X(i0:i0+kb, :)
                if (launch_gemm(ctx, false, true, L + (i0 + kb) + i0 * ldl, ldl, B + i0, ldb, B + i0 + kb, ldb, below, nrhs, kb, -1.0, 1, 0, 0, "front_gemm_dmma")) return -1;
            }
        }
    } else {
        for (int64_t bi = nb - 1; bi >= 0; --bi) {
            const int64_t i0 = bi * FNB;
            const int kb = (int)std::min<int64_t>(FNB, n - i0);
            {
                LaunchScope ls(ctx, "front_trsm_diag");
                trsm_diag_kernel<true><<<grid, 128, smem, ctx->stream>>>(L + i0 + i0 * ldl, ldl, kb, B + i0, ldb, nrhs);
            }
            if (i0 > 0) {
                // B(0:i0, :) -= L(i0:i0+kb, 0:i0)^T X(i0:i0+kb, :)
                if (launch_gemm(ctx, true, true, L + i0, ldl, B + i0, ldb, B, ldb, i0, nrhs, kb, -1.0, 1, 0, 0, "front_gemm_dmma")) return -1;
            }
        }
    }
    CUDA_TRY(cudaGetLastError());
    return 0;
}
