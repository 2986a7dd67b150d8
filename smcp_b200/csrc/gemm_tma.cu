// TMA-fed FP64 tensor-core GEMM for K-major operands (north star (1)/(3): "DMMA tiles fed by TMA"):
//     C(i, j) = [C(i, j) +] alpha * sum_k A[k + i*lda] * B[k + j*ldb]
// This is the contraction H[c0:, c0:c0+nc] = (w.Av)^T W of the Schur-complement assembly
// (src/python/solvers.py:484-486: the trailing gemv over Av[:, j:m], batched over the columns j):
// both operands are nblk x (columns) arrays with the contraction index contiguous, and leading
// dimensions that are multiples of 16 bytes, so they are legal 2-D tensor maps.
//
//  * operand tiles of 128 rows x 16 doubles (one 128-byte line per row) are fetched by
//    cp.async.bulk.tensor.2d (SASS: UTMALDG) with the 128-byte swizzle; rows and k beyond the matrix
//    are zero-filled by the copy engine, so there is no bounds code in the main loop;
//  * a ring of 6 stages (192 KB) with full/empty mbarriers: one elected thread issues the copies,
//    the 16 consumer warps never meet at a CTA-wide barrier in the main loop;
//  * fragments are read straight from the swizzled tiles.  The tensor-core instruction fixes which
//    lane holds which (row, k) of a fragment but not which MATRIX row a fragment row stands for, so
//    fragment row g of a 16-row block is matrix row 2g (+1 for the second half) and fragment column g
//    of an 8-column block is matrix column 2(g & 3) + (g >> 2): with that assignment the 16 lanes of a
//    half warp hit 16 different 8-byte slots of the XOR-swizzled lines (no bank conflicts, no padding);
//  * FP64 has no tcgen05 kind: the tensor instruction is mma.sync.m16n8k8.f64 (SASS: DMMA);
//  * triangular results (tri): tiles above the diagonal exit, warp tiles above the diagonal of a
//    diagonal tile skip their MMAs;
//  * split-K partial results go to a workspace and are summed in a fixed order (bitwise reproducible).
#include "internal.cuh"
#include <cuda.h>
#include <algorithm>

#define TM_BM 128
#define TM_BN 128
#define TM_BK 16
#define TM_STAGES 6
#define TM_THREADS 512
#define TM_TILE_BYTES (128 * TM_BK * 8)          // 16 KB per operand tile

__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long *bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, unsigned parity) {
    unsigned ok;
    do {
        asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
                     : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    } while (!ok);
}
__device__ __forceinline__ void tma_load_2d(void *dst, const CUtensorMap *map, unsigned long long *bar, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(smem_u32(dst)), "l"((unsigned long long)map), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void dmma16x8x8_m(double (&c)[4], const double (&a)[4], const double (&b)[2]) {
    asm volatile("mma.sync.aligned.m16n8k8.row.col.f64.f64.f64.f64 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+d"(c[0]), "+d"(c[1]), "+d"(c[2]), "+d"(c[3])
                 : "d"(a[0]), "d"(a[1]), "d"(a[2]), "d"(a[3]), "d"(b[0]), "d"(b[1]));
}
// element (row r, k) of a 128-byte-swizzled tile: 16-byte chunk index XOR (r & 7)
__device__ __forceinline__ double tile_ld(const unsigned char *tile, int r, int k) {
    return *reinterpret_cast<const double *>(tile + r * 128 + ((((k >> 1) ^ (r & 7)) << 4) | ((k & 1) << 3)));
}

__global__ void __launch_bounds__(TM_THREADS, 1)
gemm_tma_tn_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, double *__restrict__ C, long long ldc,
                   long long M, long long N, long long K, double alpha, int accumulate, int tri, long long tri_off, long long kchunk,
                   long long split_stride) {
    extern __shared__ unsigned char tm_raw[];
    unsigned char *base = reinterpret_cast<unsigned char *>(((unsigned long long)tm_raw + 1023ull) & ~1023ull);
    unsigned long long *full = reinterpret_cast<unsigned long long *>(base + TM_STAGES * 2 * TM_TILE_BYTES);
    unsigned long long *empty = full + TM_STAGES;
    const long long i0 = (long long)blockIdx.x * TM_BM, j0 = (long long)blockIdx.y * TM_BN;
    if (tri && (i0 + TM_BM - 1 + tri_off < j0)) return;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wm = (warp & 3) * 32, wn = (warp >> 2) * 32;
    const int g = lane >> 2, t = lane & 3;
    const bool wskip = tri && (i0 + wm + 31 + tri_off < j0 + wn);
    const long long kbeg = (long long)blockIdx.z * kchunk;
    const long long kend = (kbeg + kchunk < K) ? kbeg + kchunk : K;
    const int nk = (int)((kend - kbeg + TM_BK - 1) / TM_BK);
    C += (long long)blockIdx.z * split_stride;
    if (tid == 0) {
        for (int s = 0; s < TM_STAGES; ++s) {
            mbar_init(full + s, 1);
            mbar_init(empty + s, TM_THREADS / 32);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0) {
        for (int s = 0; s < TM_STAGES - 1 && s < nk; ++s) {
            mbar_expect_tx(full + s, 2 * TM_TILE_BYTES);
            tma_load_2d(base + s * 2 * TM_TILE_BYTES, &tmA, full + s, (int)(kbeg + (long long)s * TM_BK), (int)i0);
            tma_load_2d(base + s * 2 * TM_TILE_BYTES + TM_TILE_BYTES, &tmB, full + s, (int)(kbeg + (long long)s * TM_BK), (int)j0);
        }
    }
    double acc[2][4][4];
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b)
#pragma unroll
            for (int v = 0; v < 4; ++v) acc[a][b][v] = 0.0;
    // physical rows of this lane's fragment rows / columns inside the tiles
    const int bcol = 2 * (g & 3) + (g >> 2);
    for (int kt = 0; kt < nk; ++kt) {
        const int s = kt % TM_STAGES;
        if (tid == 0) {
            // refill the stage that was consumed in iteration kt - 1 with the tile of iteration kt + STAGES - 1
            const int nx = kt + TM_STAGES - 1;
            if (nx < nk) {
                const int sn = nx % TM_STAGES;
                if (kt >= 1) mbar_wait(empty + sn, (unsigned)(((kt - 1) / TM_STAGES) & 1));
                mbar_expect_tx(full + sn, 2 * TM_TILE_BYTES);
                tma_load_2d(base + sn * 2 * TM_TILE_BYTES, &tmA, full + sn, (int)(kbeg + (long long)nx * TM_BK), (int)i0);
                tma_load_2d(base + sn * 2 * TM_TILE_BYTES + TM_TILE_BYTES, &tmB, full + sn, (int)(kbeg + (long long)nx * TM_BK), (int)j0);
            }
        }
        mbar_wait(full + s, (unsigned)((kt / TM_STAGES) & 1));
        if (!wskip) {
            const unsigned char *as = base + s * 2 * TM_TILE_BYTES, *bs = as + TM_TILE_BYTES;
#pragma unroll
            for (int kk = 0; kk < TM_BK; kk += 8) {
                double af[2][4], bf[4][2];
#pragma unroll
                for (int a = 0; a < 2; ++a)
#pragma unroll
                    for (int v = 0; v < 4; ++v) af[a][v] = tile_ld(as, wm + a * 16 + 2 * g + (v & 1), kk + t + 4 * (v >> 1));
#pragma unroll
                for (int b = 0; b < 4; ++b)
#pragma unroll
                    for (int v = 0; v < 2; ++v) bf[b][v] = tile_ld(bs, wn + b * 8 + bcol, kk + t + 4 * v);
#pragma unroll
                for (int a = 0; a < 2; ++a)
#pragma unroll
                    for (int b = 0; b < 4; ++b) dmma16x8x8_m(acc[a][b], af[a], bf[b]);
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(empty + s);
    }
    if (wskip) return;
    // epilogue: fragment (row g + 8h, column 2t + e) of block (a, b) is matrix row 2g + h, matrix column 2((2t+e) & 3) + ((2t+e) >> 2)
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const long long i = i0 + wm + a * 16 + 2 * g + h;
            if (i >= M) continue;
#pragma unroll
            for (int b = 0; b < 4; ++b)
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const int nl = 2 * t + e;
                    const long long j = j0 + wn + b * 8 + 2 * (nl & 3) + (nl >> 2);
                    if (j >= N) continue;
                    if (tri && i + tri_off < j) continue;
                    double *c = C + i + j * ldc;
                    const double v = alpha * acc[a][b][2 * h + e];
                    *c = accumulate ? (*c + v) : v;
                }
        }
}

// fixed-order sum of the split-K partial results (same as dense.cu)
__global__ void tma_splitk_reduce_kernel(const double *__restrict__ P, long long split_stride, int splits, double *__restrict__ C,
                                         long long ldc, long long M, long long N, int tri, long long tri_off, double alpha, int accumulate) {
    const long long total = M * N;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const long long i = idx % M, j = idx / M;
        if (tri && i + tri_off < j) continue;
        double s = 0.0;
        for (int z = 0; z < splits; ++z) s += P[(long long)z * split_stride + idx];
        double *c = C + i + j * ldc;
        *c = accumulate ? (*c + alpha * s) : alpha * s;
    }
}

typedef CUresult (*PFN_tmEncodeTiled)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                      const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                      CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_tmEncodeTiled tm_encode_fn() {
    static PFN_tmEncodeTiled fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = (PFN_tmEncodeTiled)p;
    }
    return fn;
}

static bool tm_make(CUtensorMap *map, const double *G, int64_t ld, int64_t rows, int64_t K) {
    PFN_tmEncodeTiled enc = tm_encode_fn();
    if (!enc) return false;
    cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * sizeof(double)};
    cuuint32_t box[2] = {TM_BK, 128};
    cuuint32_t estr[2] = {1, 1};
    return enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, (void *)G, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// true when (A, lda) / (B, ldb) are legal tensor maps and the shape is worth the pipeline
bool gemm_tma_eligible(const double *A, int64_t lda, const double *B, int64_t ldb, int64_t M, int64_t N, int64_t K) {
    if (K < 256 || M < 1 || N < 1) return false;
    if (((uintptr_t)A & 15) || ((uintptr_t)B & 15) || (lda & 1) || (ldb & 1)) return false;
    if (K >= (1LL << 31) || M >= (1LL << 31) || N >= (1LL << 31)) return false;
    return tm_encode_fn() != nullptr;
}

int launch_gemm_tma_tn(smcp_ctx *ctx, const double *A, int64_t lda, const double *B, int64_t ldb, double *C, int64_t ldc,
                       int64_t M, int64_t N, int64_t K, double alpha, int accumulate, int tri, int64_t tri_off, const char *name) {
    CUtensorMap tmA, tmB;
    if (!tm_make(&tmA, A, lda, M, K) || !tm_make(&tmB, B, ldb, N, K)) { smcp_set_error("cuTensorMapEncodeTiled failed"); return -1; }
    dim3 grid((unsigned)((M + TM_BM - 1) / TM_BM), (unsigned)((N + TM_BN - 1) / TM_BN));
    long long ntiles = 0;
    for (unsigned bj = 0; bj < grid.y; ++bj)
        for (unsigned bi = 0; bi < grid.x; ++bi)
            if (!tri || (long long)bi * TM_BM + TM_BM - 1 + tri_off >= (long long)bj * TM_BN) ++ntiles;
    int splits = 1;
    if (K >= 2048 && ntiles > 0 && ntiles < ctx->num_sms) {
        splits = (int)(ctx->num_sms / ntiles);
        if (splits > 16) splits = 16;
        if ((long long)splits * 512 > K) splits = (int)(K / 512);
        if (splits < 1) splits = 1;
    }
    long long kchunk = K, split_stride = 0;
    double *Cout = C;
    int64_t ldout = ldc;
    if (splits > 1) {
        kchunk = ((K + splits - 1) / splits + TM_BK - 1) / TM_BK * TM_BK;
        split_stride = M * N;
        if (grow((void **)&ctx->gemm_ws, &ctx->gemm_ws_cap, (size_t)splits * M * N * sizeof(double))) return -1;
        Cout = ctx->gemm_ws;
        ldout = M;
        grid.z = splits;
    }
    const size_t smem = (size_t)TM_STAGES * 2 * TM_TILE_BYTES + 2 * TM_STAGES * 8 + 1024;
    static bool attr = false;
    if (!attr) {
        CUDA_TRY(cudaFuncSetAttribute(gemm_tma_tn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr = true;
    }
    double pairs = 0.0;
    for (int64_t j = 0; j < N; ++j) {
        int64_t lo = tri ? j - tri_off : 0;
        if (lo < 0) lo = 0;
        if (lo < M) pairs += (double)(M - lo);
    }
    LaunchScope ls(ctx, name, 1, 2.0 * (double)K * pairs);
    if (splits > 1) {
        gemm_tma_tn_kernel<<<grid, TM_THREADS, smem, ctx->stream>>>(tmA, tmB, Cout, ldout, M, N, K, 1.0, 0, tri, tri_off, kchunk, split_stride);
        ctx->launches += 1;
        long long gr = (M * N + 255) / 256;
        if (gr > (long long)ctx->num_sms * 8) gr = (long long)ctx->num_sms * 8;
        tma_splitk_reduce_kernel<<<(unsigned)gr, 256, 0, ctx->stream>>>(ctx->gemm_ws, split_stride, splits, C, ldc, M, N, tri, tri_off, alpha, accumulate);
    } else {
        gemm_tma_tn_kernel<<<grid, TM_THREADS, smem, ctx->stream>>>(tmA, tmB, C, ldc, M, N, K, alpha, accumulate, tri, tri_off, K, 0);
    }
    CUDA_TRY(cudaGetLastError());
    return 0;
}
