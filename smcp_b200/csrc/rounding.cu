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
//  * round_ls: one-flip local search of the +-1 trials (see the section before ROUND_MAX_PASS), between the packing
//    of the samples and their evaluation; the searched signs are evaluated by the same round_pack / eval / sum.
//  * round_tabu: tabu search of the +-1 trials (see the section after round_ls_kernel), after the one-flip search.
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

int launch_round_normals(smcp_ctx *ctx, uint64_t seed, int64_t col0, int n, double *B, int64_t ldb, int64_t k) {
    const long long total = (long long)((n + 3) / 4) * k;
    const long long grid = std::max(1LL, std::min((total + 255) / 256, (long long)ctx->num_sms * 16));
    {
        LaunchScope ls(ctx, "round_normal");
        round_normal_kernel<<<(unsigned)grid, 256, 0, ctx->stream>>>(seed, col0, n, k, B, ldb);
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
    if (launch_round_normals(s->ctx, seed, col0, s->d.n, B, ldb, k)) return -1;
    return k_trsm(s, L, B, ldb, k, 1);
}

// ---------------------------------------------------------------------------------------------------------------------
// One-flip local search of +-1 trials (an extension, like the rounding), f(x) = sum_ij C_ij x_i x_j minimized.
// Row i of the search's CSR holds the off-diagonal entries (i, j) of C from both triangles in increasing j, duplicates
// summed in input order (ls_rows).  Per trial, s_i = sum_{j != i} C_ij x_j in row order and g_i = x_i s_i: flipping i
// changes f by -4 g_i.  A step flips the vertex of largest g_i among those with g_i > thr_i = tol sum_{j != i} |C_ij|
// (lowest i on ties), adds 2 x_i C_ij to s_j over row i (the factor is exact, so a contraction to an FMA changes no
// bit) and negates g_i; the search stops when no vertex qualifies or after max_flips flips.
// round_ls_kernel: one CTA per trial, persistent over the T trials of a pass.  The signs are a bit array in shared
// memory, s is the trial's column of the pass buffer V (dead once the samples are packed), and the largest qualifying
// gain of every LS_CHUNK-vertex chunk is kept in shared memory.  A flip recomputes the chunks of the flipped vertex and
// of its neighbours (all chunks once the row reaches as many), one warp per chunk.  The columns of a row are distinct,
// so no two threads update the same s_j: no atomics, and every result depends on the trial's signs alone.
#define LS_THREADS 256
#define LS_WARPS (LS_THREADS / 32)
#define LS_CHUNK 256
// largest n of the shared layout: n / 8 bytes of signs + 12 bytes per chunk = 176 KiB at 2^20
#define LS_MAX_N (1 << 20)

static size_t ls_smem_bytes(int n) {
    const size_t nch = (size_t)(n + LS_CHUNK - 1) / LS_CHUNK, nxw = (size_t)(n + 31) / 32;
    return nch * (sizeof(double) + sizeof(int)) + nxw * sizeof(unsigned);
}

// (v, i) comes before (bv, bi) in the order of the search: a qualifying vertex (i >= 0), larger gain, lower index
__device__ __forceinline__ bool ls_before(double v, int i, double bv, int bi) {
    return i >= 0 && (bi < 0 || v > bv || (v == bv && i < bi));
}

// the first (v, i) of the warp lands in lane 0
__device__ __forceinline__ void ls_warp_first(double &v, int &i) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double ov = __shfl_down_sync(0xffffffffu, v, o);
        const int oi = __shfl_down_sync(0xffffffffu, i, o);
        if (ls_before(ov, oi, v, i)) { v = ov; i = oi; }
    }
}

// largest qualifying gain of chunk c (one warp); INIT: s of the chunk's vertices is summed from their rows first.
// TABU (round_tabu_kernel): a vertex qualifies when its bit in tw is clear, whatever its gain, and thr is not read.
template <bool INIT, bool TABU = false>
__device__ __forceinline__ void ls_chunk(int c, int n, int lane, const long long *__restrict__ rp, const int *__restrict__ col,
                                         const double *__restrict__ val, const double *__restrict__ thr, const unsigned *xw,
                                         double *s, double *cv, int *ci, const unsigned *tw = nullptr) {
    double bv = 0.0;
    int bi = -1;
    const int i1 = min(n, (c + 1) * LS_CHUNK);
    for (int i = c * LS_CHUNK + lane; i < i1; i += 32) {     // ascending i per lane: the first of equal gains stays
        double si;
        if (INIT) {
            si = 0.0;
            for (long long p = rp[i]; p < rp[i + 1]; ++p) {
                const int j = col[p];
                si += ((xw[j >> 5] >> (j & 31)) & 1u) ? -val[p] : val[p];
            }
            s[i] = si;
        } else {
            si = s[i];
        }
        const double g = ((xw[i >> 5] >> (i & 31)) & 1u) ? -si : si;
        const bool ok = TABU ? !((tw[i >> 5] >> (i & 31)) & 1u) : g > thr[i];
        if (ok && (bi < 0 || g > bv)) { bv = g; bi = i; }
    }
    ls_warp_first(bv, bi);
    if (lane == 0) {
        cv[c] = bv;
        ci[c] = bi;
    }
}

// trial t of the pass: signs from bit t & 63 of the word group t >> 6 of bits, s in V[t n ..], final signs back into
// V[t n + i] as +-1.0 (for round_pack_kernel), the number of flips in flips[t]
// (6 CTAs per SM: 40 registers without spills; at 8, the cap of 32 registers spills)
__global__ void __launch_bounds__(LS_THREADS, 6) round_ls_kernel(int n, int T, const unsigned long long *__restrict__ bits,
                                                              const long long *__restrict__ rp, const int *__restrict__ col,
                                                              const double *__restrict__ val, const double *__restrict__ thr,
                                                              long long max_flips, double *V, long long *__restrict__ flips) {
    extern __shared__ __align__(16) unsigned char ls_smem[];
    const int nch = (n + LS_CHUNK - 1) / LS_CHUNK, nxw = (n + 31) / 32;
    double *cv = (double *)ls_smem;                 // largest qualifying gain of each chunk
    int *ci = (int *)(cv + nch);                    // its vertex, -1: none
    unsigned *xw = (unsigned *)(ci + nch);          // bit i: x_i = -1
    __shared__ double wv[LS_WARPS];
    __shared__ int wi[LS_WARPS];
    __shared__ int pick, pneg;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int t = blockIdx.x; t < T; t += gridDim.x) {
        const unsigned long long *wg = bits + (long long)(t >> 6) * n;
        const int b = t & 63;
        double *s = V + (long long)t * n;
        for (int w = warp; w < nxw; w += LS_WARPS) {
            const int i = 32 * w + lane;
            const unsigned m = __ballot_sync(0xffffffffu, i < n && ((wg[i] >> b) & 1ULL));
            if (lane == 0) xw[w] = m;
        }
        __syncthreads();
        for (int c = warp; c < nch; c += LS_WARPS) ls_chunk<true>(c, n, lane, rp, col, val, thr, xw, s, cv, ci);
        __syncthreads();
        long long nf = 0;
        while (nf < max_flips) {
            double bv = 0.0;
            int bi = -1;
            for (int c = threadIdx.x; c < nch; c += LS_THREADS)
                if (ls_before(cv[c], ci[c], bv, bi)) { bv = cv[c]; bi = ci[c]; }
            ls_warp_first(bv, bi);
            if (lane == 0) {
                wv[warp] = bv;
                wi[warp] = bi;
            }
            __syncthreads();
            if (threadIdx.x == 0) {
                for (int w = 1; w < LS_WARPS; ++w)
                    if (ls_before(wv[w], wi[w], bv, bi)) { bv = wv[w]; bi = wi[w]; }
                if (bi >= 0) {
                    const unsigned m = 1u << (bi & 31);
                    pneg = (xw[bi >> 5] & m) == 0u;      // the new sign of x_bi
                    xw[bi >> 5] ^= m;
                }
                pick = bi;
            }
            __syncthreads();
            const int i = pick;
            if (i < 0) break;
            ++nf;
            const long long p0 = rp[i], p1 = rp[i + 1];
            const double two = pneg ? -2.0 : 2.0;
            for (long long p = p0 + threadIdx.x; p < p1; p += LS_THREADS) {
                const int j = col[p];
                s[j] = s[j] + two * val[p];
            }
            __syncthreads();
            const int d = (int)(p1 - p0), c0 = i / LS_CHUNK;
            if (d + 1 >= nch) {
                for (int c = warp; c < nch; c += LS_WARPS) ls_chunk<false>(c, n, lane, rp, col, val, thr, xw, s, cv, ci);
            } else {
                // entry d: the chunk of i; entry e < d: the chunk of the e-th neighbour unless an earlier entry has it
                // (columns ascend, so equal chunks of neighbours are adjacent)
                for (int e = warp; e <= d; e += LS_WARPS) {
                    int c = c0;
                    if (e < d) {
                        c = col[p0 + e] / LS_CHUNK;
                        if (c == c0 || (e > 0 && col[p0 + e - 1] / LS_CHUNK == c)) continue;
                    }
                    ls_chunk<false>(c, n, lane, rp, col, val, thr, xw, s, cv, ci);
                }
            }
            __syncthreads();
        }
        for (int i = threadIdx.x; i < n; i += LS_THREADS) s[i] = ((xw[i >> 5] >> (i & 31)) & 1u) ? -1.0 : 1.0;
        if (threadIdx.x == 0) flips[t] = nf;
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// Tabu search of +-1 trials: the rows, s and g of the one-flip search.  D_0 = 0; move u flips the admissible vertex i of
// largest g_i (lowest i on ties) and sets D_{u+1} = D_u - 4 g_i; D_best, the smallest D so far, changes only on a strict
// decrease.  A vertex flipped at move u is tabu during moves u+1 .. u+tenure; a tabu vertex is admissible only when
// D_u - 4 g_i < D_best (aspiration), every other vertex always is.  The search stops after iters moves or when no vertex
// is admissible (tenure >= n only) and returns the vector of the earliest move count at which D reached D_best.
// round_tabu_kernel: round_ls_kernel's layout and chunk maxima, taken over the non-tabu vertices without threshold.  The
// tabu set is a bit array tw plus a ring of the last `tenure` flips in shared memory; the flip leaving the ring clears
// its bit only if the vertex has no later entry, and only then is its chunk recomputed.  Aspiration scans the ring.  The
// best vector is a bit copy in global memory (this CTA's nxw words of bestw), taken just before the first move that
// leaves a best state, so a descent copies nothing.
#define TABU_MAX_N (1 << 19)
#define TABU_MAX_TENURE 8192

// n / 4 bytes of signs and tabu bits, 12 bytes per chunk and the ring: 184 KiB at n = 2^19, tenure = 8192
static size_t tabu_smem_bytes(int n, int tenure) {
    return ls_smem_bytes(n) + (size_t)(n + 31) / 32 * sizeof(unsigned) + (size_t)tenure * sizeof(int);
}

// the sorted columns col[0 .. d) have one in chunk c
__device__ __forceinline__ bool tabu_row_has_chunk(const int *__restrict__ col, int d, int c) {
    int lo = 0, hi = d;
    while (lo < hi) {
        const int m = (lo + hi) >> 1;
        if (col[m] < c * LS_CHUNK) lo = m + 1;
        else hi = m;
    }
    return lo < d && col[lo] < (c + 1) * LS_CHUNK;
}

// trial t of the pass: signs from bit t & 63 of the word group t >> 6 of bits, s in V[t n ..], the best vector back into
// V[t n + i] as +-1.0 (for round_pack_kernel), the number of moves in moves[t] and the move count of the best vector in
// best_iter[t]
__global__ void __launch_bounds__(LS_THREADS, 4) round_tabu_kernel(int n, int T, const unsigned long long *__restrict__ bits,
                                                                const long long *__restrict__ rp, const int *__restrict__ col,
                                                                const double *__restrict__ val, long long iters, int tenure,
                                                                double *V, unsigned *__restrict__ bestw,
                                                                long long *__restrict__ moves, long long *__restrict__ best_iter) {
    extern __shared__ __align__(16) unsigned char tabu_smem[];
    const int nch = (n + LS_CHUNK - 1) / LS_CHUNK, nxw = (n + 31) / 32;
    double *cv = (double *)tabu_smem;               // largest gain of the non-tabu vertices of each chunk
    int *ci = (int *)(cv + nch);                    // its vertex, -1: none
    unsigned *xw = (unsigned *)(ci + nch);          // bit i: x_i = -1
    unsigned *tw = xw + nxw;                        // bit i: i is tabu
    int *ring = (int *)(tw + nxw);                  // ring[u % tenure]: the vertex flipped by move u
    __shared__ double wv[LS_WARPS];
    __shared__ int wi[LS_WARPS];
    __shared__ unsigned wdup[LS_WARPS];
    __shared__ double D, Db;                        // D_u and D_best
    __shared__ long long ub;                        // the move count of D_best
    __shared__ int pick, pneg, pexp, pcopy, pend;   // pend: the current vector is the best and has no copy in bestw
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned *gb = bestw + (long long)blockIdx.x * nxw;
    for (int t = blockIdx.x; t < T; t += gridDim.x) {
        const unsigned long long *wg = bits + (long long)(t >> 6) * n;
        const int b = t & 63;
        double *s = V + (long long)t * n;
        for (int w = warp; w < nxw; w += LS_WARPS) {
            const int i = 32 * w + lane;
            const unsigned m = __ballot_sync(0xffffffffu, i < n && ((wg[i] >> b) & 1ULL));
            if (lane == 0) {
                xw[w] = m;
                tw[w] = 0u;
            }
        }
        if (threadIdx.x == 0) {
            D = 0.0;
            Db = 0.0;
            ub = 0;
            pend = 1;
        }
        __syncthreads();
        for (int c = warp; c < nch; c += LS_WARPS) ls_chunk<true, true>(c, n, lane, rp, col, val, nullptr, xw, s, cv, ci, tw);
        __syncthreads();
        long long u = 0;
        for (; u < iters; ++u) {
            const int nr = (int)min((long long)tenure, u);              // ring entries in use, all of them tabu
            const int slot = tenure > 0 ? (int)(u % tenure) : 0;
            const int ex = u >= tenure && tenure > 0 ? ring[slot] : -1;  // its flip leaves the ring with this move
            double bv = 0.0;
            int bi = -1;
            for (int c = threadIdx.x; c < nch; c += LS_THREADS)
                if (ls_before(cv[c], ci[c], bv, bi)) { bv = cv[c]; bi = ci[c]; }
            bool dup = false;
            const double d0 = D, db = Db;
            for (int r = threadIdx.x; r < nr; r += LS_THREADS) {
                const int v = ring[r];
                dup |= r != slot && v == ex;
                const double g = ((xw[v >> 5] >> (v & 31)) & 1u) ? -s[v] : s[v];
                if (d0 - 4.0 * g < db && ls_before(g, v, bv, bi)) { bv = g; bi = v; }
            }
            ls_warp_first(bv, bi);
            const unsigned wd = __ballot_sync(0xffffffffu, dup);
            if (lane == 0) {
                wv[warp] = bv;
                wi[warp] = bi;
                wdup[warp] = wd;
            }
            __syncthreads();
            if (threadIdx.x == 0) {
                bool later = false;
                for (int w = 0; w < LS_WARPS; ++w) later |= wdup[w] != 0u;
                for (int w = 1; w < LS_WARPS; ++w)
                    if (ls_before(wv[w], wi[w], bv, bi)) { bv = wv[w]; bi = wi[w]; }
                int e = -1;
                if (bi >= 0) {
                    const double dn = d0 - 4.0 * bv;
                    const bool better = dn < db;
                    pcopy = pend && !better;
                    pend = better;
                    if (better) {
                        Db = dn;
                        ub = u + 1;
                    }
                    D = dn;
                    const unsigned m = 1u << (bi & 31);
                    pneg = (xw[bi >> 5] & m) == 0u;
                    xw[bi >> 5] ^= m;
                    if (tenure > 0) {
                        tw[bi >> 5] |= m;
                        ring[slot] = bi;
                    }
                    if (ex >= 0 && ex != bi && !later) {
                        tw[ex >> 5] &= ~(1u << (ex & 31));
                        e = ex;
                    }
                }
                pick = bi;
                pexp = e;
            }
            __syncthreads();
            const int i = pick;
            if (i < 0) break;
            if (pcopy) {                                                 // the vector before this move, bit i restored
                const int wi0 = i >> 5;
                const unsigned m = 1u << (i & 31);
                for (int w = threadIdx.x; w < nxw; w += LS_THREADS) gb[w] = w == wi0 ? xw[w] ^ m : xw[w];
            }
            const long long p0 = rp[i], p1 = rp[i + 1];
            const double two = pneg ? -2.0 : 2.0;
            for (long long p = p0 + threadIdx.x; p < p1; p += LS_THREADS) {
                const int j = col[p];
                s[j] = s[j] + two * val[p];
            }
            __syncthreads();
            // entries as in round_ls_kernel, plus entry d + 1: the chunk of the vertex that left the tabu set
            const int d = (int)(p1 - p0), c0 = i / LS_CHUNK, ce = pexp >= 0 ? pexp / LS_CHUNK : -1;
            if (d + 2 >= nch) {
                for (int c = warp; c < nch; c += LS_WARPS) ls_chunk<false, true>(c, n, lane, rp, col, val, nullptr, xw, s, cv, ci, tw);
            } else {
                for (int e = warp; e <= d + 1; e += LS_WARPS) {
                    int c = c0;
                    if (e < d) {
                        c = col[p0 + e] / LS_CHUNK;
                        if (c == c0 || (e > 0 && col[p0 + e - 1] / LS_CHUNK == c)) continue;
                    } else if (e == d + 1) {
                        if (ce < 0 || ce == c0 || tabu_row_has_chunk(col + p0, d, ce)) continue;
                        c = ce;
                    }
                    ls_chunk<false, true>(c, n, lane, rp, col, val, nullptr, xw, s, cv, ci, tw);
                }
            }
            __syncthreads();
        }
        const unsigned *res = pend ? xw : gb;
        for (int i = threadIdx.x; i < n; i += LS_THREADS) s[i] = ((res[i >> 5] >> (i & 31)) & 1u) ? -1.0 : 1.0;
        if (threadIdx.x == 0) {
            moves[t] = u;
            best_iter[t] = ub;
        }
        __syncthreads();
    }
}

// largest number of trials a pass holds: bounds the word groups (grid.y) and the slice partial sums
#define ROUND_MAX_PASS 65536
// columns of one trsm call; every call of a smcp_round_pm1 has the same width, so the samples of a trial are the
// same bits whatever the pass size (k_trsm picks its kernels from the number of right-hand sides)
#define ROUND_BLOCK 256

// the objective on the device, as round_eval_kernel reads it: nc entries (r, c, coef), the factor 2 off the diagonal
// folded into coef, cut into S fixed slices of `per` entries (independent of the trials)
struct RoundObj {
    int *er = nullptr, *ec = nullptr;
    double *ev = nullptr;
    long long nc = 0, per = 1;
    int S = 1;
};

static int round_obj_upload(RoundWs &ws, const char *fn, int n, int64_t nc, const int64_t *crow, const int64_t *ccol,
                            const double *cval, RoundObj &o) {
    std::vector<int> hr((size_t)nc), hc((size_t)nc);
    std::vector<double> hv((size_t)nc);
    for (int64_t q = 0; q < nc; ++q) {
        if (crow[q] < 0 || crow[q] >= n || ccol[q] < 0 || ccol[q] >= n) {
            smcp_set_error("%s: objective entry %lld at (%lld, %lld) is outside 0..%d", fn, (long long)q, (long long)crow[q],
                           (long long)ccol[q], n - 1);
            return -2;
        }
        hr[q] = (int)crow[q];
        hc[q] = (int)ccol[q];
        hv[q] = crow[q] == ccol[q] ? cval[q] : 2.0 * cval[q];
    }
    o.nc = nc;
    o.S = (int)std::min<int64_t>(256, std::max<int64_t>(1, (nc + 511) / 512));
    o.per = std::max<long long>(1, (nc + o.S - 1) / o.S);
    o.er = (int *)ws.alloc((size_t)nc * sizeof(int));
    o.ec = (int *)ws.alloc((size_t)nc * sizeof(int));
    o.ev = (double *)ws.alloc((size_t)nc * sizeof(double));
    if (!o.er || !o.ec || !o.ev) return -1;
    if (nc) {
        CUDA_TRY(cudaMemcpyAsync(o.er, hr.data(), (size_t)nc * sizeof(int), cudaMemcpyHostToDevice, ws.ctx->stream));
        CUDA_TRY(cudaMemcpyAsync(o.ec, hc.data(), (size_t)nc * sizeof(int), cudaMemcpyHostToDevice, ws.ctx->stream));
        CUDA_TRY(cudaMemcpyAsync(o.ev, hv.data(), (size_t)nc * sizeof(double), cudaMemcpyHostToDevice, ws.ctx->stream));
    }
    return 0;
}

int ls_rows_upload(RoundWs &ws, int n, int64_t nc, const int64_t *crow, const int64_t *ccol, const double *cval, double tol,
                   LsRows &d, LsRowsHost *host) {
    std::vector<int64_t> q;
    for (int64_t e = 0; e < nc; ++e)
        if (crow[e] != ccol[e]) q.push_back(e);
    auto lo = [&](int64_t e) { return std::min(crow[e], ccol[e]); };
    auto hi = [&](int64_t e) { return std::max(crow[e], ccol[e]); };
    std::stable_sort(q.begin(), q.end(), [&](int64_t a, int64_t b) { return lo(a) < lo(b) || (lo(a) == lo(b) && hi(a) < hi(b)); });
    // merged pairs (l < h) ascending; row l gets (h, v) and row h gets (l, v).  In this order every row receives its
    // columns ascending: first the l < row (pairs of smaller l come first), then the h > row.
    std::vector<int> pl, ph;
    std::vector<double> pv;
    for (size_t a = 0; a < q.size();) {
        const int64_t l = lo(q[a]), h = hi(q[a]);
        double v = cval[q[a]];
        size_t b = a + 1;
        for (; b < q.size() && lo(q[b]) == l && hi(q[b]) == h; ++b) v += cval[q[b]];
        pl.push_back((int)l);
        ph.push_back((int)h);
        pv.push_back(v);
        a = b;
    }
    std::vector<long long> rp((size_t)n + 1, 0);
    for (size_t e = 0; e < pv.size(); ++e) {
        ++rp[pl[e] + 1];
        ++rp[ph[e] + 1];
    }
    for (int i = 0; i < n; ++i) rp[i + 1] += rp[i];
    const size_t nnz = (size_t)rp[n];
    std::vector<long long> fill(rp.begin(), rp.end() - 1);
    std::vector<int> col(nnz);
    std::vector<double> val(nnz), thr((size_t)n);
    for (size_t e = 0; e < pv.size(); ++e) {
        col[fill[pl[e]]] = ph[e];
        val[fill[pl[e]]++] = pv[e];
        col[fill[ph[e]]] = pl[e];
        val[fill[ph[e]]++] = pv[e];
    }
    for (int i = 0; i < n; ++i) {
        double a = 0.0;
        for (long long p = rp[i]; p < rp[i + 1]; ++p) a += std::fabs(val[p]);
        thr[i] = tol * a;
    }
    d.rp = (long long *)ws.alloc(rp.size() * sizeof(long long));
    d.col = (int *)ws.alloc(nnz * sizeof(int));
    d.val = (double *)ws.alloc(nnz * sizeof(double));
    d.thr = (double *)ws.alloc((size_t)n * sizeof(double));
    if (!d.rp || !d.col || !d.val || !d.thr) return -1;
    cudaStream_t st = ws.ctx->stream;
    CUDA_TRY(cudaMemcpyAsync(d.rp, rp.data(), rp.size() * sizeof(long long), cudaMemcpyHostToDevice, st));
    if (nnz) {
        CUDA_TRY(cudaMemcpyAsync(d.col, col.data(), nnz * sizeof(int), cudaMemcpyHostToDevice, st));
        CUDA_TRY(cudaMemcpyAsync(d.val, val.data(), nnz * sizeof(double), cudaMemcpyHostToDevice, st));
    }
    CUDA_TRY(cudaMemcpyAsync(d.thr, thr.data(), (size_t)n * sizeof(double), cudaMemcpyHostToDevice, st));
    if (host) {
        host->rp = std::move(rp);
        host->col = std::move(col);
    }
    return 0;
}

// what runs on every trial between its packing and the evaluation that values_host reports: the one-flip search
// (max_flips, tol; flips_host) and, with tabu, the tabu search after it (tabu_iters, tenure; moves_host, best_iter_host).
// With tabu the one-flip search runs only when max_flips > 0.  In smcp_round_pm1_ls / _tabu, values0_host receives the
// values of the rounded trials, and with tabu values1_host those before the tabu search.
struct LsArgs {
    int64_t max_flips;
    double tol;
    double *values0_host;
    int64_t *flips_host;
    bool tabu;
    int64_t tabu_iters, tenure;
    double *values1_host;
    int64_t *moves_host, *best_iter_host;
    bool one_flip() const { return !tabu || max_flips > 0; }
};

// checks shared by the entry points of the searches
static int ls_check(const char *fn, int n, const LsArgs &a) {
    const int nmax = a.tabu ? TABU_MAX_N : LS_MAX_N;
    if (n > nmax) {
        smcp_set_error("%s: n = %d exceeds %d, the largest the search's shared-memory layout holds", fn, n, nmax);
        return -2;
    }
    if (a.max_flips < 0 || !(a.tol >= 0.0) || !std::isfinite(a.tol)) {
        smcp_set_error("%s: need max_flips >= 0 and a finite tol >= 0 (got %lld, %g)", fn, (long long)a.max_flips, a.tol);
        return -2;
    }
    if (a.tabu && (a.tabu_iters < 0 || a.tenure < 0 || a.tenure > TABU_MAX_TENURE)) {
        smcp_set_error("%s: need tabu_iters >= 0 and 0 <= tenure <= %d (got %lld, %lld)", fn, TABU_MAX_TENURE,
                       (long long)a.tabu_iters, (long long)a.tenure);
        return -2;
    }
    return 0;
}

static int launch_ls(smcp_ctx *ctx, int n, int T, const unsigned long long *bits, const LsRows &d, int64_t max_flips, double *V,
                     long long *flips) {
    const size_t smem = ls_smem_bytes(n);
    CUDA_TRY(cudaFuncSetAttribute(round_ls_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, round_ls_kernel, LS_THREADS, smem));
    const int grid = std::max(1, std::min(T, std::max(1, per_sm) * ctx->num_sms));
    {
        LaunchScope ls(ctx, "round_ls");
        round_ls_kernel<<<grid, LS_THREADS, smem, ctx->stream>>>(n, T, bits, d.rp, d.col, d.val, d.thr, (long long)max_flips, V,
                                                                 flips);
    }
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// the tabu search of the T trials of a pass; bestw (one nxw-word copy per CTA) is allocated at the first pass, which has
// the most trials and so the largest grid
static int launch_tabu(RoundWs &ws, int n, int T, const unsigned long long *bits, const LsRows &d, const LsArgs &a, double *V,
                       unsigned *&bestw, long long *moves, long long *best_iter) {
    smcp_ctx *ctx = ws.ctx;
    const size_t smem = tabu_smem_bytes(n, (int)a.tenure);
    CUDA_TRY(cudaFuncSetAttribute(round_tabu_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, round_tabu_kernel, LS_THREADS, smem));
    const int grid = std::max(1, std::min(T, std::max(1, per_sm) * ctx->num_sms));
    if (!bestw && !(bestw = (unsigned *)ws.alloc((size_t)grid * ((n + 31) / 32) * sizeof(unsigned)))) return -1;
    {
        LaunchScope ls(ctx, "round_tabu");
        round_tabu_kernel<<<grid, LS_THREADS, smem, ctx->stream>>>(n, T, bits, d.rp, d.col, d.val, (long long)a.tabu_iters,
                                                                   (int)a.tenure, V, bestw, moves, best_iter);
    }
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// values[t0 + t] of the T trials whose signs are sign(V[:, t]) (packed into bits first); with `best`, the best trial so
// far and its signs x are updated
static int eval_pass(smcp_ctx *ctx, const double *V, int n, int T, unsigned long long *bits, const RoundObj &o, double *part,
                     int64_t t0, double *values, RoundBest *best, signed char *x) {
    const int nw = (T + 63) / 64;
    {
        LaunchScope ls(ctx, "round_eval", best ? 4 : 3);
        round_pack_kernel<<<dim3((unsigned)((n + 255) / 256), (unsigned)nw), 256, 0, ctx->stream>>>(V, n, n, T, bits);
        round_eval_kernel<<<dim3((unsigned)o.S, (unsigned)nw), 32 * EV_WARPS, 0, ctx->stream>>>(o.er, o.ec, o.ev, o.nc, o.per, bits,
                                                                                             n, part);
        round_sum_kernel<<<(unsigned)((T + 255) / 256), 256, 0, ctx->stream>>>(part, o.S, T, t0, values);
        if (best) round_best_kernel<<<1, BEST_THREADS, 0, ctx->stream>>>(values, t0, T, bits, n, best, x);
    }
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// device outputs of the searches over all trials; bestw is allocated by launch_tabu
struct LsOut {
    double *values1 = nullptr;
    long long *flips = nullptr, *moves = nullptr, *best_iter = nullptr;
    unsigned *bestw = nullptr;
};

// the searches of `a` on the T trials t0 .. t0 + T - 1 of a pass whose signs are packed in bits; V[:, t] then holds the
// searched signs as +-1.0.  With tabu after the one-flip search, out.values1 receives the values in between.
static int search_pass(RoundWs &ws, int n, int T, int64_t t0, unsigned long long *bits, const RoundObj &o, double *part,
                       const LsRows &d, const LsArgs &a, double *V, LsOut &out) {
    if (a.one_flip()) {
        if (launch_ls(ws.ctx, n, T, bits, d, a.max_flips, V, out.flips + t0)) return -1;
        if (a.tabu && eval_pass(ws.ctx, V, n, T, bits, o, part, t0, out.values1, nullptr, nullptr)) return -1;
    }
    if (a.tabu && launch_tabu(ws, n, T, bits, d, a, V, out.bestw, out.moves + t0, out.best_iter + t0)) return -1;
    return 0;
}

// where the samples of a pass come from: L^-T g, the normals through the chordal trsm with the completion factor L of
// s (smcp_round_pm1*), or V g, normals of length r times the factor V (n x r, row-major on the device) in one DMMA
// product (smcp_round_pm1_factor; G holds the r x tb normals of a block)
struct RoundSrc {
    smcp_sym *s;
    const double *L;
    const double *V;
    int r;
    double *G;
};

// the samples col0 .. col0 + tb - 1 into the n x tb block Vb
static int round_samples(smcp_ctx *ctx, int n, const RoundSrc &src, uint64_t seed, int64_t col0, double *Vb, int64_t tb) {
    if (src.L) {
        if (launch_round_normals(ctx, seed, col0, n, Vb, n, tb)) return -1;
        return k_trsm(src.s, src.L, Vb, n, tb, 1);
    }
    if (launch_round_normals(ctx, seed, col0, src.r, src.G, src.r, tb)) return -1;
    return launch_gemm(ctx, true, true, src.V, src.r, src.G, src.r, Vb, n, n, tb, src.r, 1.0, 0, 0, 0, "round_factor");
}

// ls == nullptr: plain rounding; otherwise the searches run on every trial between its evaluation into
// ls->values0_host and the evaluation that values_host, x_host and best_out report.  src.G is allocated here.
static int round_pm1_impl(smcp_ctx *ctx, const char *fn, int n, RoundSrc src, uint64_t seed, int64_t trials, int64_t chunk,
                          int64_t nc, const int64_t *crow, const int64_t *ccol, const double *cval, const LsArgs *ls,
                          double *values_host, int8_t *x_host, int64_t *best_out) {
    if (trials < 1 || chunk < 0 || nc < 0) {
        smcp_set_error("%s: need trials >= 1, chunk >= 0, nc >= 0 (got %lld, %lld, %lld)", fn, (long long)trials,
                       (long long)chunk, (long long)nc);
        return -2;
    }
    if (!(src.L || src.V) || !values_host || !x_host || !best_out || (nc > 0 && (!crow || !ccol || !cval)) ||
        (ls && (!ls->values0_host || !ls->flips_host)) ||
        (ls && ls->tabu && (!ls->values1_host || !ls->moves_host || !ls->best_iter_host))) {
        smcp_set_error("%s: null argument", fn);
        return -2;
    }
    if (ls && ls_check(fn, n, *ls)) return -2;
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

    RoundWs ws{ctx, fn, {}};
    if (!src.L && !(src.G = (double *)ws.alloc((size_t)src.r * tb * sizeof(double)))) return -1;
    RoundObj o;
    if (int rc = round_obj_upload(ws, fn, n, nc, crow, ccol, cval, o)) return rc;
    LsRows d;
    if (ls && ls_rows_upload(ws, n, nc, crow, ccol, cval, ls->tol, d, nullptr)) return -1;
    double *V = (double *)ws.alloc((size_t)n * pw * sizeof(double));
    unsigned long long *bits = (unsigned long long *)ws.alloc((size_t)n * nwmax * sizeof(unsigned long long));
    double *part = (double *)ws.alloc((size_t)nwmax * o.S * 64 * sizeof(double));
    double *values = (double *)ws.alloc((size_t)trials * sizeof(double));
    RoundBest *best = (RoundBest *)ws.alloc(sizeof(RoundBest));
    signed char *x = (signed char *)ws.alloc((size_t)n);
    double *values0 = ls ? (double *)ws.alloc((size_t)trials * sizeof(double)) : nullptr;
    LsOut out;
    const bool tabu = ls && ls->tabu, one_flip = ls && ls->one_flip();
    if (ls) out.flips = (long long *)ws.alloc((size_t)trials * sizeof(long long));
    if (tabu && one_flip) out.values1 = (double *)ws.alloc((size_t)trials * sizeof(double));
    if (tabu) {
        out.moves = (long long *)ws.alloc((size_t)trials * sizeof(long long));
        out.best_iter = (long long *)ws.alloc((size_t)trials * sizeof(long long));
    }
    if (!V || !bits || !part || !values || !best || !x || (ls && (!values0 || !out.flips)) ||
        (tabu && ((one_flip && !out.values1) || !out.moves || !out.best_iter)))
        return -1;
    const RoundBest none{0.0, -1};
    CUDA_TRY(cudaMemcpyAsync(best, &none, sizeof(none), cudaMemcpyHostToDevice, ctx->stream));
    if (ls && !one_flip) CUDA_TRY(cudaMemsetAsync(out.flips, 0, (size_t)trials * sizeof(long long), ctx->stream));
    for (int64_t b0 = 0; b0 < nblocks; b0 += bp) {
        const int64_t b1 = std::min(nblocks, b0 + bp);
        const int64_t t0 = b0 * tb;
        for (int64_t b = b0; b < b1; ++b) {
            double *Vb = V + (size_t)(b - b0) * tb * n;
            if (round_samples(ctx, n, src, seed, b * tb, Vb, tb)) return -1;
        }
        const int T = (int)std::min<int64_t>(trials - t0, (b1 - b0) * tb);
        if (!ls) {
            if (eval_pass(ctx, V, n, T, bits, o, part, t0, values, best, x)) return -1;
            continue;
        }
        if (eval_pass(ctx, V, n, T, bits, o, part, t0, values0, nullptr, nullptr)) return -1;
        if (search_pass(ws, n, T, t0, bits, o, part, d, *ls, V, out)) return -1;
        if (eval_pass(ctx, V, n, T, bits, o, part, t0, values, best, x)) return -1;
    }
    RoundBest hb;
    CUDA_TRY(cudaMemcpyAsync(values_host, values, (size_t)trials * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(x_host, x, (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(&hb, best, sizeof(hb), cudaMemcpyDeviceToHost, ctx->stream));
    if (ls) {
        static_assert(sizeof(long long) == sizeof(int64_t), "flip counts are copied as int64");
        CUDA_TRY(cudaMemcpyAsync(ls->values0_host, values0, (size_t)trials * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_TRY(cudaMemcpyAsync(ls->flips_host, out.flips, (size_t)trials * sizeof(long long), cudaMemcpyDeviceToHost,
                                 ctx->stream));
    }
    if (tabu) {
        CUDA_TRY(cudaMemcpyAsync(ls->values1_host, one_flip ? out.values1 : values0, (size_t)trials * sizeof(double),
                                 cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_TRY(cudaMemcpyAsync(ls->moves_host, out.moves, (size_t)trials * sizeof(long long), cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_TRY(cudaMemcpyAsync(ls->best_iter_host, out.best_iter, (size_t)trials * sizeof(long long), cudaMemcpyDeviceToHost,
                                 ctx->stream));
    }
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    if (hb.t < 0) {
        smcp_set_error("%s: no trial has a finite value", fn);
        return -1;
    }
    *best_out = hb.t;
    return 0;
}

int k_round_pm1(smcp_sym *s, const double *L, uint64_t seed, int64_t trials, int64_t chunk, int64_t nc, const int64_t *crow,
                const int64_t *ccol, const double *cval, double *values_host, int8_t *x_host, int64_t *best_out) {
    return round_pm1_impl(s->ctx, "smcp_round_pm1", s->d.n, RoundSrc{s, L, nullptr, 0, nullptr}, seed, trials, chunk, nc, crow,
                          ccol, cval, nullptr, values_host, x_host, best_out);
}

int k_round_pm1_ls(smcp_sym *s, const double *L, uint64_t seed, int64_t trials, int64_t chunk, int64_t nc, const int64_t *crow,
                   const int64_t *ccol, const double *cval, int64_t max_flips, double tol, double *values0_host,
                   double *values_host, int8_t *x_host, int64_t *best_out, int64_t *flips_host) {
    const LsArgs ls{max_flips, tol, values0_host, flips_host, false, 0, 0, nullptr, nullptr, nullptr};
    return round_pm1_impl(s->ctx, "smcp_round_pm1_ls", s->d.n, RoundSrc{s, L, nullptr, 0, nullptr}, seed, trials, chunk, nc, crow,
                          ccol, cval, &ls, values_host, x_host, best_out);
}

int k_round_pm1_tabu(smcp_sym *s, const double *L, uint64_t seed, int64_t trials, int64_t chunk, int64_t nc,
                     const int64_t *crow, const int64_t *ccol, const double *cval, int64_t max_flips, double tol,
                     double *values0_host, double *values_host, int8_t *x_host, int64_t *best_out, int64_t *flips_host,
                     int64_t tabu_iters, int64_t tenure, double *values1_host, int64_t *moves_host, int64_t *best_iter_host) {
    const LsArgs ls{max_flips, tol, values0_host, flips_host, true, tabu_iters, tenure, values1_host, moves_host, best_iter_host};
    return round_pm1_impl(s->ctx, "smcp_round_pm1_tabu", s->d.n, RoundSrc{s, L, nullptr, 0, nullptr}, seed, trials, chunk, nc, crow,
                          ccol, cval, &ls, values_host, x_host, best_out);
}

// the factor crosses to the device once; the searches are on when max_flips > 0 (one-flip) or tabu_iters > 0 (tabu, after
// the one-flip search when that is on too)
int k_round_pm1_factor(smcp_ctx *ctx, int64_t n, int64_t r, const double *V_host, uint64_t seed, int64_t trials, int64_t chunk,
                       int64_t nc, const int64_t *crow, const int64_t *ccol, const double *cval, int64_t max_flips, double tol,
                       int64_t tabu_iters, int64_t tenure, double *values0_host, double *values1_host, double *values_host,
                       int8_t *x_host, int64_t *best_out, int64_t *flips_host, int64_t *moves_host, int64_t *best_iter_host) {
    const char *fn = "smcp_round_pm1_factor";
    if (n < 1 || n > INT32_MAX || r < 1 || !V_host || max_flips < 0 || tabu_iters < 0) {
        smcp_set_error("%s: need 1 <= n < 2^31, r >= 1, a factor, max_flips >= 0 and tabu_iters >= 0 (got %lld, %lld, %lld, %lld)",
                       fn, (long long)n, (long long)r, (long long)max_flips, (long long)tabu_iters);
        return -2;
    }
    for (int64_t e = 0; e < n * r; ++e)
        if (!std::isfinite(V_host[e])) {
            smcp_set_error("%s: V[%lld][%lld] is not finite", fn, (long long)(e / r), (long long)(e % r));
            return -2;
        }
    CUDA_TRY(cudaSetDevice(ctx->device));
    RoundWs ws{ctx, fn, {}};
    double *V = (double *)ws.alloc((size_t)n * r * sizeof(double));
    if (!V) return -1;
    CUDA_TRY(cudaMemcpyAsync(V, V_host, (size_t)n * r * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    const RoundSrc src{nullptr, nullptr, V, (int)r, nullptr};
    const bool tabu = tabu_iters > 0;
    const LsArgs ls{max_flips, tol, values0_host, flips_host, tabu, tabu_iters, tenure, values1_host, moves_host, best_iter_host};
    return round_pm1_impl(ctx, fn, (int)n, src, seed, trials, chunk, nc, crow, ccol, cval, max_flips > 0 || tabu ? &ls : nullptr,
                          values_host, x_host, best_out);
}

// the searches of `a` on k caller-given vectors x_host, replaced by the searched ones
static int pm1_search_impl(smcp_ctx *ctx, const char *fn, int64_t n, int64_t k, int8_t *x_host, int64_t nc, const int64_t *crow,
                           const int64_t *ccol, const double *cval, const LsArgs &a, double *values_host) {
    if (n < 1 || k < 1 || nc < 0) {
        smcp_set_error("%s: need n >= 1, k >= 1, nc >= 0 (got %lld, %lld, %lld)", fn, (long long)n, (long long)k, (long long)nc);
        return -2;
    }
    if (!x_host || !values_host || (nc > 0 && (!crow || !ccol || !cval)) || (a.one_flip() && !a.flips_host) ||
        (a.tabu && (!a.moves_host || !a.best_iter_host))) {
        smcp_set_error("%s: null argument", fn);
        return -2;
    }
    if (ls_check(fn, (int)std::min<int64_t>(n, INT32_MAX), a)) return -2;
    for (int64_t e = 0; e < n * k; ++e)
        if (x_host[e] != 1 && x_host[e] != -1) {
            smcp_set_error("%s: x[%lld][%lld] = %d is not +-1", fn, (long long)(e / n), (long long)(e % n), (int)x_host[e]);
            return -2;
        }
    CUDA_TRY(cudaSetDevice(ctx->device));
    // trials per pass: the s workspace (n x pw doubles) within 1 GiB, as in smcp_round_pm1
    const int64_t fit = std::max<int64_t>(1, (int64_t(1) << 30) / (8 * n));
    const int64_t pw = std::min<int64_t>(k, std::min<int64_t>(fit, ROUND_MAX_PASS));
    const int64_t nwmax = (pw + 63) / 64;
    RoundWs ws{ctx, fn, {}};
    RoundObj o;
    if (int rc = round_obj_upload(ws, fn, (int)n, nc, crow, ccol, cval, o)) return rc;
    LsRows d;
    if (ls_rows_upload(ws, (int)n, nc, crow, ccol, cval, a.tol, d, nullptr)) return -1;
    double *V = (double *)ws.alloc((size_t)n * pw * sizeof(double));
    unsigned long long *bits = (unsigned long long *)ws.alloc((size_t)n * nwmax * sizeof(unsigned long long));
    double *part = (double *)ws.alloc((size_t)nwmax * o.S * 64 * sizeof(double));
    double *values = (double *)ws.alloc((size_t)k * sizeof(double));
    LsOut out;
    if (a.one_flip()) out.flips = (long long *)ws.alloc((size_t)k * sizeof(long long));
    if (a.tabu) {
        out.moves = (long long *)ws.alloc((size_t)k * sizeof(long long));
        out.best_iter = (long long *)ws.alloc((size_t)k * sizeof(long long));
    }
    if (!V || !bits || !part || !values || (a.one_flip() && !out.flips) || (a.tabu && (!out.moves || !out.best_iter))) return -1;
    std::vector<double> hx((size_t)n * pw);
    for (int64_t t0 = 0; t0 < k; t0 += pw) {
        const int T = (int)std::min<int64_t>(pw, k - t0);
        const size_t len = (size_t)n * T;
        for (size_t e = 0; e < len; ++e) hx[e] = (double)x_host[(size_t)t0 * n + e];
        CUDA_TRY(cudaMemcpyAsync(V, hx.data(), len * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        {
            LaunchScope ls(ctx, "round_eval");
            round_pack_kernel<<<dim3((unsigned)((n + 255) / 256), (unsigned)((T + 63) / 64)), 256, 0, ctx->stream>>>(V, n, (int)n, T,
                                                                                                                  bits);
        }
        CUDA_TRY(cudaGetLastError());
        if (search_pass(ws, (int)n, T, t0, bits, o, part, d, a, V, out)) return -1;
        if (eval_pass(ctx, V, (int)n, T, bits, o, part, t0, values, nullptr, nullptr)) return -1;
        CUDA_TRY(cudaMemcpyAsync(hx.data(), V, len * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_TRY(cudaStreamSynchronize(ctx->stream));
        for (size_t e = 0; e < len; ++e) x_host[(size_t)t0 * n + e] = hx[e] < 0.0 ? -1 : 1;
    }
    static_assert(sizeof(long long) == sizeof(int64_t), "counts are copied as int64");
    CUDA_TRY(cudaMemcpyAsync(values_host, values, (size_t)k * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    if (a.one_flip())
        CUDA_TRY(cudaMemcpyAsync(a.flips_host, out.flips, (size_t)k * sizeof(long long), cudaMemcpyDeviceToHost, ctx->stream));
    if (a.tabu) {
        CUDA_TRY(cudaMemcpyAsync(a.moves_host, out.moves, (size_t)k * sizeof(long long), cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_TRY(cudaMemcpyAsync(a.best_iter_host, out.best_iter, (size_t)k * sizeof(long long), cudaMemcpyDeviceToHost, ctx->stream));
    }
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int k_pm1_local_search(smcp_ctx *ctx, int64_t n, int64_t k, int8_t *x_host, int64_t nc, const int64_t *crow, const int64_t *ccol,
                       const double *cval, int64_t max_flips, double tol, double *values_host, int64_t *flips_host) {
    const LsArgs a{max_flips, tol, nullptr, flips_host, false, 0, 0, nullptr, nullptr, nullptr};
    return pm1_search_impl(ctx, "smcp_pm1_local_search", n, k, x_host, nc, crow, ccol, cval, a, values_host);
}

int k_pm1_tabu_search(smcp_ctx *ctx, int64_t n, int64_t k, int8_t *x_host, int64_t nc, const int64_t *crow, const int64_t *ccol,
                      const double *cval, int64_t iters, int64_t tenure, double *values_host, int64_t *moves_host,
                      int64_t *best_iter_host) {
    const LsArgs a{0, 0.0, nullptr, nullptr, true, iters, tenure, nullptr, moves_host, best_iter_host};
    return pm1_search_impl(ctx, "smcp_pm1_tabu_search", n, k, x_host, nc, crow, ccol, cval, a, values_host);
}
