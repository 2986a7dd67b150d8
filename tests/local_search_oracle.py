"""One-flip local search of +-1 vectors in NumPy: the twin of the device search (``smcp_pm1_local_search``,
``smcp_round_pm1_ls``), bit for bit, and of the device evaluation's fixed summation order (``round_eval_kernel`` /
``round_sum_kernel``), so that flips, signs and values can be compared exactly.

f(x) = sum_ij C_ij x_i x_j, C given by lower-triangular entries (crow, ccol, cval), minimized.  Row i holds the
off-diagonal entries (i, j) from both triangles in increasing j, duplicates summed in input order.  s_i and
a_i = sum_{j != i} |C_ij| are summed sequentially in row order, g_i = x_i s_i.  A step flips the vertex of largest
g_i among those with g_i > tol a_i (lowest index on ties) and adds 2 x_i^new C_ij to s_j over row i."""
import numpy as np

from rounding_oracle import RoundingOracleBackend

EV_WARPS = 8          # warps of round_eval_kernel


def search_rows(n, crow, ccol, cval):
    """CSR (rp, col, val) of the off-diagonal entries of C in both triangles, duplicates merged in input order."""
    crow, ccol = np.asarray(crow, dtype=np.int64), np.asarray(ccol, dtype=np.int64)
    cval = np.asarray(cval, dtype=np.float64)
    q = np.flatnonzero(crow != ccol)
    lo, hi = np.minimum(crow[q], ccol[q]), np.maximum(crow[q], ccol[q])
    o = np.lexsort((q, hi, lo))                         # by pair, input order within a pair
    lo, hi, v = lo[o], hi[o], cval[q][o]
    first = np.ones(len(o), dtype=bool)
    first[1:] = (lo[1:] != lo[:-1]) | (hi[1:] != hi[:-1])
    start = np.flatnonzero(first)
    cnt = np.diff(np.append(start, len(o)))
    pv = v[start].copy()
    for m in range(1, int(cnt.max()) if len(cnt) else 0):   # sequential sum within each pair
        g = np.flatnonzero(cnt > m)
        pv[g] = pv[g] + v[start[g] + m]
    pl, ph = lo[start], hi[start]
    R, Cc, V = np.concatenate([pl, ph]), np.concatenate([ph, pl]), np.concatenate([pv, pv])
    o = np.lexsort((Cc, R))
    rp = np.zeros(n + 1, dtype=np.int64)
    np.add.at(rp, R + 1, 1)
    return np.cumsum(rp), Cc[o], V[o]


def _row_sums(rp, col, term, k, n):
    """out[:, i] = sum over row i, in row order, of term(p) (shape (k, len(p)) for entry positions p)."""
    out = np.zeros((k, n))
    deg = np.diff(rp)
    for m in range(int(deg.max()) if n else 0):
        rows = np.flatnonzero(deg > m)
        out[:, rows] = out[:, rows] + term(rp[rows] + m)
    return out


def local_search(x, crow, ccol, cval, max_flips, tol):
    """Search of the rows of x (k x n, +-1).  Returns (x, flips)."""
    x = np.array(x, dtype=np.int8, ndmin=2)
    k, n = x.shape
    rp, col, val = search_rows(n, crow, ccol, cval)
    thr = tol * _row_sums(rp, col, lambda p: np.abs(val[p])[None, :], 1, n)[0]
    s = _row_sums(rp, col, lambda p: np.where(x[:, col[p]] < 0, -val[p], val[p]), k, n)
    g = np.where(x < 0, -s, s)
    deg = np.diff(rp)
    flips = np.zeros(k, dtype=np.int64)
    active = np.full(k, max_flips > 0)
    while active.any():
        a = np.flatnonzero(active)
        ga = g[a]
        ok = ga > thr
        i = np.where(ok, ga, -np.inf).argmax(axis=1)          # first of equal maxima: lowest index
        has = ok[np.arange(len(a)), i]
        active[a[~has]] = False
        a, i = a[has], i[has]
        if len(a) == 0:
            break
        x[a, i] = -x[a, i]
        g[a, i] = -g[a, i]
        cnt = deg[i]
        tt = np.repeat(a, cnt)
        pp = np.repeat(rp[i] - np.cumsum(cnt) + cnt, cnt) + np.arange(cnt.sum())
        jj = col[pp]
        two = np.repeat(np.where(x[a, i] < 0, -2.0, 2.0), cnt)
        s[tt, jj] = s[tt, jj] + two * val[pp]
        g[tt, jj] = np.where(x[tt, jj] < 0, -s[tt, jj], s[tt, jj])
        flips[a] += 1
        active[a[flips[a] >= max_flips]] = False
    return x, flips


def eval_values(x, crow, ccol, cval):
    """C . x x^T of the rows of x summed in the order of round_eval_kernel and round_sum_kernel: S fixed slices of
    the entries, EV_WARPS warps per slice taking 32-entry tiles in turn, each warp's sum sequential, then the warp
    sums and the slice sums in order."""
    x = np.array(x, dtype=np.int8, ndmin=2)
    crow, ccol = np.asarray(crow, dtype=np.int64), np.asarray(ccol, dtype=np.int64)
    cval = np.asarray(cval, dtype=np.float64)
    k, nc = x.shape[0], len(cval)
    coef = np.where(crow == ccol, cval, 2.0 * cval)
    S = min(256, max(1, (nc + 511) // 512))
    per = max(1, -(-nc // S))
    e0 = np.arange(S) * per
    e1 = np.minimum(nc, e0 + per)
    acc = np.zeros((S, EV_WARPS, k))
    base = e0[:, None] + 32 * np.arange(EV_WARPS)[None, :]
    for m in range(-(-per // (32 * EV_WARPS)) * 32):
        e = base + 32 * EV_WARPS * (m // 32) + m % 32
        ok = e < e1[:, None]
        ec = np.where(ok, e, 0)
        neg = x[:, crow[ec]] != x[:, ccol[ec]]              # (k, S, EV_WARPS)
        term = np.where(ok, np.where(neg, -coef[ec], coef[ec]), 0.0)
        acc = acc + np.moveaxis(term, 0, -1)
    part = np.zeros((S, k))
    for w in range(EV_WARPS):
        part = part + acc[:, w]
    values = np.zeros(k)
    for sl in range(S):
        values = values + part[sl]
    return values


class LocalSearchOracleBackend(RoundingOracleBackend):
    """``RoundingOracleBackend`` with the two search methods of ``DeviceBackend``."""

    def round_pm1_ls(self, Lbuf, crow, ccol, cval, trials, seed, chunk=0, max_flips=None, tol=1e-12):
        V = self.completion_sample(Lbuf, trials, seed)
        x0 = np.where(V.T < 0.0, -1, 1).astype(np.int8)
        mf = self.symb.n if max_flips is None else max_flips
        x, flips = local_search(x0, crow, ccol, cval, mf, tol)
        values0 = eval_values(x0, crow, ccol, cval)
        values = eval_values(x, crow, ccol, cval)
        best = int(np.argmin(values))
        return values0, values, flips, x[best].copy(), best

    def pm1_local_search(self, x, crow, ccol, cval, max_flips=None, tol=1e-12):
        x = np.array(x, dtype=np.int8, ndmin=2)
        mf = x.shape[1] if max_flips is None else max_flips
        xs, flips = local_search(x, crow, ccol, cval, mf, tol)
        return xs, eval_values(xs, crow, ccol, cval), flips
