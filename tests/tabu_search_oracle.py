"""Tabu search of +-1 vectors in NumPy: the twin of the device search (``smcp_pm1_tabu_search``,
``smcp_round_pm1_tabu``), bit for bit.  Rows, s_i and g_i = x_i s_i are those of the one-flip search
(tests/local_search_oracle.py).

D_0 = 0.  Move u flips the admissible vertex i with the largest g_i (lowest index on ties) and sets
D_{u+1} = D_u - 4.0 * g_i; D_best, the smallest D so far, changes on a strict decrease only.  A vertex flipped by move u
is tabu during moves u+1 .. u+tenure.  A vertex that is not tabu is always admissible; a tabu vertex only when
D_u - 4.0 * g_i < D_best (aspiration).  The search stops after `iters` moves or when no vertex is admissible, and
returns the vector at the earliest move count where D reached D_best."""
import numpy as np

from local_search_oracle import LocalSearchOracleBackend, _row_sums, eval_values, local_search, search_rows


def tabu_search(x, crow, ccol, cval, iters, tenure):
    """Search of the rows of x (k x n, +-1).  Returns (x, moves, best_iter): the returned vectors, the numbers of moves
    made and the move count of each returned vector."""
    x = np.array(x, dtype=np.int8, ndmin=2)
    k, n = x.shape
    rp, col, val = search_rows(n, crow, ccol, cval)
    deg = np.diff(rp)
    s = _row_sums(rp, col, lambda p: np.where(x[:, col[p]] < 0, -val[p], val[p]), k, n)
    g = np.where(x < 0, -s, s)
    last = np.full((k, n), -1 - tenure, dtype=np.int64)   # move of the latest flip: tabu at move u iff last >= u - tenure
    ring = np.zeros((k, max(tenure, 1)), dtype=np.int64)   # ring[:, u % tenure]: the vertex flipped by move u
    gm = g.copy()                                          # g where not tabu at the next move, -inf where tabu
    D, Db = np.zeros(k), np.zeros(k)
    best = x.copy()
    pend = np.ones(k, dtype=bool)                          # the current vector is the best one and `best` lacks it
    best_iter = np.zeros(k, dtype=np.int64)
    moves = np.zeros(k, dtype=np.int64)
    active = np.ones(k, dtype=bool)
    for u in range(iters):
        a = np.flatnonzero(active)
        if len(a) == 0:
            break
        i = gm[a].argmax(axis=1)                           # first of equal maxima: lowest index
        gi = gm[a, i]
        nr = min(u, tenure)
        if nr > 0:                                         # aspiration: the tabu vertices are the last nr flips
            R = ring[a, :nr]
            gR = g[a[:, None], R]
            ok = D[a, None] - 4.0 * gR < Db[a, None]
            sc = np.where(ok, gR, -np.inf)
            m = sc.max(axis=1)
            j = np.where(ok & (sc == m[:, None]), R, n).min(axis=1)
            take = ok.any(axis=1) & ((m > gi) | ((m == gi) & (j < i)))
            i, gi = np.where(take, j, i), np.where(take, m, gi)
        has = gi > -np.inf
        active[a[~has]] = False
        a, i, gi = a[has], i[has], gi[has]
        if len(a) == 0:
            break
        dn = D[a] - 4.0 * gi
        better = dn < Db[a]
        keep = a[pend[a] & ~better]                        # the move leaves a best vector: keep a copy
        best[keep] = x[keep]
        pend[a] = better
        Db[a[better]] = dn[better]
        best_iter[a[better]] = u + 1
        D[a] = dn
        x[a, i] = -x[a, i]
        g[a, i] = -g[a, i]
        cnt = deg[i]
        tt = np.repeat(a, cnt)
        pp = np.repeat(rp[i] - np.cumsum(cnt) + cnt, cnt) + np.arange(cnt.sum())
        jj = col[pp]
        two = np.repeat(np.where(x[a, i] < 0, -2.0, 2.0), cnt)
        s[tt, jj] = s[tt, jj] + two * val[pp]
        g[tt, jj] = np.where(x[tt, jj] < 0, -s[tt, jj], s[tt, jj])
        last[a, i] = u
        rows, cols = [a, tt], [i, jj]
        if tenure > 0:
            if u >= tenure:                                # the flip of move u - tenure leaves the tabu list
                rows.append(a)
                cols.append(ring[a, u % tenure].copy())
            ring[a, u % tenure] = i
        tr, vc = np.concatenate(rows), np.concatenate(cols)
        gm[tr, vc] = np.where(last[tr, vc] >= u + 1 - tenure, -np.inf, g[tr, vc])
        moves[a] += 1
    out = np.where(pend[:, None], x, best)
    return out.astype(np.int8), moves, best_iter


class TabuSearchOracleBackend(LocalSearchOracleBackend):
    """``LocalSearchOracleBackend`` with the two tabu methods of ``DeviceBackend``."""

    def round_pm1_tabu(self, Lbuf, crow, ccol, cval, trials, seed, tabu_iters, tenure, chunk=0, max_flips=0, tol=1e-12):
        V = self.completion_sample(Lbuf, trials, seed)
        x0 = np.where(V.T < 0.0, -1, 1).astype(np.int8)
        mf = self.symb.n if max_flips is None else max_flips
        if mf > 0:
            x1, flips = local_search(x0, crow, ccol, cval, mf, tol)
        else:
            x1, flips = x0, np.zeros(len(x0), dtype=np.int64)
        x, moves, best_iter = tabu_search(x1, crow, ccol, cval, tabu_iters, tenure)
        values = eval_values(x, crow, ccol, cval)
        best = int(np.argmin(values))
        return (eval_values(x0, crow, ccol, cval), eval_values(x1, crow, ccol, cval), values, flips, moves, best_iter,
                x[best].copy(), best)

    def pm1_tabu_search(self, x, crow, ccol, cval, iters, tenure):
        xs, moves, best_iter = tabu_search(x, crow, ccol, cval, iters, tenure)
        return xs, eval_values(xs, crow, ccol, cval), moves, best_iter
