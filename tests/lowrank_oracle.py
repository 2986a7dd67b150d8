"""Low-rank (mixing-method) solve in NumPy: the twin of the device solve (``smcp_lowrank_solve``, csrc/lowrank.cu), bit
for bit: the greedy colouring, the start, the sweeps with separately rounded products and sums, the warp sums (lane l
sums components l, l + 32, ... in order, then an xor butterfly over 16, 8, 4, 2, 1), the objective's summation order
(per-vertex terms, partial sums of OBJ_VB consecutive vertices, the partials in order) and y."""
import numpy as np

from local_search_oracle import search_rows
from rounding_oracle import RoundingOracleBackend, normals

OBJ_VB = 64           # vertices per block of lowrank_obj_kernel


def colouring(n, rp, col):
    """Greedy colouring in increasing vertex index: vertex i takes the smallest colour none of its lower-index
    neighbours has."""
    colour = np.zeros(n, dtype=np.int64)
    for i in range(n):
        taken = {int(colour[j]) for j in col[rp[i]:rp[i + 1]] if j < i}
        c = 0
        while c in taken:
            c += 1
        colour[i] = c
    return colour


def warp_sum(T):
    """Row sums of T (k x r) in the order of a warp: lane l sums columns l, l + 32, ... in order, then the xor butterfly."""
    k, r = T.shape
    P = np.zeros((k, 32))
    lanes = np.arange(32)
    for q in range(-(-r // 32)):
        m = 32 * q + lanes < r
        P[:, m] = P[:, m] + T[:, 32 * q + lanes[m]]
    for o in (16, 8, 4, 2, 1):
        P = P + P[:, lanes ^ o]
    return P[:, 0].copy()


def start(G, b):
    """The start from the raw normals G (n x r, row i = sample i): each row scaled to norm sqrt(b_i)."""
    V = np.array(G, dtype=np.float64)
    ss = warp_sum(V * V)
    ok = ss > 0.0
    a = np.sqrt(b[ok]) / np.sqrt(ss[ok])
    V[ok] = a[:, None] * V[ok]
    return V


def _w(V, rows, rp, col, val):
    """w_i = sum_{j != i} C_ij v_j for the vertices ``rows``, summed in row order."""
    W = np.zeros((len(rows), V.shape[1]))
    deg = rp[rows + 1] - rp[rows]
    for m in range(int(deg.max()) if len(rows) else 0):
        a = np.flatnonzero(deg > m)
        p = rp[rows[a]] + m
        W[a] = W[a] + val[p][:, None] * V[col[p]]
    return W


def diag_sums(n, crow, ccol, cval):
    """C_ii, duplicates summed in input order."""
    cd = np.zeros(n)
    for r, c, v in zip(crow, ccol, cval):
        if r == c:
            cd[r] += v
    return cd


def objective(V, rp, col, val, cd, b):
    """(f, e): e_i = C_ii b_i + <v_i, w_i> and f summed as lowrank_obj_kernel / lowrank_sum_kernel sum it."""
    n = V.shape[0]
    W = _w(V, np.arange(n), rp, col, val)
    e = cd * b + warp_sum(V * W)
    f = 0.0
    for i0 in range(0, n, OBJ_VB):
        s = 0.0
        for x in e[i0:i0 + OBJ_VB]:
            s = s + x
        f = f + s
    return f, e


def lowrank_solve(n, crow, ccol, cval, b, r, seed, max_sweeps, tol, G=None):
    """The device solve.  G: the raw normals (n x r); None: ``rounding_oracle.normals`` (equal to the device's to
    about 1e-15, not bitwise).  Returns (V, f, y, sweeps, colors, converged)."""
    b = np.asarray(b, dtype=np.float64)
    rp, col, val = search_rows(n, crow, ccol, cval)
    colour = colouring(n, rp, col)
    ncol = int(colour.max()) + 1 if n else 0
    groups = [np.flatnonzero(colour == c) for c in range(ncol)]
    cd = diag_sums(n, crow, ccol, cval)
    V = start(normals(r, n, seed).T if G is None else G, b)
    sb = np.sqrt(b)
    f0, e = objective(V, rp, col, val, cd, b)
    f = [f0]
    converged = False
    for k in range(1, max_sweeps + 1):
        for vs in groups:
            W = _w(V, vs, rp, col, val)
            ss = warp_sum(W * W)
            ok = ss > 0.0
            a = -sb[vs[ok]] / np.sqrt(ss[ok])
            V[vs[ok]] = a[:, None] * W[ok]
        fk, e = objective(V, rp, col, val, cd, b)
        f.append(fk)
        if f[-2] - fk <= tol * max(1.0, abs(fk)):
            converged = True
            break
    return V, np.array(f), e / b, len(f) - 1, ncol, converged


class LowrankOracleBackend(RoundingOracleBackend):
    """``RoundingOracleBackend`` with ``DeviceBackend.lowrank_solve`` restated by the twin."""

    def lowrank_solve(self, crow, ccol, cval, b, rank, seed, max_sweeps, tol):
        V, f, y, sweeps, colors, _ = lowrank_solve(len(b), crow, ccol, cval, b, rank, seed, max_sweeps, tol)
        return V, f, y, sweeps, colors
