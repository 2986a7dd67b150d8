"""SMCP's chordal interior-point drivers on the B200 backend (host control flow only).

Public surface (drop-in for ``smcp.solvers``, reference ``src/python/solvers.py``):

* ``options``                      – same keys and defaults (``solvers.py:22-44``)
* ``chordalsolver_feas(A, b, ...)`` – feasible-start barrier method (``solvers.py:49-1327``)
* ``chordalsolver_esd(A, b, ...)``  – extended self-dual embedding (``solvers.py:1330-2467``)
* ``conelp(c, G, h, dims)``         – CVXOPT-style cone-LP front end (``solvers.py:2470-2599``)

``kktsolver='chol'`` is the north-star path; ``'qr'`` is provided in its SYRK form (``_KKTqr``, the default)
and, with ``options['qr_method'] = 'householder'``, in the reference's Householder form (``_KKTqrh``).

The numerical work of every iteration — chordal Cholesky / completion / projected inverse,
the barrier Hessian, the dense Schur complement and its Cholesky, step-length probes and
reductions — runs in CUDA behind ``include/smcp_b200.h`` through ``smcp_b200.device``.  The
drivers below reproduce the reference's *decisions* (the order of solves, refinement
rounds, line-search probes, stopping tests and all constants) so that the iteration
sequence is the reference's; they hold no arithmetic of their own beyond scalars and
m-vectors.  Data layout follows CVXOPT: ``A`` is CCS ``n^2 x (m+1)`` with column 0 = vec(C),
column i = vec(A_i), lower-triangular entries at row ``i + n*j``; ``b`` is dense.
"""
from __future__ import annotations

import math
from time import perf_counter, process_time

import numpy as np
import scipy.sparse as sp

from . import misc
from .symbolic import Symbolic, amalgamate, embed, maxcardsearch, min_degree, lower_pattern
from .chordal import (cspmatrix, cholesky, completion, projected_inverse, llt, hessian,
                      hessian_norm, dot, schur_token)

__version__ = "smcp-b200 0.1"

# DEFAULT OPTIONS (solvers.py:22-44)
options = {
    "debug": False, "maxiters": 100, "abstol": 1e-6, "reltol": 1e-6, "feastol": 1e-8,
    "refinement": 2, "cholmod": False, "order": "AMD", "tnzcols": 0.1,
    "show_progress": True, "dimacs": True, "eta": None, "delta": 0.9, "alpha": 1e-1,
    "beta": 0.7, "minstep": 1e-8, "lifting": True, "t0": 1e-1, "equalsteps": True,
    "prediction": True, "step": 0.98,
    # extension (not in the reference): relaxed supernodes, see smcp_b200.symbolic.amalgamate; 0 = the reference's pattern
    "amalgamation": 0.0,
    # extension: how kktsolver='qr' factors Z = [G(A_1) ... G(A_m)]: 'syrk' (H = Z^T Z and its Cholesky factor)
    # or 'householder' (Z = Q R on the device, Newton solves through Q and R like the reference's kkt_qr)
    "qr_method": "syrk",
}

_backend_factory = None
_iteration_hook = None      # optional callable(solver_name, iteration) used by bench.py for timing
_last_problem = None        # the _Problem of the most recent driver call (instrumentation: pattern / flop statistics)


def set_backend_factory(factory):
    """Install the factory ``symb -> backend`` used by the drivers.  ``None`` restores the
    product default (the CUDA backend).  The parity tests use this seam to run the drivers
    on the CPU oracle; nothing in the package itself ever installs a non-CUDA backend."""
    global _backend_factory
    _backend_factory = factory


def _make_backend(symb):
    if _backend_factory is not None:
        return _backend_factory(symb)
    from .device import DeviceBackend      # raises loudly if the CUDA library is missing
    return DeviceBackend(symb)


# --------------------------------------------------------------------------------------
# option validation (solvers.py:112-223, 1399-1464)
# --------------------------------------------------------------------------------------
class _Opt:
    pass


def _check(cond, exc, msg):
    if not cond:
        raise exc(msg)


def _read_options(n, feas):
    o = _Opt()
    g = options
    o.debug = g["debug"]
    _check(isinstance(o.debug, bool), TypeError, "options['debug'] must be a bool")
    o.maxiters = g["maxiters"]
    _check(type(o.maxiters) is int, TypeError, "options['maxiters'] must be a positive integer")
    _check(o.maxiters >= 1, ValueError, "options['maxiters'] must be positive")
    o.abstol, o.reltol, o.feastol = g["abstol"], g["reltol"], g["feastol"]
    for key in ("abstol", "reltol"):
        _check(type(g[key]) in (float, int), TypeError, "options['%s'] must be a scalar" % key)
    _check(o.reltol > 0.0 or o.abstol > 0.0, ValueError,
           "at least one of options['reltol'] and options['abstol'] must be positive")
    _check(type(o.feastol) in (float, int), TypeError, "options['feastol'] must be a positive scalar")
    _check(o.feastol > 0.0, ValueError, "options['feastol'] must be positive")
    o.cholmod = g["cholmod"]
    _check(type(o.cholmod) is bool, TypeError, "options['cholmod'] must be bool")
    _check(not o.cholmod, NotImplementedError, "the CHOLMOD embedding is not available (no SuiteSparse)")
    o.order = g["order"]
    _check(o.order in ("AMD", "METIS"), ValueError, "options['order'] must be 'AMD' or 'METIS'")
    o.show_progress = g["show_progress"]
    _check(type(o.show_progress) is bool, TypeError, "options['show_progress'] must be a bool")
    o.refinement = g["refinement"]
    _check(type(o.refinement) is int, TypeError, "options['refinement'] must be a nonnegative integer")
    _check(o.refinement >= 0, ValueError, "options['refinement'] must be nonnegative ")
    tz = g["tnzcols"]
    _check(type(tz) is float, TypeError, "tnzcols must be a float between 0.0 and 1.0")
    _check(0.0 <= tz <= 1.0, ValueError, "tnzcols must be between 0.0 and 1.0")
    o.tnzcols = int(n * tz)
    o.dimacs = g["dimacs"]
    _check(type(o.dimacs) is bool, TypeError, "dimacs must be a bool")
    o.amalgamation = g.get("amalgamation", 0.0)
    _check(type(o.amalgamation) in (float, int) and 0.0 <= o.amalgamation < 1.0, ValueError,
           "options['amalgamation'] must be a number in [0, 1)")
    o.qr_method = g.get("qr_method", "syrk")
    _check(o.qr_method in ("syrk", "householder"), ValueError,
           "options['qr_method'] must be 'syrk' or 'householder'")
    if feas:
        o.alpha = g["alpha"]
        _check(type(o.alpha) is float and 0.0 < o.alpha < 0.5, TypeError,
               "options['alpha'] must be a float in the interval (0.0,0.5)")
        o.beta = g["beta"]
        _check(type(o.beta) is float and 0.0 < o.beta < 1.0, TypeError,
               "options['beta'] must be a float in the interval (0.0,1.0)")
        o.minstep = g["minstep"]
        _check(type(o.minstep) is float and o.minstep >= 0.0, TypeError,
               "options['minstep'] must be a nonnegative float")
        o.delta = g["delta"]
        _check(type(o.delta) is float and 0.0 < o.delta < 1.0, TypeError,
               "options['delta'] must be a float in the interval (0.0,1.0)")
        o.eta = g["eta"]
        if o.eta is not None:
            _check(type(o.eta) is float and o.eta > 0.0, TypeError, "options['eta'] must be a positive float")
            o.etatol = 0.10 * o.eta
        o.t0 = g["t0"]
        _check(type(o.t0) is float, TypeError, "options['t0'] must be a positive float")
        _check(o.t0 > 0.0, ValueError, "options['t0'] must be a positive float")
        for key in ("lifting", "equalsteps", "prediction"):
            _check(type(g[key]) is bool, TypeError, "options['%s'] must be True or False" % key)
        o.lifting, o.equalsteps, o.prediction = g["lifting"], g["equalsteps"], g["prediction"]
        o.step = g["step"]
        _check(type(o.step) is float, TypeError, "options['step'] must be a float")
        _check(0 < o.step <= 1, ValueError, "options['step'] must be between 0 and 1.")
    return o


# --------------------------------------------------------------------------------------
# setup shared by both drivers (solvers.py:234-367 == 1475-1608)
# --------------------------------------------------------------------------------------
class _Problem:
    """Ordering, chordal embedding, vector-space layout and the operators A / A^adj."""

    def __init__(self, A, b, opt, kktsolver, p):
        if kktsolver not in ("chol", "qr"):
            raise ValueError("Unknown 'kktsolver'.")
        self.kktsolver = kktsolver
        self.qr_method = opt.qr_method
        A = misc.as_csc(A)
        self.m = m = A.shape[1] - 1
        self.n = n = int(math.sqrt(A.shape[0]))
        b = np.array(b, dtype=np.float64).ravel()
        _check(len(b) == m, ValueError, "b must have m entries")

        # aggregate sparsity pattern (lower triangle of the union of all columns of A)
        Ia, Ja = misc.ind2sub(n, np.unique(A.indices))
        keep = Ia >= Ja
        va_colptr, va_rowind = lower_pattern(n, Ia[keep], Ja[keep])
        self.nnz_Va = int(va_colptr[-1])

        # constraint permutation: "dense" constraints first, "sparse" ones last; each group by
        # decreasing nnz, ties by decreasing index (solvers.py:246-268)
        if kktsolver == "chol":
            Nz = misc.nzcolumns(A)
            pm, Ns = misc.matperm(Nz, opt.tnzcols)
            nnz_col = np.diff(A.indptr)[1:]
            for lo, hi in ((0, m - Ns), (m - Ns, m)):
                if hi > lo:
                    grp = sorted(((int(nnz_col[j]), int(j)) for j in pm[lo:hi]), reverse=True)
                    pm[lo:hi] = [j for _, j in grp]
        else:
            # kktsolver='qr': no sparse-constraint technique, constraints keep their order (solvers.py:269-271)
            pm, Ns = np.arange(m, dtype=np.int64), 0
        self.pm, self.Ns = pm, Ns
        self.b = b = b[pm].copy()
        if m:
            self.bmax, self.ii = max(zip(np.abs(b).tolist(), range(m)))
        else:
            self.bmax, self.ii = 0.0, 0

        # ordering and embedding (solvers.py:278-315)
        pmcs = maxcardsearch(n, va_colptr, va_rowind)
        fc, fr, _ = embed(n, va_colptr, va_rowind, pmcs)
        if int(fc[-1]) == self.nnz_Va:
            self.chordal = True
            p = pmcs
        else:
            self.chordal = False
            if p is None:
                p = min_degree(n, va_colptr, va_rowind)
            p = np.asarray(p, dtype=np.int64).ravel()
            _check(len(p) == n and np.array_equal(np.sort(p), np.arange(n)), ValueError,
                   "p must be a permutation of 0..n-1")
            fc, fr, _ = embed(n, va_colptr, va_rowind, p)
        if opt.amalgamation > 0.0:
            # opt-in: merge supernodes into their parents (explicit zeros in exchange for larger dense blocks);
            # the embedding stays a filled pattern in the same elimination ordering
            fc, fr = amalgamate(n, fc, fr, float(opt.amalgamation))
        self.p = p
        self.ip = np.empty(n, dtype=np.int64)
        self.ip[p] = np.arange(n, dtype=np.int64)
        self.symb = symb = Symbolic(n, fc, fr)
        _check(m <= symb.nvp, ValueError, "more constraints than nonzeros")

        # vector space: q-th non-zero (Ip[q], Jp[q]) of Vp  <->  row LI[q] of A (solvers.py:318-346)
        oi, oj = p[symb.Ip], p[symb.Jp]
        LI = np.maximum(oi, oj) + n * np.minimum(oi, oj)
        order = np.argsort(LI, kind="stable")
        LIs = LI[order]
        coo = A.tocoo()
        pos = np.searchsorted(LIs, coo.row)
        pos[pos >= len(LIs)] = 0
        hit = LIs[pos] == coo.row
        q = order[pos[hit]]
        col = coo.col[hit]
        val = coo.data[hit]
        c = np.zeros(symb.nvp)
        is0 = col == 0
        c[q[is0]] = val[is0]
        self.c = c
        inv_pm = np.empty(m, dtype=np.int64)
        inv_pm[pm] = np.arange(m, dtype=np.int64)
        self.inv_pm = inv_pm
        self.Av = misc.as_csc(sp.csc_matrix((val[~is0], (q[~is0], inv_pm[col[~is0] - 1])),
                                            shape=(symb.nvp, m)))

        self.ops = ops = _make_backend(symb)
        ops.set_operator(self.Av, Ns)
        self.C = cspmatrix.from_vec(ops, c)
        global _last_problem
        _last_problem = self

    # operators (solvers.py:369-384)
    def Amap(self, X, i=None):
        if i is None:
            return self.ops.Amap(X.buf)
        return self.ops.Amap_col(X.buf, int(i))

    def Aadj(self, y):
        return cspmatrix(self.ops, self.ops.Aadj(np.ascontiguousarray(y, dtype=np.float64)))

    def zeros(self):
        return cspmatrix(self.ops)

    def identity(self, alpha=1.0):
        return cspmatrix.identity(self.ops, alpha)

    def from_original(self, Xs):
        """cspmatrix(symb) + tril(perm(symmetrize(tril(X)), p))  (solvers.py:693, 1629)."""
        Xs = sp.csc_matrix(Xs)
        lo = sp.tril(Xs, format="csc")
        full = (lo + sp.tril(lo, -1).T).tocsr()
        symb = self.symb
        v = np.asarray(full[self.p[symb.Ip], self.p[symb.Jp]]).ravel()
        return cspmatrix.from_vec(self.ops, v)

    def to_original(self, X):
        """perm(symmetrize(X.spmatrix(reordered=False, symmetric=False)), ip)."""
        symb = self.symb
        v = X.to_vec()
        r, c = self.p[symb.Ip], self.p[symb.Jp]
        off = r != c
        rows = np.concatenate([r, c[off]])
        cols = np.concatenate([c, r[off]])
        vals = np.concatenate([v, v[off]])
        return sp.csc_matrix((vals, (rows, cols)), shape=(self.n, self.n))


class _KKT:
    """``kkt_chol`` (solvers.py:477-541 == 1906-1969): assemble the Schur complement
    H_ij = A_i . Hess(A_j) on the device, factor it, and solve
        [ -kk*Hess^{-1}  A^adj ] [x]   [bx]
        [  A             0     ] [y] = [by]
    by  y = H^{-1}(kk*by + A(Hess(bx))),  x = (1/kk) Hess(A^adj(y) - bx)."""

    def __init__(self, prob, L, Y, scaling):
        self.prob, self.L, self.Y, self.scaling = prob, L, Y, scaling
        prob.ops.schur_factor(schur_token(L, Y))     # raises ArithmeticError if H is not PD

    def solve(self, bx, by, t):
        kk = 1.0 / t if self.scaling == "primal" else t
        prob = self.prob
        r1 = bx.copy()
        hessian(self.L, self.Y, r1, inv=False, adj=None)
        y = prob.ops.schur_solve(kk * by + prob.Amap(r1))
        x = prob.Aadj(y) - bx
        hessian(self.L, self.Y, [x], inv=False, adj=None)
        x.scale(1.0 / kk)
        return x, y


class _KKTqr:
    """``kkt_qr`` (solvers.py:413-475 == 1843-1904): with the half factor G of the Hessian
    (``hessian = G^adj o G``) and Z = [G(A_1) ... G(A_m)], the Schur complement is H = Z^T Z in the trace
    inner product.  The reference takes the QR factorisation of Z (``lapack.geqrf``); here H = Z^T Z is
    formed by one triangular DMMA product (SYRK form, SURVEY 8f rank 3: half the Hessian work of
    ``kkt_chol``, H positive semidefinite by construction) and factored by the same Cholesky, i.e. R of
    Z = Q R without Q (Q is only ever applied as Z R^-1):
        y = H^{-1}(kk*by + Z^T G(bx)),   x = (1/kk) G^adj(Z y - G(bx))."""

    def __init__(self, prob, L, Y, scaling):
        self.prob, self.L, self.Y, self.scaling = prob, L, Y, scaling
        prob.ops.schur_factor_qr(schur_token(L, Y))      # raises ArithmeticError if Z is rank deficient

    def solve(self, bx, by, t):
        kk = 1.0 / t if self.scaling == "primal" else t
        ops = self.prob.ops
        r1 = bx.copy()
        hessian(self.L, self.Y, [r1], inv=False, adj=False)
        y = ops.schur_solve(kk * by + ops.z_tmul(r1.buf))
        x = cspmatrix(ops, ops.z_mul(np.ascontiguousarray(y, dtype=np.float64)))
        x -= r1
        hessian(self.L, self.Y, [x], inv=False, adj=True)
        x.scale(1.0 / kk)
        return x, y


class _KKTqrh:
    """``kkt_qr`` as the reference computes it (``lapack.geqrf / ormqr / trtrs``), ``options['qr_method'] =
    'householder'``: with the weights w of the trace inner product, Zw = diag(sqrt(w)) Z = Q1 R by a blocked
    Householder QR on the device, and the solve goes through Q1 and R:
        gw = sqrt(w) G(bx),  v = R^-T (kk*by) + Q1^T gw,  y = R^-1 v,  x = (1/kk) G^adj((Q1 v - gw) / sqrt(w)).
    This equals ``_KKTqr.solve`` in exact arithmetic (Z y = Q1 R y = Q1 v); it never forms Z^T Z, whose
    condition number is that of Z squared."""

    def __init__(self, prob, L, Y, scaling):
        self.prob, self.L, self.Y, self.scaling = prob, L, Y, scaling
        prob.ops.schur_factor_householder(schur_token(L, Y))      # raises ArithmeticError if Z is rank deficient

    def solve(self, bx, by, t):
        kk = 1.0 / t if self.scaling == "primal" else t
        ops = self.prob.ops
        r1 = bx.copy()
        hessian(self.L, self.Y, [r1], inv=False, adj=False)
        y, xbuf = ops.qr_solve(r1.buf, kk * np.asarray(by, dtype=np.float64))
        x = cspmatrix(ops, xbuf)
        hessian(self.L, self.Y, [x], inv=False, adj=True)
        x.scale(1.0 / kk)
        return x, y


def _make_kkt(prob, L, Y, scaling):
    if prob.kktsolver == "qr":
        return (_KKTqrh if prob.qr_method == "householder" else _KKTqr)(prob, L, Y, scaling)
    return _KKT(prob, L, Y, scaling)


def _nrm2(v):
    return float(np.sqrt(np.dot(v, v)))


def _frob(X):
    return math.sqrt(dot(X, X))


_tree_cache = {}


def _bisection_tree(minstep, depth=8):
    """Step lengths of every node of the bisection on [minstep, 1] in heap order (node 1 = first
    midpoint; child 2i after a failed probe, 2i+1 after a successful one), computed with the
    same floating-point expression ``(gmin + gmax) / 2`` as the sequential loop."""
    key = (float(minstep), depth)
    if key not in _tree_cache:
        gam = np.zeros(2 ** depth)
        lo = np.zeros(2 ** depth)
        hi = np.zeros(2 ** depth)
        lo[1], hi[1] = minstep, 1.0
        for i in range(1, 2 ** depth):
            gam[i] = (lo[i] + hi[i]) / 2.0
            if 2 * i + 1 < 2 ** depth:
                lo[2 * i], hi[2 * i] = lo[i], gam[i]              # failure: gmax = gam
                lo[2 * i + 1], hi[2 * i + 1] = gam[i], hi[i]      # success: gmin = gam
        _tree_cache[key] = gam
    return _tree_cache[key]


def _in_cone(X, test):
    """True iff ``test`` (cholesky or completion) succeeds on a copy of X; returns the
    factor as well."""
    Lt = X.copy()
    try:
        test(Lt)
    except ArithmeticError:
        return None
    return Lt


# --------------------------------------------------------------------------------------
# feasible-start barrier method
# --------------------------------------------------------------------------------------
def chordalsolver_feas(A, b, primalstart=None, dualstart=None, scaling="primal",
                       kktsolver="chol", p=None):
    """Chordal SDP solver (feasible start):

        minimize   c'*x        maximize   b'*y
        subject to A*x = b     subject to A'*y + s = c
                   x in C                 s in K

    with C the cone of matrices with pattern V that have a PSD completion and K the PSD
    matrices with pattern V.  Same arguments and result dictionary as the reference
    (``solvers.py:49-1327``).
    """
    T0wall, T0 = perf_counter(), process_time()
    A = misc.as_csc(A)
    n = int(math.sqrt(A.shape[0]))
    opt = _read_options(n, feas=True)
    _check(scaling in ("primal", "dual"), ValueError, "scaling must be 'primal' or 'dual'")
    prob = _Problem(A, b, opt, kktsolver, p)
    m, b, C = prob.m, prob.b, prob.C
    Amap, Aadj = prob.Amap, prob.Aadj
    ALPHA, BETA, MINSTEP, DELTA = opt.alpha, opt.beta, opt.minstep, opt.delta
    REFINEMENT = opt.refinement
    say = print if opt.show_progress else (lambda *a, **k: None)

    st = _Opt()                 # mutable solver state shared with the helpers below
    st.t = opt.t0
    st.scaling = scaling
    status = "unknown"

    def Omega(Lsh, Ls, gap):
        # Omega(X,S) = phi_p(X) + phi_d(S) + n log(<X,S>/n)      (solvers.py:386-395)
        return 2.0 * Lsh.sumlogdiag() - 2.0 * Ls.sumlogdiag() + n * math.log(gap / n)

    resy0 = max(1, _nrm2(b))
    resx0 = max(1, _frob(C))

    def kkt_res(L, Y, x, y, bx, by):
        # residual of the KKT system (solvers.py:401-411)
        r = x.copy()
        hessian(L, Y, r, inv=True, adj=None)
        r.scale(-1.0 / st.t if st.scaling == "primal" else -st.t)
        r += Aadj(y) - bx
        return r, Amap(x) - by

    def solve_refined(f, L, Y, bx, by, tt=None):
        """One KKT solve followed by REFINEMENT rounds of iterative refinement
        (solvers.py:907-913, 968-974, 1037-1043, 1109-1115)."""
        t_of = (lambda: st.t) if tt is None else (lambda: tt)
        x, y = f.solve(bx, by, t_of())
        for _ in range(REFINEMENT):
            r1, r2 = kkt_res(L, Y, x, y, bx, by)
            dx_, dy_ = f.solve(r1, r2, t_of())
            x -= dx_
            y = y - dy_
        return x, y

    def bisect(X, dX, test):
        # 8 halvings on [MINSTEP, 1] (solvers.py:615-647).  The verdict of a probe depends only on
        # its step length, so on a backend with batched probes the whole decision tree of the
        # bisection (255 candidate steps) is evaluated as ONE device batch and the reference's
        # decisions are replayed on the verdicts; otherwise the probes run one after the other.
        ops = prob.ops
        if getattr(ops, "batched_probes", False):
            tree = _bisection_tree(MINSTEP)
            ok, _ = ops.probe("completion" if test is completion else "cholesky", X.buf, dX.buf, tree[1:])
            gmin, gmax = MINSTEP, 1.0
            g_ok = gmin
            node = 1
            for _ in range(8):
                gam = tree[node]
                if ok[node - 1]:
                    gmin = gam
                    g_ok = gam
                    node = 2 * node + 1
                else:
                    gmax = gam
                    g_ok = gmin
                    node = 2 * node
            return g_ok
        gmin, gmax = MINSTEP, 1.0
        g_ok = gmin
        for _ in range(8):
            gam = (gmin + gmax) / 2.0
            if _in_cone(X.copy() + gam * dX, test) is not None:
                gmin = gam
                g_ok = gam
            else:
                gmax = gam
                g_ok = gmin
        return g_ok

    def linesearch(X, dx, S, ds, a=1.0):
        return a * bisect(X, dx, completion), a * bisect(S, ds, cholesky)

    def linesearch_Omega(X, dx, S, ds, eta):
        # bisection that keeps Omega within eta +- ETATOL (solvers.py:662-689)
        gmin, gmax = MINSTEP, 1.0
        g_ok = None
        for _ in range(8):
            gam = (gmin + gmax) / 2.0
            Xt = X.copy() + gam * dx
            St = S.copy() + gam * ds
            Lt = _in_cone(Xt, completion)
            Lst = _in_cone(St, cholesky) if Lt is not None else None
            if Lt is None or Lst is None:
                gmax = gam
                g_ok = None
                continue
            g_ok = gam
            Ot = Omega(Lt, Lst, dot(St, Xt))
            if Ot - eta > opt.etatol:
                gmax = gam
            elif Ot - eta < -opt.etatol:
                gmin = gam
            else:
                break
        return g_ok if g_ok else gmin

    def damped_primal(X, dx, L, ntdecr):
        # backtracking on the primal barrier (solvers.py:924-942, 1134-1153)
        gam = 1.0
        logdetL = L.sumlogdiag()
        tdcdx = st.t * dot(C, dx)
        Xt = X
        while gam > MINSTEP:
            Xt = X.copy() + gam * dx
            val = tdcdx + gam * ALPHA * ntdecr ** 2
            Lt = _in_cone(Xt, completion)
            if Lt is not None and gam * val < 2 * (logdetL - Lt.sumlogdiag()):
                break
            gam *= BETA
        return Xt, gam

    def damped_dual(y, dy, L, ntdecr):
        # backtracking on the dual barrier (solvers.py:985-1005, 1175-1196)
        gam = 1.0
        logdetL = L.sumlogdiag()
        ddyb = -st.t * float(np.dot(dy, b))
        yt, St = y, None
        while gam > MINSTEP:
            yt = y + gam * dy
            St = Aadj(-yt) + C
            val = ddyb + gam * ALPHA * ntdecr ** 2
            Lt = _in_cone(St, cholesky)
            if Lt is not None and gam * val < 2 * (Lt.sumlogdiag() - logdetL):
                break
            gam *= BETA
        return yt, St, gam

    # ---- starting point (solvers.py:691-814) -------------------------------------
    X = y = S = None
    if primalstart is not None:
        X = prob.from_original(primalstart["x"])
        if _nrm2(b - Amap(X)) / resy0 > 1e-8:
            raise ValueError("infeasible primal starting point")
        if _in_cone(X, completion) is None:
            raise ValueError("infeasible primal starting point")
    if dualstart is not None:
        if "y" in dualstart and "s" in dualstart:
            y = np.array(dualstart["y"], dtype=np.float64).ravel()[prob.pm]
            S = prob.from_original(dualstart["s"])
            if _frob(Aadj(-y) + C - S) / resx0 > 1e-8:
                raise ValueError("infeasible dual starting point")
        elif "y" in dualstart:
            y = np.array(dualstart["y"], dtype=np.float64).ravel()[prob.pm]
            S = Aadj(-y) + C
        if S is None or _in_cone(S, cholesky) is None:
            raise ValueError("infeasible dual starting point")

    if primalstart is None and dualstart is None:
        # heuristics at the identity (solvers.py:722-802)
        Xt = prob.identity()
        Lt = Xt.copy()
        completion(Lt)
        fI = _make_kkt(prob, Lt, Xt, st.scaling)
        X0, _nu = fI.solve(prob.zeros(), b, st.t)
        if _in_cone(X0, completion) is not None:
            X = X0
            print("Primal least-norm solution is feasible.")
        else:
            dvec = prob.symb.diag_vec
            trA = np.asarray(prob.Av[dvec, :].sum(axis=0)).ravel()
            Xb, _nu = fI.solve(prob.zeros(), trA, st.t)
            Xb -= Xt
            for sign in (1.0, -1.0):
                if sign < 0:
                    Xb.scale(-1.0)
                if _in_cone(Xb, completion) is None:
                    continue
                gam = 2.0
                while True:
                    X = X0.copy() + gam * Xb
                    if _in_cone(X, cholesky) is not None:
                        break
                    gam *= 2
                print("Feasible primal solution found.")
                break
        _nu, y = fI.solve(C, np.zeros(m), st.t)
        S = Aadj(-y) + C
        if _in_cone(S, cholesky) is not None:
            print("Dual least-squares solution is feasible.")
        else:
            _nu, y = fI.solve(prob.identity(-1.0), np.zeros(m), st.t)
            if _in_cone(Aadj(-y), cholesky) is not None:
                while True:
                    S = Aadj(-y) + C
                    if _in_cone(S, cholesky) is not None:
                        break
                    y = y * 1.4
                print("Feasible dual solution found.")
            else:
                S = y = None
        del fI, Lt, Xt

    if y is None and X is None:
        raise ValueError("could not find a feasible starting point (solve Phase I problem instead)")
    elif X is None and st.scaling == "primal":
        print("Switching to dual scaling.")
        st.scaling = "dual"
    elif S is None and st.scaling == "dual":
        print("Switching to primal scaling.")
        st.scaling = "primal"
    primal = st.scaling == "primal"

    if opt.show_progress:
        tag = "Chol." + (",lifting" if opt.lifting else "") + (",prediction" if opt.prediction else "")
        print("%-20s Barrier method, %s scaling (%s)" % (__version__, st.scaling, tag))
        print("-" * 79)
        print("SDP var. size:       %i " % n)
        print("Constraints:         %i (%i|%i)" % (m, m - prob.Ns, prob.Ns))
        print("Aggregate sparsity:  %-14s NNZ(tril(V)) = %7i"
              % ("Chordal" if prob.chordal else "Nonchordal", prob.nnz_Va))
        if not prob.chordal:
            print("Embedding:           %-14s       NNZ(L) = %7i" % ("min. degree", prob.symb.nvp))
        print("-" * 79)
        print(" it  pcost       dcost      gap     pres    dres    ntdecr  Omega   pstep dstep")

    gap = n / st.t
    pres = dres = pcost = dcost = relgap = None
    ntdecr = Ot = pstep = dstep = gam = None
    stype = None
    CENTER = True
    dxL = dyL = None
    Shat = None
    trace = []
    it = 0

    for it in range(1, opt.maxiters + 2):
        # residuals and convergence statistics (solvers.py:833-869)
        if primal:
            pres = _nrm2(b - Amap(X)) / resy0
            pcost = dot(C, X)
        else:
            dres = _frob(Aadj(-y) + C - S) / resx0
            dcost = float(np.dot(b, y))
        if pcost is not None and pcost < 0.0:
            relgap = gap / -pcost
        elif dcost is not None and dcost > 0.0:
            relgap = gap / dcost
        else:
            relgap = None

        if it == opt.maxiters + 1:
            say("Terminated (maximum number of iterations reached).")
            status = "unknown"
            break
        elif dres is not None and pres is not None:
            feasible = pres < opt.feastol and dres < opt.feastol
            if feasible and (gap < opt.abstol or (relgap is not None and relgap < opt.reltol)):
                say("Optimal solution found.")
                status = "optimal"
                break

        # scaling point (solvers.py:871-891)
        if primal:
            L = _in_cone(X, completion)
            if L is None:
                say("*** Completion failed.")
                status = "unknown"
                break
            Y = X.copy()
        else:
            L = _in_cone(S, cholesky)
            if L is None:
                say("*** Factorization of S failed.")
                status = "unknown"
                break
            Y = L.copy()
            projected_inverse(Y)

        try:
            f = _make_kkt(prob, L, Y, st.scaling)
        except ArithmeticError:
            # reference: "*** Factorization failed" and a dict that makes the next call fail
            print("*** Factorization failed")
            status = "unknown"
            break

        if CENTER:
            if primal:
                # centering (solvers.py:899-959)
                Shat = L.copy()
                llt(Shat)
                bx = C.copy() - (1.0 / st.t) * Shat
                by = b - Amap(X)
                dx, lam = solve_refined(f, L, Y, bx, by)
                ntdecr = hessian_norm(L, Y, dx, inv=True)
                if ntdecr > DELTA:
                    if ntdecr >= 1.0:
                        X, gam = damped_primal(X, dx, L, ntdecr)
                    else:
                        X += dx
                        gam = 1.0
                    stype = "c"
                else:
                    if opt.lifting:
                        X -= dx
                        dxL = dx
                    else:
                        X += dx
                    y = lam
                    S = Aadj(-y) + C
                    CENTER = False
            else:
                # dual centering (solvers.py:961-1024)
                bx = S.copy()
                bx.scale(-1.0)
                by = b
                nu, dy = solve_refined(f, L, Y, bx, by)
                ntdecr = hessian_norm(L, Y, Aadj(dy), inv=False)
                if ntdecr > DELTA:
                    if ntdecr >= 1.0:
                        y, S, gam = damped_dual(y, dy, L, ntdecr)
                    else:
                        y = y + dy
                        S = Aadj(-y) + C
                        gam = 1.0
                    stype = "c"
                else:
                    if opt.lifting:
                        y = y - dy
                        S = Aadj(-y) + C
                        dyL = dy
                    else:
                        y = y + dy
                        S = Aadj(-y) + C
                    X = nu
                    CENTER = False

        if not CENTER:
            # approximate tangent direction (solvers.py:1026-1044)
            bx = S.copy()
            by = b - Amap(X)
            dx, dy = solve_refined(f, L, Y, bx, by)
            ds = Aadj(-dy)

            if opt.eta is not None:
                gam = linesearch_Omega(X, dx, S, ds, opt.eta)
                X += gam * dx
                y = y + gam * dy
                S = Aadj(-y) + C
                pstep = dstep = gam
            else:
                pstep, dstep = linesearch(X, dx, S, ds, opt.step)
                if opt.equalsteps:
                    pstep = min(pstep, dstep)
                    dstep = pstep
                Xt = X.copy() + pstep * dx
                yt = y + dstep * dy
                St = Aadj(-yt) + C

                if not opt.prediction:
                    X, S, y = Xt, St, yt
                else:
                    gapt = dot(Xt, St)
                    if opt.lifting:
                        if primal:
                            X += dxL
                        else:
                            y = y + dyL
                            S = Aadj(-y) + C
                    st.t = n / gapt

                    if primal:
                        bx = S.copy() - (1.0 / st.t) * Shat
                        by = b - Amap(X)
                    else:
                        bx = X.copy()
                        hessian(L, Y, bx, inv=True, adj=None)
                        bx.scale(st.t)
                        bx -= S
                        by = b - Amap(X)
                    dx, dy = solve_refined(f, L, Y, bx, by, tt=st.t)
                    ds = Aadj(-dy)

                    if primal:
                        ntdecr = hessian_norm(L, Y, dx, inv=True)
                    else:
                        ntdecr = hessian_norm(L, Y, Aadj(dy), inv=False)

                    if primal:
                        if ntdecr >= 1.0:
                            X, pstep = damped_primal(X, dx, L, ntdecr)
                        else:
                            pstep = 1.0
                            X += dx
                        gam = 1.0
                        while True:
                            yt = y + gam * dy
                            St = Aadj(-yt) + C
                            if _in_cone(St, cholesky) is not None:
                                break
                            gam *= BETA
                        dstep = gam
                        y, S = yt, St
                    else:
                        if ntdecr >= 1.0:
                            y, S, dstep = damped_dual(y, dy, L, ntdecr)
                        else:
                            y = y + dy
                            S = Aadj(-y) + C
                            dstep = 1.0
                        gam = 1.0
                        while True:
                            Xt = X.copy() + gam * dx
                            if _in_cone(Xt, completion) is not None:
                                break
                            gam *= BETA
                        pstep = gam
                        X = Xt

            # new gap and Omega (solvers.py:1214-1239)
            Lt = X.copy()
            completion(Lt)
            Lst = S.copy()
            cholesky(Lst)
            gapt = dot(X, S)
            Ot = Omega(Lt, Lst, gapt)
            gap = min(n / st.t, gapt)
            st.t = n / gap
            stype = "a"
            pres = _nrm2(Amap(X) - b) / resy0
            dres = _frob(Aadj(y) + S - C) / resx0
            pcost = dot(C, X)
            dcost = float(np.dot(b, y))
            CENTER = True

        trace.append(dict(iter=it, stype=stype, pcost=pcost, dcost=dcost, gap=gap, pres=pres,
                          dres=dres, ntdecr=ntdecr, pstep=pstep, dstep=dstep, gam=gam, t=st.t))
        if _iteration_hook is not None:
            _iteration_hook("feas", it)
        if opt.show_progress:
            if stype == "c":
                print("%3i %-11s %-11s %.1e %-7s %-7s %.1e %7s %4.2f" % (
                    it, "% .4e" % pcost if pcost is not None else " ",
                    "% .4e" % dcost if dcost is not None else " ", gap,
                    "%.1e" % pres if pres is not None else " ",
                    "%.1e" % dres if dres is not None else " ", ntdecr, " ", gam))
            else:
                print("%3i % .4e % .4e %.1e %.1e %.1e %.1e %.1e %4.2f  %4.2f"
                      % (it, pcost, dcost, gap, pres, dres, ntdecr, Ot, pstep, dstep))

    Tcpu = process_time() - T0
    Twall = perf_counter() - T0wall

    dimacs = None
    if opt.dimacs and X is not None and y is not None and S is not None:
        cmax = float(np.max(np.abs(prob.c))) if len(prob.c) else 0.0
        dimacs = [_nrm2(Amap(X) - b) / (1.0 + float(np.max(np.abs(b)))), 0.0,
                  _frob(Aadj(y) + S - C) / (1.0 + cmax), 0.0,
                  (pcost - dcost) / (1 + abs(pcost) + abs(dcost)),
                  gap / (1 + abs(pcost) + abs(dcost))]

    Xo = prob.to_original(X) if X is not None else None
    yo = y[prob.inv_pm] if y is not None else None
    So = prob.to_original(S) if S is not None else None

    if opt.show_progress:
        _print_exit(status, pcost, dcost, gap, relgap, pres, dres, it, Tcpu, Twall, dimacs)

    return {"status": status, "x": Xo, "y": yo, "s": So, "primal objective": pcost,
            "dual objective": dcost, "gap": gap, "relative gap": relgap,
            "primal infeasibility": pres, "dual infeasibility": dres, "iterations": it,
            "cputime": Tcpu, "time": Twall, "trace": trace, "dimacs": dimacs}


def _print_exit(status, pcost, dcost, gap, relgap, pres, dres, it, Tcpu, Twall, dimacs):
    if status in ("optimal", "unknown"):
        if pcost is not None:
            print("   Primal objective:                % .8e" % pcost)
        if dcost is not None:
            print("   Dual objective:                  % .8e" % dcost)
    for label, v in (("Gap:                 ", gap), ("Relative gap:        ", relgap),
                     ("Primal infeasibility:", pres), ("Dual infeasibility:  ", dres)):
        if v is not None:
            print("   %s            % .8e" % (label, v))
    if it:
        print("   Iterations:                       %i" % it)
        print("   CPU time:                         %.2f" % Tcpu)
        print("   CPU time per iteration:           %.2f" % (Tcpu / it))
        print("   Real time:                        %.2f" % Twall)
        print("   Real time per iteration:          %.2f\n" % (Twall / it))
    if dimacs is not None:
        print("   DIMACS:  %.2e %.2e %.2e %.2e %.2e %.2e\n" % tuple(dimacs))


# --------------------------------------------------------------------------------------
# extended self-dual embedding
# --------------------------------------------------------------------------------------
def chordalsolver_esd(A, b, primalstart=None, dualstart=None, scaling="primal",
                      kktsolver="chol", p=None):
    """Chordal SDP solver, extended self-dual embedding with a predictor/corrector step
    (``solvers.py:1330-2467``).  Same arguments and result dictionary as the reference."""
    BETA, EXPON, STEP, MINSTEP = 0.7, 3.0, 0.99, 1e-12        # solvers.py:1384-1387
    T0wall, T0 = perf_counter(), process_time()
    A = misc.as_csc(A)
    n = int(math.sqrt(A.shape[0]))
    opt = _read_options(n, feas=False)
    _check(scaling in ("primal", "dual"), ValueError, "scaling must be 'primal' or 'dual'")
    prob = _Problem(A, b, opt, kktsolver, p)
    m, b, C = prob.m, prob.b, prob.C
    Amap, Aadj = prob.Amap, prob.Aadj
    REFINEMENT = opt.refinement
    primal = scaling == "primal"
    bmax, ii = prob.bmax, prob.ii
    say = print if opt.show_progress else (lambda *a, **k: None)
    status = "unknown"

    # starting point (solvers.py:1627-1637)
    X = prob.from_original(primalstart["x"]) if primalstart is not None else prob.identity()
    if dualstart is not None:
        y = np.array(dualstart["y"], dtype=np.float64).ravel()[prob.pm]
        S = prob.from_original(dualstart["s"])
    else:
        S = prob.identity()
        y = np.zeros(m)

    st = _Opt()
    st.tau = st.kappa = 1.0
    gap = dot(X, S) / st.tau ** 2
    st.t = (n + 1.0) / (gap * st.tau ** 2 + st.tau * st.kappa)
    resy0 = max(1, _nrm2(b))
    resx0 = max(1, _frob(C))

    def bres(sigma, dz=None):
        # right-hand side of the Newton system (solvers.py:1712-1770)
        t, tau, kappa = st.t, st.tau, st.kappa
        rby = (1 - sigma) * st.ry
        rbx = st.rx.copy()
        rbx.scale(1 - sigma)
        rbt = (1 - sigma) * st.rt
        if primal:
            rbs = st.L.copy()
            llt(rbs)
            rbs.scale(sigma / t)
            rbs -= S
            rbk = -kappa + sigma / (t * tau)
        else:
            rbs = st.Y.copy()
            rbs.scale(sigma / t)
            rbs -= X
            rbk = -tau + sigma / (t * kappa)
        if dz:
            ddy_, ddX_, ddtau_, ddS_, ddkappa_ = dz
            rby = rby + (b * ddtau_ - Amap(ddX_))
            if primal:
                rbx += Aadj(ddy_) + ddS_ - ddtau_ * C
            else:
                rbx += -ddtau_ * C + ddS_ + Aadj(ddy_)
            rbt += dot(C, ddX_) - float(np.dot(b, ddy_)) + ddkappa_
            if primal:
                rbs -= ddS_
                u = ddX_.copy()
                hessian(st.L, st.Y, [u], inv=True, adj=None)
                rbs -= (1.0 / t) * u
                rbk -= ddkappa_ + 1.0 / (t * tau ** 2) * ddtau_
            else:
                rbs -= ddX_
                u = ddS_.copy()
                hessian(st.L, st.Y, [u], inv=False, adj=None)
                rbs -= (1.0 / t) * u
                rbk -= ddtau_ + 1.0 / (t * kappa ** 2) * ddkappa_
        return (rby, rbx, rbt, rbs, rbk)

    def tres(rbz):
        # reduced right-hand side (solvers.py:1774-1797)
        t, tau, kappa = st.t, st.tau, st.kappa
        if primal:
            a = tau ** 2 * t * (rbz[2] + rbz[4])
            rtx = C.copy()
            rtx.scale(a)
            rtx -= rbz[1] + rbz[3]
        else:
            a = rbz[4] + 1.0 / (t * kappa ** 2) * rbz[2]
            rtx = rbz[3].copy()
            hessian(st.L, st.Y, rtx, inv=True, adj=None)
            rtx.scale(-t)
            rtx += a * C - rbz[1]
        return rtx, rbz[0] + a * b

    def direction(sigma, dz):
        """One reduced solve + back-substitution (solvers.py:1997-2022 / 2062-2086)."""
        t, tau, kappa = st.t, st.tau, st.kappa
        rbz = bres(sigma, dz)
        rtx, rty = tres(rbz)
        u1, u2 = st.f.solve(rtx, rty, t)
        den = (1.0 / (t * tau ** 2)) if primal else (t * kappa ** 2)
        gamma = (-float(np.dot(b, u2)) + dot(C, u1)) / (den + float(np.dot(b, st.v2)) - dot(C, st.v1))
        dy = u2 + gamma * st.v2
        dX = u1.copy() + gamma * st.v1
        dkappa = -rbz[2] + float(np.dot(b, dy)) - dot(C, dX)
        if bmax > 1e-5:
            dtau = (Amap(dX, ii) - rbz[0][ii]) / b[ii]
        elif primal:
            dtau = (rbz[4] - dkappa) * t * tau ** 2
        else:
            dtau = rbz[4] - dkappa / (t * kappa ** 2)
        if primal:
            dS = dX.copy()
            dS.scale(-1.0 / t)
            hessian(st.L, st.Y, dS, inv=True, adj=None)
            dS += rbz[3]
        else:
            dS = rbz[3].copy() - dX
            dS.scale(t)
            hessian(st.L, st.Y, [dS], inv=True, adj=None)
        return dy, dX, dtau, dS, dkappa

    def newton(sigma):
        dy, dX, dtau, dS, dkappa = direction(sigma, None)
        for _ in range(REFINEMENT):
            ddy, ddX, ddtau, ddS, ddkappa = direction(sigma, (dy, dX, dtau, dS, dkappa))
            dy = dy + ddy
            dX += ddX
            dtau += ddtau
            dS += ddS
            dkappa += ddkappa
        return dy, dX, dtau, dS, dkappa

    def newton_res(sigma, dy, dX, dtau, dS, dkappa):
        # residuals of the five Newton equations, options['debug'] (solvers.py:1813-1841)
        t, tau, kappa = st.t, st.tau, st.kappa
        rbz = bres(sigma)
        r1 = _nrm2(Amap(dX) - dtau * b - rbz[0])
        r2 = _frob(Aadj(-dy) + dtau * C - dS - rbz[1])
        r3 = abs(float(np.dot(b, dy)) - dot(C, dX) - dkappa - rbz[2])
        if primal:
            r4 = dX.copy()
            hessian(st.L, st.Y, r4, inv=True, adj=None)
            r4.scale(1.0 / t)
            r4 += dS - rbz[3]
            r5 = abs(dtau / (t * tau ** 2) + dkappa - rbz[4])
        else:
            r4 = dS.copy()
            hessian(st.L, st.Y, r4, inv=False, adj=None)
            r4.scale(1.0 / t)
            r4 += dX - rbz[3]
            r5 = abs(dkappa / (t * kappa ** 2) + dtau - rbz[4])
        print(" Newton:   % .2e % .2e % .2e % .2e % .2e" % (r1, r2, r3, _frob(r4), r5))

    def linesearch(dX, dS, dtau, dkappa):
        # backtracking: kappa, tau, X, S must stay in their cones (solvers.py:2172-2209)
        t = 1.0
        while (st.kappa + t * dkappa <= 0) or (st.tau + t * dtau <= 0):
            t *= BETA
            if t < MINSTEP:
                return None
        for Z, dZ, test in ((X, dX, completion), (S, dS, cholesky)):
            while _in_cone(Z.copy() + t * dZ, test) is None:
                t *= BETA
                if t < MINSTEP:
                    return None
        return t

    if opt.show_progress:
        print("%-20s Extended self-dual embedding, %s scaling (%s)" % (__version__, scaling, "Cholesky"))
        print("-" * 76)
        print("SDP var. size:       %i " % n)
        print("Constraints:         %i (%i|%i)" % (m, m - prob.Ns, prob.Ns))
        print("Aggregate sparsity:  %-14s NNZ(tril(V)) = %7i"
              % ("Chordal" if prob.chordal else "Nonchordal", prob.nnz_Va))
        if not prob.chordal:
            print("Embedding:           %-14s       NNZ(L) = %7i" % ("min. degree", prob.symb.nvp))
        print("-" * 76)
        print(" it  pcost       dcost      gap     pres    dres    k/t     step    cputime")

    pinfres = dinfres = None
    step = None
    trace = []
    it = 0
    for it in range(opt.maxiters + 1):
        # residuals and convergence statistics (solvers.py:2219-2263)
        tau, kappa = st.tau, st.kappa
        hry = Amap(X)
        st.ry = b * tau - hry
        hrx = Aadj(y) + S
        st.rx = hrx.copy() - tau * C
        cx = dot(C, X)
        by = float(np.dot(b, y))
        st.rt = kappa - by + cx
        pres = (_nrm2(st.ry) / tau) / resy0
        dres = (_frob(st.rx) / tau) / resx0
        pcost = cx / tau
        dcost = by / tau
        gap = dot(X, S) / tau ** 2
        if pcost < 0.0:
            relgap = gap / -pcost
        elif dcost > 0.0:
            relgap = gap / dcost
        else:
            relgap = None
        pinfres = (_frob(hrx) / resx0 / by) if -by < 0.0 else None
        dinfres = (_nrm2(hry) / resy0 / (-cx)) if cx < 0.0 else None

        trace.append(dict(iter=it, pcost=pcost, dcost=dcost, gap=gap, pres=pres, dres=dres,
                          kt=kappa / tau, step=step))
        if opt.show_progress:
            print("%3d % .4e % .4e %.1e %.1e %.1e %.1e %-7s %7.1f" % (
                it, pcost, dcost, gap, pres, dres, kappa / tau,
                "%.1e" % step if it else " ", process_time() - T0))

        # stopping criteria (solvers.py:2289-2336)
        if dres <= opt.feastol and pres <= opt.feastol and (
                gap <= opt.abstol or (relgap is not None and relgap <= opt.reltol)):
            say("Optimal solution found.")
            status = "optimal"
            break
        elif pinfres is not None and pinfres <= opt.feastol:
            say("Certificate of primal infeasibility found.")
            status = "primal infeasibility"
            X, pcost, dcost = None, None, 1
            gap = relgap = pres = dres = dinfres = None
            break
        elif dinfres is not None and dinfres <= opt.feastol:
            say("Certificate of dual infeasibility found.")
            status = "dual infeasibility"
            y, S, pcost, dcost = None, None, -1, None
            gap = relgap = pres = dres = pinfres = None
            break
        elif it == opt.maxiters:
            say("Terminated (maximum number of iterations reached).")
            status = "unknown"
            break

        st.t = (n + 1) / (gap * tau ** 2 + kappa * tau)

        # scaling point (solvers.py:2341-2361)
        if primal:
            st.L = _in_cone(X, completion)
            if st.L is None:
                say("*** Completion failed")
                status = "unknown"
                break
            st.Y = X
        else:
            st.L = _in_cone(S, cholesky)
            if st.L is None:
                say("*** Factorization of S failed")
                status = "unknown"
                break
            st.Y = st.L.copy()
            projected_inverse(st.Y)

        try:
            st.f = _make_kkt(prob, st.L, st.Y, scaling)
        except ArithmeticError:
            print("*** Factorization failed")
            status = "unknown"
            break
        st.v1, st.v2 = st.f.solve(C, b, st.t)

        # predictor (affine scaling) direction and step
        dy, dX, dtau, dS, dkappa = newton(0.0)
        if opt.debug:
            newton_res(0.0, dy, dX, dtau, dS, dkappa)
        step = linesearch(dX, dS, dtau, dkappa)
        if not step:
            say("Terminated (small step size detected).")
            status = "unknown"
            break

        St = S.copy() + step * dS
        Xt = X.copy() + step * dX
        taut = tau + step * dtau
        kappat = kappa + step * dkappa
        sigma = ((dot(Xt, St) + taut * kappat) / (gap * tau ** 2 + kappa * tau)) ** EXPON

        # corrector direction and step
        dy, dX, dtau, dS, dkappa = newton(sigma)
        if opt.debug:
            newton_res(sigma, dy, dX, dtau, dS, dkappa)
        step = linesearch(dX, dS, dtau, dkappa)
        if not step:
            say("Terminated (small step size detected).")
            break

        if primal:
            # Y aliases X in the reference (solvers.py:2350); X is updated in place only here
            st.Y = None
        X += (STEP * step) * dX
        y = y + STEP * step * dy
        S += (STEP * step) * dS
        st.tau += STEP * step * dtau
        st.kappa += STEP * step * dkappa
        if _iteration_hook is not None:
            _iteration_hook("esd", it + 1)

    Tcpu = process_time() - T0
    Twall = perf_counter() - T0wall
    tau = st.tau

    dimacs = None
    if opt.dimacs and X is not None and y is not None and S is not None:
        R = Aadj(y) + S
        R.scale(1.0 / tau)
        R -= C
        cmax = float(np.max(np.abs(prob.c))) if len(prob.c) else 0.0
        dimacs = [_nrm2(Amap(X) / tau - b) / (1 + float(np.max(np.abs(b)))), 0.0,
                  _frob(R) / (1 + cmax), 0.0,
                  (pcost - dcost) / (1 + abs(pcost) + abs(dcost)),
                  gap / (1 + abs(pcost) + abs(dcost))]

    Xo = yo = So = None
    if X is not None:
        Xo = prob.to_original(X * (1.0 / tau))
    if y is not None:
        yo = y[prob.inv_pm] / tau
    if S is not None:
        So = prob.to_original(S * (1.0 / tau))

    if opt.show_progress:
        _print_exit(status, pcost, dcost, gap, relgap, pres, dres, it, Tcpu, Twall, dimacs)

    return {"status": status, "x": Xo, "y": yo, "s": So, "primal objective": pcost,
            "dual objective": dcost, "gap": gap, "relative gap": relgap,
            "primal infeasibility": pres, "dual infeasibility": dres,
            "residual as primal infeasibility certificate": pinfres,
            "residual as dual infeasibility certificate": dinfres,
            "iterations": it, "cputime": Tcpu, "time": Twall, "trace": trace, "dimacs": dimacs}


# --------------------------------------------------------------------------------------
# CVXOPT-style cone LP front end
# --------------------------------------------------------------------------------------
def conelp(c, G, h, dims=None, kktsolver="chol"):
    """Cone LP  min c'x  s.t. Gx + s = h, s in K  with K = R^l_+ x SOC(q_1) x ... x PSD(s_1)...
    embedded in one block-diagonal / arrow chordal SDP and solved with the self-dual
    driver (``solvers.py:2470-2599``).  ``G`` is N x m (dense or sparse), ``h`` has N entries,
    's' blocks are stored column-major (lower triangle used)."""
    from .base import SDP

    Nl = dims.get("l", 0) or 0
    Nq = list(dims.get("q", []) or [])
    Nsd = list(dims.get("s", []) or [])
    n = Nl + sum(Nq) + sum(Nsd)
    G = sp.csc_matrix(G)
    m = G.shape[1]
    h = np.asarray(h, dtype=np.float64).ravel()
    c = np.asarray(c, dtype=np.float64).ravel()

    rows, cols, vals = [], [], []

    def put(r, cidx, k, v):
        rows.append(r + n * cidx)
        cols.append(k)
        vals.append(v)

    for k in range(m + 1):
        v = h if k == 0 else np.asarray(G[:, k - 1].todense()).ravel()
        ptr = 0
        base = 0
        for i in range(Nl):
            if v[i] != 0.0:
                put(i, i, k, v[i])
        ptr += Nl
        base += Nl
        for nq in Nq:                       # arrow: u0 on the diagonal, u1 in the last row
            u0 = v[ptr]
            u1 = v[ptr + 1:ptr + nq]
            if u0 != 0.0:
                for i in range(nq):
                    put(base + i, base + i, k, u0)
            for i in range(nq - 1):
                if u1[i] != 0.0:
                    put(base + nq - 1, base + i, k, u1[i])
            ptr += nq
            base += nq
        for ns in Nsd:                      # lower triangle of the ns x ns block
            u = v[ptr:ptr + ns * ns]
            for jj in range(ns):
                for i in range(jj, ns):
                    if u[i + ns * jj] != 0.0:
                        put(base + i, base + jj, k, u[i + ns * jj])
            ptr += ns * ns
            base += ns
    P = SDP()
    P._A = misc.as_csc(sp.csc_matrix((np.array(vals, dtype=np.float64),
                                      (np.array(rows, dtype=np.int64), np.array(cols, dtype=np.int64))),
                                     shape=(n * n, m + 1)))
    P._b = -c
    P._blockstruct = ([-Nl] if Nl else []) + Nq + Nsd
    sol = P.solve_esd(kktsolver=kktsolver)

    x, s = sol["x"], sol["s"]

    def unpack(M, soc):
        if M is None:
            return None
        M = np.asarray(M.todense())
        out = [np.diag(M)[:Nl]]
        N = Nl
        for nq in Nq:
            out.append(soc(M, N, nq))
            N += nq
        for ns in Nsd:
            out.append(M[N:N + ns, N:N + ns].reshape(-1, order="F"))
            N += ns
        return np.concatenate(out) if out else np.zeros(0)

    z = unpack(x, lambda M, N, nq: np.concatenate([[np.trace(M[N:N + nq, N:N + nq])],
                                                    2 * M[N + nq - 1, N:N + nq - 1]]))
    sv = unpack(s, lambda M, N, nq: np.concatenate([[M[N + nq - 1, N + nq - 1]],
                                                     M[N + nq - 1, N:N + nq - 1]]))
    sol["x"] = sol.pop("y")
    sol["z"] = z
    sol["s"] = sv
    return sol


def lp(c, G, h, kktsolver="chol"):
    """Linear program  min c'x  s.t. Gx + s = h, s >= 0  through ``conelp`` (``solvers.py:2602-2603``)."""
    G = sp.csc_matrix(G)
    return conelp(c, G, h, dims={"l": G.shape[0], "q": [], "s": []}, kktsolver=kktsolver)


def _stack(blocks_G, blocks_h):
    G = sp.vstack([sp.csc_matrix(g) for g in blocks_G], format="csc")
    h = np.concatenate([np.asarray(v, dtype=np.float64).reshape(-1, order="F") for v in blocks_h])
    return G, h


def socp(c, Gl=None, hl=None, Gq=None, hq=None, kktsolver="chol"):
    """Second-order cone program through ``conelp`` (``solvers.py:2606-2648``; the reference's version
    fails on its first ``dims['l'].append`` — this one follows its documented contract): ``Gq[k]``,
    ``hq[k]`` describe the k-th cone ``s_k = hq[k] - Gq[k] x`` with ``s_k[0] >= ||s_k[1:]||``.
    Returns ``conelp``'s dictionary with ``zl, sl`` and the lists ``zq, sq`` instead of ``z, s``."""
    if Gq is None or hq is None:
        raise ValueError("'Gq' and 'hq' cannot be zero")
    dims = {"l": 0, "q": [], "s": []}
    Gs_, hs_ = [], []
    if Gl is not None and hl is not None:
        dims["l"] = sp.csc_matrix(Gl).shape[0]
        Gs_.append(Gl)
        hs_.append(hl)
    for Gk, hk in zip(Gq, hq):
        dims["q"].append(sp.csc_matrix(Gk).shape[0])
        Gs_.append(Gk)
        hs_.append(hk)
    G, h = _stack(Gs_, hs_)
    sol = conelp(c, G, h, dims=dims, kktsolver=kktsolver)
    z, s = sol.pop("z"), sol.pop("s")
    N = dims["l"]
    sol["zl"] = z[:N] if (N and z is not None) else None
    sol["sl"] = s[:N] if (N and s is not None) else None
    sol["zq"], sol["sq"] = [], []
    for nq in dims["q"]:
        sol["zq"].append(z[N:N + nq] if z is not None else None)
        sol["sq"].append(s[N:N + nq] if s is not None else None)
        N += nq
    return sol


def sdp(c, Gl=None, hl=None, Gs=None, hs=None, kktsolver="chol"):
    """Semidefinite program through ``conelp`` (``solvers.py:2651-2699``): ``Gs[k]`` is
    ns_k^2 x n (column j = vec of the symmetric matrix multiplying x_j, column-major), ``hs[k]``
    an ns_k x ns_k matrix.  Returns ``conelp``'s dictionary with ``zl, sl`` and the lists
    ``zs, ss`` of ns_k x ns_k arrays instead of ``z, s``."""
    if Gs is None or hs is None:
        raise ValueError("'Gs' and 'hs' cannot be zero")
    dims = {"l": 0, "q": [], "s": []}
    G_, h_ = [], []
    if Gl is not None and hl is not None:
        dims["l"] = sp.csc_matrix(Gl).shape[0]
        G_.append(Gl)
        h_.append(hl)
    for Gk, hk in zip(Gs, hs):
        dims["s"].append(int(round(math.sqrt(sp.csc_matrix(Gk).shape[0]))))
        G_.append(Gk)
        h_.append(hk)
    G, h = _stack(G_, h_)
    sol = conelp(c, G, h, dims=dims, kktsolver=kktsolver)
    z, s = sol.pop("z"), sol.pop("s")
    N = dims["l"]
    sol["zl"] = z[:N] if (N and z is not None) else None
    sol["sl"] = s[:N] if (N and s is not None) else None
    sol["zs"], sol["ss"] = [], []
    for ns in dims["s"]:
        sol["zs"].append(z[N:N + ns * ns].reshape(ns, ns, order="F") if z is not None else None)
        sol["ss"].append(s[N:N + ns * ns].reshape(ns, ns, order="F") if s is not None else None)
        N += ns * ns
    return sol
