"""Problem containers and random problem builders (API surface of ``smcp.base``,
reference ``src/python/base.py``).

``SDP`` keeps the reference's data layout — ``A`` CCS ``n^2 x (m+1)`` with column 0 = vec(C)
and lower-triangular entries only, ``b`` dense — and its three solve entry points on the
hot path: ``solve_feas`` (``base.py:346-368``), ``solve_esd`` (``316-344``) and
``solve_phase1`` (``370-470``), plus SDPA (dat-s) / pickle I/O with the reference's signatures.
``solve_cvxopt`` and the robust-LS converters are outside the path and not provided.

The generators restate ``band_SDP`` (``base.py:598-636``), ``mtxnorm_SDP`` (``707-778``),
``rand_SDP`` (``879-949``) and ``mk_rand`` (``514-560``) with NumPy's ``default_rng``:
cvxopt's RNG stream (``setseed``/``normal``) cannot be reproduced, so instances differ from
the reference's for the same seed but follow the same construction.  ``maxcut_SDP`` builds
the max-cut relaxation the reference reads from SDPLIB files.
"""
from __future__ import annotations

import numpy as np
import scipy.sparse as sp
import scipy.sparse.linalg as spla

from . import misc, solvers
from .symbolic import Symbolic, embed, maxcardsearch, min_degree, lower_pattern

__all__ = ["SDP", "band_SDP", "mtxnorm_SDP", "rand_SDP", "maxcut_SDP", "mk_rand", "completion", "completion_sample"]


class SDP(object):
    """SDP object: ``n``, ``m``, ``A`` (CCS n^2 x (m+1)), ``b``, aggregate sparsity ``I``."""

    def __init__(self, A=None, b=None, name=None, filename=None):
        """``SDP(A, b)`` from problem data, or ``SDP(filename)`` / ``SDP(filename='x.dat-s')`` from a sparse
        SDPA (dat-s) or pickle file (``base.py:62-85, 177-195``: the file's primal is negated into SMCP's
        standard form)."""
        if filename is not None:
            if A is not None and not isinstance(A, str):
                raise TypeError("give either problem data or a file name")
            A = filename
        self._I = None
        self._ischordal = None
        self._blockstruct = None
        self._X0 = self._y0 = self._S0 = None
        if isinstance(A, str):
            import os
            fp, ext = os.path.splitext(A)
            if ext == ".bz2" and fp.endswith(".pkl"):
                self._load(A)
                return
            if ext == ".bz2":
                # compressed SDPLIB files (``base.py:180-190``): decompress next to a temporary name
                import bz2, tempfile
                with open(A, "rb") as fc, tempfile.NamedTemporaryFile("wb", suffix=".dat-s", delete=False) as fo:
                    fo.write(bz2.decompress(fc.read()))
                    tmp = fo.name
                try:
                    self._A, self._b, self._blockstruct = misc.sdpa_read(tmp, neg=True)
                finally:
                    os.remove(tmp)
                fp = os.path.splitext(fp)[0]
            elif ext == ".dat-s":
                self._A, self._b, self._blockstruct = misc.sdpa_read(A, neg=True)
            elif ext == ".pkl":
                self._load(A)
                return
            else:
                raise NameError("Unknown file extension")
            self._pname = name or os.path.basename(fp)
            return
        self._A = misc.as_csc(A) if A is not None else None
        self._b = np.asarray(b, dtype=np.float64).ravel() if b is not None else None
        self._pname = name

    def _load(self, fname):
        """Load problem data saved by ``save`` (``base.py:219-238``)."""
        import bz2, pickle
        raw = open(fname, "rb").read()
        D = pickle.loads(bz2.decompress(raw) if fname.endswith(".bz2") else raw)
        self._A = misc.as_csc(D["A"])
        self._b = np.asarray(D["b"], dtype=np.float64).ravel()
        self._X0, self._y0, self._S0, self._pname = D["X0"], D["y0"], D["S0"], D["pname"]

    def save(self, fname=None, compress=False):
        """Save problem data (and the generator's strictly feasible point, if any) to a pickle file
        ``<fname>.pkl`` or ``<fname>.pkl.bz2`` (``base.py:240-270``); refuses to overwrite."""
        import bz2, os, pickle
        fname = (fname or self._pname) + (".pkl.bz2" if compress else ".pkl")
        if os.path.isfile(fname):
            raise IOError("file %s already exists" % fname)
        D = {"A": self._need(), "b": self._b, "X0": self._X0, "y0": self._y0, "S0": self._S0, "pname": self._pname}
        raw = pickle.dumps(D)
        with open(fname, "wb") as f:
            f.write(bz2.compress(raw) if compress else raw)
        return fname

    def write_sdpa(self, fname=None, compress=False):
        """Writes the problem to the sparse SDPA file ``<fname>.dat-s`` (``<fname>`` defaults to the problem
        name; ``compress=True``: ``<fname>.dat-s.bz2``), refusing to overwrite an existing file
        (``base.py:197-217``; one block unless the object was read from a file with a block structure).
        Returns the name of the file written."""
        import bz2, os
        bs = self._blockstruct if self._blockstruct is not None else np.array([self.n], dtype=np.int64)
        if fname is None:
            fname = self._pname
        if fname is None:
            raise ValueError("the problem has no name: give a file name")
        fname += ".dat-s"
        if os.path.isfile(fname):
            raise IOError("file %s already exists" % fname)
        if compress and os.path.isfile(fname + ".bz2"):
            raise IOError("file %s already exists" % (fname + ".bz2"))
        misc.sdpa_write(fname, self._need(), self.b, bs, neg=True)
        if compress:
            with open(fname, "rb") as fi, open(fname + ".bz2", "wb") as fo:
                fo.write(bz2.compress(fi.read()))
            os.remove(fname)
            fname += ".bz2"
        return fname

    def __str__(self):
        return "<SDP: n=%i, m=%i, nnz=%i> %s" % (self.n, self.m, self.nnz, self._pname)

    def _need(self):
        if self._A is None:
            raise AttributeError("SDP object has not been initialized")
        return self._A

    @property
    def n(self):
        return int(np.sqrt(self._need().shape[0]))

    @property
    def m(self):
        return self._need().shape[1] - 1

    @property
    def A(self):
        return self._need()

    def get_A(self, i=None):
        """A if i is None, otherwise A_i as an n x n lower-triangular sparse matrix."""
        A = self._need()
        if i is None:
            return A
        if not 0 <= i <= self.m:
            raise ValueError("index is out of range")
        r = A.indices[A.indptr[i]:A.indptr[i + 1]]
        v = A.data[A.indptr[i]:A.indptr[i + 1]]
        Il, Jl = misc.ind2sub(self.n, r)
        return sp.csc_matrix((v, (Il, Jl)), shape=(self.n, self.n))

    @property
    def b(self):
        if self._b is None:
            raise AttributeError("SDP object has not been initialized")
        return self._b

    @property
    def I(self):
        """Aggregate sparsity pattern as absolute (linear) indices."""
        if self._I is None:
            self._I = np.unique(self._need().indices)
        return self._I

    @property
    def V(self):
        I, J = misc.ind2sub(self.n, self.I)
        return sp.csc_matrix((np.zeros(len(I)), (I, J)), shape=(self.n, self.n))

    @property
    def nnz(self):
        return len(self.I)

    @property
    def issparse(self):
        return len(self.I) <= 0.5 * (self.n * (self.n + 1) / 2)

    def get_nnz(self, i=None):
        """Number of non-zeros in the lower triangle of A_0 .. A_m, or of A_i (``base.py:279-293``)."""
        cnt = np.diff(self._need().indptr)
        if i is None:
            return cnt
        if not 0 <= i <= self.m:
            raise ValueError("index out of range")
        return int(cnt[i])

    nnzs = property(get_nnz, doc="Vector with number of nonzeros in lower triangle of A0,A1,...,Am")

    def get_nzcols(self, i=None):
        """Number of non-zero columns of A_1 .. A_m, or of A_i, i >= 1 (``base.py:299-310``)."""
        nzc = misc.nzcolumns(self._need())
        if i is None:
            return nzc
        if not 0 < i <= self.m:
            raise ValueError("index out of range")
        return int(nzc[i - 1])

    nzcols = property(get_nzcols, doc="Vector with number of nonzero columns in A1,..,Am")

    @property
    def ischordal(self):
        if self._ischordal is None:
            I, J = misc.ind2sub(self.n, self.I)
            cp, ri = lower_pattern(self.n, I, J)
            p = maxcardsearch(self.n, cp, ri)
            fc, _, _ = embed(self.n, cp, ri, p)
            self._ischordal = bool(fc[-1] == cp[-1])
        return self._ischordal

    # -- solvers ------------------------------------------------------------------
    def solve_esd(self, kktsolver="chol", scaling="primal", primalstart=None, dualstart=None, p=None):
        return solvers.chordalsolver_esd(self.A, self.b, kktsolver=kktsolver, scaling=scaling,
                                         primalstart=primalstart, dualstart=dualstart, p=p)

    def solve_feas(self, kktsolver="chol", scaling="primal", primalstart=None, dualstart=None):
        return solvers.chordalsolver_feas(self.A, self.b, kktsolver=kktsolver, scaling=scaling,
                                          primalstart=primalstart, dualstart=dualstart)

    def solve_phase1(self, kktsolver="chol", MM=1e5):
        """Primal Phase I with the feasible-start solver; returns ``(X0, sol)`` with a primal
        feasible ``X0`` (``base.py:370-470``).  The least-norm start (``base.py:383-396``: sparse
        ``syrk`` + CHOLMOD in the reference) runs on the backend: Gram matrix of the constraints by one
        triangular product, dense Cholesky, ``A^adj``."""
        from .chordal import cspmatrix, completion
        n, m = self.n, self.m
        k = 1e-3
        A = self._need()
        Id = np.arange(n, dtype=np.int64) * (n + 1)
        # least-norm start X0 = sum_j u_j A_j with G u = b, G_ij = <A_i, A_j> (base.py:383-396: the reference
        # forms As^T As with syrk and solves with CHOLMOD).  On the backend: G as ONE triangular product of
        # the constraint vectors (DMMA / TMA on the device), the dense Cholesky of the Schur complement, and
        # A^adj for the combination -- on the same embedding the completability test below needs.
        opt = solvers._read_options(n, True)
        prob = solvers._Problem(A, self.b, opt, "qr", None)          # 'qr': no constraint reordering (Ns = 0)
        ops, symb, pm = prob.ops, prob.symb, prob.p
        # the product runs over the rows of the backend's dense constraint copy: all of blkval, or on filled
        # patterns only the rows the constraints touch (a backend without dense_rows() contracts over all)
        rows = ops.dense_rows() if hasattr(ops, "dense_rows") else symb.nblk
        dense_bytes = 8.0 * rows * m
        if dense_bytes <= (16 << 30):
            ops.gram_factor()
            u = ops.schur_solve(prob.b)
            Xc = prob.Aadj(u)
            X0 = sp.tril(prob.to_original(Xc), format="csc")
            X0.eliminate_zeros()
        else:
            # constraint vectors too large for the dense product: sparse normal equations on the host
            As = A[:, 1:].tocsc().copy()
            scale = np.ones(A.shape[0])
            scale[Id] = 1.0 / np.sqrt(2.0)
            As = (sp.diags(scale) @ As).tocsc()
            u = spla.spsolve((As.T @ As).tocsc(), self.b)
            x = 0.5 * (A[:, 1:] @ u)
            I, J = misc.ind2sub(n, self.I)
            X0 = sp.csc_matrix((x[self.I], (I, J)), shape=(n, n))
            Xc = prob.from_original(X0)

        def completable(Z):
            L = Z.copy()
            try:
                completion(L)
                return True
            except ArithmeticError:
                return False

        if completable(Xc):
            return X0, None

        trA = np.zeros(m + 1)
        trA[:m] = np.asarray(A[Id, 1:].sum(axis=0)).ravel()
        trA[-1] = MM
        P1 = SDP(misc.phase1_sdp(A, trA), np.concatenate([self.b - k * trA[:m], [MM]]))

        tMIN, tMAX = 0.0, 1.0
        while True:
            t = (tMIN + tMAX) / 2.0
            if completable(Xc.copy() + cspmatrix.identity(ops, t)):
                tMAX = t
                if tMAX - tMIN < 1e-1:
                    break
            else:
                tMAX *= 2.0
                tMIN = t
        tt = t + 1.0
        U = (X0 + tt * sp.identity(n, format="csc")).tocsc()
        trU = U.diagonal().sum()
        Z0 = sp.block_diag([U, sp.diags([tt + k, MM - trU])], format="csc")
        sol = P1.solve_feas(primalstart={"x": Z0}, kktsolver=kktsolver)
        s = sol["x"][n, n] - k
        if s > 0:
            return None, P1
        sol.pop("y")
        sol.pop("s")
        Xz = sol.pop("x")
        X0 = (Xz[:n, :n] - s * sp.identity(n, format="csc")).tocsc()
        return X0, sol

    # -- rounding (an extension: the reference has none) ---------------------------------
    def round_pm1(self, sol, trials=256, seed=0, chunk=0, local_search=False, max_flips=None, tol=1e-12, tabu_iters=0,
                  tenure=None):
        """Goemans-Williamson rounding of a solution with diag(X) = 1: ``trials`` sign vectors
        s_t = sign(v_t), v_t drawn with covariance the max-det completion of ``sol['x']``
        (``completion_sample``), evaluated against the objective C on the device; ``chunk`` trials per pass
        (0: as many as fit in 1 GiB), with no effect on the result.  Returns a dict: ``x`` (int8 +-1, original
        order) of the smallest C . x x^T (lowest trial on ties), ``value`` = C . x x^T, ``values`` of every
        trial and ``trial``, the index of the best one.  Raises ``ArithmeticError`` if X has no positive
        definite completion.

        ``local_search=True`` runs the one-flip local search of ``local_search_pm1`` (``max_flips``, ``tol``) on
        every trial on the device, in the internal order of the completion (which decides ties); ``x``, ``value``,
        ``values`` and ``trial`` then refer to the searched trials, ``values_rounded`` holds the values before the
        search and ``flips`` the number of flips of every trial.

        ``tabu_iters > 0`` runs the tabu search of ``tabu_search_pm1`` (``tabu_iters`` moves, ``tenure``) on every
        trial on the device, after the one-flip search when that is on; ``x``, ``value``, ``values`` and ``trial``
        then refer to the trials after the tabu search, ``values_before_tabu`` holds the values before it, ``moves``
        the number of moves and ``best_iter`` the move count of every returned vector.

        When ``sol`` holds ``V`` (a low-rank solution from ``solve_lowrank``), trial t is sign(V g_t) instead, g_t the
        length-r normal sample t under ``seed``: the samples are one DMMA product per block of trials on the device, in
        the original order, and need no completion; everything else is as above."""
        trials = _check_count(trials, "trials", 1)
        seed = _check_seed(seed)
        chunk = _check_count(chunk, "chunk", 0)
        if not isinstance(local_search, (bool, np.bool_)):
            raise TypeError("local_search must be a bool")
        if max_flips is not None:
            max_flips = _check_count(max_flips, "max_flips", 0)
        tol = _check_tol(tol)
        tabu_iters = _check_count(tabu_iters, "tabu_iters", 0)
        tenure = _tabu_tenure(self.n) if tenure is None else _check_count(tenure, "tenure", 0)
        if not isinstance(sol, dict) or ("x" not in sol and "V" not in sol):
            raise ValueError("sol must be a solution dict holding 'x' or 'V'")
        if "V" in sol:
            return self._round_pm1_factor(sol["V"], trials, seed, chunk, local_search, max_flips, tol, tabu_iters, tenure)
        L, order = _completion_factor(sol["x"])
        n = self.n
        if len(order) != n:
            raise ValueError("sol['x'] is %d x %d, the problem has n = %d" % (len(order), len(order), n))
        I, J, v = self._objective_entries()
        pos = np.empty(n, dtype=np.int64)
        pos[order] = np.arange(n, dtype=np.int64)
        out = {}
        if tabu_iters > 0:
            mf = (n if max_flips is None else max_flips) if local_search else 0
            values0, values1, values, flips, moves, best_iter, xi, best = L.ops.round_pm1_tabu(
                L.buf, pos[I], pos[J], v, trials, seed, tabu_iters, tenure, chunk, mf, tol)
            out = {"values_before_tabu": values1, "moves": moves, "best_iter": best_iter}
            if local_search:
                out.update({"values_rounded": values0, "flips": flips})
        elif local_search:
            values0, values, flips, xi, best = L.ops.round_pm1_ls(L.buf, pos[I], pos[J], v, trials, seed, chunk,
                                                                  max_flips, tol)
            out = {"values_rounded": values0, "flips": flips}
        else:
            values, xi, best = L.ops.round_pm1(L.buf, pos[I], pos[J], v, trials, seed, chunk)
        x = np.empty(n, dtype=np.int8)
        x[order] = xi
        out.update({"x": x, "value": float(values[best]), "values": values, "trial": int(best)})
        return out

    def _round_pm1_factor(self, V, trials, seed, chunk, local_search, max_flips, tol, tabu_iters, tenure):
        """``round_pm1`` from the factor V (checked arguments)."""
        n = self.n
        V = np.asarray(V, dtype=np.float64)
        if V.ndim != 2 or V.shape[0] != n or not 1 <= V.shape[1] <= _LOWRANK_MAX_RANK:
            raise ValueError("sol['V'] must be n x r with n = %d and 1 <= r <= %d" % (n, _LOWRANK_MAX_RANK))
        I, J, v = self._objective_entries()
        ops = solvers._make_backend(Symbolic(n, np.arange(n + 1), np.arange(n)))
        mf = (n if max_flips is None else max_flips) if local_search else 0
        values0, values1, values, flips, moves, best_iter, x, best = ops.round_pm1_factor(
            V, I, J, v, trials, seed, chunk, mf, tol, tabu_iters, tenure)
        out = {}
        if tabu_iters > 0:
            out.update({"values_before_tabu": values1, "moves": moves, "best_iter": best_iter})
        if local_search:
            if values0 is None:                     # max_flips = 0 and no tabu search: nothing ran
                values0, flips = values.copy(), np.zeros(len(values), dtype=np.int64)
            out.update({"values_rounded": values0, "flips": flips})
        out.update({"x": x, "value": float(values[best]), "values": values, "trial": int(best)})
        return out

    # -- low-rank solve (an extension: the reference has none) ----------------------------
    def solve_lowrank(self, rank=None, seed=0, tol=1e-6, max_sweeps=1000, bound=True):
        """Low-rank (Burer-Monteiro) solve of  min C . X  s.t.  X_ii = b_i, X >= 0  on the device, for an SDP whose m = n
        constraints each hold one entry, coefficient 1 at a diagonal position (d_k, d_k), d a permutation of 0..n-1, and
        b > 0 (``maxcut_SDP`` has this form; any other problem raises ``ValueError``).

        X = V V^T with V n x ``rank`` (None: the smallest r with r(r+1)/2 > n, at most 512), solved by the mixing method:
        with the rows of C's off-diagonal entries (both triangles, duplicates summed in input order) and a greedy
        colouring in increasing vertex index (vertex i takes the smallest colour none of its lower-index neighbours
        has), each sweep takes the colours in order and sets v_i <- -sqrt(b_i) w_i / ||w_i|| for every vertex i of the
        colour, w_i = sum_{j != i} C_ij v_j (v_i stays when w_i = 0).  Row i of the start is the standard normal sample
        i (length r) under ``seed`` of ``completion_sample``'s generator, scaled to norm sqrt(b_i).  The objective
        f = sum_i C_ii b_i + <v_i, w_i> is evaluated at the start and after every sweep; the run stops after the first
        sweep k with f_{k-1} - f_k <= ``tol`` max(1, |f_k|), or after ``max_sweeps`` sweeps.  csrc/lowrank.cu states the
        summation orders: every result is bitwise reproducible.

        ``bound=True`` certifies a lower bound on the optimum (``_lowrank_certificate``): with y_i = (C_ii b_i +
        <v_i, w_i>) / b_i, the smallest shift t >= 0 found by bisection with C - Diag(y) + tI >= 0 proven by chordal
        Cholesky factorizations on the backend, so y - t is dual feasible and b^T y - t sum(b) a lower bound.

        Returns a dict: ``V`` (n x r, original order), ``x`` = P_V(V V^T) on the chordal embedding of C's pattern (the
        form ``solve_feas`` returns), ``y`` (constraint order, shifted by t), ``primal objective`` f, ``dual objective``
        (the certified bound, None when bound=False), ``gap`` (their difference, None without a bound), ``converged``,
        ``sweeps``, ``objective history`` (f_0 .. f_sweeps), ``colors`` (the number of colours), ``rank``, ``shift`` (t)
        and ``probes`` (Cholesky factorizations of the certificate)."""
        n = self.n
        d, bk = self._lowrank_form()
        if rank is None:
            rank = min(_LOWRANK_MAX_RANK, next(r for r in range(1, n + 2) if r * (r + 1) // 2 > n))
        rank = _check_count(rank, "rank", 1)
        if rank > _LOWRANK_MAX_RANK:
            raise ValueError("rank must be at most %d" % _LOWRANK_MAX_RANK)
        seed = _check_seed(seed)
        tol = _check_tol(tol)
        max_sweeps = _check_count(max_sweeps, "max_sweeps", 0)
        bv = np.empty(n)
        bv[d] = bk                                  # b per vertex
        I, J, v = self._objective_entries()
        ops = solvers._make_backend(Symbolic(n, np.arange(n + 1), np.arange(n)))
        V, f, yv, sweeps, colors = ops.lowrank_solve(I, J, v, bv, rank, seed, max_sweeps, tol)
        fk = float(f[-1])
        converged = sweeps > 0 and float(f[-2]) - fk <= tol * max(1.0, abs(fk))
        symb, p, _ = _chordal_embedding(sp.coo_matrix((np.concatenate([v, np.ones(n)]),
                                                       (np.concatenate([I, np.arange(n)]),
                                                        np.concatenate([J, np.arange(n)]))), shape=(n, n)))
        ri, ci = p[symb.Ip], p[symb.Jp]
        xv = np.empty(len(ri))
        step = max(1, (1 << 24) // rank)
        for a in range(0, len(ri), step):
            xv[a:a + step] = np.einsum("ij,ij->i", V[ri[a:a + step]], V[ci[a:a + step]])
        off = ri != ci
        x = sp.csc_matrix((np.concatenate([xv, xv[off]]), (np.concatenate([ri, ci[off]]), np.concatenate([ci, ri[off]]))),
                          shape=(n, n))
        t, probes, dual = 0.0, 0, None
        if bound:
            t, probes = _lowrank_certificate(n, I, J, v, yv, bv, fk)
            bsum = float(bv.sum())
            dual = float(np.dot(bv, yv)) - t * bsum
            # rounding of the two sums above (gamma_{n+2} of their absolute terms): the bound stays a bound
            dual -= _gamma(n + 2) * (float(np.abs(bv * yv).sum()) + t * bsum)
        return {"V": V, "x": x, "y": yv[d] - t, "primal objective": fk, "dual objective": dual,
                "gap": None if dual is None else fk - dual, "converged": bool(converged), "sweeps": int(sweeps),
                "objective history": f, "colors": int(colors), "rank": rank, "shift": t, "probes": probes}

    def _lowrank_form(self):
        """(d, b) of an SDP whose constraint k holds the single entry 1 at (d_k, d_k), d a permutation, b > 0; raises
        ``ValueError`` for any other problem."""
        A, n, m = self._need(), self.n, self.m
        if m != n:
            raise ValueError("solve_lowrank needs m = n constraints X_ii = b_i (got m = %d, n = %d)" % (m, n))
        cnt = np.diff(A.indptr)[1:]
        if (cnt != 1).any():
            raise ValueError("solve_lowrank needs constraints with one entry each (constraint %d has %d)" % (
                int(np.flatnonzero(cnt != 1)[0]), int(cnt[cnt != 1][0])))
        pos = A.indices[A.indptr[1]:A.indptr[m + 1]]
        val = A.data[A.indptr[1]:A.indptr[m + 1]]
        r, c = misc.ind2sub(n, pos)
        if (np.asarray(r) != np.asarray(c)).any() or (val != 1.0).any():
            raise ValueError("solve_lowrank needs constraints X_ii = b_i: coefficient 1 at a diagonal position")
        d = np.asarray(r, dtype=np.int64)
        if len(np.unique(d)) != n:
            raise ValueError("solve_lowrank needs one constraint per diagonal entry")
        b = self.b
        if not (np.isfinite(b).all() and (b > 0).all()):
            raise ValueError("solve_lowrank needs b > 0")
        return d, b

    def local_search_pm1(self, x, max_flips=None, tol=1e-12):
        """One-flip local search of +-1 vectors against f(x) = C . x x^T (minimized), on the device (an
        extension).  ``x``: integers +-1 of shape (n,) or (k, n), original order.  With s_i = sum_{j != i} C_ij x_j
        and a_i = sum_{j != i} |C_ij|, each step flips the vertex with the largest gain g_i = x_i s_i among those
        with g_i > ``tol`` a_i (lowest index on ties), which lowers f by 4 g_i; a vector's search stops when no
        vertex qualifies or after ``max_flips`` flips (None: n).  Returns a dict: ``x`` (int8, the shape of the
        input), ``values`` = f of the searched vectors and ``flips``, their numbers of flips (shape x.shape[:-1])."""
        n = self.n
        xa = _check_pm1(x, n)
        max_flips = n if max_flips is None else _check_count(max_flips, "max_flips", 0)
        tol = _check_tol(tol)
        I, J, v = self._objective_entries()
        ops = solvers._make_backend(Symbolic(n, np.arange(n + 1), np.arange(n)))
        xs, values, flips = ops.pm1_local_search(xa.reshape(-1, n), I, J, v, max_flips, tol)
        shape = np.shape(x)
        return {"x": xs.reshape(shape), "values": values.reshape(shape[:-1]), "flips": flips.reshape(shape[:-1])}

    def tabu_search_pm1(self, x, iters, tenure=None):
        """Tabu search of +-1 vectors against f(x) = C . x x^T (minimized), on the device (an extension).
        ``x``: integers +-1 of shape (n,) or (k, n), original order.  With s_i and the gain g_i = x_i s_i of
        ``local_search_pm1``, D_0 = 0 and move u flips the admissible vertex i with the largest g_i (lowest index on
        ties), setting D_{u+1} = D_u - 4 g_i, the change of f.  A vertex flipped by move u is tabu during moves
        u+1 .. u+``tenure`` (None: min(n - 1, 10 + n // 100)); a tabu vertex is admissible only when the move would
        bring D below its smallest value so far (aspiration), every other vertex always is, even when its flip
        raises f.  A vector's search stops after ``iters`` moves, or when no vertex is admissible, and returns the
        earliest vector with the smallest D.  Returns a dict: ``x`` (int8, the shape of the input), ``values`` = f
        of the returned vectors, ``moves``, the numbers of moves made, and ``best_iter``, the move count of each
        returned vector (0: the input); the last three of shape x.shape[:-1].  Needs n <= 2**19 and
        tenure <= 8192."""
        n = self.n
        xa = _check_pm1(x, n)
        iters = _check_count(iters, "iters", 0)
        tenure = _tabu_tenure(n) if tenure is None else _check_count(tenure, "tenure", 0)
        I, J, v = self._objective_entries()
        ops = solvers._make_backend(Symbolic(n, np.arange(n + 1), np.arange(n)))
        xs, values, moves, best_iter = ops.pm1_tabu_search(xa, I, J, v, iters, tenure)
        shape = np.shape(x)
        return {"x": xs.reshape(shape), "values": values.reshape(shape[:-1]), "moves": moves.reshape(shape[:-1]),
                "best_iter": best_iter.reshape(shape[:-1])}

    def _objective_entries(self):
        """Lower-triangular entries (row, col, value) of C in the original order."""
        A = self._need()
        I, J = misc.ind2sub(self.n, A.indices[A.indptr[0]:A.indptr[1]])
        return np.asarray(I, dtype=np.int64), np.asarray(J, dtype=np.int64), A.data[A.indptr[0]:A.indptr[1]]


# --------------------------------------------------------------------------------------
# generators
# --------------------------------------------------------------------------------------
def _pattern_cols(n, colptr):
    return np.repeat(np.arange(n, dtype=np.int64), np.diff(colptr))


def mk_rand(n, colptr, rowind, cone="posdef", seed=0):
    """Random matrix with the given lower pattern that is positive definite ('posdef') or
    has a positive definite completion ('completable'): U = P_V(sum_i u_i u_i^T) with
    u_i ~ N(0, I/n), plus the first shift t*I, t in {0.1, 0.2, 0.4, ...}, that puts it in
    the cone (``base.py:514-560``).  The cone tests run on the solver backend (the chordal
    Cholesky / completion kernels), as in the reference.  Returns values in pattern order."""
    from .chordal import cspmatrix, cholesky, completion
    if cone not in ("posdef", "completable"):
        raise ValueError("cone must be 'posdef' (default) or 'completable' ")
    rng = np.random.default_rng(seed)
    colptr = np.asarray(colptr, dtype=np.int64)
    rowind = np.asarray(rowind, dtype=np.int64)
    cols = _pattern_cols(n, colptr)
    U = np.zeros(len(rowind))
    chunk = max(1, min(n, (1 << 24) // max(n, 1)))
    for i0 in range(0, n, chunk):
        G = rng.standard_normal((n, min(chunk, n - i0))) / np.sqrt(n)
        U += np.einsum("ij,ij->i", G[rowind], G[cols])
    # embedding + symbolic for the cone test
    pm = maxcardsearch(n, colptr, rowind)
    fc, fr, _ = embed(n, colptr, rowind, pm)
    if fc[-1] != colptr[-1]:
        pm = min_degree(n, colptr, rowind)
        fc, fr, _ = embed(n, colptr, rowind, pm)
    symb = Symbolic(n, fc, fr)
    ops = solvers._make_backend(symb)
    ip = np.empty(n, dtype=np.int64)
    ip[pm] = np.arange(n, dtype=np.int64)
    pr, pc = ip[rowind], ip[cols]
    key = np.minimum(pr, pc) * n + np.maximum(pr, pc)
    vkey = symb.Jp * n + symb.Ip
    pos = np.searchsorted(vkey, key)            # Vp is CCS-sorted: keys ascending
    diag = rowind == cols
    test = cholesky if cone == "posdef" else completion
    t = 0.1
    Ut = U.copy()
    while True:
        v = np.zeros(symb.nvp)
        v[pos] = Ut
        Z = cspmatrix.from_vec(ops, v)
        try:
            test(Z)
            return Ut
        except ArithmeticError:
            Ut = U.copy()
            Ut[diag] += t
            t *= 2.0


def _band_pattern(n, bw):
    I = np.concatenate([np.arange(j, min(j + bw + 1, n)) for j in range(n)])
    J = np.concatenate([np.full(min(j + bw + 1, n) - j, j) for j in range(n)])
    return I.astype(np.int64), J.astype(np.int64)


class band_SDP(SDP):
    """Random SDP with band structure, ``band_SDP(n, m, bw, seed=0)`` (``base.py:563-636``):
    pattern {(i,j): j <= i <= j+bw}; every A_i dense on the band with N(0, 1/|V|^2) entries;
    A_0 = S0 + sum y0_i A_i and b_i = A_i . X0 with S0 > 0 and X0 completable, so a strictly
    feasible primal-dual pair is known."""

    def __init__(self, n, m, bw, seed=0):
        SDP.__init__(self)
        if type(seed) is not int:
            raise ValueError("seed must be an integer")
        self._bw = bw
        rng = np.random.default_rng(seed)
        I1, J1 = _band_pattern(n, bw)
        N = len(I1)
        Il = misc.sub2ind((n, n), I1, J1)
        diag = I1 == J1
        cp, ri = lower_pattern(n, I1, J1)
        y0 = rng.standard_normal(m)
        y0 /= np.linalg.norm(y0)
        S0 = mk_rand(n, cp, ri, "posdef", seed)
        X0 = mk_rand(n, cp, ri, "completable", seed)
        A_ = rng.standard_normal((N, m + 1)) * (1.0 / N)
        A_[:, 0] = S0 + A_[:, 1:] @ y0
        x = X0.copy()
        x[diag] *= 0.5
        self._b = 2.0 * (A_[:, 1:].T @ x)
        rows = np.tile(Il, m + 1)
        cols = np.repeat(np.arange(m + 1, dtype=np.int64), N)
        self._A = misc.as_csc(sp.csc_matrix((A_.T.reshape(-1), (rows, cols)), shape=(n * n, m + 1)))
        self._X0 = sp.csc_matrix((X0, (I1, J1)), shape=(n, n))
        self._S0 = sp.csc_matrix((S0, (I1, J1)), shape=(n, n))
        self._y0 = y0
        self._pname = "band_n%i_m%i_bw%i" % (n, m, bw)

    @property
    def bw(self):
        return self._bw


class mtxnorm_SDP(SDP):
    """Matrix-norm minimisation  min ||F(x) + G||_2  as an SDP of order n = p+q
    (``base.py:639-778``): the p x q block (rows q..n-1, columns 0..q-1) holds G (column 0,
    dense N(0,1)) and F_i (columns 1..r, ``nz = round(density*p*q)`` random positions,
    N(0,1)); the last column is -I and b = (0,...,0,-1), so m = r+1."""

    def __init__(self, p, q, r, density=1.0, seed=0):
        SDP.__init__(self)
        if type(seed) is not int:
            raise ValueError("seed must be an integer")
        # density: one float for all F_i or a list with one float per F_i (base.py:718-760)
        if type(density) is float and 0.0 < density <= 1.0:
            dens = [density] * r
        elif isinstance(density, (list, tuple)) and len(density) == r and all(0.0 < float(v) <= 1.0 for v in density):
            dens = [float(v) for v in density]
        else:
            raise TypeError("density must be a float between 0 and 1 or a list of r such floats")
        rng = np.random.default_rng(seed)
        n = p + q
        self._p, self._q = p, q
        I1 = np.tile(np.arange(q, n, dtype=np.int64), q)
        J1 = np.repeat(np.arange(q, dtype=np.int64), p)
        Il = misc.sub2ind((n, n), I1, J1)
        rows = [Il]
        cols = [np.zeros(p * q, dtype=np.int64)]
        vals = [rng.standard_normal(p * q)]
        for j in range(1, r + 1):
            nz = min(max(1, int(round(dens[j - 1] * p * q))), p * q)
            sel = Il if nz == p * q else rng.choice(Il, size=nz, replace=False)
            rows.append(sel)
            cols.append(np.full(nz, j, dtype=np.int64))
            vals.append(rng.standard_normal(nz))
        rows.append(np.arange(0, n * n, n + 1, dtype=np.int64))
        cols.append(np.full(n, r + 1, dtype=np.int64))
        vals.append(-np.ones(n))
        self._A = misc.as_csc(sp.csc_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))),
                                            shape=(n * n, r + 2)))
        self._b = np.zeros(r + 1)
        self._b[-1] = -1.0
        self._pname = "mtxnorm_p%i_q%i_r%i_d%s" % (p, q, r, density if type(density) is float else "list")


class rand_SDP(SDP):
    """Random SDP on an arbitrary pattern, ``rand_SDP(V, m, density=1.0, seed=0)``
    (``base.py:864-949``): ``V`` is an n x n sparse matrix (its lower triangle is the
    pattern); each A_i has ``nz = round(density*|V|)`` entries at random pattern positions;
    A_0 = S0 + sum y0_k A_k, b_k = A_k . X0 — strictly feasible by construction."""

    def __init__(self, V, m, density=1.0, seed=0):
        SDP.__init__(self)
        if type(seed) is not int:
            raise ValueError("seed must be an integer")
        rng = np.random.default_rng(seed)
        V = sp.tril(sp.csc_matrix(V), format="coo")
        n = V.shape[0]
        cp, ri = lower_pattern(n, V.row, V.col)
        J1 = _pattern_cols(n, cp)
        I1 = ri
        N = len(I1)
        Il = misc.sub2ind((n, n), I1, J1)
        diag = I1 == J1
        y0 = rng.standard_normal(m)
        y0 /= np.linalg.norm(y0)
        S0 = mk_rand(n, cp, ri, "posdef", seed)
        X0 = mk_rand(n, cp, ri, "completable", seed)
        # density: one float for all constraints or a list with one float per constraint
        # (``base.py:903-931``)
        if isinstance(density, float):
            nzs = [min(max(1, int(round(density * N))), N)] * m
        elif isinstance(density, (list, tuple)) and len(density) == m:
            nzs = [min(max(1, int(round(float(v) * N))), N) for v in density]
        else:
            raise TypeError("density must be a float or a list of m floats")
        pos = [np.arange(N) if nz == N else rng.choice(N, size=nz, replace=False) for nz in nzs]
        vals = [rng.standard_normal(nz) for nz in nzs]
        x = X0.copy()
        x[diag] *= 0.5
        a0 = S0.copy()
        self._b = np.empty(m)
        for j in range(m):
            np.add.at(a0, pos[j], vals[j] * y0[j])
            self._b[j] = 2.0 * np.dot(vals[j], x[pos[j]])
        pos_all = np.concatenate(pos) if m else np.zeros(0, dtype=np.int64)
        rows = np.concatenate([Il, Il[pos_all]])
        cols = np.concatenate([np.zeros(N, dtype=np.int64), np.repeat(np.arange(1, m + 1, dtype=np.int64), nzs)])
        data = np.concatenate([a0] + vals)
        self._A = misc.as_csc(sp.csc_matrix((data, (rows, cols)), shape=(n * n, m + 1)))
        self._X0 = sp.csc_matrix((X0, (I1, J1)), shape=(n, n))
        self._S0 = sp.csc_matrix((S0, (I1, J1)), shape=(n, n))
        self._y0 = y0
        self._pname = "rand_n%i_m%i" % (n, m)


class maxcut_SDP(SDP):
    """Max-cut relaxation  min C.X  s.t. X_ii = 1, X >= 0  with C = -(1/4) Laplacian of a
    graph given by its edge list (the SDPLIB ``maxG*``/``mcp*`` family the reference
    benchmarks read from ``dat-s`` files; ``doc/source/benchmarks/index.rst``)."""

    def __init__(self, n, edges, weights=None):
        SDP.__init__(self)
        edges = np.asarray(edges, dtype=np.int64).reshape(-1, 2)
        e = edges[edges[:, 0] != edges[:, 1]]
        i = np.maximum(e[:, 0], e[:, 1])
        j = np.minimum(e[:, 0], e[:, 1])
        w = np.ones(len(e)) if weights is None else np.asarray(weights, dtype=np.float64)
        Lap = sp.coo_matrix((np.concatenate([-w, w, w]),
                             (np.concatenate([i, i, j]), np.concatenate([j, i, j]))), shape=(n, n)).tocsc()
        Lap.sum_duplicates()
        C = (-0.25 * sp.tril(Lap)).tocoo()
        d = np.arange(n, dtype=np.int64)
        rows = np.concatenate([misc.sub2ind((n, n), C.row, C.col), d * (n + 1)])
        cols = np.concatenate([np.zeros(len(C.row), dtype=np.int64), d + 1])
        vals = np.concatenate([C.data, np.ones(n)])
        self._A = misc.as_csc(sp.csc_matrix((vals, (rows, cols)), shape=(n * n, n + 1)))
        self._b = np.ones(n)
        self._pname = "maxcut_n%i" % n

    def cut(self, sol, trials=256, seed=0, local_search=False, tabu_iters=0):
        """A cut from a solution of the relaxation by Goemans-Williamson rounding (``SDP.round_pm1``):
        returns ``(x, weight, bound)`` with the +-1 vector x of the heaviest of ``trials`` random hyperplane
        cuts, its weight (= -C . x x^T) and the certified upper bound -``sol['dual objective']`` on every
        cut's weight.  ``local_search=True`` improves every cut by single-vertex moves first (one-flip local
        search, see ``SDP.local_search_pm1``) and returns the heaviest improved cut.  ``tabu_iters > 0`` then
        runs that many moves of tabu search on every cut (``SDP.tabu_search_pm1``, default tenure) and returns
        the heaviest cut it visited."""
        r = self.round_pm1(sol, trials=trials, seed=seed, local_search=local_search, tabu_iters=tabu_iters)
        return r["x"], -r["value"], -float(sol["dual objective"])


def _chordal_embedding(X):
    """``symbolic`` of the pattern of the sparse symmetric ``X`` (lower triangle used) under a fill-reducing ordering
    (maximum cardinality search when it adds no fill, else minimum degree).  Returns ``(symb, p, full)``: the symbolic,
    the ordering (vertex p[k] is the k-th of the embedding) and X with both triangles as CSR."""
    X = sp.tril(sp.csc_matrix(X), format="coo")
    n = X.shape[0]
    cp, ri = lower_pattern(n, X.row, X.col)
    p = maxcardsearch(n, cp, ri)
    fc, fr, _ = embed(n, cp, ri, p)
    if fc[-1] != cp[-1]:
        p = min_degree(n, cp, ri)
        fc, fr, _ = embed(n, cp, ri, p)
    lo = sp.tril(X, format="csc")
    return Symbolic(n, fc, fr), p, (lo + sp.tril(lo, -1).T).tocsr()


def _completion_factor(X):
    """``symbolic`` of the pattern of ``X`` (``_chordal_embedding``) and ``chompack.completion`` on the backend: returns
    the factor L (a cspmatrix, P_V((L L^T)^-1) = X) and ``order``, the original vertex at each internal position.  Raises
    ``ArithmeticError`` if X has no positive definite completion."""
    from .chordal import cspmatrix
    from . import chordal
    symb, p, full = _chordal_embedding(X)
    ops = solvers._make_backend(symb)
    L = cspmatrix.from_vec(ops, np.asarray(full[p[symb.Ip], p[symb.Jp]]).ravel())
    chordal.completion(L)                       # ArithmeticError if X has no PD completion
    return L, p[symb.perm]                      # internal order: vertex p[perm[i]] at position i


_LOWRANK_MAX_RANK = 512
_U = 2.0 ** -53                                 # unit roundoff of IEEE double


def _gamma(k):
    """gamma_k = k u / (1 - k u) (Higham, Accuracy and Stability of Numerical Algorithms, 3.1)."""
    return k * _U / (1.0 - k * _U)


def _lowrank_delta(n, sdiag_abs, t):
    """Backward-error margin delta(t) of a probe of ``_lowrank_certificate`` that factors M = fl(S + (t - delta) I).

    If floating-point Cholesky runs to completion on a symmetric M of order n, the computed factor satisfies
    L L^T = M + dM with |dM| <= gamma_{n+1} |L| |L^T| (Higham, Thm 10.3; any order of the inner sums, blocked and
    supernodal included, FMA or not), and ||l_i||^2 <= M_ii / (1 - gamma_{n+1}) from the diagonal equation.  Hence
    ||dM||_2 <= gamma_{n+1} sum_i ||l_i||^2 <= alpha tr(M) with alpha = gamma_{n+1} / (1 - gamma_{n+1}), and
    lambda_min(M) >= -alpha tr(M) (Rump, "Verification of positive definiteness", BIT 46 (2006), Lemma 2.1 and
    Theorem 2.3; no underflow term is needed at these magnitudes).  M differs from the exact S + (t - delta) I only on
    the diagonal, by at most 2u |M_ii| (the rounded t - delta and the rounded sum), and the rounded S_ii = fl(C_ii - y_i)
    differs from the exact C_ii - y_i by at most u |S_ii|.  With |M_ii| <= (|S_ii| + |t|)(1 + 2u) this gives

        lambda_min(C - Diag(y) + t I) >= delta - alpha sum_i (|S_ii| + |t|)(1 + 2u) - 3u (1 + 2u) max_i (|S_ii| + |t|),

    so delta = (1 + 1e-6) (alpha sum_i (|S_ii| + |t|) + 3u max_i (|S_ii| + |t|)) makes a successful probe prove
    C - Diag(y) + t I >= 0; the factor 1 + 1e-6 covers 2u and the rounding of this evaluation."""
    alpha = _gamma(n + 1) / (1.0 - _gamma(n + 1))
    a = sdiag_abs + abs(t)
    return (1.0 + 1e-6) * (alpha * float(a.sum()) + 3.0 * _U * float(a.max()))


def _lowrank_certificate(n, I, J, v, y, b, f):
    """The smallest shift t >= 0 (up to the bisection tolerance) with C - Diag(y) + t I >= 0 proven, and the number of
    Cholesky probes spent.  S = C - Diag(y) lives on the chordal embedding of C's pattern (``_chordal_embedding``); a
    probe at t factors S + (t - delta(t)) I (``_lowrank_delta``) with the backend's chordal ``cholesky``, and its
    success proves S + t I >= 0.  t = 0 is probed first; otherwise the bracket [0, t_hi] starts from the Gershgorin
    shift max_i (sum_{j != i} |S_ij| - S_ii) plus a margin, and is halved until (t_hi - t_lo) sum(b) <= 1e-6 max(1, |f|).
    Returns t_hi, the upper end: a probe at it succeeded."""
    from .chordal import cspmatrix, cholesky
    S = sp.coo_matrix((np.concatenate([v, -y]), (np.concatenate([I, np.arange(n)]), np.concatenate([J, np.arange(n)]))),
                      shape=(n, n))
    symb, p, full = _chordal_embedding(S)
    ops = solvers._make_backend(symb)
    sv = np.asarray(full[p[symb.Ip], p[symb.Jp]]).ravel()
    dpos = symb.diag_vec
    sdiag = sv[dpos]
    sabs = np.abs(sdiag)
    probes = 0

    def ok(t):
        nonlocal probes
        probes += 1
        w = sv.copy()
        w[dpos] = sdiag + (t - _lowrank_delta(n, sabs, t))
        try:
            cholesky(cspmatrix.from_vec(ops, w))
            return True
        except ArithmeticError:
            return False

    if ok(0.0):
        return 0.0, probes
    Sf = full.tocoo()
    offd = np.zeros(n)
    np.add.at(offd, Sf.row[Sf.row != Sf.col], np.abs(Sf.data[Sf.row != Sf.col]))
    g = max(0.0, float((offd - full.diagonal()).max()))
    lo, hi = 0.0, g + 4.0 * _lowrank_delta(n, sabs, g) + 1e-12 * max(1.0, g)
    while not ok(hi):
        lo, hi = hi, 2.0 * hi
    tol = 1e-6 * max(1.0, abs(f)) / float(b.sum())
    while hi - lo > tol:
        mid = 0.5 * (lo + hi)
        if ok(mid):
            hi = mid
        else:
            lo = mid
    return hi, probes


def completion(X):
    """Maximum-determinant positive definite completion of the sparse symmetric matrix ``X``
    (lower triangle used) as a dense n x n array; raises ``ArithmeticError`` if none exists
    (``base.py:952-973``: ``symbolic`` under a fill-reducing ordering, ``chompack.completion``,
    then two ``chompack.trsm`` on the identity: X_hat = L^{-T} L^{-1})."""
    L, order = _completion_factor(X)
    n = len(order)
    Z = L.ops.trsm(L.buf, np.eye(n), "N")
    Z = L.ops.trsm(L.buf, Z, "T")
    out = np.empty((n, n))
    out[np.ix_(order, order)] = Z
    return out


def _check_seed(seed):
    if isinstance(seed, bool) or not isinstance(seed, (int, np.integer)):
        raise TypeError("seed must be an integer")
    if not 0 <= int(seed) < 1 << 64:
        raise ValueError("seed must be in [0, 2**64)")
    return int(seed)


def _check_count(k, name, lo):
    if isinstance(k, bool) or not isinstance(k, (int, np.integer)) or int(k) < lo:
        raise ValueError("%s must be an integer >= %d" % (name, lo))
    return int(k)


def _tabu_tenure(n):
    """The default tabu tenure of an n-vertex search."""
    return min(n - 1, 10 + n // 100)


def _check_tol(tol):
    if isinstance(tol, bool) or not isinstance(tol, (int, float, np.integer, np.floating)):
        raise TypeError("tol must be a real number")
    if not (np.isfinite(tol) and tol >= 0):
        raise ValueError("tol must be finite and >= 0")
    return float(tol)


def _check_pm1(x, n):
    """x as a (k, n) int8 array, k >= 1, for x of shape (n,) or (k, n) holding integers +-1 only."""
    a = np.asarray(x)
    if a.dtype == bool or a.dtype.kind not in "iu":
        raise TypeError("x must be an integer array")
    if a.ndim not in (1, 2) or a.shape[-1] != n or a.size == 0:
        raise ValueError("x must have shape (%d,) or (k, %d) with k >= 1, got %s" % (n, n, a.shape))
    if not np.all((a == 1) | (a == -1)):
        raise ValueError("x must hold +-1 only")
    return np.ascontiguousarray(a.reshape(-1, n), dtype=np.int8)


def completion_sample(X, k, seed=0):
    """``k`` Gaussian samples whose covariance is the maximum-determinant positive definite completion X_hat
    of the sparse symmetric matrix ``X`` (lower triangle used), as an n x k array in the original order
    (an extension: the reference has no sampling).  With L from ``chompack.completion``, X_hat = L^-T L^-1,
    so column j is L^-T g_j: one chordal triangular solve, nothing dense of size n x n.  g_j is the standard
    normal vector of sample j under ``seed`` (Philox4x64-10 and Box-Muller; entry i depends on (seed, j, i)
    only).  Raises ``ArithmeticError`` where ``completion`` does."""
    k = _check_count(k, "k", 0)
    seed = _check_seed(seed)
    L, order = _completion_factor(X)
    out = np.empty((len(order), k))
    out[order] = L.ops.completion_sample(L.buf, k, seed)
    return out
