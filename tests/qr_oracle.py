"""The Q-form of kktsolver='qr' on the CPU oracle: ``OracleBackend`` with the two methods the Householder form
needs (``schur_factor_householder``, ``qr_solve``), in NumPy / LAPACK.  The oracle's own ``schur_factor_qr``
(R of Zw only, the solve through Z) is left as it is."""
import numpy as np
import scipy.linalg as sl

from oracle import supernodal as sn
from oracle.backend import OracleBackend


class QROracleBackend(OracleBackend):

    def schur_factor_householder(self, hf):
        """Zw = Q1 R with diag(R) >= 0 (the matching columns of Q1 change sign); Hf = R^T."""
        symb, Av, m = self.symb, self.Av, self.m
        Z = np.zeros((m, symb.nblk))
        for j in range(m):
            c0, c1 = Av.indptr[j], Av.indptr[j + 1]
            Z[j, symb.vec2blk[Av.indices[c0:c1]]] = Av.data[c0:c1]
        sn.hessian_half(hf, Z, False, False)
        self.Zw = (Z * np.sqrt(symb.wdot)[None, :]).T.copy()
        Q1, R = np.linalg.qr(self.Zw)
        s = np.where(np.diag(R) < 0.0, -1.0, 1.0)
        R = R * s[:, None]
        Q1 = Q1 * s[None, :]
        if not np.all(np.isfinite(R)):
            raise ArithmeticError("Z is rank deficient")
        d = np.diag(R)
        bad = np.flatnonzero(~(d > 1e-14 * d.max()))
        if bad.size:
            raise ArithmeticError("Z is rank deficient (info=%d)" % (bad[0] + 1))
        self.Q1 = Q1
        self.Hf = np.ascontiguousarray(R.T)
        self.H = None

    def qr_solve(self, g, r):
        """gw = sqrt(w) g, v = R^-T r + Q1^T gw, y = R^-1 v, x = (Q1 v - gw) / sqrt(w) (-g where w = 0)."""
        w = np.sqrt(self.symb.wdot)
        g = np.asarray(g, dtype=np.float64)
        gw = w * g
        a = sl.solve_triangular(self.Hf, np.asarray(r, dtype=np.float64).ravel(), lower=True, check_finite=False)
        v = a + self.Q1.T @ gw
        y = sl.solve_triangular(self.Hf, v, lower=True, trans="T", check_finite=False)
        x = np.divide(self.Q1 @ v - gw, w, out=-g.copy(), where=w > 0)
        return y, x
