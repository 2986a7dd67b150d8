"""Goemans-Williamson rounding on the CPU oracle: ``OracleBackend`` with the two methods the rounding needs
(``completion_sample``, ``round_pm1``), in NumPy, with the same counter-based normals as the device
(Philox4x64-10 with key (seed, 0) and counter (i // 4, j, 0, 0), Box-Muller on pairs of 53-bit uniforms)."""
import numpy as np

from oracle import supernodal as sn
from oracle.backend import OracleBackend

_M32 = np.uint64(0xFFFFFFFF)
_PM0, _PM1 = np.uint64(0xD2E7470EE14C6C93), np.uint64(0xCA5A826395121157)
_PW0, _PW1 = np.uint64(0x9E3779B97F4A7C15), np.uint64(0xBB67AE8584CAA73B)


def _mulhilo(a, b):
    """(high, low) 64-bit halves of the 128-bit products a * b (elementwise, uint64)."""
    s32 = np.uint64(32)
    al, ah = a & _M32, a >> s32
    bl, bh = b & _M32, b >> s32
    p0, p1, p2, p3 = al * bl, al * bh, ah * bl, ah * bh
    mid = (p0 >> s32) + (p1 & _M32) + (p2 & _M32)
    return p3 + (p1 >> s32) + (p2 >> s32) + (mid >> s32), a * b


def philox4x64(ctr, key):
    """Philox4x64-10 of the counters ``ctr`` (uint64, shape (..., 4)) under ``key`` = (k0, k1)."""
    c = [np.array(ctr[..., q], dtype=np.uint64) for q in range(4)]
    k0 = np.full(c[0].shape, key[0], dtype=np.uint64)
    k1 = np.full(c[0].shape, key[1], dtype=np.uint64)
    with np.errstate(over="ignore"):
        for rnd in range(10):
            if rnd:
                k0, k1 = k0 + _PW0, k1 + _PW1
            hi0, lo0 = _mulhilo(_PM0, c[0])
            hi1, lo1 = _mulhilo(_PM1, c[2])
            c = [hi1 ^ c[1] ^ k0, lo1, hi0 ^ c[3] ^ k1, lo0]
    return np.stack(c, axis=-1)


def normals(n, k, seed, col0=0):
    """n x k standard normals: entry i of column c is entry i of sample col0 + c under ``seed``."""
    nr = -(-n // 4)
    ctr = np.zeros((nr, k, 4), dtype=np.uint64)
    ctr[..., 0] = np.arange(nr, dtype=np.uint64)[:, None]
    ctr[..., 1] = np.arange(col0, col0 + k, dtype=np.uint64)[None, :]
    w = philox4x64(ctr, (np.uint64(seed), np.uint64(0)))
    u = ((w >> np.uint64(11)).astype(np.float64) + 0.5) * 2.0 ** -53
    z = np.empty((nr, 4, k))
    for q in (0, 2):
        r = np.sqrt(-2.0 * np.log(u[..., q]))
        z[:, q] = r * np.cos(2.0 * np.pi * u[..., q + 1])
        z[:, q + 1] = r * np.sin(2.0 * np.pi * u[..., q + 1])
    return z.reshape(4 * nr, k)[:n]


def pm1_values(V, crow, ccol, cval):
    """values[t] = sum_q c_q s[r_q, t] s[c_q, t] (x2 off the diagonal) with s = sign(V), sign(0) = +1."""
    s = np.where(V < 0.0, -1.0, 1.0)
    coef = np.where(crow == ccol, 1.0, 2.0) * cval
    return (coef[:, None] * s[crow] * s[ccol]).sum(axis=0)


class RoundingOracleBackend(OracleBackend):

    def completion_sample(self, Lbuf, k, seed, col0=0):
        """L^-T g_{col0 + c}, c = 0..k-1: n x k, rows in the internal order."""
        B = normals(self.symb.n, k, seed, col0)
        sn.trsm(self.symb, Lbuf, B, "T")
        return B

    def round_pm1(self, Lbuf, crow, ccol, cval, trials, seed, chunk=0):
        V = self.completion_sample(Lbuf, trials, seed)
        values = pm1_values(V, np.asarray(crow), np.asarray(ccol), np.asarray(cval, dtype=np.float64))
        best = int(np.argmin(values))
        x = np.where(V[:, best] < 0.0, -1, 1).astype(np.int8)
        return values, x, best
