"""Low-rank solve of max-cut-type SDPs (``SDP.solve_lowrank``) and rounding from its factor (``SDP.round_pm1`` on a
solution holding ``V``).  On the CPU: the NumPy twin (tests/lowrank_oracle.py) against a vertex-by-vertex restatement
of the definition, the colouring, monotone objective, the start, the certificate against dense eigenvalues and the
twin's bounds against the interior-point optimum, argument validation.  On the device: V, the objective history, y,
sweeps and colours bitwise against the twin, grouping independence, ABI errors, the certificate on the device Cholesky,
and rounding from V against the twin evaluation and the standalone searches."""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse as sp

from local_search_oracle import eval_values, search_rows
from lowrank_oracle import LowrankOracleBackend, colouring, diag_sums, lowrank_solve, objective, start, warp_sum
from rounding_oracle import normals
from test_local_search import _entries, _graph


def _twin():
    from smcp_b200 import solvers
    solvers.set_backend_factory(lambda symb: LowrankOracleBackend(symb))


def _device():
    from smcp_b200 import solvers
    solvers.set_backend_factory(None)


@pytest.fixture(autouse=True)
def _restore_backend():
    yield
    from smcp_b200 import solvers
    solvers.set_backend_factory(None)


def _family(n, fam, seed):
    """Objective entries (row, col, value) of a test graph: the one-flip tests' 'sparse' / 'hub' families with unit or
    real weights, a star (hub of degree n - 1), 'isolated' (edges among the first half only) and 'negdup' (negative
    and duplicate weights)."""
    rng = np.random.default_rng(seed)
    if fam in ("sparse-unit", "sparse-real", "hub-unit", "hub-real"):
        s, w = fam.split("-")
        return _entries(n, s, w, seed)
    if fam == "star":
        o = np.arange(1, n, dtype=np.int64)
        return o, np.zeros(n - 1, dtype=np.int64), -np.ones(n - 1)
    if fam == "isolated":
        m = max(1, n // 2)
        r, c = rng.integers(0, m, 2 * n), rng.integers(0, m, 2 * n)
        k = r != c
        return np.maximum(r[k], c[k]), np.minimum(r[k], c[k]), rng.standard_normal(int(k.sum()))
    if fam == "negdup":
        r, c = rng.integers(0, n, 3 * n), rng.integers(0, n, 3 * n)
        r, c = np.concatenate([r, r[: n]]), np.concatenate([c, c[: n]])
        return np.maximum(r, c), np.minimum(r, c), -np.abs(rng.standard_normal(len(r))) - 0.1
    raise ValueError(fam)


def _b(n, kind, seed):
    return np.ones(n) if kind == "unit" else 0.5 + np.random.default_rng(seed).random(n) * 2.0


def _slow(n, crow, ccol, cval, b, G, sweeps):
    """The definition, one vertex at a time in colour order, scalar arithmetic."""
    rp, col, val = search_rows(n, crow, ccol, cval)
    colour = colouring(n, rp, col)
    r = G.shape[1]

    def wsum(t):
        lanes = [0.0] * 32
        for c, x in enumerate(t):
            lanes[c % 32] = lanes[c % 32] + x
        for o in (16, 8, 4, 2, 1):
            lanes = [lanes[l] + lanes[l ^ o] for l in range(32)]
        return lanes[0]

    def w(V, i):
        out = [0.0] * r
        for p in range(rp[i], rp[i + 1]):
            for c in range(r):
                out[c] = out[c] + float(val[p]) * V[col[p]][c]
        return out

    V = [list(map(float, g)) for g in G]
    for i in range(n):
        ss = wsum([x * x for x in V[i]])
        if ss > 0.0:
            a = float(np.sqrt(b[i])) / float(np.sqrt(ss))
            V[i] = [a * x for x in V[i]]
    for _ in range(sweeps):
        for c in range(int(colour.max()) + 1):
            for i in range(n):
                if colour[i] != c:
                    continue
                wi = w(V, i)
                ss = wsum([x * x for x in wi])
                if ss > 0.0:
                    a = -float(np.sqrt(b[i])) / float(np.sqrt(ss))
                    V[i] = [a * x for x in wi]
    return np.array(V)


# ---------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,r,fam", [(1, 3, "star"), (7, 1, "sparse-real"), (25, 5, "hub-unit"), (30, 33, "negdup"),
                                     (40, 70, "isolated")])
def test_twin_matches_vertex_by_vertex_definition(n, r, fam):
    crow, ccol, cval = _family(n, fam, n)
    b = _b(n, "real", n)
    G = normals(r, n, 3).T
    for sweeps in (0, 1, 3):
        V, f, y, k, _, _ = lowrank_solve(n, crow, ccol, cval, b, r, 3, sweeps, 0.0, G=G)
        if k == sweeps:
            assert np.array_equal(V, _slow(n, crow, ccol, cval, b, G, sweeps))
    rp, col, val = search_rows(n, crow, ccol, cval)
    f0, e = objective(V, rp, col, val, diag_sums(n, crow, ccol, cval), b)
    assert f0 == f[-1] and np.array_equal(y, e / b)


@pytest.mark.parametrize("fam", ["sparse-unit", "hub-real", "star", "isolated", "negdup"])
def test_colouring_is_proper_and_greedy(fam):
    n = 300
    rp, col, _ = search_rows(n, *_family(n, fam, 5))
    colour = colouring(n, rp, col)
    for i in range(n):
        nb = col[rp[i]:rp[i + 1]]
        assert (colour[nb] != colour[i]).all()
        lower = set(colour[nb[nb < i]].tolist())
        assert colour[i] not in lower and all(c in lower for c in range(colour[i]))


@pytest.mark.parametrize("fam", ["sparse-real", "hub-unit", "negdup"])
@pytest.mark.parametrize("r", [1, 4, 20])
def test_objective_never_rises(fam, r):
    n = 200
    crow, ccol, cval = _family(n, fam, 11)
    _, f, _, k, _, _ = lowrank_solve(n, crow, ccol, cval, _b(n, "real", 2), r, 0, 60, 0.0)
    assert k >= 1
    assert (np.diff(f) <= 1e-12 * np.abs(f[:-1]).max()).all(), np.diff(f).max()


def test_max_sweeps_zero_returns_normalised_start():
    _twin()
    n, r = 50, 9
    P = _graph(n, 3 * n, 4)
    sol = P.solve_lowrank(rank=r, seed=5, max_sweeps=0, bound=False)
    G = normals(r, n, 5).T
    assert sol["sweeps"] == 0 and len(sol["objective history"]) == 1 and not sol["converged"]
    assert np.array_equal(sol["V"], start(G, np.ones(n)))
    assert np.abs(np.linalg.norm(sol["V"], axis=1) - 1.0).max() < 1e-14
    assert sol["dual objective"] is None and sol["gap"] is None
    assert abs(sol["x"].diagonal() - 1.0).max() < 1e-14


def _dense_C(P):
    I, J, v = P._objective_entries()
    C = np.zeros((P.n, P.n))
    np.add.at(C, (I, J), v)
    np.add.at(C, (J[I != J], I[I != J]), v[I != J])
    return C


@pytest.mark.parametrize("n,seed", [(12, 1), (25, 2), (40, 3)])
def test_certificate_against_dense_eigenvalues(n, seed):
    from smcp_b200.base import _lowrank_delta
    _twin()
    P = _graph(n, 3 * n, seed)
    sol = P.solve_lowrank(rank=3, max_sweeps=8, tol=0.0)           # far from optimal: t > 0
    C = _dense_C(P)
    y = sol["y"]                                                    # constraint k is X_kk: vertex order
    lam = np.linalg.eigvalsh(C - np.diag(y))[0]
    assert lam >= -1e-12 * max(1.0, np.abs(C).max())
    t = sol["shift"]
    lam0 = np.linalg.eigvalsh(C - np.diag(y + t))[0]
    S = C - np.diag(y + t)
    dmax = _lowrank_delta(n, np.abs(np.diag(S)), t)
    btol = 1e-6 * max(1.0, abs(sol["primal objective"])) / n
    assert t >= -lam0 - 1e-12
    assert t <= max(0.0, -lam0) + btol + dmax + 1e-12
    b = P.b
    assert sol["dual objective"] <= float(b @ y) + 1e-9 and sol["dual objective"] <= sol["primal objective"]
    assert sol["probes"] >= 1


LOWRANK_GAP = 1e-5      # relative gap (f - bound) / max(1, |f|) the low-rank solve reaches on the small instances


@pytest.mark.parametrize("n,seed", [(8, 0), (15, 1), (22, 2), (30, 3)])
def test_twin_brackets_interior_point_optimum(n, seed):
    from smcp_b200 import solvers
    _twin()
    solvers.options["show_progress"] = False
    P = _graph(n, 2 * n, seed)
    ipm = P.solve_feas(primalstart={"x": sp.identity(n, format="csc")})
    assert ipm["status"] == "optimal"
    sol = P.solve_lowrank(tol=1e-12, max_sweeps=5000)
    f, lb = sol["primal objective"], sol["dual objective"]
    p_ipm, d_ipm = ipm["primal objective"], ipm["dual objective"]
    assert lb <= p_ipm + 1e-9 * abs(p_ipm)
    assert f >= d_ipm - 1e-9 * abs(d_ipm)
    assert (f - lb) / max(1.0, abs(f)) <= LOWRANK_GAP, (f, lb)


def test_form_and_argument_validation():
    import smcp_b200 as S
    _twin()
    P = _graph(10, 20, 0)
    for bad in (dict(rank=0), dict(rank=513), dict(tol=-1.0), dict(max_sweeps=-1), dict(tol=float("nan"))):
        with pytest.raises((ValueError, TypeError)):
            P.solve_lowrank(**bad)
    n = 4
    C = sp.coo_matrix(([-1.0], ([1], [0])), shape=(n, n))
    rows0 = list(C.row * n + C.col)
    d = np.arange(n)

    def sdp(rows, cols, vals, b):
        return S.SDP(sp.csc_matrix((vals, (rows, cols)), shape=(n * n, n + 1)), b)

    ok = sdp(rows0 + list(d * (n + 1)), [0] + list(d + 1), [-1.0] + [1.0] * n, np.ones(n))
    assert ok.solve_lowrank(rank=2, max_sweeps=3)["sweeps"] >= 1
    offdiag = list(d * (n + 1))
    offdiag[2] = 1 * n + 0                                            # constraint 3 at (1, 0)
    with pytest.raises(ValueError):
        sdp(rows0 + offdiag, [0] + list(d + 1), [-1.0] + [1.0] * n, np.ones(n)).solve_lowrank()
    dup = list(d * (n + 1))
    dup[3] = 0                                                        # two constraints on X_00
    with pytest.raises(ValueError):
        sdp(rows0 + dup, [0] + list(d + 1), [-1.0] + [1.0] * n, np.ones(n)).solve_lowrank()
    with pytest.raises(ValueError):
        sdp(rows0 + list(d * (n + 1)), [0] + list(d + 1), [-1.0] + [1.0] * n, np.array([1.0, 0.0, 1.0, 1.0])).solve_lowrank()
    with pytest.raises(ValueError):
        sdp(rows0 + list(d * (n + 1)), [0] + list(d + 1), [-1.0] + [2.0] * n, np.ones(n)).solve_lowrank()
    with pytest.raises(ValueError):
        S.band_SDP(8, 3, 1).solve_lowrank()


# ---------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------
def _device_normals(r, n, seed):
    """The device's raw normals (n x r, row i = sample i): samples of the identity's completion, L = I."""
    import smcp_b200 as S
    return S.completion_sample(sp.identity(r, format="csc"), n, seed).T.copy()


def _run_device(n, crow, ccol, cval, b, r, seed, max_sweeps, tol):
    from smcp_b200 import solvers
    from smcp_b200.symbolic import Symbolic
    ops = solvers._make_backend(Symbolic(n, np.arange(n + 1), np.arange(n)))
    return ops.lowrank_solve(crow, ccol, cval, b, r, seed, max_sweeps, tol)


_GPU_CASES = [
    (1, 1, "star", "unit"), (2, 2, "sparse-real", "unit"), (33, 31, "hub-unit", "real"), (33, 32, "star", "unit"),
    (33, 33, "negdup", "real"), (257, 512, "isolated", "unit"), (257, 200, "sparse-unit", "real"),
    (1000, 1, "hub-real", "unit"), (1000, 33, "star", "real"), (1000, 200, "negdup", "unit"),
    (5000, 32, "sparse-real", "real"), (5000, 512, "isolated", "unit"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("n,r,fam,bk", _GPU_CASES)
def test_device_matches_twin(n, r, fam, bk):
    _device()
    crow, ccol, cval = _family(n, fam, n + r)
    b = _b(n, bk, n)
    G = _device_normals(r, n, 9)
    max_sweeps = 20 if n * r > 100000 else 60
    V, f, y, sweeps, colors = _run_device(n, crow, ccol, cval, b, r, 9, max_sweeps, 1e-6)
    Vt, ft, yt, st, ct, _ = lowrank_solve(n, crow, ccol, cval, b, r, 9, max_sweeps, 1e-6, G=G)
    assert (sweeps, colors) == (st, ct)
    assert np.array_equal(V, Vt) and np.array_equal(f, ft) and np.array_equal(y, yt)


@pytest.mark.gpu
def test_device_grouping_independent_and_tol_zero():
    _device()
    n, r = 1000, 2
    crow, ccol, cval = _family(n, "sparse-real", 3)
    b = _b(n, "real", 3)
    G = _device_normals(r, n, 1)
    Vl, fl, yl, sl, _ = _run_device(n, crow, ccol, cval, b, r, 1, 40, 0.0)
    assert sl == 40
    for ms in (0, 15, 16, 17, 33):
        V, f, y, s, _ = _run_device(n, crow, ccol, cval, b, r, 1, ms, 0.0)
        Vt, ft, yt, st, _, _ = lowrank_solve(n, crow, ccol, cval, b, r, 1, ms, 0.0, G=G)
        assert s == ms == st
        assert np.array_equal(f, fl[:ms + 1]) and np.array_equal(f, ft)
        assert np.array_equal(V, Vt) and np.array_equal(y, yt)


@pytest.mark.gpu
def test_device_abi_errors():
    from smcp_b200.device import Context, _i64
    ctx = Context.get()
    lib = ctx.lib
    n = 4
    crow, ccol, cval = _i64([1, 2]), _i64([0, 1]), np.array([-1.0, -1.0])
    b = np.ones(n)
    V, f, y = np.empty((n, 512)), np.empty(4), np.empty(n)
    s, c = C.c_int64(), C.c_int64()

    def call(r=2, bb=b, ms=3, tol=1e-6, rows=crow):
        return lib.smcp_lowrank_solve(ctx.h, n, r, len(cval), rows, ccol, cval, bb, 0, ms, tol, V, f, y, C.byref(s), C.byref(c))

    assert call() == 0
    for rc in (call(r=0), call(r=513), call(bb=np.array([1.0, 0.0, 1.0, 1.0])), call(bb=np.array([1.0, np.inf, 1.0, 1.0])),
               call(ms=-1), call(tol=-1e-3), call(tol=float("nan")), call(rows=_i64([1, 4]))):
        assert rc == -2
    assert lib.smcp_round_pm1_factor(ctx.h, n, 0, V, 0, 8, 0, len(cval), crow, ccol, cval, 0, 1e-12, 0, 0, None, None,
                                     np.empty(8), np.empty(n, dtype=np.int8), C.byref(s), None, None, None) == -2
    bufs = [np.empty(8), np.empty(8)] + [np.zeros(8, dtype=np.int64) for _ in range(3)]
    p = [a.ctypes.data for a in bufs]
    assert lib.smcp_round_pm1_factor(ctx.h, n, 2, V, 0, 8, 0, len(cval), crow, ccol, cval, 0, 1e-12, 5, 9000, p[0], p[1],
                                     np.empty(8), np.empty(n, dtype=np.int8), C.byref(s), p[2], p[3], p[4]) == -2


@pytest.mark.gpu
def test_device_certificate_matches_oracle():
    _device()
    P = _graph(300, 900, 7)
    dev = P.solve_lowrank(rank=4, max_sweeps=10, tol=0.0)
    dev_cert = (dev["shift"], dev["dual objective"])
    _twin()
    from smcp_b200.base import _lowrank_certificate
    I, J, v = P._objective_entries()
    y = dev["y"] + dev["shift"]
    t, _ = _lowrank_certificate(P.n, I, J, v, y, np.ones(P.n), dev["primal objective"])
    btol = 1e-6 * max(1.0, abs(dev["primal objective"])) / P.n
    assert abs(t - dev_cert[0]) <= 2 * btol + 1e-9
    assert dev_cert[1] <= dev["primal objective"]


def _rounded_signs(V, trials, seed):
    Z = V @ _device_normals(V.shape[1], trials, seed).T
    return Z, np.where(Z < 0.0, -1, 1).astype(np.int8).T


@pytest.mark.gpu
@pytest.mark.parametrize("n,r", [(257, 33), (2000, 64)])
def test_round_from_factor(n, r):
    _device()
    P = _graph(n, 3 * n, n)
    sol = P.solve_lowrank(rank=r, max_sweeps=30, bound=False)
    V = sol["V"]
    trials = 300
    Z, X0 = _rounded_signs(V, trials, 4)
    I, J, v = P._objective_entries()
    clear = (np.abs(Z) > 1e-9).all(axis=0)                 # trials whose signs cannot depend on the product's order
    assert clear.sum() >= trials // 2
    plain = P.round_pm1(sol, trials=trials, seed=4)
    ref = eval_values(X0, I, J, v)
    assert np.array_equal(plain["values"][clear], ref[clear])
    if clear[plain["trial"]]:
        assert np.array_equal(plain["x"], X0[plain["trial"]])
    ls = P.round_pm1(sol, trials=trials, seed=4, local_search=True)
    assert np.array_equal(ls["values_rounded"], plain["values"])
    one = P.local_search_pm1(X0)
    assert np.array_equal(ls["values"][clear], one["values"][clear]) and np.array_equal(ls["flips"][clear], one["flips"][clear])
    tb = P.round_pm1(sol, trials=trials, seed=4, local_search=True, tabu_iters=n)
    two = P.tabu_search_pm1(one["x"], n)
    assert np.array_equal(tb["values_before_tabu"][clear], one["values"][clear])
    assert np.array_equal(tb["values"][clear], two["values"][clear]) and np.array_equal(tb["moves"][clear], two["moves"][clear])
    for chunk in (64, 256, 0):
        for kw, res in ((dict(), plain), (dict(local_search=True, tabu_iters=n), tb)):
            o = P.round_pm1(sol, trials=trials, seed=4, chunk=chunk, **kw)
            assert np.array_equal(o["values"], res["values"]) and np.array_equal(o["x"], res["x"])


@pytest.mark.gpu
def test_cut_from_lowrank():
    from test_rounding import _brute_max_cut
    _device()
    P = _graph(10, 20, 2)
    sol = P.solve_lowrank()
    assert sol["converged"] and sol["gap"] >= 0
    x, w, ub = P.cut(sol, local_search=True)
    assert w == _brute_max_cut(P) and w <= ub + 1e-9
    P = _graph(3000, 9000, 1)
    sol = P.solve_lowrank()
    x, w, ub = P.cut(sol, local_search=True)
    assert w <= ub and (sol["primal objective"] - sol["dual objective"]) / abs(sol["primal objective"]) < 1e-3
