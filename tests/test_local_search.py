"""One-flip local search of +-1 vectors (``SDP.local_search_pm1``, ``SDP.round_pm1(local_search=True)``,
``maxcut_SDP.cut(local_search=True)``).  On the CPU: the NumPy twin (tests/local_search_oracle.py) ends at a one-flip
local optimum without raising f, keeps brute-force optima, honours max_flips; argument validation.  On the device:
flips, signs and values bitwise against the twin over chunk and word boundaries, the standalone search against the
one inside round_pm1, and the integrated path against the plain rounding."""
import itertools

import numpy as np
import pytest
import scipy.sparse as sp

from local_search_oracle import LocalSearchOracleBackend, eval_values, local_search, search_rows


def _twin():
    from smcp_b200 import solvers
    solvers.set_backend_factory(lambda symb: LocalSearchOracleBackend(symb))


def _device():
    from smcp_b200 import solvers
    from smcp_b200.device import DeviceBackend
    solvers.set_backend_factory(lambda symb: DeviceBackend(symb))


def _entries(n, structure, weights, seed):
    """Lower-triangular objective entries (row, col, value) of a test graph on n vertices.
    'sparse': random edges among the first 3/4 of the vertices (the rest isolated), a nonzero diagonal, and duplicate
    entries, some given in the upper triangle.  'hub': random edges plus vertex n // 3 adjacent to all others.
    weights 'unit': +-1 (exact arithmetic), 'real': normal values of both signs."""
    rng = np.random.default_rng(seed)
    m = max(1, (3 * n) // 4) if structure == "sparse" else n
    ne = 2 * n
    r, c = rng.integers(0, m, size=ne), rng.integers(0, m, size=ne)
    keep = r != c
    r, c = r[keep], c[keep]
    if structure == "hub" and n > 1:
        h = n // 3
        others = np.delete(np.arange(n), h)
        r, c = np.concatenate([r, np.full(n - 1, h)]), np.concatenate([c, others])
    else:
        dup = rng.integers(0, len(r), size=len(r) // 4) if len(r) else np.zeros(0, dtype=np.int64)
        r, c = np.concatenate([r, c[dup]]), np.concatenate([c, r[dup]])     # duplicates
    d = rng.choice(n, size=max(1, n // 5), replace=False)
    big, small = np.maximum(r, c), np.minimum(r, c)
    upper = rng.random(len(r)) < 0.5 if structure == "sparse" else np.zeros(len(r), dtype=bool)
    rows = np.where(upper, small, big)
    cols = np.where(upper, big, small)
    rows, cols = np.concatenate([rows, d]), np.concatenate([cols, d])
    if weights == "unit":
        v = rng.choice([-1.0, 1.0], size=len(rows))
    else:
        v = rng.standard_normal(len(rows))
    return rows.astype(np.int64), cols.astype(np.int64), v


def _dense(n, crow, ccol, cval):
    C = np.zeros((n, n))
    for r, c, v in zip(crow, ccol, cval):
        C[r, c] += v
        if r != c:
            C[c, r] += v
    return C


def _f(C, x):
    x = np.asarray(x, dtype=np.float64)
    return np.einsum("ti,ij,tj->t", np.atleast_2d(x), C, np.atleast_2d(x))


def _gains(C, x):
    """g = x * s and a of the definition, from the dense C (off-diagonal part)."""
    Co = C - np.diag(np.diag(C))
    x = np.atleast_2d(np.asarray(x, dtype=np.float64))
    return x * (x @ Co), np.abs(Co).sum(axis=1)


def _random_pm1(k, n, seed):
    return np.where(np.random.default_rng(seed).random((k, n)) < 0.5, -1, 1).astype(np.int8)


def _graph(n, ne, seed):
    import smcp_b200 as S
    rng = np.random.default_rng(seed)
    return S.maxcut_SDP(n, rng.integers(0, n, size=(ne, 2)))


# ---------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------
def test_twin_rows_merge_duplicates_in_input_order():
    rp, col, val = search_rows(4, [1, 0, 2, 1, 3, 3], [0, 1, 2, 0, 1, 3], [0.1, 0.2, 5.0, 0.3, -1.0, 7.0])
    assert rp.tolist() == [0, 1, 3, 3, 4]
    assert col.tolist() == [1, 0, 3, 1]
    assert val[0] == (0.1 + 0.2) + 0.3 and val[1] == val[0] and val[2] == -1.0 and val[3] == -1.0


@pytest.mark.parametrize("structure", ["sparse", "hub"])
@pytest.mark.parametrize("weights", ["unit", "real"])
@pytest.mark.parametrize("n", [2, 40, 300])
def test_twin_ends_at_local_optimum(structure, weights, n):
    crow, ccol, cval = _entries(n, structure, weights, n)
    C = _dense(n, crow, ccol, cval)
    x0 = _random_pm1(20, n, 1)
    x, flips = local_search(x0, crow, ccol, cval, n, 1e-12)
    g, a = _gains(C, x)
    scale = np.abs(C).sum()
    assert (flips < n).all()
    assert (g <= 1e-12 * a + 1e-13 * scale).all(), (g - 1e-12 * a).max()
    assert (_f(C, x) <= _f(C, x0) + 1e-12 * scale).all()
    assert ((flips > 0) | (x == x0).all(axis=1)).all()
    ev = eval_values(x, crow, ccol, cval)
    assert np.abs(ev - _f(C, x)).max() <= 1e-12 * scale


@pytest.mark.parametrize("weights", ["unit", "real"])
@pytest.mark.parametrize("n", [5, 9, 14])
def test_twin_keeps_brute_force_optimum(weights, n):
    crow, ccol, cval = _entries(n, "sparse", weights, 100 + n)
    C = _dense(n, crow, ccol, cval)
    X = np.array(list(itertools.product((1, -1), repeat=n)), dtype=np.int8)
    best = X[int(np.argmin(_f(C, X)))]
    x, flips = local_search(best[None, :], crow, ccol, cval, n, 1e-12)
    assert flips.tolist() == [0] and np.array_equal(x[0], best)


def test_twin_max_flips_zero_and_one():
    n = 60
    crow, ccol, cval = _entries(n, "sparse", "unit", 7)
    C = _dense(n, crow, ccol, cval)
    x0 = _random_pm1(10, n, 2)
    x, flips = local_search(x0, crow, ccol, cval, 0, 1e-12)
    assert np.array_equal(x, x0) and not flips.any()
    x, flips = local_search(x0, crow, ccol, cval, 1, 1e-12)
    g, a = _gains(C, x0)
    for t in range(len(x0)):
        ok = g[t] > 1e-12 * a[t]
        if not ok.any():
            assert flips[t] == 0 and np.array_equal(x[t], x0[t])
            continue
        i = int(np.argmax(np.where(ok, g[t], -np.inf)))
        ref = x0[t].copy()
        ref[i] = -ref[i]
        assert flips[t] == 1 and np.array_equal(x[t], ref), t
        assert _f(C, x[t])[0] == _f(C, x0[t])[0] - 4 * g[t, i]


def test_argument_validation():
    P = _graph(6, 8, 0)
    sol = {"x": sp.identity(6, format="csc")}
    x = np.ones(6, dtype=np.int8)
    for bad, exc in ((-1, ValueError), (1.5, ValueError), (True, ValueError), ("2", ValueError)):
        with pytest.raises(exc):
            P.round_pm1(sol, local_search=True, max_flips=bad)
        with pytest.raises(exc):
            P.local_search_pm1(x, max_flips=bad)
    for bad, exc in ((-1e-3, ValueError), (np.inf, ValueError), (np.nan, ValueError), (True, TypeError), ("0", TypeError),
                     (None, TypeError)):
        with pytest.raises(exc):
            P.round_pm1(sol, local_search=True, tol=bad)
        with pytest.raises(exc):
            P.local_search_pm1(x, tol=bad)
    for bad in (1, None, "yes"):
        with pytest.raises(TypeError):
            P.round_pm1(sol, local_search=bad)
        with pytest.raises(TypeError):
            P.cut(sol, local_search=bad)
    for bad, exc in ((np.zeros(6, dtype=np.int8), ValueError), (np.ones(5, dtype=np.int8), ValueError),
                     (np.ones((2, 7), dtype=np.int8), ValueError), (np.ones((0, 6), dtype=np.int8), ValueError),
                     (np.ones((1, 2, 6), dtype=np.int8), ValueError), (np.full(6, 3), ValueError),
                     (np.ones(6), TypeError), (np.ones(6, dtype=bool), TypeError)):
        with pytest.raises(exc):
            P.local_search_pm1(bad)


def test_twin_public_methods():
    from smcp_b200 import solvers
    _twin()
    solvers.options["show_progress"] = False
    P = _graph(12, 20, 3)
    I, J, v = P._objective_entries()
    C = _dense(P.n, I, J, v)
    x0 = _random_pm1(5, P.n, 4)
    r = P.local_search_pm1(x0)
    xs, flips = local_search(x0, I, J, v, P.n, 1e-12)
    assert r["x"].dtype == np.int8 and np.array_equal(r["x"], xs) and np.array_equal(r["flips"], flips)
    assert np.array_equal(r["values"], eval_values(xs, I, J, v))
    one = P.local_search_pm1(x0[2])
    assert one["x"].shape == (P.n,) and np.array_equal(one["x"], xs[2]) and one["values"].shape == ()
    sol = P.solve_esd()
    assert sol["status"] == "optimal"
    plain = P.round_pm1(sol, trials=64, seed=1)
    q = P.round_pm1(sol, trials=64, seed=1, local_search=True)
    assert np.array_equal(q["values_rounded"], plain["values"])        # unit weights: exact sums
    assert (q["values"] <= q["values_rounded"]).all()
    assert q["value"] == q["values"].min() and abs(q["value"] - _f(C, q["x"])[0]) <= 1e-12
    g, a = _gains(C, q["x"])
    assert (g <= 1e-12 * a).all()
    _, w0, _ = P.cut(sol, trials=64, seed=1)
    _, w1, ub = P.cut(sol, trials=64, seed=1, local_search=True)
    assert w0 <= w1 <= ub + 1e-6


# ---------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------
def _device_ops(n):
    from smcp_b200.device import DeviceBackend
    from smcp_b200.symbolic import Symbolic
    return DeviceBackend(Symbolic(n, np.arange(n + 1), np.arange(n)))


def _check_against_twin(ops, x0, crow, ccol, cval, max_flips, tol=1e-12):
    xd, vd, fd = ops.pm1_local_search(x0, crow, ccol, cval, max_flips, tol)
    xt, ft = local_search(x0, crow, ccol, cval, x0.shape[1] if max_flips is None else max_flips, tol)
    vt = eval_values(xt, crow, ccol, cval)
    assert np.array_equal(fd, ft), (max_flips, np.flatnonzero(fd != ft)[:5])
    assert np.array_equal(xd, xt), max_flips
    assert np.array_equal(vd.view(np.int64), vt.view(np.int64)), max_flips
    return fd


# (n, k): n across the 256-vertex chunks, k across the 64-trial words
SIZES = [(1, 1), (1, 65), (2, 63), (2, 64), (255, 65), (256, 64), (257, 63), (257, 300), (1000, 1), (1000, 300),
         (5000, 65)]


@pytest.mark.gpu
@pytest.mark.parametrize("n,k", SIZES)
@pytest.mark.parametrize("structure", ["sparse", "hub"])
@pytest.mark.parametrize("weights", ["unit", "real"])
def test_device_matches_twin(n, k, structure, weights):
    _device()
    crow, ccol, cval = _entries(n, structure, weights, 11 * n + k)
    x0 = _random_pm1(k, n, n + k)
    ops = _device_ops(n)
    full = _check_against_twin(ops, x0, crow, ccol, cval, None)
    for mf in (0, 1):
        f = _check_against_twin(ops, x0, crow, ccol, cval, mf)
        assert (f <= mf).all()
    if full.max() >= 2:
        cap = int(full.max()) // 2
        f = _check_against_twin(ops, x0, crow, ccol, cval, cap)
        assert (f == cap).any() and (f <= cap).all()


@pytest.mark.gpu
def test_device_tol_and_usage_errors():
    from smcp_b200.device import DeviceError
    _device()
    n = 400
    crow, ccol, cval = _entries(n, "sparse", "real", 5)
    x0 = _random_pm1(70, n, 6)
    ops = _device_ops(n)
    for tol in (0.0, 1e-3, 0.25):
        _check_against_twin(ops, x0, crow, ccol, cval, None, tol)
    bad = x0.copy()
    bad[3, 17] = 0
    for args in ((bad, crow, ccol, cval, None, 1e-12), (x0, [0], [n], [1.0], None, 1e-12), (x0, [-1], [0], [1.0], None, 1e-12),
                 (x0, crow, ccol, cval, -1, 1e-12), (x0, crow, ccol, cval, None, -1.0), (x0, crow, ccol, cval, None, np.nan),
                 (x0, crow, ccol, cval, None, np.inf), (np.ones((1, (1 << 20) + 1), dtype=np.int8), [0], [0], [1.0], 0, 0.0)):
        with pytest.raises(DeviceError):
            ops.pm1_local_search(*args)
    xa, va, fa = ops.pm1_local_search(np.ones((1, 1 << 20), dtype=np.int8), [5, 7], [0, 5], [1.0, 2.0], None, 1e-12)
    assert fa.tolist() == [1] and xa[0, 5] == -1 and (np.delete(xa[0], 5) == 1).all()


def _round_case(seed, n=60):
    from test_rounding import _unit_diag_on_pattern
    P = _graph(n, 2 * n, seed)
    return P, {"x": _unit_diag_on_pattern(P, seed)}


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [1, 2])
def test_round_pm1_local_search(seed):
    _device()
    P, sol = _round_case(seed, 300)
    trials = 600
    plain = P.round_pm1(sol, trials=trials, seed=seed)
    off = P.round_pm1(sol, trials=trials, seed=seed, local_search=False)
    assert set(off) == set(plain)
    for key in ("x", "values"):
        assert np.array_equal(off[key], plain[key])
    assert off["trial"] == plain["trial"] and off["value"] == plain["value"]
    q = P.round_pm1(sol, trials=trials, seed=seed, local_search=True)
    assert np.array_equal(q["values_rounded"].view(np.int64), plain["values"].view(np.int64))
    assert (q["values"] <= q["values_rounded"]).all() and (q["values"] < q["values_rounded"]).any()
    assert q["flips"].dtype == np.int64 and ((q["flips"] > 0) == (q["values"] < q["values_rounded"])).all()
    t = int(np.flatnonzero(q["values"] == q["values"].min())[0])
    assert q["trial"] == t and q["value"] == q["values"][t]
    I, J, v = P._objective_entries()
    C = _dense(P.n, I, J, v)
    assert _f(C, q["x"])[0] == q["value"]
    g, a = _gains(C, q["x"])
    assert (g <= 1e-12 * a).all()
    for chunk in (1, 7, 250):
        c = P.round_pm1(sol, trials=trials, seed=seed, chunk=chunk, local_search=True)
        for key in ("x", "values", "values_rounded", "flips"):
            assert np.array_equal(c[key], q[key]), (chunk, key)
        assert c["trial"] == q["trial"]
    c = P.round_pm1(sol, trials=trials, seed=seed, local_search=True, max_flips=1)
    assert (c["flips"] <= 1).all() and np.array_equal(c["values_rounded"], q["values_rounded"])


@pytest.mark.gpu
def test_standalone_matches_integrated_and_twin():
    """The same trials through smcp_pm1_local_search and smcp_round_pm1_ls, in the internal coordinates."""
    from smcp_b200.base import _completion_factor
    _device()
    P, sol = _round_case(4, 500)
    L, order = _completion_factor(sol["x"])
    ops = L.ops
    I, J, v = P._objective_entries()
    pos = np.empty(P.n, dtype=np.int64)
    pos[order] = np.arange(P.n)
    crow, ccol = pos[I], pos[J]
    trials, seed = 200, 8                               # one solve block: the samples of completion_sample
    V = ops.completion_sample(L.buf, trials, seed)
    x0 = np.where(V.T < 0.0, -1, 1).astype(np.int8)
    ops.ctx.prof_reset()
    ops.ctx.prof_enable(True)
    try:
        values0, values, flips, xb, best = ops.round_pm1_ls(L.buf, crow, ccol, v, trials, seed)
        names = ops.ctx.prof_names()
    finally:
        ops.ctx.prof_enable(False)
    assert "round_ls" in names and "round_eval" in names, names
    plain, _, _ = ops.round_pm1(L.buf, crow, ccol, v, trials, seed)
    assert np.array_equal(values0, plain)
    _, v0, f0 = ops.pm1_local_search(x0, crow, ccol, v, 0)
    assert np.array_equal(v0, values0) and not f0.any()
    xs, vs, fs = ops.pm1_local_search(x0, crow, ccol, v)
    assert np.array_equal(vs, values) and np.array_equal(fs, flips)
    assert best == int(np.argmin(values)) and np.array_equal(xb, xs[best])
    xt, ft = local_search(x0, crow, ccol, v, P.n, 1e-12)
    assert np.array_equal(xs, xt) and np.array_equal(fs, ft)
    assert np.array_equal(vs, eval_values(xt, crow, ccol, v)) and np.array_equal(values0, eval_values(x0, crow, ccol, v))
    # the public standalone call, in the original order
    r = P.local_search_pm1(x0[:, pos])
    xo, fo = local_search(x0[:, pos], I, J, v, P.n, 1e-12)
    assert np.array_equal(r["x"], xo) and np.array_equal(r["flips"], fo)
    assert np.array_equal(r["values"], eval_values(xo, I, J, v))


def _maxcut_cases():
    # the end-to-end cases of test_rounding.py
    return [(12, 1), (12, 3), (16, 0), (16, 1), (18, 0), (18, 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("n,seed", _maxcut_cases())
@pytest.mark.parametrize("method", ["feas", "esd"])
def test_cut_local_search_end_to_end(n, seed, method):
    from smcp_b200 import solvers
    from test_rounding import _brute_max_cut
    _device()
    solvers.options["show_progress"] = False
    P = _graph(n, 2 * n, seed)
    if method == "feas":
        sol = P.solve_feas(primalstart={"x": sp.identity(n, format="csc")})
    else:
        sol = P.solve_esd()
    assert sol["status"] == "optimal", sol["status"]
    x0, w0, ub = P.cut(sol, trials=256)
    x1, w1, ub1 = P.cut(sol, trials=256, local_search=True)
    best = _brute_max_cut(P)
    assert ub1 == ub
    assert w0 <= w1 <= best + 1e-9 and best <= ub + 1e-6, (w0, w1, best, ub)
