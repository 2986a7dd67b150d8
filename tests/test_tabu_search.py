"""Tabu search of +-1 vectors (``SDP.tabu_search_pm1``, ``SDP.round_pm1(tabu_iters=...)``,
``maxcut_SDP.cut(tabu_iters=...)``).  On the CPU: the NumPy twin (tests/tabu_search_oracle.py) against a direct
restatement of the definition, never above the start's f, iters = 0, tenure = 0 and tenure >= n, the optimum of a small
graph where the one-flip search stops short of it; argument validation.  On the device: signs, values, moves and best
iterations bitwise against the twin over chunk and word boundaries, the shared-memory limits, the standalone search
against the one inside round_pm1, and cut(tabu_iters) against cut(local_search=True), brute force and the dual bound."""
import itertools
from fractions import Fraction

import numpy as np
import pytest
import scipy.sparse as sp

from local_search_oracle import eval_values, local_search
from tabu_search_oracle import TabuSearchOracleBackend, tabu_search
from test_local_search import _dense, _entries, _f, _graph, _random_pm1


def _twin():
    from smcp_b200 import solvers
    solvers.set_backend_factory(lambda symb: TabuSearchOracleBackend(symb))


def _device():
    from smcp_b200 import solvers
    from smcp_b200.device import DeviceBackend
    solvers.set_backend_factory(lambda symb: DeviceBackend(symb))


def _tenure(n):
    from smcp_b200.base import _tabu_tenure
    return _tabu_tenure(n)


def _definition(C, x0, iters, tenure):
    """The search of one vector as defined, with g recomputed from the dense C at every move (exact for integer C)."""
    Co = C - np.diag(np.diag(C))
    x = np.asarray(x0, dtype=np.float64).copy()
    n = len(x)
    last = np.full(n, -1 - tenure)
    D = Db = 0.0
    best, best_iter, moves = x.copy(), 0, 0
    for u in range(iters):
        g = x * (Co @ x)
        adm = (last < u - tenure) | (D - 4.0 * g < Db)
        if not adm.any():
            break
        i = int(np.argmax(np.where(adm, g, -np.inf)))
        D -= 4.0 * g[i]
        x[i] = -x[i]
        last[i] = u
        moves += 1
        if D < Db:
            Db, best, best_iter = D, x.copy(), u + 1
    return best.astype(np.int8), moves, best_iter


def _f_exact(n, crow, ccol, cval, x):
    """C . x x^T in exact rational arithmetic."""
    tot = Fraction(0)
    for r, c, v in zip(crow, ccol, cval):
        term = Fraction(float(v)) * (1 if r == c else 2)
        tot += term if x[r] == x[c] else -term
    return tot


# ---------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("structure", ["sparse", "hub"])
@pytest.mark.parametrize("n", [1, 2, 7, 20, 60])
def test_twin_follows_definition(structure, n):
    crow, ccol, cval = _entries(n, structure, "unit", n)
    C = _dense(n, crow, ccol, cval)
    x0 = _random_pm1(6, n, n + 1)
    for tenure in sorted({0, 1, max(n - 1, 0), n, n + 3, _tenure(n)}):
        for iters in (0, 1, n, 5 * n + 3):
            xs, moves, best_iter = tabu_search(x0, crow, ccol, cval, iters, tenure)
            for t in range(len(x0)):
                xr, mr, br = _definition(C, x0[t], iters, tenure)
                assert np.array_equal(xs[t], xr) and moves[t] == mr and best_iter[t] == br, (tenure, iters, t)


@pytest.mark.parametrize("structure", ["sparse", "hub"])
@pytest.mark.parametrize("weights", ["unit", "real"])
@pytest.mark.parametrize("n", [2, 40, 300])
def test_twin_never_above_start(structure, weights, n):
    crow, ccol, cval = _entries(n, structure, weights, 3 * n)
    x0 = _random_pm1(12, n, 5)
    for tenure in (0, 1, _tenure(n), n):
        xs, moves, best_iter = tabu_search(x0, crow, ccol, cval, 3 * n, tenure)
        assert (moves <= 3 * n).all() and (best_iter <= moves).all()
        for t in range(len(x0)):
            if best_iter[t] == 0:
                assert np.array_equal(xs[t], x0[t])
            assert _f_exact(n, crow, ccol, cval, xs[t]) <= _f_exact(n, crow, ccol, cval, x0[t]), (tenure, t)


def test_twin_iters_zero_and_tenure_limits():
    n = 50
    crow, ccol, cval = _entries(n, "sparse", "unit", 9)
    C = _dense(n, crow, ccol, cval)
    x0 = _random_pm1(8, n, 3)
    xs, moves, best_iter = tabu_search(x0, crow, ccol, cval, 0, 5)
    assert np.array_equal(xs, x0) and not moves.any() and not best_iter.any()
    # tenure 0: nothing is ever tabu, every move takes the largest gain, even one that is not positive
    x1, _ = local_search(x0, crow, ccol, cval, n, 1e-12)
    Co = C - np.diag(np.diag(C))
    xs, moves, best_iter = tabu_search(x1, crow, ccol, cval, 1, 0)
    assert (moves == 1).all() and not best_iter.any() and np.array_equal(xs, x1)
    assert ((x1 * (x1 @ Co)).max(axis=1) <= 0).all()
    xs, moves, best_iter = tabu_search(x1, crow, ccol, cval, 3 * n, 0)
    assert (moves == 3 * n).all()
    for t in range(len(x1)):
        xr, mr, br = _definition(C, x1[t], 3 * n, 0)
        assert np.array_equal(xs[t], xr) and mr == moves[t] and br == best_iter[t]
    # tenure >= n: the search stops before iters once every vertex is tabu and none passes the aspiration test
    xs, moves, best_iter = tabu_search(x1, crow, ccol, cval, 3 * n, n)
    assert (moves >= n).all() and (moves < 3 * n).all()
    for t in range(len(x1)):
        xr, mr, br = _definition(C, x1[t], 3 * n, n)
        assert np.array_equal(xs[t], xr) and mr == moves[t] and br == best_iter[t]
    # an isolated vertex: with tenure >= 1 its second move is tabu and has no gain to aspire with
    xs, moves, best_iter = tabu_search(np.ones((1, 1), dtype=np.int8), [0], [0], [2.0], 10, 1)
    assert moves.tolist() == [1] and best_iter.tolist() == [0] and xs.tolist() == [[1]]
    xs, moves, best_iter = tabu_search(np.ones((1, 1), dtype=np.int8), [0], [0], [2.0], 10, 0)
    assert moves.tolist() == [10] and best_iter.tolist() == [0] and xs.tolist() == [[1]]


def test_twin_escapes_one_flip_optimum():
    """n = 10: from this start the one-flip search stops at f = -11, the optimum is -15; tabu search reaches it."""
    from test_rounding import _brute_max_cut
    n = 10
    P = _graph(n, 2 * n, 2)
    I, J, v = P._objective_entries()
    C = _dense(n, I, J, v)
    X = np.array(list(itertools.product((1, -1), repeat=n)), dtype=np.int8)
    fopt = _f(C, X).min()
    assert -fopt == _brute_max_cut(P)
    x1, _ = local_search(_random_pm1(1, n, 2), I, J, v, n, 1e-12)
    assert _f(C, x1)[0] > fopt
    xt, moves, best_iter = tabu_search(x1, I, J, v, 4 * n, _tenure(n))
    assert _f(C, xt)[0] == fopt and 0 < best_iter[0] <= moves[0]


def test_argument_validation():
    P = _graph(6, 8, 0)
    sol = {"x": sp.identity(6, format="csc")}
    x = np.ones(6, dtype=np.int8)
    for bad in (-1, 1.5, True, "2", None):
        with pytest.raises(ValueError):
            P.round_pm1(sol, tabu_iters=bad)
        with pytest.raises(ValueError):
            P.tabu_search_pm1(x, bad)
        with pytest.raises(ValueError):
            P.cut(sol, tabu_iters=bad)
    for bad in (-1, 2.0, True, "3"):
        with pytest.raises(ValueError):
            P.round_pm1(sol, tabu_iters=3, tenure=bad)
        with pytest.raises(ValueError):
            P.tabu_search_pm1(x, 3, tenure=bad)
    for bad, exc in ((np.zeros(6, dtype=np.int8), ValueError), (np.ones(5, dtype=np.int8), ValueError),
                     (np.ones((2, 7), dtype=np.int8), ValueError), (np.ones((0, 6), dtype=np.int8), ValueError),
                     (np.full(6, 3), ValueError), (np.ones(6), TypeError), (np.ones(6, dtype=bool), TypeError)):
        with pytest.raises(exc):
            P.tabu_search_pm1(bad, 3)


def test_twin_public_methods():
    from smcp_b200 import solvers
    _twin()
    solvers.options["show_progress"] = False
    P = _graph(12, 20, 3)
    I, J, v = P._objective_entries()
    C = _dense(P.n, I, J, v)
    x0 = _random_pm1(5, P.n, 4)
    r = P.tabu_search_pm1(x0, 30)
    xs, moves, best_iter = tabu_search(x0, I, J, v, 30, _tenure(P.n))
    assert r["x"].dtype == np.int8 and np.array_equal(r["x"], xs)
    assert np.array_equal(r["moves"], moves) and np.array_equal(r["best_iter"], best_iter)
    assert np.array_equal(r["values"], eval_values(xs, I, J, v))
    one = P.tabu_search_pm1(x0[2], 30, tenure=0)
    xs0, _, _ = tabu_search(x0[2:3], I, J, v, 30, 0)
    assert one["x"].shape == (P.n,) and np.array_equal(one["x"], xs0[0]) and one["values"].shape == ()
    sol = P.solve_esd()
    assert sol["status"] == "optimal"
    plain = P.round_pm1(sol, trials=64, seed=1)
    ls = P.round_pm1(sol, trials=64, seed=1, local_search=True)
    q = P.round_pm1(sol, trials=64, seed=1, tabu_iters=2 * P.n)
    assert "values_rounded" not in q and np.array_equal(q["values_before_tabu"], plain["values"])
    assert (q["values"] <= q["values_before_tabu"]).all() and (q["best_iter"] <= q["moves"]).all()
    assert q["value"] == q["values"].min() and abs(q["value"] - _f(C, q["x"])[0]) <= 1e-12
    b = P.round_pm1(sol, trials=64, seed=1, local_search=True, tabu_iters=2 * P.n)
    assert np.array_equal(b["values_rounded"], plain["values"]) and np.array_equal(b["flips"], ls["flips"])
    assert np.array_equal(b["values_before_tabu"], ls["values"]) and (b["values"] <= ls["values"]).all()
    _, w1, _ = P.cut(sol, trials=64, seed=1, local_search=True)
    _, w2, ub = P.cut(sol, trials=64, seed=1, tabu_iters=P.n)
    assert w1 <= w2 <= ub + 1e-6


# ---------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------
def _device_ops(n):
    from smcp_b200.device import DeviceBackend
    from smcp_b200.symbolic import Symbolic
    return DeviceBackend(Symbolic(n, np.arange(n + 1), np.arange(n)))


def _check_against_twin(ops, x0, crow, ccol, cval, iters, tenure):
    xd, vd, md, bd = ops.pm1_tabu_search(x0, crow, ccol, cval, iters, tenure)
    xt, mt, bt = tabu_search(x0, crow, ccol, cval, iters, tenure)
    vt = eval_values(xt, crow, ccol, cval)
    key = (iters, tenure)
    assert np.array_equal(md, mt), (key, np.flatnonzero(md != mt)[:5])
    assert np.array_equal(bd, bt), (key, np.flatnonzero(bd != bt)[:5])
    assert np.array_equal(xd, xt), key
    assert np.array_equal(vd.view(np.int64), vt.view(np.int64)), key
    return md, bd


# (n, k): n across the 256-vertex chunks, k across the 64-trial words
SIZES = [(1, 1), (1, 65), (2, 63), (2, 64), (255, 65), (256, 64), (257, 63), (257, 300), (1000, 1), (1000, 300),
         (5000, 65)]


@pytest.mark.gpu
@pytest.mark.parametrize("n,k", SIZES)
@pytest.mark.parametrize("structure", ["sparse", "hub"])
@pytest.mark.parametrize("weights", ["unit", "real"])
def test_device_matches_twin(n, k, structure, weights):
    _device()
    crow, ccol, cval = _entries(n, structure, weights, 13 * n + k)
    ops = _device_ops(n)
    x0 = _random_pm1(k, n, n + k)
    x1, _ = local_search(x0, crow, ccol, cval, n, 1e-12)     # from one-flip optima too, where moves go uphill
    long = 10 * n if n * k <= 100000 else n
    cases = [(x0, 0, _tenure(n)), (x0, 1, _tenure(n)), (x0, n, _tenure(n)), (x1, long, _tenure(n)), (x1, n, 0),
             (x1, long, 1), (x1, n, max(n - 1, 0)), (x1, 2 * n + 5, 8192)]
    for x, iters, tenure in cases:
        moves, best_iter = _check_against_twin(ops, x, crow, ccol, cval, iters, tenure)
        assert (moves <= iters).all() and (best_iter <= moves).all()
        if tenure < n:
            assert (moves == iters).all()
        if iters == 0:
            assert not moves.any()


@pytest.mark.gpu
def test_device_limits_and_usage_errors():
    from smcp_b200.device import DeviceError
    _device()
    n = 1 << 19
    ops = _device_ops(n)
    rng = np.random.default_rng(0)
    r, c = rng.integers(0, n, size=3 * n), rng.integers(0, n, size=3 * n)
    keep = r != c
    crow, ccol = np.maximum(r, c)[keep], np.minimum(r, c)[keep]
    cval = rng.choice([-1.0, 1.0], size=len(crow))
    x0 = _random_pm1(1, n, 1)
    _check_against_twin(ops, x0, crow, ccol, cval, 6, 8192)
    big = _device_ops(n + 1)
    with pytest.raises(DeviceError):
        big.pm1_tabu_search(np.ones((1, n + 1), dtype=np.int8), [0], [0], [1.0], 1, 0)
    m = 300
    crow, ccol, cval = _entries(m, "sparse", "real", 5)
    x0 = _random_pm1(3, m, 6)
    small = _device_ops(m)
    bad = x0.copy()
    bad[1, 7] = 0
    for args in ((x0, crow, ccol, cval, 5, 8193), (x0, crow, ccol, cval, 5, -1), (x0, crow, ccol, cval, -1, 5),
                 (bad, crow, ccol, cval, 5, 5), (x0, [0], [m], [1.0], 5, 5), (x0, [-1], [0], [1.0], 5, 5)):
        with pytest.raises(DeviceError):
            small.pm1_tabu_search(*args)


def _round_case(seed, n=60):
    from test_rounding import _unit_diag_on_pattern
    P = _graph(n, 2 * n, seed)
    return P, {"x": _unit_diag_on_pattern(P, seed)}


@pytest.mark.gpu
def test_standalone_matches_integrated_and_twin():
    """The same trials through smcp_pm1_tabu_search and smcp_round_pm1_tabu, in the internal coordinates, with and
    without the one-flip search before the tabu search."""
    from smcp_b200.base import _completion_factor
    from smcp_b200.device import DeviceError
    _device()
    P, sol = _round_case(4, 500)
    L, order = _completion_factor(sol["x"])
    ops = L.ops
    I, J, v = P._objective_entries()
    pos = np.empty(P.n, dtype=np.int64)
    pos[order] = np.arange(P.n)
    crow, ccol = pos[I], pos[J]
    trials, seed, iters, tenure = 200, 8, 2 * P.n, _tenure(P.n)   # one solve block: the samples of completion_sample
    V = ops.completion_sample(L.buf, trials, seed)
    x0 = np.where(V.T < 0.0, -1, 1).astype(np.int8)
    plain, _, _ = ops.round_pm1(L.buf, crow, ccol, v, trials, seed)
    l0, lv, lf, _, _ = ops.round_pm1_ls(L.buf, crow, ccol, v, trials, seed)
    x1, _, _ = ops.pm1_local_search(x0, crow, ccol, v)
    for start, max_flips in ((x0, 0), (x1, None)):
        ops.ctx.prof_reset()
        ops.ctx.prof_enable(True)
        try:
            values0, values1, values, flips, moves, best_iter, xb, best = ops.round_pm1_tabu(
                L.buf, crow, ccol, v, trials, seed, iters, tenure, max_flips=max_flips)
            names = ops.ctx.prof_names()
        finally:
            ops.ctx.prof_enable(False)
        assert "round_tabu" in names and "round_eval" in names, names
        assert ("round_ls" in names) == (max_flips is None), names
        assert np.array_equal(values0, plain)
        if max_flips is None:
            assert np.array_equal(values1, lv) and np.array_equal(flips, lf)
        else:
            assert np.array_equal(values1, plain) and not flips.any()
        xs, vs, ms, bs = ops.pm1_tabu_search(start, crow, ccol, v, iters, tenure)
        assert np.array_equal(vs, values) and np.array_equal(ms, moves) and np.array_equal(bs, best_iter)
        assert best == int(np.argmin(values)) and np.array_equal(xb, xs[best])
        xt, mt, bt = tabu_search(start, crow, ccol, v, iters, tenure)
        assert np.array_equal(xs, xt) and np.array_equal(ms, mt) and np.array_equal(bs, bt)
        assert np.array_equal(vs, eval_values(xt, crow, ccol, v))
    with pytest.raises(DeviceError):
        ops.round_pm1_tabu(L.buf, crow, ccol, v, trials, seed, iters, 8193)
    # the public standalone call, in the original order
    r = P.tabu_search_pm1(x0[:, pos], iters)
    xo, mo, bo = tabu_search(x0[:, pos], I, J, v, iters, tenure)
    assert np.array_equal(r["x"], xo) and np.array_equal(r["moves"], mo) and np.array_equal(r["best_iter"], bo)
    assert np.array_equal(r["values"], eval_values(xo, I, J, v))


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [1, 2])
def test_round_pm1_tabu(seed):
    _device()
    P, sol = _round_case(seed, 300)
    trials = 600
    plain = P.round_pm1(sol, trials=trials, seed=seed)
    off = P.round_pm1(sol, trials=trials, seed=seed, tabu_iters=0, tenure=5)
    assert set(off) == set(plain)
    for key in ("x", "values"):
        assert np.array_equal(off[key], plain[key])
    ls = P.round_pm1(sol, trials=trials, seed=seed, local_search=True)
    for local_search in (False, True):
        q = P.round_pm1(sol, trials=trials, seed=seed, local_search=local_search, tabu_iters=P.n)
        before = ls["values"] if local_search else plain["values"]
        assert np.array_equal(q["values_before_tabu"].view(np.int64), before.view(np.int64))
        assert (q["values"] <= q["values_before_tabu"]).all() and (q["values"] < q["values_before_tabu"]).any()
        assert q["moves"].dtype == np.int64 and (q["moves"] == P.n).all()
        assert ((q["best_iter"] > 0) == (q["values"] < q["values_before_tabu"])).all()
        t = int(np.flatnonzero(q["values"] == q["values"].min())[0])
        assert q["trial"] == t and q["value"] == q["values"][t]
        I, J, v = P._objective_entries()
        assert _f(_dense(P.n, I, J, v), q["x"])[0] == q["value"]
        for chunk in (1, 7, 250):
            c = P.round_pm1(sol, trials=trials, seed=seed, chunk=chunk, local_search=local_search, tabu_iters=P.n)
            for key in ("x", "values", "values_before_tabu", "moves", "best_iter"):
                assert np.array_equal(c[key], q[key]), (chunk, key)
            assert c["trial"] == q["trial"]


def _maxcut_cases():
    # the end-to-end cases of test_rounding.py
    return [(12, 1), (12, 3), (16, 0), (16, 1), (18, 0), (18, 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("n,seed", _maxcut_cases())
@pytest.mark.parametrize("method", ["feas", "esd"])
def test_cut_tabu_end_to_end(n, seed, method):
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
    _, w1, ub = P.cut(sol, trials=256, local_search=True)
    _, w2, ub2 = P.cut(sol, trials=256, tabu_iters=n)
    best = _brute_max_cut(P)
    assert ub2 == ub
    assert w1 <= w2 <= best + 1e-9 and best <= ub + 1e-6, (w1, w2, best, ub)
