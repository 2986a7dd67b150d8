"""Goemans-Williamson rounding: Gaussian samples of the max-det completion (``completion_sample``) and batched
+-1 evaluation (``SDP.round_pm1``, ``maxcut_SDP.cut``).  On the CPU: the NumPy twin's generator against
np.random.Philox, argument validation, and the twin end to end.  On the device: the generator, the samples
against the dense completion, the trial values against a host evaluation and the twin, end-to-end cuts against
brute force, and the ArithmeticError of an X without a positive definite completion."""
import itertools

import numpy as np
import pytest
import scipy.linalg as sl
import scipy.sparse as sp

from conftest import random_pattern
from rounding_oracle import RoundingOracleBackend, normals, philox4x64, pm1_values


def _twin():
    from smcp_b200 import solvers
    solvers.set_backend_factory(lambda symb: RoundingOracleBackend(symb))


def _device():
    from smcp_b200 import solvers
    from smcp_b200.device import DeviceBackend
    solvers.set_backend_factory(lambda symb: DeviceBackend(symb))


def _graph(n, ne, seed):
    import smcp_b200 as S
    rng = np.random.default_rng(seed)
    return S.maxcut_SDP(n, rng.integers(0, n, size=(ne, 2)))


def _objective(P):
    """Lower-triangular entries (row, col, value) of C in the original order."""
    from smcp_b200 import misc
    A = P.A
    I, J = misc.ind2sub(P.n, A.indices[A.indptr[0]:A.indptr[1]])
    return np.asarray(I, dtype=np.int64), np.asarray(J, dtype=np.int64), A.data[A.indptr[0]:A.indptr[1]]


def _brute_max_cut(P):
    """Largest -C . x x^T over all x in {-1, 1}^n (x_0 = 1)."""
    I, J, v = _objective(P)
    coef = np.where(I == J, 1.0, 2.0) * v
    best = -np.inf
    X = np.array(list(itertools.product((1.0, -1.0), repeat=P.n - 1)))
    X = np.hstack([np.ones((len(X), 1)), X])
    for c0 in range(0, len(X), 1 << 14):
        x = X[c0:c0 + (1 << 14)]
        best = max(best, float((-(x[:, I] * x[:, J]) @ coef).max()))
    return best


def _unit_diag_on_pattern(P, seed):
    """X = P_V(M), M = (I + G G^T) / 2 with unit rows g_i: unit diagonal and a positive definite completion."""
    rng = np.random.default_rng(seed)
    n = P.n
    G = rng.standard_normal((n, 4))
    G /= np.linalg.norm(G, axis=1)[:, None]
    M = 0.5 * (np.eye(n) + G @ G.T)
    V = sp.tril(P.V, format="coo")
    return sp.csc_matrix((M[V.row, V.col], (V.row, V.col)), shape=(n, n))


# ---------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed", [0, 1, 12345, 2 ** 63 + 11, 2 ** 64 - 1])
def test_twin_philox_matches_numpy(seed):
    """Counter c of the generator is NumPy's first block after counter c - 1 (NumPy increments first)."""
    rng = np.random.default_rng(seed % 1000)
    for c, j in [(1, 0), (1, 7), (2, 0), (3, 123)] + [(int(a), int(b)) for a, b in rng.integers(1, 2 ** 62, size=(6, 2))]:
        w = philox4x64(np.array([[c, j, 0, 0]], dtype=np.uint64), (np.uint64(seed), np.uint64(0)))[0]
        ref = np.random.Philox(key=np.array([seed, 0], dtype=np.uint64),
                               counter=np.array([c - 1, j, 0, 0], dtype=np.uint64)).random_raw(4)
        assert np.array_equal(w, ref), (seed, c, j)


def test_twin_normals_are_counter_based():
    a = normals(37, 9, 5)
    assert np.array_equal(a[:, 4:], normals(37, 5, 5, col0=4))
    assert np.array_equal(a[:21], normals(21, 9, 5))
    assert not np.array_equal(a, normals(37, 9, 6))


def test_argument_validation():
    import smcp_b200 as S
    P = _graph(6, 8, 0)
    sol = {"x": sp.identity(6, format="csc")}
    for bad in (0, -1, 1.5, True, "4"):
        with pytest.raises(ValueError):
            P.round_pm1(sol, trials=bad)
        with pytest.raises(ValueError):
            P.cut(sol, trials=bad)
    for bad, exc in ((-1, ValueError), (2 ** 64, ValueError), (1.0, TypeError), ("1", TypeError), (None, TypeError)):
        with pytest.raises(exc):
            P.round_pm1(sol, seed=bad)
        with pytest.raises(exc):
            P.cut(sol, seed=bad)
        with pytest.raises(exc):
            S.completion_sample(sol["x"], 3, seed=bad)
    with pytest.raises(ValueError):
        P.round_pm1(sol, chunk=-1)
    for bad in ({}, {"y": 1}, None):
        with pytest.raises(ValueError):
            P.round_pm1(bad)
        with pytest.raises(ValueError):
            P.cut(bad)
    for bad in (-1, 2.0, None):
        with pytest.raises(ValueError):
            S.completion_sample(sol["x"], bad)


def test_twin_cut_within_brute_force():
    from smcp_b200 import solvers
    _twin()
    solvers.options["show_progress"] = False
    P = _graph(12, 20, 3)
    sol = P.solve_esd()
    assert sol["status"] == "optimal"
    x, w, ub = P.cut(sol, trials=64, seed=1)
    best = _brute_max_cut(P)
    I, J, v = _objective(P)
    assert x.dtype == np.int8 and set(np.unique(x)) <= {-1, 1}
    assert abs(w + float(((x[I] * x[J]).astype(float) * np.where(I == J, 1.0, 2.0) * v).sum())) <= 1e-12
    assert w <= best + 1e-9 and best <= ub + 1e-6, (w, best, ub)


# ---------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_generator_on_diagonal_pattern():
    """X = I: L = I, the samples are the raw normals (in the internal order)."""
    from smcp_b200.base import _completion_factor
    _device()
    n, k, seed = 1000, 300, 2024
    L, order = _completion_factor(sp.identity(n, format="csc"))
    ops = L.ops
    Z = ops.completion_sample(L.buf, k, seed)
    ref = normals(n, k, seed)
    assert np.abs(Z - ref).max() <= 1e-13 * max(1.0, np.abs(ref).max())
    assert np.array_equal(Z, ops.completion_sample(L.buf, k, seed))
    halves = np.hstack([ops.completion_sample(L.buf, 150, seed, col0=0), ops.completion_sample(L.buf, 150, seed, col0=150)])
    assert np.array_equal(Z, halves)
    N = Z.size
    assert abs(Z.mean()) <= 5.0 / np.sqrt(N) and abs(Z.var() - 1.0) <= 5.0 / np.sqrt(N), (Z.mean(), Z.var())
    # the public function: the same numbers in the original order
    import smcp_b200 as S
    out = S.completion_sample(sp.identity(n, format="csc"), 20, seed=seed)
    assert np.array_equal(out[order], Z[:, :20])


# (n, extra edges, bandwidth, seed): band, sparse random with fill, filled pattern with a dense top set (bigfront.cu)
SAMPLE_PATTERNS = [(200, 0, 4, 0), (150, 120, 2, 6), (700, 6000, 2, 3)]


def _completable(n, nextra, bw, seed):
    cp, ri = random_pattern(n, nextra, bw, seed)
    cols = np.repeat(np.arange(n), np.diff(cp))
    rng = np.random.default_rng(seed + 100)
    G = rng.standard_normal((n, n + 5)) / np.sqrt(n)
    M = G @ G.T + 0.5 * np.eye(n)
    return sp.csc_matrix((M[ri, cols], (ri, cols)), shape=(n, n))


@pytest.mark.gpu
@pytest.mark.parametrize("pat", SAMPLE_PATTERNS)
@pytest.mark.parametrize("k", [1, 31, 32, 257])
def test_samples_match_dense_factor(pat, k):
    """V = L^-T G with L the dense factor of X_hat^-1 and G from the twin (both sides of k_trsm's nrhs >= 32)."""
    import smcp_b200 as S
    from smcp_b200.base import _completion_factor
    _device()
    X = _completable(*pat)
    L, order = _completion_factor(X)
    if pat[1] > 1000:
        big = np.diff(L.ops.symb.rowptr).max()
        assert big >= 300, big                  # the top set goes through the dense multi-CTA path
    V = L.ops.completion_sample(L.buf, k, 77)
    Xh = S.completion(X)[np.ix_(order, order)]
    Ld = np.linalg.cholesky(np.linalg.inv(Xh))
    ref = sl.solve_triangular(Ld, normals(X.shape[0], k, 77), lower=True, trans="T")
    assert np.linalg.norm(V - ref) <= 1e-10 * np.linalg.norm(ref)


@pytest.mark.gpu
def test_sample_covariance_is_the_completion():
    import smcp_b200 as S
    _device()
    X = _completable(30, 20, 1, 4)
    Z = S.completion_sample(X, 20000, seed=9)
    C = Z @ Z.T / Z.shape[1]
    assert np.abs(C - S.completion(X)).max() <= 0.05


def _round_case(seed):
    P = _graph(60, 100, seed)
    return P, {"x": _unit_diag_on_pattern(P, seed)}


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [1, 2])
def test_round_values_match_host_evaluation(seed):
    import smcp_b200 as S
    _device()
    P, sol = _round_case(seed)
    trials = 600
    r = P.round_pm1(sol, trials=trials, seed=seed)
    V = S.completion_sample(sol["x"], trials, seed=seed)
    assert (np.abs(V) > 1e-9 * np.linalg.norm(V, axis=0)).all()        # no sign is decided by rounding error
    I, J, v = _objective(P)
    host = pm1_values(V, I, J, v)
    scale = 2.0 * np.abs(v).sum()
    assert np.abs(r["values"] - host).max() <= 1e-12 * scale
    t = int(np.flatnonzero(r["values"] == r["values"].min())[0])
    assert r["trial"] == t and r["value"] == r["values"][t]
    assert np.array_equal(r["x"], np.where(V[:, t] < 0.0, -1, 1).astype(np.int8))
    # pass sizes: 1 and 7 (one 200-column solve block per pass), 250 (two), 0 (everything)
    for chunk in (1, 7, 250, 0):
        q = P.round_pm1(sol, trials=trials, seed=seed, chunk=chunk)
        assert np.array_equal(q["values"], r["values"]) and np.array_equal(q["x"], r["x"]) and q["trial"] == r["trial"], chunk
    # the twin
    _twin()
    o = P.round_pm1(sol, trials=trials, seed=seed)
    assert np.abs(o["values"] - r["values"]).max() <= 1e-12 * scale
    assert o["trial"] == r["trial"] and np.array_equal(o["x"], r["x"])


@pytest.mark.gpu
def test_round_profile_families_and_usage_errors():
    from smcp_b200.base import _completion_factor
    from smcp_b200.device import DeviceError
    _device()
    P, sol = _round_case(3)
    L, order = _completion_factor(sol["x"])
    ops = L.ops
    ops.ctx.prof_reset()
    ops.ctx.prof_enable(True)
    try:
        ops.round_pm1(L.buf, [0, 1], [0, 0], [1.0, -0.5], 70, 1)
        names = ops.ctx.prof_names()
    finally:
        ops.ctx.prof_enable(False)
    assert "round_normal" in names and "round_eval" in names, names
    n = P.n
    for args in (([0], [n], [1.0], 4, 0, 0), ([-1], [0], [1.0], 4, 0, 0), ([0], [0], [1.0], 0, 0, 0), ([0], [0], [1.0], 4, 0, -1)):
        with pytest.raises(DeviceError):
            ops.round_pm1(L.buf, *args)


def _maxcut_cases():
    # graph seeds whose relaxation both drivers solve to optimal on the device: on the 12-vertex graph of seed 0,
    # solve_esd exits 'unknown' on the device (optimal on the oracle), and without a certified dual the bound
    # -dual objective of cut() means nothing
    return [(12, 1), (12, 3), (16, 0), (16, 1), (18, 0), (18, 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("n,seed", _maxcut_cases())
@pytest.mark.parametrize("method", ["feas", "esd"])
def test_cut_end_to_end(n, seed, method):
    from smcp_b200 import solvers
    _device()
    solvers.options["show_progress"] = False
    P = _graph(n, 2 * n, seed)
    if method == "feas":
        sol = P.solve_feas(primalstart={"x": sp.identity(n, format="csc")})
    else:
        sol = P.solve_esd()
    assert sol["status"] == "optimal", sol["status"]
    x, w, ub = P.cut(sol, trials=256)
    best = _brute_max_cut(P)
    assert w <= best + 1e-9 and best <= ub + 1e-6, (w, best, ub)
    assert w >= 0.878 * (-sol["primal objective"]) - 1e-6, (w, sol["primal objective"])


@pytest.mark.gpu
def test_cut_on_solver_graph():
    """The 40-vertex graph of test_gpu_solver.py."""
    import smcp_b200 as S
    from smcp_b200 import solvers
    _device()
    solvers.options["show_progress"] = False
    rng = np.random.default_rng(5)
    P = S.maxcut_SDP(40, rng.integers(0, 40, size=(70, 2)))
    sol = P.solve_esd()
    x, w, ub = P.cut(sol, trials=256, seed=3)
    assert w <= ub and w >= 0.878 * (-sol["primal objective"]) - 1e-6, (w, ub, sol["primal objective"])


@pytest.mark.gpu
def test_no_completion_raises():
    import smcp_b200 as S
    _device()
    X = sp.csc_matrix(np.array([[1.0, 2.0], [2.0, 1.0]]))
    with pytest.raises(ArithmeticError):
        S.completion(X)
    with pytest.raises(ArithmeticError):
        S.completion_sample(X, 4)
    P = S.maxcut_SDP(2, [(0, 1)])
    with pytest.raises(ArithmeticError):
        P.round_pm1({"x": X}, trials=4)
