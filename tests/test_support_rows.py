"""Dense-constraint copy on the support rows (the rows of blkval some constraint touches): selection, Schur
assembly, A(X), the phase-1 Gram matrix and end-to-end solves against the full copy and the CPU oracle."""
import contextlib
import os

import numpy as np
import pytest
import scipy.sparse as sp

pytestmark = pytest.mark.gpu

ENV = "SMCP_B200_AVW_SUPPORT"


@contextlib.contextmanager
def _support(mode):
    """SMCP_B200_AVW_SUPPORT around operator creation: None = automatic, "0" full copy, "1" support copy."""
    old = os.environ.pop(ENV, None)
    if mode is not None:
        os.environ[ENV] = mode
    try:
        yield
    finally:
        os.environ.pop(ENV, None)
        if old is not None:
            os.environ[ENV] = old


def _oracle():
    from oracle.backend import OracleBackend
    return lambda symb: OracleBackend(symb, batch_columns=16)


def _device():
    from smcp_b200.device import DeviceBackend
    return lambda symb: DeviceBackend(symb, small_work=5000)


def _problem(P, factory, mode=None, kkt="chol"):
    from smcp_b200 import solvers
    from smcp_b200.solvers import _Problem, _read_options
    solvers.set_backend_factory(factory)
    with _support(mode):
        return _Problem(P.A, P.b, _read_options(P.n, False), kkt, None)


def _pattern(n, seed=0):
    """Tridiagonal plus 6n random pairs (the aggregate pattern of the rand workloads): heavy fill."""
    rng = np.random.default_rng(seed)
    e = rng.integers(0, n, size=(6 * n, 2))
    I = np.concatenate([np.maximum(e[:, 0], e[:, 1]), np.arange(n), np.arange(1, n)])
    J = np.concatenate([np.minimum(e[:, 0], e[:, 1]), np.arange(n), np.arange(0, n - 1)])
    return sp.coo_matrix((np.ones(len(I)), (I, J)), shape=(n, n))


_CACHE = {}


def _make(kind):
    if kind in _CACHE:
        return _CACHE[kind]
    import smcp_b200 as S
    from smcp_b200 import solvers
    from test_gpu_solver import _make as make_existing
    solvers.set_backend_factory(_oracle())        # the generators probe the cone
    if kind == "dense300":
        P = S.rand_SDP(_pattern(300), 700, density=1.0, seed=0)
    elif kind == "dense80":
        P = S.rand_SDP(_pattern(80, seed=1), 60, density=1.0, seed=2)
    elif kind == "dense500":
        P = S.rand_SDP(_pattern(500, seed=3), 2100, density=1.0, seed=4)
    elif kind == "mixed80":
        P = S.rand_SDP(_pattern(80, seed=5), 50, density=[0.9] * 15 + [0.002] * 35, seed=6)
    else:
        P = make_existing(kind)
    _CACHE[kind] = P
    return P


def _support_rows(pr):
    return len(np.unique(pr.symb.vec2blk[pr.Av.indices]))


def _scaling_point(symb, seed=0):
    rng = np.random.default_rng(seed)
    s = np.zeros(symb.nvp)
    s[symb.diag_vec] = 2.0
    s += 0.05 * rng.standard_normal(symb.nvp)
    return s


def _token(pr, s):
    from smcp_b200.chordal import cspmatrix, cholesky, projected_inverse, schur_token
    L = cspmatrix.from_vec(pr.ops, s)
    cholesky(L)
    Y = L.copy()
    projected_inverse(Y)
    return schur_token(L, Y), (L, Y)


def _schur(pr, s):
    tok, keep = _token(pr, s)
    pr.ops.schur_assemble(tok)
    if getattr(pr.ops, "lib", None) is None:
        return np.tril(pr.ops.H.copy())
    return np.tril(pr.ops.get_H())


def _rel(a, b):
    return np.linalg.norm(a - b) / np.linalg.norm(b)


def _set_H_zero(ops):
    from smcp_b200.device import _ck
    _ck(ops.lib, ops.lib.smcp_kkt_set_H(ops._op, np.zeros(ops.m * ops.m)))


def test_selection():
    P = _make("dense300")
    pd = _problem(P, _device())
    assert pd.Ns == 0 and pd.m == 700
    nsup = _support_rows(pd)
    assert nsup <= 0.25 * pd.symb.nblk
    assert pd.ops.dense_rows() == nsup
    assert _problem(P, _device(), "0").ops.dense_rows() == pd.symb.nblk
    assert _problem(P, _device(), "1").ops.dense_rows() == nsup
    for kind in ("band", "mtxnorm", "rand_mixed"):
        pr = _problem(_make(kind), _device())
        assert pr.ops.dense_rows() == pr.symb.nblk, kind
        assert _problem(_make(kind), _device(), "1").ops.dense_rows() == _support_rows(pr), kind
    # no dense constraint: no copy
    pr = _problem(_make("rand_sparse"), _device())
    assert pr.m > 0 and pr.Ns == pr.m and pr.ops.dense_rows() == 0


def test_schur_and_amap_support_vs_full():
    """dense300: H from the support copy matches the full copy, two assemblies give the same bits, the gather has
    its own profile family and the contraction stays schur_gemm_dmma; A(X) on both copies."""
    from smcp_b200.chordal import cspmatrix
    P = _make("dense300")
    pf, ps = _problem(P, _device(), "0"), _problem(P, _device())
    assert ps.ops.dense_rows() < pf.ops.dense_rows()
    s = _scaling_point(ps.symb)
    Hf = _schur(pf, s)
    ctx = ps.ops.ctx
    ctx.prof_enable(True)
    ctx.prof_reset()
    Hs = _schur(ps, s)
    fam = {nm for nm in ctx.prof_names() if ctx.prof_get(nm)[1] > 0}
    ctx.prof_enable(False)
    assert "support_gather" in fam and "schur_gemm_dmma" in fam, sorted(fam)
    assert _rel(Hs, Hf) <= 1e-12
    assert np.array_equal(_schur(ps, s), Hs)
    v = np.random.default_rng(1).standard_normal(ps.symb.nvp)
    af = pf.Amap(cspmatrix.from_vec(pf.ops, v))
    as_ = ps.Amap(cspmatrix.from_vec(ps.ops, v))
    assert _rel(as_, af) <= 1e-12


@pytest.mark.parametrize("kind", ["dense80", "mixed80"])
def test_schur_and_amap_against_oracle(kind):
    """Support copy forced on a filled pattern: H against the oracle to 1e-11 and the full copy to 1e-12; Amap (all
    columns and one column) against the oracle.  mixed80 has dense and sparse constraints together."""
    from smcp_b200.chordal import cspmatrix
    P = _make(kind)
    po = _problem(P, _oracle())
    pf, ps = _problem(P, _device(), "0"), _problem(P, _device(), "1")
    assert ps.ops.dense_rows() == _support_rows(ps) < ps.symb.nblk
    if kind == "mixed80":
        assert 0 < ps.Ns < ps.m and po.Ns == ps.Ns
    s = _scaling_point(po.symb, 3)
    Ho, Hf, Hs = _schur(po, s), _schur(pf, s), _schur(ps, s)
    assert _rel(Hs, Ho) <= 1e-11
    assert _rel(Hs, Hf) <= 1e-12
    v = np.random.default_rng(2).standard_normal(po.symb.nvp)
    ao = po.Amap(cspmatrix.from_vec(po.ops, v))
    assert _rel(ps.Amap(cspmatrix.from_vec(ps.ops, v)), ao) <= 1e-12
    for i in (0, ps.m // 2, ps.m - 1):
        assert abs(ps.Amap(cspmatrix.from_vec(ps.ops, v), i) - ao[i]) <= 1e-12 * np.linalg.norm(ao)


def test_chunks_ranges_and_cyclic():
    """m = 2100 crosses a batch boundary of the Hessian workspace (2048 columns).  Column ranges of
    smcp_kkt_assemble and the block-cyclic columns of smcp_kkt_assemble_cyclic (3 ranks, block 128) match the
    full assembly on the support copy, which matches the full copy."""
    from smcp_b200.device import _ck
    P = _make("dense500")
    ps = _problem(P, _device(), "1")
    m = ps.m
    assert m > 2048 and ps.Ns == 0 and ps.ops.dense_rows() < ps.symb.nblk
    s = _scaling_point(ps.symb, 5)
    tok, keep = _token(ps, s)          # keep: the factors the token refers to
    ops = ps.ops
    ops.schur_assemble(tok)
    H = np.tril(ops.get_H())
    scale = np.linalg.norm(H)
    assert np.isfinite(H).all()
    for j0, j1 in ((0, 1), (5, 700), (700, 2050), (2040, 2100)):
        _set_H_zero(ops)
        ops.schur_assemble(tok, j0, j1)
        Hr = np.tril(ops.get_H())
        assert np.linalg.norm(Hr[:, j0:j1] - H[:, j0:j1]) <= 1e-12 * scale, (j0, j1)
        assert not Hr[:, :j0].any() and not Hr[:, j1:].any()
    for rank in range(3):
        _set_H_zero(ops)
        _ck(ops.lib, ops.lib.smcp_kkt_assemble_cyclic(ops._op, tok, 128, rank, 3))
        Hr = np.tril(ops.get_H())
        own = np.zeros(m, dtype=bool)
        for c0 in range(rank * 128, m, 3 * 128):
            own[c0:c0 + 128] = True
        assert np.linalg.norm(Hr[:, own] - H[:, own]) <= 1e-12 * scale, rank
        assert not Hr[:, ~own].any()
    pf = _problem(P, _device(), "0")
    assert _rel(H, _schur(pf, s)) <= 1e-12


def _gram(P):
    """<A_i, A_j> (trace inner product) from the lower-triangle columns of P.A."""
    n = P.n
    A = P.A[:, 1:].tocsc()
    I, J = np.arange(A.shape[0]) % n, np.arange(A.shape[0]) // n
    w = np.where(I == J, 1.0, 2.0)
    return (A.T @ sp.diags(w) @ A).toarray()


def test_gram_support():
    from smcp_b200.device import DeviceError
    P = _make("dense80")
    pq = _problem(P, _device(), "1", kkt="qr")
    assert pq.Ns == 0 and pq.ops.dense_rows() == _support_rows(pq)
    pq.ops.gram_factor()
    L = np.tril(pq.ops.get_H())
    G = _gram(P)
    pm = np.argsort(pq.inv_pm)          # column k of Av is constraint pm[k]
    G = G[np.ix_(pm, pm)]
    assert _rel(L @ L.T, G) <= 1e-12
    with pytest.raises(DeviceError):
        pq.ops.z_tmul(pq.C.buf)


def _feas(P, factory, mode, kktsolver="chol"):
    from smcp_b200 import solvers
    solvers.options["show_progress"] = False
    solvers.set_backend_factory(factory)
    with _support(mode):
        return P.solve_feas(kktsolver=kktsolver, primalstart={"x": P._X0} if P._X0 is not None else None)


def _agree(a, b, tol):
    assert a["status"] == b["status"], (a["status"], b["status"])
    assert abs(a["iterations"] - b["iterations"]) <= 1, (a["iterations"], b["iterations"])
    for key in ("primal objective", "dual objective"):
        assert abs(a[key] - b[key]) <= tol * max(1.0, abs(a[key])), (key, a[key], b[key])


def test_solve_feas_support_vs_full():
    P = _make("dense300")
    a = _feas(P, _device(), "0")
    b = _feas(P, _device(), None)
    assert a["status"] == "optimal"
    _agree(a, b, 1e-8)


def test_solve_feas_support_vs_oracle():
    P = _make("dense80")
    a = _feas(P, _oracle(), None)
    b = _feas(P, _device(), "1")
    assert a["status"] == "optimal"
    _agree(a, b, 1e-8)


def test_solve_phase1_support():
    from smcp_b200 import solvers
    P = _make("dense80")
    solvers.options["show_progress"] = False
    solvers.set_backend_factory(_device())
    with _support("1"):
        X0, sol = P.solve_phase1()
    assert X0 is not None
    n = P.n
    x = X0.toarray().ravel(order="F")
    I, J = np.arange(n * n) % n, np.arange(n * n) // n
    w = np.where(I == J, 1.0, 2.0)
    r = P.A[:, 1:].T @ (w * x) - P.b
    assert np.linalg.norm(r) <= 1e-9 * np.linalg.norm(P.b), (np.linalg.norm(r), sol is None)


def test_solve_esd_qr_support_vs_full():
    """kktsolver='qr' (SYRK form) on a problem that selects the support copy against the full copy.  Z^T Z squares
    the condition of Z, and near the optimum this instance sits on the edge (one run may stop 'unknown', the other
    'optimal'), so the first 12 iterates are compared: the same iterations, costs and gaps to 1e-8."""
    from smcp_b200 import solvers
    P = _make("dense80")
    out = []
    for mode in ("0", None):
        solvers.options["show_progress"] = False
        solvers.options["maxiters"] = 12
        solvers.set_backend_factory(_device())
        with _support(mode):
            out.append(P.solve_esd(kktsolver="qr"))
        assert solvers._last_problem.ops.dense_rows() == (_support_rows(solvers._last_problem) if mode is None
                                                          else solvers._last_problem.symb.nblk)
    a, b = out
    assert a["iterations"] == b["iterations"] and len(a["trace"]) == len(b["trace"]) >= 8
    for ra, rb in zip(a["trace"], b["trace"]):
        for key in ("pcost", "dcost", "gap"):
            if ra.get(key) is not None:
                assert abs(ra[key] - rb[key]) <= 1e-8 * max(1.0, abs(ra[key])), (key, ra, rb)
