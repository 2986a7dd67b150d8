"""kktsolver='qr' in Householder form (options['qr_method'] = 'householder'): the oracle's Q-form on the CPU,
and on the device the blocked Householder QR (lapack.geqrf / orgqr parity), the KKT-level factor and solve,
and end-to-end runs against the oracle."""
import numpy as np
import pytest
import scipy.sparse as sp


def _oracle_factory():
    from qr_oracle import QROracleBackend
    return lambda symb: QROracleBackend(symb)


def _make(kind):
    import smcp_b200 as S
    from smcp_b200 import solvers
    solvers.set_backend_factory(_oracle_factory())      # the generators probe the cone
    if kind == "band":
        return S.band_SDP(40, 12, 3, seed=2)
    if kind == "mtxnorm":
        return S.mtxnorm_SDP(12, 4, 9, density=0.6, seed=1)
    if kind.startswith("rand25-s"):
        return S.rand_SDP(sp.csc_matrix(np.tril(np.ones((25, 25)))), 8, density=1.0, seed=int(kind[len("rand25-s"):]))
    raise ValueError(kind)


def _problem(P, factory, A=None, b=None):
    from smcp_b200 import solvers
    solvers.set_backend_factory(factory)
    opt = solvers._read_options(P.n, False)
    return solvers._Problem(P.A if A is None else A, P.b if b is None else b, opt, "qr", None)


def _scaling_point(prob, seed):
    """L = chol(S), Y = the projected inverse, for S = 2I + a small symmetric perturbation on the pattern."""
    from smcp_b200.chordal import cspmatrix, cholesky, projected_inverse
    symb = prob.symb
    rng = np.random.default_rng(seed)
    s = np.zeros(symb.nvp)
    s[symb.diag_vec] = 2.0
    s += 0.05 * rng.standard_normal(symb.nvp)
    L = cspmatrix.from_vec(prob.ops, s)
    cholesky(L)
    Y = L.copy()
    projected_inverse(Y)
    return L, Y


def _rel(a, b):
    return np.linalg.norm(np.asarray(a) - np.asarray(b)) / max(np.linalg.norm(np.asarray(b)), 1e-300)


E2E = ["band", "mtxnorm", "rand25-s1", "rand25-s2", "rand25-s7"]


# ---------------------------------------------------------------------------------------------------------
# CPU: the oracle's Q-form
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", E2E)
def test_oracle_householder_exits_optimal(kind):
    """The Q-form exits where the SYRK form may not (rand25 seed 1 ends 'unknown' in the SYRK form)."""
    from smcp_b200 import solvers
    P = _make(kind)
    solvers.options["show_progress"] = False
    solvers.options["qr_method"] = "householder"
    sol = P.solve_esd(kktsolver="qr")
    assert sol["status"] == "optimal", (kind, sol["status"], sol["iterations"])


@pytest.mark.parametrize("kind", E2E)
def test_oracle_qform_solve_matches_syrk_form(kind):
    """One KKT system at a scaling point, solved by _KKTqr (H = Z^T Z, Cholesky) and by _KKTqrh (through Q and R):
    the same x and y to 1e-10."""
    from smcp_b200 import solvers
    from smcp_b200.chordal import cspmatrix
    P = _make(kind)
    prob = _problem(P, _oracle_factory())
    L, Y = _scaling_point(prob, 3)
    rng = np.random.default_rng(7)
    bx = cspmatrix.from_vec(prob.ops, rng.standard_normal(prob.symb.nvp))
    by = rng.standard_normal(prob.m)
    out = []
    for cls in (solvers._KKTqr, solvers._KKTqrh):
        f = cls(prob, L, Y, "primal")
        x, y = f.solve(bx, by, 0.7)
        out.append((x.to_vec(), np.asarray(y)))
    (xs, ys), (xh, yh) = out
    assert _rel(yh, ys) <= 1e-10, _rel(yh, ys)
    assert _rel(xh, xs) <= 1e-10, _rel(xh, xs)


def test_qr_method_option_is_validated():
    from smcp_b200 import solvers
    P = _make("band")
    solvers.options["show_progress"] = False
    solvers.options["qr_method"] = "bogus"
    with pytest.raises(ValueError, match="qr_method"):
        P.solve_esd(kktsolver="qr")


def test_qr_method_picks_the_kkt_class(monkeypatch):
    """'householder' selects _KKTqrh for kktsolver='qr' only; kktsolver='chol' ignores the option."""
    from smcp_b200 import solvers
    P = _make("band")
    prob = _problem(P, _oracle_factory())
    L, Y = _scaling_point(prob, 1)
    for method, cls in (("syrk", solvers._KKTqr), ("householder", solvers._KKTqrh)):
        prob.qr_method = method
        assert type(solvers._make_kkt(prob, L, Y, "primal")) is cls
    chol = type("Chol", (), {"__init__": lambda self, *args: None})
    monkeypatch.setattr(solvers, "_KKT", chol)
    prob.kktsolver = "chol"
    prob.qr_method = "householder"
    assert type(solvers._make_kkt(prob, L, Y, "primal")) is chol


# ---------------------------------------------------------------------------------------------------------
# GPU: dense geqrf / orgqr
# ---------------------------------------------------------------------------------------------------------
def _dev_geqrf(A):
    import ctypes as C
    from smcp_b200.device import Context, _ck
    ctx = Context.get()
    M, N = A.shape
    a = np.asfortranarray(A, dtype=np.float64).copy(order="F")
    flat = a.reshape(-1, order="F")
    tau = np.zeros(N)
    ms = C.c_double()
    _ck(ctx.lib, ctx.lib.smcp_dense_geqrf(ctx.h, flat, M, M, N, tau, C.byref(ms)))
    return flat.reshape((M, N), order="F"), tau


def _dev_orgqr(QR, tau):
    import ctypes as C
    from smcp_b200.device import Context, _ck
    ctx = Context.get()
    M, N = QR.shape
    flat = np.asfortranarray(QR).copy(order="F").reshape(-1, order="F")
    ms = C.c_double()
    _ck(ctx.lib, ctx.lib.smcp_dense_orgqr(ctx.h, flat, M, M, N, np.ascontiguousarray(tau), C.byref(ms)))
    return flat.reshape((M, N), order="F")


SHAPES = [(1, 1), (7, 3), (160, 12), (513, 65), (4097, 257), (30000, 1000), (300000, 40)]


@pytest.mark.gpu
@pytest.mark.parametrize("M,N", SHAPES)
def test_dense_geqrf_orgqr_match_lapack(M, N):
    """Same convention as LAPACK (R, Householder vectors, tau, Q1) to 1e-12 in relative Frobenius norm.
    300000 x 40: the panel slab of a CTA does not fit in shared memory and is read from global memory."""
    from scipy.linalg import lapack
    A = np.random.default_rng(M + N).standard_normal((M, N))
    qr_ref, tau_ref, _, info = lapack.dgeqrf(A)
    assert info == 0
    q_ref, _, info = lapack.dorgqr(qr_ref, tau_ref)
    assert info == 0
    qr, tau = _dev_geqrf(A)
    assert _rel(np.triu(qr), np.triu(qr_ref)) <= 1e-12
    assert _rel(np.tril(qr, -1), np.tril(qr_ref, -1)) <= 1e-12 or M == 1
    assert np.abs(tau - tau_ref).max() <= 1e-12 * max(1.0, np.abs(tau_ref).max())
    q = _dev_orgqr(qr, tau)
    assert _rel(q, q_ref) <= 1e-12


@pytest.mark.gpu
@pytest.mark.parametrize("M,N", [(4097, 257), (30000, 1000)])
def test_dense_qr_ill_conditioned_is_backward_stable(M, N):
    rng = np.random.default_rng(5)
    U, _ = np.linalg.qr(rng.standard_normal((M, N)))
    V, _ = np.linalg.qr(rng.standard_normal((N, N)))
    A = (U * np.logspace(0, -12, N)[None, :]) @ V.T          # cond(A) = 1e12
    qr, tau = _dev_geqrf(A)
    R = np.triu(qr[:N])
    Q = _dev_orgqr(qr, tau)
    assert _rel(Q @ R, A) <= 1e-12
    assert np.abs(Q.T @ Q - np.eye(N)).max() <= 1e-12


@pytest.mark.gpu
def test_dense_qr_is_deterministic():
    A = np.random.default_rng(9).standard_normal((30000, 300))
    a1, t1 = _dev_geqrf(A)
    a2, t2 = _dev_geqrf(A)
    assert np.array_equal(a1, a2) and np.array_equal(t1, t2)
    assert np.array_equal(_dev_orgqr(a1, t1), _dev_orgqr(a2, t2))


# ---------------------------------------------------------------------------------------------------------
# GPU: KKT level and end to end
# ---------------------------------------------------------------------------------------------------------
def _dev_factory():
    from smcp_b200.device import DeviceBackend
    return lambda symb: DeviceBackend(symb, small_work=5000)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["band", "mtxnorm", "rand25-s2"])
def test_kkt_factor_and_solve_match(kind):
    """L L^T equals the SYRK-form H; qr_solve equals the oracle's Q-form; the SYRK-form products refuse while
    Zq holds Q1."""
    from smcp_b200.chordal import schur_token
    from smcp_b200.device import DeviceError, _ck
    P = _make(kind)
    po, pd = _problem(P, _oracle_factory()), _problem(P, _dev_factory())
    Lo, Yo = _scaling_point(po, 2)
    Ld, Yd = _scaling_point(pd, 2)
    td, to = schur_token(Ld, Yd), schur_token(Lo, Yo)
    with pytest.raises(DeviceError):
        pd.ops.qr_solve(Ld.buf, np.zeros(pd.m))               # no factorisation yet
    _ck(pd.ops.lib, pd.ops.lib.smcp_kkt_assemble_syrk(pd.ops._op, td))       # H = Z^T Z, not yet factored
    H = np.tril(pd.ops.get_H())
    pd.ops.schur_factor_householder(td)
    Lf = np.tril(pd.ops.get_H())
    assert np.all(np.diag(Lf) > 0)
    assert _rel(np.tril(Lf @ Lf.T), H) <= 1e-12
    with pytest.raises(DeviceError):
        pd.ops.z_tmul(Ld.buf)
    with pytest.raises(DeviceError):
        pd.ops.z_mul(np.zeros(pd.m))
    po.ops.schur_factor_householder(to)
    rng = np.random.default_rng(4)
    g = rng.standard_normal(po.symb.nblk)
    r = rng.standard_normal(po.m)
    yo, xo = po.ops.qr_solve(g, r)
    gbuf = pd.ops.set_blk(g)
    yd, xbuf = pd.ops.qr_solve(gbuf, r)
    xd = pd.ops.get_blk(xbuf)
    pd.ops.release(xbuf)
    pd.ops.release(gbuf)
    assert _rel(yd, yo) <= 1e-10, _rel(yd, yo)
    assert _rel(xd, xo) <= 1e-10, _rel(xd, xo)


@pytest.mark.gpu
def test_kkt_factor_rank_deficient_raises():
    """A duplicated constraint makes Z rank deficient: R has a zero on its diagonal."""
    from smcp_b200.chordal import schur_token
    P = _make("band")
    A = sp.csc_matrix(P.A)
    A2 = sp.hstack([A, A[:, 1]], format="csc")
    b2 = np.append(np.asarray(P.b, dtype=np.float64).ravel(), float(np.ravel(P.b)[0]))
    pd = _problem(P, _dev_factory(), A2, b2)
    L, Y = _scaling_point(pd, 2)
    with pytest.raises(ArithmeticError):
        pd.ops.schur_factor_householder(schur_token(L, Y))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", E2E)
def test_esd_householder_gpu(kind):
    """solve_esd(kktsolver='qr') in Householder form on the device exits optimal where the oracle's Q-form does
    (band: the instance the SYRK form lets go 'unknown' on the device).  The objectives agree to 1e-7 when both
    runs exit at the same iteration.  The self-dual embedding's exit iteration is not reproducible across
    rounding (DESIGN.md section 2); when the runs exit at different iterations, each objective is only as
    accurate as the duality gap its run certifies, and they must agree to the larger of the two gaps."""
    from smcp_b200 import solvers
    P = _make(kind)
    out = []
    for fac in (_oracle_factory(), _dev_factory()):
        solvers.options["show_progress"] = False
        solvers.options["qr_method"] = "householder"
        solvers.set_backend_factory(fac)
        out.append(P.solve_esd(kktsolver="qr"))
    a, b = out
    assert a["status"] == "optimal", a["status"]
    assert b["status"] == "optimal", (b["status"], b["iterations"])
    for key in ("primal objective", "dual objective"):
        tol = 1e-7 * max(1.0, abs(a[key]))
        if a["iterations"] != b["iterations"]:
            tol = max(tol, a["gap"], b["gap"])
        assert abs(a[key] - b[key]) <= tol, (key, a[key], b[key], a["iterations"], b["iterations"], a["gap"], b["gap"])


@pytest.mark.gpu
def test_feas_householder_gpu():
    from smcp_b200 import solvers
    P = _make("band")
    out = []
    for fac in (_oracle_factory(), _dev_factory()):
        solvers.options["show_progress"] = False
        solvers.options["qr_method"] = "householder"
        solvers.set_backend_factory(fac)
        out.append(P.solve_feas(kktsolver="qr", primalstart={"x": P._X0} if P._X0 is not None else None))
    a, b = out
    assert a["status"] == "optimal" and b["status"] == "optimal", (a["status"], b["status"])
    assert abs(a["iterations"] - b["iterations"]) <= 1, (a["iterations"], b["iterations"])
    for key in ("primal objective", "dual objective"):
        assert abs(a[key] - b[key]) <= 1e-7 * max(1.0, abs(a[key])), (key, a[key], b[key])
