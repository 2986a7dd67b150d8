"""Sparse-constraint columns of the Schur complement (misc.SCMcolumn2 on the dense inverse Z = S^-1) in every
dispatch bucket of assemble_sparse_range (csrc/capi.cu), against H_ij = tr(A_i Z A_j Z) in float64 on the host.

The kernel form is picked from the shape of the constraint data:

* E = min(64, 25600 / 2n) columns of Z staged per round; E < 2 (n > 6400), more than 32 * 512 = 16384 positions,
  or fewer than 3 entries per sparse column on average: the pairwise form scm_sparse;
* otherwise kpos = ceil(npos / 512) picks the template KPOS = 8 / 16 / 32 of scm_position and scm_kstream;
* nnz_sp >= 2 npos (and K within SMCP_B200_SCM_KMAT_GB): the materialised K (scm_kmat + scm_kstream), otherwise
  scm_position, which stages Z in ceil(nnz_j / E) rounds;
* the longest sparse column w <= 2 avg + 8: the ELL row walk of scm_rows, otherwise the CSR walk.

Every case below is built from the symbolic pattern, S and Av directly, so that it lands in exactly one bucket;
test_case_buckets recomputes the rule from Av without a GPU.  The reference forms the position kernel matrix
K[(p,q),(r,c)] = Z_pr Z_qc + [p != q] Z_qr Z_pc by blocks of positions and takes H = B^T K A' (A' doubled off the
diagonal), with the same sums on |Z|, |A'|, |B| as the error scale; test_reference_has_teeth shows that the check
rejects each of the ways a kernel could be subtly wrong."""
import contextlib
import os

import numpy as np
import pytest
import scipy.sparse as sp

CAP = 25600          # doubles of dynamic shared memory the position kernels stage (assemble_sparse_range)
SCM_T = 512          # threads (positions per register slot) of scm_position / scm_kstream
KMAT_ENV = "SMCP_B200_SCM_KMAT_GB"
FAMILY = {"kstream": "scm_kstream", "position": "scm_position", "pairwise": "scm_sparse"}
RTOL, CTOL = 1e-12, 1e-14
SENTINEL = -7.25e77

# name: n, band half-width (None: dense lower pattern), npos, per-column entry counts (cycled over Ns sparse
# columns), Ns, md dense columns in front, expected (form, KPOS, row walk); `last` overrides the last count
CASES = {
    # E = 64 at n = 200: columns of 65 and 129 entries stage Z in 2 and 3 rounds, 64 in exactly one
    "kpos8_npos512": dict(n=200, npos=512, counts=[1, 3, 63, 64, 65, 129, 100, 100, 100, 100], Ns=40,
                          expect=("kstream", 8, "ell")),
    "kpos8_npos4096": dict(n=200, npos=4096, counts=[1, 3, 63, 64, 65, 129, 100, 100, 100, 100], Ns=120,
                           expect=("kstream", 8, "ell")),
    "kpos16_npos4097": dict(n=200, npos=4097, counts=[3, 7, 20, 33, 40, 17], Ns=420, expect=("kstream", 16, "ell")),
    "kpos16_npos8192": dict(n=200, npos=8192, counts=[3, 7, 20, 33, 40, 17], Ns=840, expect=("kstream", 16, "ell")),
    "kpos32_npos8193": dict(n=200, npos=8193, counts=[3, 7, 20, 33, 40, 17], Ns=840, expect=("kstream", 32, "ell")),
    "kpos32_npos16384": dict(n=200, npos=16384, counts=[3, 7, 20, 33, 40, 17], Ns=1650, expect=("kstream", 32, "ell")),
    "npos_cap_16385": dict(n=200, npos=16385, counts=[3, 7, 20, 33, 40, 17], Ns=1650, expect=("pairwise", None, None)),
    # average exactly 3.0, then one entry fewer (nnz_sp < 2 npos: the direct position form)
    "avg_3": dict(n=200, npos=401, counts=[3], Ns=200, expect=("position", 8, "ell")),
    "avg_below_3": dict(n=200, npos=401, counts=[3], Ns=200, last=2, expect=("pairwise", None, None)),
    # nnz_sp = 2 npos = 1024 over 322 columns (1024 / 322 * 322 rounds below 1024), then 1023
    "kform_edge": dict(n=200, npos=512, counts=[4] * 58 + [3] * 264, Ns=322, expect=("kstream", 8, "ell")),
    "kform_below": dict(n=200, npos=512, counts=[4] * 57 + [3] * 265, Ns=322, expect=("position", 8, "ell")),
    # one column of 40 entries among columns of 8: w > 2 avg + 8
    "csr_kpos8": dict(n=200, npos=2000, counts=[8], Ns=600, last=40, expect=("kstream", 8, "csr")),
    "csr_kpos16": dict(n=200, npos=6000, counts=[8], Ns=1600, last=40, expect=("kstream", 16, "csr")),
    # the C3 shape: E = 6, 80 entries per column = 13 full staging rounds and a partial one
    "c3_staging": dict(n=2000, bw=6, npos=12000, counts=[80], Ns=320, expect=("kstream", 32, "ell")),
    # E = 2 at n = 6400 (2 E n = 25600: the whole staging buffer), odd column lengths; E = 1 at n = 6401
    "e_edge_6400": dict(n=6400, bw=2, npos=600, counts=[3, 5, 7], Ns=300, expect=("kstream", 8, "ell")),
    "e_edge_6401": dict(n=6401, bw=2, npos=600, counts=[3, 5, 7], Ns=300, expect=("pairwise", None, None)),
    # dense-technique columns in front of sparse ones
    "mixed": dict(n=200, npos=6000, counts=[3, 9, 15], Ns=1500, md=24, md_nnz=400, expect=("kstream", 16, "ell")),
}


class Case:
    """Pattern, constraints and the entry coordinates (original order) of one dispatch case."""

    def __init__(self, name):
        from smcp_b200.symbolic import Symbolic, lower_pattern
        spec = CASES[name]
        self.name = name
        self.spec = spec
        n, npos, Ns, md = spec["n"], spec["npos"], spec["Ns"], spec.get("md", 0)
        self.n, self.Ns, self.md, self.m = n, Ns, md, md + Ns
        bw = spec.get("bw")
        if bw is None:                          # dense lower pattern: one supernode, n (n + 1) / 2 positions
            I, J = np.tril_indices(n)
        else:
            J = np.repeat(np.arange(n), bw + 1)
            I = J + np.tile(np.arange(bw + 1), n)
            keep = I < n
            I, J = I[keep], J[keep]
        colptr, rowind = lower_pattern(n, I, J)
        self.symb = symb = Symbolic(n, colptr, rowind)
        self.Ip, self.Jp = symb.Ip, symb.Jp          # (row, col) of every vector-space entry, row >= col
        rng = np.random.default_rng(sum(map(ord, name)))
        # the positions: a quarter diagonal (as far as there are diagonal entries), the rest off the diagonal
        diag = symb.diag_vec
        off = np.setdiff1d(np.arange(symb.nvp), diag)
        nd = min(len(diag), npos // 4)
        pos = rng.permutation(np.concatenate([rng.choice(diag, nd, replace=False),
                                              rng.choice(off, npos - nd, replace=False)]))
        counts = np.resize(np.asarray(spec["counts"], dtype=np.int64), Ns)
        if "last" in spec:
            counts[-1] = spec["last"]
        assert counts.sum() >= npos and counts.max() <= npos
        # sparse column j takes the next counts[j] positions of the cyclic sequence pos: distinct within a column,
        # and every position is used
        rows = pos[np.arange(counts.sum()) % npos]
        cols = md + np.repeat(np.arange(Ns), counts)
        if md:
            rows = np.concatenate([np.concatenate([rng.choice(pos, spec["md_nnz"], replace=False) for _ in range(md)]),
                                   rows])
            cols = np.concatenate([np.repeat(np.arange(md), spec["md_nnz"]), cols])
        vals = rng.uniform(0.5, 1.5, len(rows)) * rng.choice([-1.0, 1.0], len(rows))
        self.Av = sp.csc_matrix((vals, (rows, cols)), shape=(symb.nvp, self.m))
        self.Av.sort_indices()
        assert self.Av.nnz == len(rows)

    def scaling_point(self, seed):
        """Values (vector space) of a strictly diagonally dominant S with cond(S) < 5 on the pattern: on the dense
        pattern diag + two rank-one terms whose sum never cancels, so that no entry of Z is tiny."""
        rng = np.random.default_rng(seed)
        n, Ip, Jp = self.n, self.Ip, self.Jp
        if self.spec.get("bw") is None:
            u1 = rng.uniform(0.5, 1.0, n) * rng.choice([-1.0, 1.0], n)
            u2 = 0.3 * rng.uniform(0.5, 1.0, n) * rng.choice([-1.0, 1.0], n)
            d = n * rng.uniform(2.0, 3.0, n)
            return (u1[Ip] * u1[Jp] + u2[Ip] * u2[Jp] + np.where(Ip == Jp, d[Ip], 0.0)) / n
        s = rng.uniform(0.5, 1.0, len(Ip)) * rng.choice([-1.0, 1.0], len(Ip))
        offd = Ip != Jp
        rowsum = np.zeros(n)
        np.add.at(rowsum, Ip[offd], np.abs(s[offd]))
        np.add.at(rowsum, Jp[offd], np.abs(s[offd]))
        s[~offd] = 1.5 * rowsum[Ip[~offd]] + 1.0
        return s


_CASES = {}
_REFS = {}


def _case(name):
    if name not in _CASES:
        _CASES[name] = Case(name)
    return _CASES[name]


def rule(case):
    """The dispatch rule of assemble_sparse_range, recomputed in exact arithmetic from Av."""
    Av, md, m, n = case.Av, case.md, case.m, case.n
    rows = Av.indices[Av.indptr[md]:]
    lens = np.diff(Av.indptr)[md:]
    npos, nnz_sp, Ns = len(np.unique(rows)), len(rows), m - md
    E = min(64, CAP // (2 * n))
    w = int(lens.max())
    kpos = -(-npos // SCM_T)
    ldk = npos + (npos & 1)
    position = E >= 2 and npos <= 32 * SCM_T and nnz_sp >= 3 * Ns
    if not position:
        form = "pairwise"
    elif ldk * npos * 8 <= 4 * 2 ** 30 and 2 * n <= CAP and nnz_sp >= 2 * npos:
        form = "kstream"
    else:
        form = "position"
    ell = w * Ns <= 2 * nnz_sp + 8 * Ns and w * Ns * 12 <= 2 ** 31        # w <= 2 avg + 8, ELL copy <= 2 GB
    return dict(form=form, npos=npos, nnz_sp=nnz_sp, avg=nnz_sp / Ns, E=E, w=w,
                kpos=(8 if kpos <= 8 else 16 if kpos <= 16 else 32) if position else None,
                walk=("ell" if ell else "csr") if position else None,
                rounds=-(-w // E))


def reference(case, s, block=2048):
    """(H, H_abs): H = B^T K A' over the positions every column touches, by blocks of `block` positions."""
    Z, pr, pc = _inverse(case, s)
    Ap, B = _operands(case)
    return _kform(Z, pr, pc, Ap, B, block=block)


def _inverse(case, s):
    """Z = S^-1 (float64) on the indices the positions touch, and the positions in those local indices."""
    Av, Ip, Jp, n = case.Av, case.Ip, case.Jp, case.n
    pos = np.unique(Av.indices)
    idx, loc = np.unique(np.concatenate([Ip[pos], Jp[pos]]), return_inverse=True)
    S = sp.csc_matrix((s, (Ip, Jp)), shape=(n, n))
    S = S + sp.triu(S.T, 1)
    if n <= 2000:
        Z = np.linalg.inv(S.toarray())[np.ix_(idx, idx)]
    else:
        from scipy.sparse.linalg import splu
        E = np.zeros((n, len(idx)))
        E[idx, np.arange(len(idx))] = 1.0
        Z = splu(S.tocsc(), permc_spec="NATURAL").solve(E)[idx]
    return Z, loc[:len(pos)], loc[len(pos):]


def _operands(case):
    """A' (values doubled off the diagonal) and B (undoubled) with one row per position of np.unique(Av.indices)."""
    Av = case.Av
    pos, rows = np.unique(Av.indices, return_inverse=True)
    B = sp.csc_matrix((Av.data, rows, Av.indptr), shape=(len(pos), case.m))
    Ap = B.copy()
    Ap.data = Ap.data * np.where(case.Ip[Av.indices] != case.Jp[Av.indices], 2.0, 1.0)
    return Ap, B


def _kform(Z, pr, pc, Ap, B, block=2048, sym=True):
    npos, m = len(pr), Ap.shape[1]
    # the block of K for the positions a = (p, q) is formed transposed, KT[k, a] = K[(p_a, q_a), (r_k, c_k)]:
    # Zr[k, x] = Z(x, r_k), Zc[k, x] = Z(x, c_k)
    Zr, Zc = np.ascontiguousarray(Z[:, pr].T), np.ascontiguousarray(Z[:, pc].T)
    Apt, Aat = Ap.T.tocsr(), abs(Ap).T.tocsr()
    B = B.tocsr()
    H, Habs = np.zeros((m, m)), np.zeros((m, m))
    for b0 in range(0, npos, block):
        p, q = pr[b0:b0 + block], pc[b0:b0 + block]
        KT = np.take(Zr, p, axis=1) * np.take(Zc, q, axis=1)
        KTabs = np.abs(KT)
        if sym:
            T = np.take(Zr, q, axis=1) * np.take(Zc, p, axis=1)
            T[:, p == q] = 0.0
            KT += T
            KTabs += np.abs(T)
            del T
        Bb = B[b0:b0 + block]
        H += Bb.T @ (Apt @ KT).T             # G_j on the block's positions, weighted by beta of A_i
        Habs += abs(Bb).T @ (Aat @ KTabs).T
    return np.tril(H), np.tril(Habs)


def _trace_reference(case, s, cols):
    """tr(A_i Z A_j Z) for i, j in `cols`, with the A_i formed as dense symmetric matrices."""
    Z, pr, pc = _inverse(case, s)
    Ap, B = _operands(case)
    k = len(Z)
    A = []
    for i in cols:
        col = B[:, i]
        M = np.zeros((k, k))
        M[pr[col.indices], pc[col.indices]] = col.data          # lower triangle: local indices keep row >= col
        A.append(M + np.tril(M, -1).T)
    W = [Z @ a @ Z for a in A]
    return np.tril(np.array([[np.sum(A[i] * W[j]) for j in range(len(cols))] for i in range(len(cols))]))


def violations(H, Href, Habs):
    """Entries outside |H - H_ref| <= 1e-12 H_abs + 1e-14 max(H_abs of the column), for columns of lower triangles."""
    return np.abs(H - Href) > RTOL * Habs + CTOL * Habs.max(axis=0)[None, :]


def assert_close(H, Href, Habs, what=""):
    bad = violations(H, Href, Habs)
    if bad.any():
        i, j = np.argwhere(bad)[0]
        ratio = np.abs(H - Href) / (Habs + Habs.max(axis=0)[None, :] * (CTOL / RTOL))
        raise AssertionError("%s: %d entries outside the bound, first (%d, %d): %r vs %r (H_abs %r); worst "
                             "|dH| / (H_abs + 1e-2 max col) = %.3e" % (what, bad.sum(), i, j, H[i, j], Href[i, j],
                                                                      Habs[i, j], np.nanmax(ratio)))


# ------------------------------------------------------------------------------------------------------------
# CPU: the buckets and the reference
# ------------------------------------------------------------------------------------------------------------
def test_case_buckets():
    """Every case lands in the bucket it is named for, by the rule of assemble_sparse_range."""
    by = {name: rule(_case(name)) for name in CASES}
    for name, r in by.items():
        assert (r["form"], r["kpos"], r["walk"]) == CASES[name]["expect"], (name, r)
        assert r["npos"] == CASES[name]["npos"], (name, r)
    # the edges sit exactly on the thresholds
    assert by["npos_cap_16385"]["npos"] == 32 * SCM_T + 1 and by["kpos32_npos16384"]["npos"] == 32 * SCM_T
    assert by["avg_3"]["avg"] == 3.0 and by["avg_below_3"]["avg"] < 3.0
    assert by["kform_edge"]["nnz_sp"] == 2 * 512 and by["kform_below"]["nnz_sp"] == 2 * 512 - 1
    assert by["kpos16_npos4097"]["npos"] % 2 == 1 and by["kpos32_npos8193"]["npos"] % 2 == 1
    assert by["e_edge_6400"]["E"] == 2 and by["e_edge_6401"]["E"] == 1
    assert 2 * by["e_edge_6400"]["E"] * 6400 == CAP
    # staging rounds: 3 at n = 200 (129 entries, E = 64), 14 on the C3 shape (80 entries, E = 6), 4 at E = 2
    assert by["kpos8_npos512"]["E"] == 64 and by["kpos8_npos512"]["rounds"] == 3
    assert by["c3_staging"]["E"] == 6 and by["c3_staging"]["rounds"] == 14
    assert by["e_edge_6400"]["rounds"] == 4
    assert by["csr_kpos8"]["w"] > 2 * by["csr_kpos8"]["avg"] + 8
    # scm_position<16> and <32> run on the kstream cases under SMCP_B200_SCM_KMAT_GB=0
    seen = {spec["expect"] for spec in CASES.values()}
    for fk in [("kstream", 8, "ell"), ("kstream", 16, "ell"), ("kstream", 32, "ell"), ("position", 8, "ell"),
               ("kstream", 8, "csr"), ("kstream", 16, "csr"), ("pairwise", None, None)]:
        assert fk in seen, fk


@pytest.mark.parametrize("name", ["kpos8_npos512", "avg_3", "mixed"])
def test_reference_matches_trace(name):
    """The K-form reference (several blocks) equals tr(A_i Z A_j Z) with dense A_i."""
    c = _case(name)
    s = c.scaling_point(1)
    Href, Habs = reference(c, s, block=c.spec["npos"] // 3 + 1)
    cols = np.arange(c.m) if c.m <= 200 else np.r_[np.arange(c.md), np.arange(c.md, c.m, 97), c.m - 1]
    sub = np.ix_(cols, cols)
    assert_close(_trace_reference(c, s, cols), Href[sub], Habs[sub], name)
    assert np.abs(Href).max() > 0 and (Habs >= np.abs(Href)).all()


@pytest.mark.parametrize("name", ["kpos8_npos512", "avg_3"])
def test_reference_has_teeth(name):
    """The check rejects H_ref computed with each defect a kernel of the sparse technique could have."""
    c = _case(name)
    s = c.scaling_point(1)
    Z, pr, pc = _inverse(c, s)
    Ap, B = _operands(c)
    Href, Habs = _kform(Z, pr, pc, Ap, B)
    assert not violations(Href, Href, Habs).any()
    E = min(64, CAP // (2 * c.n))
    defects = {}
    # alpha not doubled for one off-diagonal entry of a column
    j = c.md + c.Ns // 2
    k = next(k for k in range(Ap.indptr[j], Ap.indptr[j + 1]) if pr[Ap.indices[k]] != pc[Ap.indices[k]])
    A1 = Ap.copy()
    A1.data[k] *= 0.5
    defects["alpha not doubled"] = _kform(Z, pr, pc, A1, B)[0]
    # the symmetric term dropped for p != q
    defects["no symmetric term"] = _kform(Z, pr, pc, Ap, B, sym=False)[0]
    # the contribution of the last position in the kernels' order (sorted by internal (col, row)) zeroed
    pos = np.unique(c.Av.indices)
    iperm = c.symb.iperm
    last = int(np.argmax(iperm[c.Jp[pos]] * c.n + iperm[c.Ip[pos]]))
    B1 = B.tocsr()
    B1.data[B1.indptr[last]:B1.indptr[last + 1]] = 0.0
    defects["last position zeroed"] = _kform(Z, pr, pc, Ap, B1.tocsc())[0]
    # one entry dropped from a row walk
    B2 = B.copy()
    B2.data[B2.indptr[c.m - 1]] = 0.0
    defects["row walk short"] = _kform(Z, pr, pc, Ap, B2)[0]
    # one staging round skipped: entries E .. 2E-1 of a column dropped
    lens = np.diff(Ap.indptr)
    long_cols = np.nonzero(lens > E)[0]
    if len(long_cols):
        j = int(long_cols[0])
        A2 = Ap.copy()
        A2.data[A2.indptr[j] + E:A2.indptr[j] + 2 * E] = 0.0
        defects["staging round skipped"] = _kform(Z, pr, pc, A2, B)[0]
    else:
        assert name != "kpos8_npos512"
    for what, Hbad in defects.items():
        assert violations(Hbad, Href, Habs).any(), (name, what)


# ------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------
@contextlib.contextmanager
def _kmat_gb(value):
    """SMCP_B200_SCM_KMAT_GB around an assembly (read on every call): None = the default budget."""
    old = os.environ.pop(KMAT_ENV, None)
    if value is not None:
        os.environ[KMAT_ENV] = value
    try:
        yield
    finally:
        os.environ.pop(KMAT_ENV, None)
        if old is not None:
            os.environ[KMAT_ENV] = old


def _device(case):
    from smcp_b200.device import DeviceBackend
    ops = DeviceBackend(case.symb)
    ops.set_operator(case.Av, case.Ns)
    return ops


def _token(ops, s):
    from smcp_b200.chordal import cspmatrix, cholesky, projected_inverse, schur_token
    L = cspmatrix.from_vec(ops, s)
    cholesky(L)
    Y = L.copy()
    projected_inverse(Y)
    return schur_token(L, Y), (L, Y)


def _assemble(ops, run, kmat=None):
    """Runs `run()` (an assembly) with the profiler on: (lower triangle of H, families that launched)."""
    ctx = ops.ctx
    ctx.prof_enable(True)
    ctx.prof_reset()
    try:
        with _kmat_gb(kmat):
            run()
        fam = {nm for nm in ctx.prof_names() if ctx.prof_get(nm)[1] > 0}
    finally:
        ctx.prof_enable(False)
    return ops.get_H(), fam


def _ref(name, seed=1):
    key = (name, seed)
    if key not in _REFS:
        c = _case(name)
        _REFS[key] = reference(c, c.scaling_point(seed))
    return _REFS[key]


def _assert_family(fam, form, what):
    assert FAMILY[form] in fam, (what, form, sorted(fam))
    for other in set(FAMILY) - {form}:
        assert FAMILY[other] not in fam, (what, form, sorted(fam))
    assert ("scm_kmat" in fam) == (form == "kstream"), (what, sorted(fam))


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_bucket_on_device(name):
    """The expected kernel family runs, H passes the check against tr(A_i Z A_j Z), a second assembly gives the same
    bits, and where both K-forms apply, SMCP_B200_SCM_KMAT_GB=0 (scm_position) gives the bits of scm_kstream."""
    c = _case(name)
    form = c.spec["expect"][0]
    ops = _device(c)
    s = c.scaling_point(1)
    tok, keep = _token(ops, s)
    Href, Habs = _ref(name)
    H, fam = _assemble(ops, lambda: ops.schur_assemble(tok))
    _assert_family(fam, form, name)
    if c.md:
        assert "scatter_cols" in fam, sorted(fam)
    H = np.tril(H)
    assert_close(H, Href, Habs, name)
    H2, _ = _assemble(ops, lambda: ops.schur_assemble(tok))
    assert np.array_equal(np.tril(H2), H), name
    if form == "kstream":
        Hp, fam = _assemble(ops, lambda: ops.schur_assemble(tok), kmat="0")
        _assert_family(fam, "position", name)
        assert np.array_equal(np.tril(Hp), H), name


def _set_sentinel(ops):
    from smcp_b200.device import _ck
    _ck(ops.lib, ops.lib.smcp_kkt_set_H(ops._op, np.full(ops.m * ops.m, SENTINEL)))


@pytest.mark.gpu
def test_column_ranges_keep_the_rest():
    """schur_assemble(tok, j0, j1) across md writes only the columns [j0, j1), and in the sparse ones only the rows
    i >= j; the sparse columns have the bits of the full assembly, the dense ones pass the check."""
    c = _case("mixed")
    ops = _device(c)
    tok, keep = _token(ops, c.scaling_point(1))
    Href, Habs = _ref("mixed")
    ops.schur_assemble(tok)
    Hfull = np.tril(ops.get_H())
    m, md = c.m, c.md
    upper = np.triu(np.ones((m, m), dtype=bool), 1)
    for j0, j1 in ((10, 300), (md - 1, md + 1), (md, m)):
        _set_sentinel(ops)
        ops.schur_assemble(tok, j0, j1)
        H = ops.get_H()
        assert (H[:, :j0] == SENTINEL).all() and (H[:, j1:] == SENTINEL).all(), (j0, j1)
        sl = slice(max(j0, md), j1)
        assert (H[:, sl][upper[:, sl]] == SENTINEL).all(), (j0, j1)
        assert np.array_equal(np.tril(H)[:, sl], Hfull[:, sl]), (j0, j1)
        if j0 < md:
            d = slice(j0, md)
            assert_close(np.tril(H)[:, d], Href[:, d], Habs[:, d], "dense columns of [%d, %d)" % (j0, j1))


@pytest.mark.gpu
@pytest.mark.parametrize("block", [128, 37])
def test_cyclic_ranks(block):
    """smcp_kkt_assemble_cyclic for rank 0..2 of 3 (no communicator: each rank builds Z itself): owned sparse columns
    have the bits of the full assembly, owned dense columns pass the check, the others keep the sentinel."""
    from smcp_b200.device import _ck
    c = _case("mixed")
    ops = _device(c)
    tok, keep = _token(ops, c.scaling_point(1))
    Href, Habs = _ref("mixed")
    ops.schur_assemble(tok)
    Hfull = np.tril(ops.get_H())
    m, md = c.m, c.md
    upper = np.triu(np.ones((m, m), dtype=bool), 1)
    covered = np.zeros(m, dtype=bool)
    for rank in range(3):
        _set_sentinel(ops)
        _ck(ops.lib, ops.lib.smcp_kkt_assemble_cyclic(ops._op, tok, block, rank, 3))
        H = ops.get_H()
        own = np.zeros(m, dtype=bool)
        for c0 in range(rank * block, m, 3 * block):
            own[c0:c0 + block] = True
        assert not (covered & own).any()
        covered |= own
        assert (H[:, ~own] == SENTINEL).all(), rank
        sparse = own & (np.arange(m) >= md)
        assert np.array_equal(np.tril(H)[:, sparse], Hfull[:, sparse]), rank
        assert (H[:, sparse][upper[:, sparse]] == SENTINEL).all(), rank
        dense = own & (np.arange(m) < md)
        if dense.any():
            assert_close(np.tril(H)[:, dense], Href[:, dense], Habs[:, dense], "rank %d dense columns" % rank)
    assert covered.all()


@pytest.mark.gpu
def test_second_scaling_point():
    """A second scaling point on the same operator rebuilds the materialised K: H at S2 passes the check at S2."""
    name = "kpos16_npos4097"
    c = _case(name)
    ops = _device(c)
    tok1, keep1 = _token(ops, c.scaling_point(1))
    H1, fam = _assemble(ops, lambda: ops.schur_assemble(tok1))
    _assert_family(fam, "kstream", name)
    del tok1, keep1
    tok2, keep2 = _token(ops, c.scaling_point(2))
    H2, fam = _assemble(ops, lambda: ops.schur_assemble(tok2))
    _assert_family(fam, "kstream", name)
    Href, Habs = _ref(name, seed=2)
    assert_close(np.tril(H2), Href, Habs, "second scaling point")
    assert violations(np.tril(H1), Href, Habs).any()
