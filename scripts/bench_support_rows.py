"""Dense-constraint copy on the support rows (the rows of blkval some constraint touches) against the full copy.

    python scripts/bench_support_rows.py [--m 10000] [--m-big 15000] [--skip-a] [--skip-b] [--skip-c] [--out FILE.json]

(a) rand_SDP on the C3 pattern (n = 2000, tridiagonal + 6n random pairs) with density 1.0 and m constraints:
    one operator per copy, created, timed and destroyed one after the other (they do not fit side by side).
    Each: 1 warm-up and 3 timed smcp_kkt_assemble calls at one scaling point (kkt_assemble region, profiling
    off), then one more call with the per-family profile on (schur_gemm_dmma, support_gather); bytes of the copy
    and the relative Frobenius difference of the two H.
(b) the same pattern at m-big constraints: solve_feas for 3 iterations on the support copy (status, ms per
    iteration); the full copy's size is printed, not allocated.
(c) solve_phase1 on the bench's C3 problem (density 0.005, m = 10^4): wall time, the Gram path taken and
    ||A(X0) - b|| / ||b||.
The card's name and power limit are read in the same run.  Needs a CUDA device: there is no CPU fallback.
"""
import argparse
import gc
import json
import os
import subprocess
import sys
import time

import numpy as np
import scipy.sparse as sp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ENV = "SMCP_B200_AVW_SUPPORT"


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return out[1] if len(out) > 1 else "unknown"
    except Exception as e:
        return "nvidia-smi unavailable (%s)" % e


def c3_pattern(n=2000):
    """The aggregate pattern of bench.py's rand workloads."""
    rng = np.random.default_rng(0)
    e = rng.integers(0, n, size=(6 * n, 2))
    I = np.concatenate([np.maximum(e[:, 0], e[:, 1]), np.arange(n), np.arange(1, n)])
    J = np.concatenate([np.minimum(e[:, 0], e[:, 1]), np.arange(n), np.arange(0, n - 1)])
    return sp.coo_matrix((np.ones(len(I)), (I, J)), shape=(n, n))


def log(*a):
    print(*a, flush=True)


def problem(P, mode):
    from smcp_b200.solvers import _Problem, _read_options
    os.environ[ENV] = mode
    try:
        return _Problem(P.A, P.b, _read_options(P.n, False), "chol", None)
    finally:
        os.environ.pop(ENV, None)


def part_a(m):
    import smcp_b200 as S
    from smcp_b200.chordal import cspmatrix, cholesky, projected_inverse, schur_token
    t0 = time.perf_counter()
    P = S.rand_SDP(c3_pattern(), m, density=1.0, seed=0)
    log("(a) generated rand_SDP n=2000 m=%d density=1.0 in %.1f s" % (m, time.perf_counter() - t0))
    res, H = {}, {}
    for tag, mode in (("support", "1"), ("full", "0")):
        t0 = time.perf_counter()
        pr = problem(P, mode)
        ops, ctx, symb = pr.ops, pr.ops.ctx, pr.symb
        rows = ops.dense_rows()
        lds = rows + (rows & 1) if tag == "support" else rows
        r = {"create_s": time.perf_counter() - t0, "nblk": symb.nblk, "dense_rows": rows,
             "copy_bytes": 8 * lds * m}
        rng = np.random.default_rng(0)
        s = np.zeros(symb.nvp)
        s[symb.diag_vec] = 2.0
        s += 0.05 * rng.standard_normal(symb.nvp)
        L = cspmatrix.from_vec(ops, s)
        cholesky(L)
        Y = L.copy()
        projected_inverse(Y)
        tok = schur_token(L, Y)
        ops.schur_assemble(tok)                 # warm-up
        ctx.sync()
        ctx.region_reset()
        t0 = time.perf_counter()
        for _ in range(3):
            ops.schur_assemble(tok)
        ctx.sync()
        r["wall_ms_per_call"] = 1e3 * (time.perf_counter() - t0) / 3
        ms, n = ctx.region_get("kkt_assemble")
        r["kkt_assemble_ms_per_call"] = ms / max(n, 1)
        ctx.prof_enable(True)
        ctx.prof_reset()
        ops.schur_assemble(tok)
        ctx.sync()
        r["families_ms_one_call"] = {nm: ctx.prof_get(nm)[0] for nm in ctx.prof_names() if ctx.prof_get(nm)[1] > 0}
        ctx.prof_enable(False)
        H[tag] = np.tril(ops.get_H())
        res[tag] = r
        log("(a) %s: %s" % (tag, json.dumps(r)))
        del tok, L, Y, pr, ops
        gc.collect()
    res["rel_frobenius_H"] = float(np.linalg.norm(H["support"] - H["full"]) / np.linalg.norm(H["full"]))
    log("(a) ||H_support - H_full||_F / ||H_full||_F = %.3e" % res["rel_frobenius_H"])
    return res


def part_b(m):
    import smcp_b200 as S
    from smcp_b200 import solvers
    t0 = time.perf_counter()
    P = S.rand_SDP(c3_pattern(), m, density=1.0, seed=0)
    log("(b) generated rand_SDP n=2000 m=%d density=1.0 in %.1f s" % (m, time.perf_counter() - t0))
    old = solvers.options["maxiters"]
    solvers.options["maxiters"] = 3
    os.environ[ENV] = "1"
    try:
        t0 = time.perf_counter()
        sol = P.solve_feas(kktsolver="chol", primalstart={"x": P._X0})
        wall = time.perf_counter() - t0
    finally:
        os.environ.pop(ENV, None)
        solvers.options["maxiters"] = old
    pr = solvers._last_problem
    rows = pr.ops.dense_rows()
    r = {"status": sol["status"], "iterations": sol["iterations"], "wall_s_incl_setup": wall,
         "ms_per_iteration_incl_setup": 1e3 * wall / max(sol["iterations"], 1),
         "nblk": pr.symb.nblk, "dense_rows": rows, "support_copy_bytes": 8 * (rows + (rows & 1)) * m,
         "full_copy_bytes_not_allocated": 8 * pr.symb.nblk * m}
    log("(b) %s" % json.dumps(r))
    return r


def part_c():
    import smcp_b200 as S
    from smcp_b200 import solvers
    P = S.rand_SDP(c3_pattern(), 10000, density=0.005, seed=0)
    t0 = time.perf_counter()
    X0, sol = P.solve_phase1()
    wall = time.perf_counter() - t0
    n = P.n
    X = X0.tocoo()
    lin = X.row + n * X.col
    w = np.where(X.row == X.col, 1.0, 2.0)
    x = sp.csc_matrix((w * X.data, (lin, np.zeros(len(lin), dtype=np.int64))), shape=(n * n, 1))
    res = np.asarray((P.A[:, 1:].T @ x).todense()).ravel() - P.b
    r = {"wall_s": wall, "phase1_sdp_solved": sol is not None,
         "rel_residual": float(np.linalg.norm(res) / np.linalg.norm(P.b))}
    # the least-norm start runs on the first operator solve_phase1 builds (kktsolver 'qr': Ns = 0)
    from smcp_b200.solvers import _Problem, _read_options
    pr = _Problem(P.A, P.b, _read_options(n, True), "qr", None)
    rows = pr.ops.dense_rows()
    r.update(nblk=pr.symb.nblk, dense_rows=rows, gram_path="device" if 8.0 * rows * P.m <= (16 << 30) else "host")
    log("(c) %s" % json.dumps(r))
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--m", type=int, default=10000)
    ap.add_argument("--m-big", type=int, default=15000)
    ap.add_argument("--skip-a", action="store_true")
    ap.add_argument("--skip-b", action="store_true")
    ap.add_argument("--skip-c", action="store_true")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    from smcp_b200 import solvers
    from smcp_b200.device import DeviceBackend
    solvers.options["show_progress"] = False
    solvers.set_backend_factory(lambda symb: DeviceBackend(symb))
    out = {"card": card()}
    log("card: %s" % out["card"])
    for key, skip, fn in (("a", a.skip_a, lambda: part_a(a.m)), ("b", a.skip_b, lambda: part_b(a.m_big)),
                          ("c", a.skip_c, part_c)):
        if skip:
            continue
        out[key] = fn()
        if a.out:                       # after every part, so that a long run keeps what it measured
            os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
            with open(a.out, "w") as f:
                json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
