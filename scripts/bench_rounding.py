"""Goemans-Williamson rounding on the device against the dense host route.

    python scripts/bench_rounding.py [--n 20000] [--ks 64,256,1024] [--reps 5] [--no-dense] [--out FILE.json]

Graph: the C5 max-cut graph as scripts/run_config.py builds it (n vertices, 3n/2 random edges, seed 0).  Input:
mk_rand(..., 'completable') on its pattern scaled to unit diagonal, a completable X with diag(X) = 1 like a
solution of the relaxation, so no solve is needed.
  completion   _completion_factor(X) (symbolic + device completion): wall time, and the device time of the
               op_completion region; 1 warm-up, --reps timed.
  per k        SDP.round_pm1's device call (smcp_round_pm1) with k trials: 1 warm-up, then --reps calls with the
               profile off (wall time, device time of the op_trsm region) and --reps with the per-family profile
               on (round_normal: the normals, round_eval: packing, evaluation, best trial).  The evaluation's
               effective bandwidth counts 8 n k bytes of samples read once plus 16 bytes per objective entry.
  dense        completion(X) (the dense n x n max-det completion through the host) followed by
               numpy.linalg.cholesky of it, the route that existed before: one run, wall time.
Times are median [min, max] over the repetitions.  The card's name and power limit are read in the same run.
Needs a CUDA device: there is no CPU fallback.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import scipy.sparse as sp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return out[1] if len(out) > 1 else "unknown"
    except Exception as e:
        return "nvidia-smi unavailable (%s)" % e


def log(*a):
    print(*a, flush=True)


def spread(xs):
    xs = sorted(xs)
    return {"median": xs[len(xs) // 2], "min": xs[0], "max": xs[-1], "n": len(xs)}


def c5_problem(n):
    import smcp_b200 as S
    rng = np.random.default_rng(0)
    e = rng.integers(0, n, size=(3 * n // 2, 2))
    return S.maxcut_SDP(n, e)


def unit_diag_x(P):
    """mk_rand(..., 'completable') on the pattern of P, scaled to unit diagonal (D X D keeps it completable)."""
    import smcp_b200 as S
    from smcp_b200.symbolic import lower_pattern
    n = P.n
    V = sp.tril(P.V, format="coo")
    cp, ri = lower_pattern(n, V.row, V.col)
    cols = np.repeat(np.arange(n, dtype=np.int64), np.diff(cp))
    u = S.mk_rand(n, cp, ri, "completable", seed=0)
    d = np.empty(n)
    d[cols[ri == cols]] = u[ri == cols]
    u = u / np.sqrt(d[ri] * d[cols])
    return sp.csc_matrix((u, (ri, cols)), shape=(n, n))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=20000)
    ap.add_argument("--ks", default="64,256,1024")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--no-dense", action="store_true")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    from smcp_b200 import misc, solvers
    from smcp_b200.base import _completion_factor, completion
    from smcp_b200.device import Context, DeviceBackend
    solvers.set_backend_factory(lambda symb: DeviceBackend(symb))
    ctx = Context.get()
    res = {"card (name, power limit)": card(), "n": a.n}
    log("card:", res["card (name, power limit)"])
    t0 = time.perf_counter()
    P = c5_problem(a.n)
    X = unit_diag_x(P)
    log("C5 graph n = %d, |V| = %d, X built in %.1f s" % (a.n, X.nnz, time.perf_counter() - t0))

    # completion
    L, order = _completion_factor(X)
    walls, devs = [], []
    for _ in range(a.reps):
        del L
        ctx.region_reset()
        t0 = time.perf_counter()
        L, order = _completion_factor(X)
        ctx.sync()
        walls.append(time.perf_counter() - t0)
        devs.append(ctx.region_get("op_completion")[0])
    ops = L.ops
    symb = ops.symb
    nj = np.diff(symb.rowptr)
    res["pattern"] = {"nsn": int(symb.nsn), "nblk": int(symb.nblk), "largest front": int(nj.max())}
    res["completion"] = {"wall_s": spread(walls), "device_ms": spread(devs)}
    log("pattern:", res["pattern"])
    log("completion: wall %s s, device %s ms" % (res["completion"]["wall_s"], res["completion"]["device_ms"]))

    A = P.A
    I, J = misc.ind2sub(a.n, A.indices[A.indptr[0]:A.indptr[1]])
    pos = np.empty(a.n, dtype=np.int64)
    pos[order] = np.arange(a.n, dtype=np.int64)
    crow, ccol, cval = pos[np.asarray(I)], pos[np.asarray(J)], A.data[A.indptr[0]:A.indptr[1]]
    nc = len(cval)
    res["objective entries"] = nc
    res["rounding"] = {}
    for k in [int(v) for v in a.ks.split(",")]:
        values, x, best = ops.round_pm1(L.buf, crow, ccol, cval, k, 1)          # warm-up
        walls, trsm = [], []
        for _ in range(a.reps):
            ctx.region_reset()
            t0 = time.perf_counter()
            v2, _, _ = ops.round_pm1(L.buf, crow, ccol, cval, k, 1)
            walls.append(time.perf_counter() - t0)
            trsm.append(ctx.region_get("op_trsm")[0])
            assert np.array_equal(v2, values)
        fam = {"round_normal": [], "round_eval": []}
        ctx.prof_enable(True)
        try:
            for _ in range(a.reps):
                ctx.prof_reset()
                ops.round_pm1(L.buf, crow, ccol, cval, k, 1)
                for f in fam:
                    fam[f].append(ctx.prof_get(f)[0])
        finally:
            ctx.prof_enable(False)
        ev = spread(fam["round_eval"])
        byts = 8.0 * a.n * k + 16.0 * nc
        r = {"wall_s": spread(walls), "trsm_device_ms": spread(trsm),
             "normal_device_ms": spread(fam["round_normal"]), "eval_device_ms": ev,
             "eval_bytes": byts, "eval_GBps_at_median": byts / (ev["median"] * 1e-3) / 1e9 if ev["median"] > 0 else None,
             "best_value": float(values[best]), "best_cut_weight": -float(values[best]), "best_trial": int(best)}
        res["rounding"][str(k)] = r
        log("k = %d: wall %s s | trsm %s ms | normals %s ms | eval %s ms (%.1f GB/s) | best cut %.1f" % (
            k, r["wall_s"], r["trsm_device_ms"], r["normal_device_ms"], ev, r["eval_GBps_at_median"] or 0.0, r["best_cut_weight"]))

    if not a.no_dense:
        del L, ops
        t0 = time.perf_counter()
        Xd = completion(X)
        t1 = time.perf_counter()
        np.linalg.cholesky(Xd)
        t2 = time.perf_counter()
        res["dense route"] = {"completion_s": t1 - t0, "host_cholesky_s": t2 - t1, "total_s": t2 - t0, "runs": 1}
        log("dense route: completion(X) %.1f s + numpy.linalg.cholesky %.1f s" % (t1 - t0, t2 - t1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
