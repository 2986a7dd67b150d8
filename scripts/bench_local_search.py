"""One-flip local search of the Goemans-Williamson trials on the device (smcp_round_pm1_ls).

    python scripts/bench_local_search.py [--n 20000] [--ks 64,256,1024] [--reps 3] [--out FILE.json]

Input: the C5 graph (n vertices, 3n/2 random edges, seed 0) and the unit-diagonal completable X of
scripts/bench_rounding.py, so no solve is needed.  Per k: one warm-up of round_pm1 with local_search, then --reps
calls with the per-family profile on; reported are the device time of the search kernel (profile family round_ls),
of the evaluations (round_eval: pre- and post-search packing, evaluation, best trial) and the call's wall time,
median [min, max]; flips per trial (median, max) and the best cut weight before and after the search.  The NumPy
twin (tests/local_search_oracle.py) runs once at the smallest k on the device's rounded trials: its wall time, and
whether flips, signs and values agree bit for bit.  The card's name and power limit are read in the same run.
Needs a CUDA device: there is no CPU fallback.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

from bench_rounding import c5_problem, card, log, spread, unit_diag_x  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=20000)
    ap.add_argument("--ks", default="64,256,1024")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    from smcp_b200 import solvers
    from smcp_b200.base import _completion_factor
    from smcp_b200.device import Context, DeviceBackend
    from local_search_oracle import eval_values, local_search
    solvers.set_backend_factory(lambda symb: DeviceBackend(symb))
    ctx = Context.get()
    res = {"card (name, power limit)": card(), "n": a.n}
    log("card:", res["card (name, power limit)"])
    P = c5_problem(a.n)
    X = unit_diag_x(P)
    L, order = _completion_factor(X)
    ops = L.ops
    I, J, cval = P._objective_entries()
    pos = np.empty(a.n, dtype=np.int64)
    pos[order] = np.arange(a.n, dtype=np.int64)
    crow, ccol = pos[I], pos[J]
    res["objective entries"] = len(cval)
    res["search"] = {}
    ks = [int(v) for v in a.ks.split(",")]
    for k in ks:
        ref = ops.round_pm1_ls(L.buf, crow, ccol, cval, k, 1)                 # warm-up
        fam = {"round_ls": [], "round_eval": []}
        walls = []
        ctx.prof_enable(True)
        try:
            for _ in range(a.reps):
                ctx.prof_reset()
                t0 = time.perf_counter()
                out = ops.round_pm1_ls(L.buf, crow, ccol, cval, k, 1)
                walls.append(time.perf_counter() - t0)
                for f in fam:
                    fam[f].append(ctx.prof_get(f)[0])
                assert all(np.array_equal(u, v) for u, v in zip(out, ref))
        finally:
            ctx.prof_enable(False)
        values0, values, flips = ref[0], ref[1], ref[2]
        r = {"search_device_ms": spread(fam["round_ls"]), "eval_device_ms": spread(fam["round_eval"]),
             "wall_s": spread(walls), "flips_median": float(np.median(flips)), "flips_max": int(flips.max()),
             "flips_total": int(flips.sum()),
             "best_cut_before": -float(values0.min()), "best_cut_after": -float(values.min()),
             "mean_cut_before": -float(values0.mean()), "mean_cut_after": -float(values.mean())}
        res["search"][str(k)] = r
        log("k = %d: search %s ms | eval %s ms | wall %s s | flips median %.0f max %d | best cut %.1f -> %.1f" % (
            k, r["search_device_ms"], r["eval_device_ms"], r["wall_s"], r["flips_median"], r["flips_max"],
            r["best_cut_before"], r["best_cut_after"]))

    k = ks[0]
    V = ops.completion_sample(L.buf, k, 1)
    x0 = np.where(V.T < 0.0, -1, 1).astype(np.int8)
    xd, vd, fd = ops.pm1_local_search(x0, crow, ccol, cval)
    t0 = time.perf_counter()
    xt, ft = local_search(x0, crow, ccol, cval, a.n, 1e-12)
    vt = eval_values(xt, crow, ccol, cval)
    tw = time.perf_counter() - t0
    res["host twin"] = {"k": k, "wall_s": tw, "runs": 1,
                        "bitwise equal to the device": bool(np.array_equal(xd, xt) and np.array_equal(fd, ft)
                                                            and np.array_equal(vd, vt))}
    log("host twin at k = %d: %.2f s, bitwise equal: %s" % (k, tw, res["host twin"]["bitwise equal to the device"]))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
