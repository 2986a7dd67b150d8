"""Low-rank solve of the C5 max-cut relaxation on the device (SDP.solve_lowrank), its certified bound, and rounding from
the factor (round_pm1 on a solution holding V).

    python scripts/bench_lowrank.py [--n 20000] [--ks 64,256,1024] [--reps 3] [--out FILE.json]

Input: the C5 graph of scripts/bench_rounding.py (n = 20 000, 30 000 random edges, seed 0) at the default rank
(smallest r with r(r+1)/2 > n) and the default tol = 1e-6, max_sweeps = 1000.  One warm-up solve (max_sweeps = 2, no
bound), then the timed solve: the host time of the greedy colouring (region lowrank_colour_host), the device time of the
sweep loop including the host reads of the stop flag between groups (region lowrank_loop), the solve's wall time,
sweeps, colours, f, and the certificate's wall time, bound, shift and number of Cholesky probes; f - bound.  Then
round_pm1 from V for each k: one warm-up and --reps calls, wall time median [min, max], and the best cut; and the best cut
with local_search=True and with tabu_iters=n (default tenure) at the largest k, medians of --reps runs.  The card's name
and power limit are read in the same run.  Needs a CUDA device: there is no CPU fallback.
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

from bench_rounding import c5_problem, card, log, spread  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=20000)
    ap.add_argument("--ks", default="64,256,1024")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    from smcp_b200 import base, solvers
    from smcp_b200.device import Context
    solvers.set_backend_factory(None)
    ctx = Context.get()
    res = {"card (name, power limit)": card(), "n": a.n}
    log("card:", res["card (name, power limit)"])
    P = c5_problem(a.n)
    P.solve_lowrank(max_sweeps=2, bound=False)                     # warm-up: modules, allocations

    ctx.region_reset()
    t0 = time.perf_counter()
    sol = P.solve_lowrank(bound=False)
    wall = time.perf_counter() - t0
    colour_ms, _ = ctx.region_get("lowrank_colour_host")
    loop_ms, _ = ctx.region_get("lowrank_loop")
    I, J, v = P._objective_entries()
    bv = np.ones(a.n)
    yv = sol["y"]                                                  # maxcut_SDP: constraint k is X_kk
    t0 = time.perf_counter()
    t, probes = base._lowrank_certificate(a.n, I, J, v, yv, bv, sol["primal objective"])
    cert = time.perf_counter() - t0
    dual = float(bv @ yv) - t * a.n - base._gamma(a.n + 2) * (float(np.abs(yv).sum()) + t * a.n)
    f = sol["primal objective"]
    res["solve"] = {"rank": sol["rank"], "colours": sol["colors"], "sweeps": sol["sweeps"], "converged": sol["converged"],
                    "colouring host ms": colour_ms, "sweep loop device ms (events)": loop_ms,
                    "solve wall s (no bound)": wall, "f": f, "f_0": float(sol["objective history"][0])}
    res["certificate"] = {"wall s": cert, "probes": probes, "shift t": t, "bound": dual, "f - bound": f - dual,
                          "relative gap": (f - dual) / abs(f)}
    log("solve:", res["solve"])
    log("certificate:", res["certificate"])
    sol["y"] = yv - t
    sol["dual objective"] = dual

    res["round_pm1 from V"] = {}
    for k in [int(s) for s in a.ks.split(",")]:
        P.round_pm1(sol, trials=k)
        ts, best = [], None
        for _ in range(a.reps):
            t0 = time.perf_counter()
            r = P.round_pm1(sol, trials=k)
            ts.append(1e3 * (time.perf_counter() - t0))
            best = -r["value"]
        res["round_pm1 from V"][str(k)] = {"wall ms": spread(ts), "best cut": best}
        log("round_pm1 k=%d:" % k, res["round_pm1 from V"][str(k)])
    k = max(int(s) for s in a.ks.split(","))
    for name, kw in (("local_search=True", dict(local_search=True)), ("tabu_iters=n", dict(tabu_iters=a.n))):
        ws, ts = [], []
        for seed in range(a.reps):
            t0 = time.perf_counter()
            _, w, ub = P.cut(sol, trials=k, seed=seed, **kw)
            ts.append(time.perf_counter() - t0)
            ws.append(w)
        res["cut k=%d %s" % (k, name)] = {"best cut (median over seeds)": spread(ws)["median"], "cuts": sorted(ws),
                                          "wall s": spread(ts), "bound": ub}
        log("cut", name, res["cut k=%d %s" % (k, name)])
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
