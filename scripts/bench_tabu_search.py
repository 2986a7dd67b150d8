"""Tabu search of the Goemans-Williamson trials on the device, after the one-flip search (smcp_round_pm1_tabu).

    python scripts/bench_tabu_search.py [--n 20000] [--ks 64,256,1024] [--iters N] [--reps 3] [--out FILE.json]

Input: the C5 graph and the unit-diagonal completable X of scripts/bench_local_search.py, so no solve is needed; that X
is a random completable matrix, not a solution of the relaxation.  Per k: one warm-up of round_pm1 with the one-flip
search and --iters tabu moves per trial (default n, default tenure), then --reps calls with the per-family profile on;
reported are the device time of the tabu kernel (profile family round_tabu), of the one-flip kernel (round_ls) and the
call's wall time, median [min, max]; moves per microsecond of round_tabu device time over all trials; the best and mean
cut weight after the one-flip search and after the tabu search, and the move counts of the returned vectors.  The NumPy
twin (tests/tabu_search_oracle.py) runs once at the smallest k on the device's one-flip optima: its wall time, and
whether signs, values, moves and best iterations agree bit for bit.  The card's name and power limit are read in the
same run.  Needs a CUDA device: there is no CPU fallback.
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
    ap.add_argument("--iters", type=int, default=None, help="tabu moves per trial (default n)")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    from smcp_b200 import solvers
    from smcp_b200.base import _completion_factor, _tabu_tenure
    from smcp_b200.device import Context, DeviceBackend
    from local_search_oracle import eval_values
    from tabu_search_oracle import tabu_search
    solvers.set_backend_factory(lambda symb: DeviceBackend(symb))
    ctx = Context.get()
    iters = a.n if a.iters is None else a.iters
    tenure = _tabu_tenure(a.n)
    res = {"card (name, power limit)": card(), "n": a.n, "iters": iters, "tenure": tenure}
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

    def call(k):
        return ops.round_pm1_tabu(L.buf, crow, ccol, cval, k, 1, iters, tenure, max_flips=None)

    for k in ks:
        ref = call(k)                                                           # warm-up
        fam = {"round_tabu": [], "round_ls": []}
        walls = []
        ctx.prof_enable(True)
        try:
            for _ in range(a.reps):
                ctx.prof_reset()
                t0 = time.perf_counter()
                out = call(k)
                walls.append(time.perf_counter() - t0)
                for f in fam:
                    fam[f].append(ctx.prof_get(f)[0])
                assert all(np.array_equal(u, v) for u, v in zip(out, ref))
        finally:
            ctx.prof_enable(False)
        values1, values, moves, best_iter = ref[1], ref[2], ref[4], ref[5]
        tabu_ms = spread(fam["round_tabu"])
        r = {"tabu_device_ms": tabu_ms, "one_flip_device_ms": spread(fam["round_ls"]), "wall_s": spread(walls),
             "moves_total": int(moves.sum()), "moves_per_us": float(moves.sum()) / (tabu_ms["median"] * 1e3),
             "best_iter_median": float(np.median(best_iter)), "best_iter_max": int(best_iter.max()),
             "best_cut_one_flip": -float(values1.min()), "best_cut_tabu": -float(values.min()),
             "mean_cut_one_flip": -float(values1.mean()), "mean_cut_tabu": -float(values.mean())}
        res["search"][str(k)] = r
        log("k = %d: tabu %s ms | one-flip %s ms | wall %s s | %.1f moves/us | best cut %.1f -> %.1f | mean %.2f -> %.2f" % (
            k, r["tabu_device_ms"], r["one_flip_device_ms"], r["wall_s"], r["moves_per_us"], r["best_cut_one_flip"],
            r["best_cut_tabu"], r["mean_cut_one_flip"], r["mean_cut_tabu"]))

    k = ks[0]
    V = ops.completion_sample(L.buf, k, 1)
    x0 = np.where(V.T < 0.0, -1, 1).astype(np.int8)
    x1, _, _ = ops.pm1_local_search(x0, crow, ccol, cval)
    xd, vd, md, bd = ops.pm1_tabu_search(x1, crow, ccol, cval, iters, tenure)
    t0 = time.perf_counter()
    xt, mt, bt = tabu_search(x1, crow, ccol, cval, iters, tenure)
    vt = eval_values(xt, crow, ccol, cval)
    tw = time.perf_counter() - t0
    equal = bool(np.array_equal(xd, xt) and np.array_equal(md, mt) and np.array_equal(bd, bt)
                 and np.array_equal(vd.view(np.int64), vt.view(np.int64)))
    res["host twin"] = {"k": k, "wall_s": tw, "runs": 1, "bitwise equal to the device": equal}
    log("host twin at k = %d: %.2f s, bitwise equal: %s" % (k, tw, equal))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
