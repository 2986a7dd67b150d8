"""Convergence diagnostic: full solve of a band SDP with the per-iteration trace, and the consistency
of the forward / inverse Hessian pair along the way.   python scripts/diag_convergence.py n m bw"""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import smcp_b200 as S
from smcp_b200 import solvers
n, m, bw = (int(a) for a in sys.argv[1:4])
P = S.band_SDP(n, m, bw, seed=0)
solvers.options["show_progress"] = False
solvers.options["maxiters"] = int(sys.argv[4]) if len(sys.argv) > 4 else 60
t0 = time.time()
sol = P.solve_feas(kktsolver="chol", primalstart={"x": P._X0})
print("n=%d m=%d bw=%d env NO_CHAIN=%s: status %s, %d iterations, %.2f s; pobj %.10e dobj %.10e gap %.2e pres %.1e dres %.1e" % (
    n, m, bw, os.environ.get("SMCP_B200_NO_CHAIN"), sol["status"], sol["iterations"], time.time() - t0, sol["primal objective"],
    sol["dual objective"], sol["gap"], sol["primal infeasibility"] or 0, sol["dual infeasibility"] or 0))
for r in sol["trace"]:
    if r["iter"] % 4 == 0 or r["iter"] >= sol["iterations"] - 3:
        f = lambda k: float(r.get(k) or 0.0)
        print("  it %3d %s gap %.2e pres %.1e dres %.1e ntdecr %.2e pstep %.2e t %.2e" % (
            r["iter"], r.get("stype"), f("gap"), f("pres"), f("dres"), f("ntdecr"), f("pstep"), f("t")))
