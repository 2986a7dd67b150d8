"""Blocked Householder QR on the device (kktsolver='qr', options['qr_method'] = 'householder').

    python scripts/bench_qr.py [--iters 8] [--reps 3] [--skip-c4] [--out FILE.json]

(a) smcp_dense_geqrf + smcp_dense_orgqr: device time (CUDA events around the kernels, host copies excluded)
    and FP64 TFLOP/s (4 M N^2 - 4/3 N^3 flops) at the shapes of kktsolver='qr' (C2: 30000 x 1000, C4:
    80400 x 501) and two larger ones, beside torch.linalg.qr (cuSOLVER geqrf + orgqr) on the same input in
    the same process; the per-family split of one device factorisation at each shape (qr_panel: the
    cooperative panel kernel, qr_wy_dmma: the block-reflector GEMMs).
(b) C4 (mtxnorm p = q = 200, r = 500) through solve_esd(kktsolver='qr') for a fixed number of iterations with
    both qr_method values: status, iterations, ms per iteration and the kkt_* API regions per iteration.
The card's name and power limit are read in the same run.  Needs a CUDA device: there is no CPU fallback.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

SHAPES = [(30000, 1000), (80400, 501), (200000, 1000), (100000, 2000)]


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:          # the name still comes from torch below
        return "nvidia-smi unavailable (%s)" % e


def qr_flops(M, N):
    return 4.0 * M * N * N - 4.0 / 3.0 * N ** 3


def dense(ctx, reps):
    import torch
    from smcp_b200.device import _ck
    lib = ctx.lib
    rows = []
    for M, N in SHAPES:
        A = np.random.default_rng(M + N).standard_normal((M, N))
        flat = np.asfortranarray(A).reshape(-1, order="F")
        ours = []
        for r in range(reps + 1):           # the first run warms up (module load, workspace growth)
            a = flat.copy()
            tau = np.zeros(N)
            t1, t2 = C.c_double(), C.c_double()
            _ck(lib, lib.smcp_dense_geqrf(ctx.h, a, M, M, N, tau, C.byref(t1)))
            _ck(lib, lib.smcp_dense_orgqr(ctx.h, a, M, M, N, tau, C.byref(t2)))
            if r:
                ours.append((t1.value, t2.value))
        # per-family split of one more factorisation (per-launch event timing serialises the launches)
        ctx.prof_reset()
        ctx.prof_enable(True)
        a = flat.copy()
        tau = np.zeros(N)
        _ck(lib, lib.smcp_dense_geqrf(ctx.h, a, M, M, N, tau, None))
        _ck(lib, lib.smcp_dense_orgqr(ctx.h, a, M, M, N, tau, None))
        ctx.prof_enable(False)
        fam = {nm: ctx.prof_get(nm) for nm in ctx.prof_names()}
        fam = {nm: (round(ms, 3), cnt) for nm, (ms, cnt) in fam.items() if cnt}
        Qd = a.reshape((M, N), order="F")
        At = torch.from_numpy(A).cuda()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ref = []
        for r in range(reps + 1):
            torch.cuda.synchronize()
            ev0.record()
            Qt, Rt = torch.linalg.qr(At, mode="reduced")
            ev1.record()
            torch.cuda.synchronize()
            if r:
                ref.append(ev0.elapsed_time(ev1))
        # the two Q factors agree up to column signs (LAPACK's beta convention in both)
        Qt_h = Qt.cpu().numpy()
        s = np.sign(np.sum(Qt_h[:64] * Qd[:64], axis=0))
        dq = float(np.abs(Qt_h * s[None, :] - Qd).max())
        del At, Qt, Rt
        torch.cuda.empty_cache()
        geq = float(np.median([o[0] for o in ours]))
        org = float(np.median([o[1] for o in ours]))
        tref = float(np.median(ref))
        fl = qr_flops(M, N)
        row = {"M": M, "N": N, "geqrf_ms": round(geq, 3), "orgqr_ms": round(org, 3), "ms": round(geq + org, 3),
               "tflops": round(fl / (geq + org) / 1e9, 2), "cusolver_ms": round(tref, 3),
               "cusolver_tflops": round(fl / tref / 1e9, 2), "ratio_vs_cusolver": round((geq + org) / tref, 2),
               "max_abs_dQ_vs_cusolver": dq, "families": fam}
        print("  %6d x %4d  geqrf %8.2f ms  orgqr %8.2f ms  total %8.2f ms  %6.2f TFLOP/s | torch.linalg.qr %8.2f ms %6.2f TFLOP/s"
              " | ours/cuSOLVER %.2f | max|dQ| %.1e" % (M, N, geq, org, geq + org, row["tflops"], tref, row["cusolver_tflops"],
                                                      row["ratio_vs_cusolver"], dq), flush=True)
        print("      families: " + ", ".join("%s %.2f ms/%d" % (nm, ms, cnt) for nm, (ms, cnt) in sorted(fam.items(), key=lambda kv: -kv[1][0])),
              flush=True)
        rows.append(row)
    return rows


def c4(ctx, iters):
    import smcp_b200 as S
    from smcp_b200 import solvers
    t0 = time.time()
    P = S.mtxnorm_SDP(200, 200, 500, density=1.0, seed=0)
    print("  C4 generated in %.1f s" % (time.time() - t0), flush=True)
    out = {}
    for method in ("syrk", "householder"):
        solvers.options["maxiters"] = iters
        solvers.options["show_progress"] = False
        solvers.options["qr_method"] = method
        stamps = {}

        def hook(name, it):
            ctx.sync()
            stamps[it] = time.perf_counter()
        solvers._iteration_hook = hook
        ctx.region_reset()
        sol = P.solve_esd(kktsolver="qr")
        solvers._iteration_hook = None
        its = sorted(stamps)
        n_t = len(its) - 1
        ms_it = 1e3 * (stamps[its[-1]] - stamps[its[0]]) / n_t if n_t > 0 else float("nan")
        nit = max(1, sol["iterations"])
        regions = {nm: ctx.region_get(nm) for nm in ctx.region_names()}
        regions = {nm: (round(ms / nit, 3), calls) for nm, (ms, calls) in regions.items() if calls and nm.startswith("kkt_")}
        out[method] = {"status": sol["status"], "iterations": sol["iterations"], "ms_per_iteration": round(ms_it, 2),
                       "timed_iterations": n_t, "regions_ms_per_iteration": regions,
                       "primal_objective": sol["primal objective"], "gap": sol["gap"]}
        print("  C4 qr_method=%-11s status %-8s %3d iterations  %9.2f ms/iteration (%d timed; the first is not)  regions/iteration: %s"
              % (method, sol["status"], sol["iterations"], ms_it, n_t,
                 ", ".join("%s %.2f ms" % (nm, v[0]) for nm, v in sorted(regions.items()))), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=8)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--skip-c4", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_qr.py needs a CUDA device")
    from smcp_b200.device import Context
    ctx = Context.get()
    res = {"card": card(), "torch_device": torch.cuda.get_device_name(0)}
    print("card: %s (%s)" % (res["card"], res["torch_device"]), flush=True)
    print("(a) geqrf + orgqr, FP64, device time (median of %d after one warm-up run)" % args.reps, flush=True)
    res["dense"] = dense(ctx, args.reps)
    if not args.skip_c4:
        print("(b) C4 through solve_esd(kktsolver='qr'), maxiters = %d" % args.iters, flush=True)
        res["c4"] = c4(ctx, args.iters)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
