"""Cost and benefit of stopping at a relative tolerance (Session.solve(..., tol=)).

    python tools/tol_bench.py [--repeats 5] [--out profiles/tol_bench_b200.json]

1. Overhead: µs per iteration (info loop_ms / iterations) of PR-CG with no tolerance against the same run
   with a tolerance that is not reached (tol = 1e-150: the threshold is ~1e-300 nu_0), so that both runs
   do the same iterations; the difference is what the device test and, on the stream path, the chunked
   polling cost.  (The updated residual keeps falling after convergence and can still cross that
   threshold: a case whose tolerance run stops at k is then timed with max_iter = k on both sides.)
   One warm-up of each, then `repeats` alternating pairs; median / min / max.
2. Benefit: wall time of a solve (host copies in and out included, no histories) with a tolerance that
   is reached (tol = 1e-8) against the fixed max_iter the reference's protocol runs (figure_gen case
   tables; the 64^3 Poisson problem's 2000, SURVEY.md section 8d).  bcsstk18_None runs 1 750 000
   iterations (~30 s), so its fixed run is timed once.
The GPU name and power limit are read in the same process as the measurements."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import helpers                                                          # noqa: E402
from helpers import orc                                                 # noqa: E402
from new_cg_variants_b200 import PoissonStencil, Session                # noqa: E402

NEVER, REACHED = 1e-150, 1e-8


def problems():
    """name -> (operator, dinv, b, x0, reference max_iter)."""
    out = {}
    for case in ("bcsstk15_jacobi", "nos2_None", "bcsstk18_None"):
        A, b, x0, _, dinv, max_iter = helpers.case_problem(case)
        out[case] = (A, dinv, b, x0, max_iter)
    for n, it in ((64, 2000), (256, 300)):
        S = PoissonStencil(n, n, n, dim=3)
        rng = np.random.default_rng(0)
        out[f"poisson3d_{n}"] = (S, np.full(S.shape[0], 1.0 / S.diag), rng.standard_normal(S.shape[0]),
                                 np.zeros(S.shape[0]), it)
    return out


# (problem, path, iterations for the overhead runs)
OVERHEAD = [("poisson3d_64", "stream", 2000), ("poisson3d_64", "persistent", 2000),
            ("bcsstk15_jacobi", "persistent", 2000), ("nos2_None", "persistent", 5000),
            ("bcsstk18_None", "persistent", 20000), ("poisson3d_256", "stream", 300)]
# (problem, path, timed repeats of the fixed-max_iter run)
SOLUTION = [("poisson3d_64", "stream", None), ("poisson3d_64", "persistent", None),
            ("bcsstk15_jacobi", "persistent", None), ("nos2_None", "persistent", None),
            ("bcsstk18_None", "persistent", 1), ("poisson3d_256", "stream", None)]


def stat(v):
    return {"median": float(np.median(v)), "min": float(min(v)), "max": float(max(v)), "n": len(v)}


def overhead(sess, b, x0, path, iters, repeats):
    def run(tol):
        info = sess.solve("pr", b, x0, iters, histories=(), path=path, return_x=False, tol=tol)[2]
        assert info["path"] == (1 if path == "stream" else 2)
        return info

    def us(tol):
        info = run(tol)
        assert info["stop_iter"] == -1
        return 1e3 * info["loop_ms"] / info["iterations"]
    stop = run(NEVER)["stop_iter"]
    if stop >= 0:
        iters = stop
    us(None)
    off, on = [], []
    for _ in range(repeats):
        off.append(us(None))
        on.append(us(NEVER))
    rec = {"iterations": iters, "us_per_iter_tol_off": stat(off), "us_per_iter_tol_never_reached": stat(on)}
    rec["overhead_median_pct"] = 100.0 * (rec["us_per_iter_tol_never_reached"]["median"] / rec["us_per_iter_tol_off"]["median"] - 1)
    return rec


def solution(sess, b, x0, path, max_iter, repeats):
    def run(tol):
        t0 = time.perf_counter()
        info = sess.solve("pr", b, x0, max_iter, histories=(), path=path, return_x=True, tol=tol)[2]
        return time.perf_counter() - t0, info
    run(REACHED)
    t_tol, t_fix, info_tol, info_fix = [], [], None, None
    for _ in range(repeats):
        t, info_tol = run(REACHED)
        t_tol.append(t)
        t, info_fix = run(None)
        t_fix.append(t)
    return {"max_iter": max_iter, "tol": REACHED, "stop_iter": info_tol["stop_iter"],
            "wall_s_tol": stat(t_tol), "wall_s_fixed": stat(t_fix),
            "loop_ms_tol": info_tol["loop_ms"], "loop_ms_fixed": info_fix["loop_ms"],
            "speedup_median": float(np.median(t_fix) / np.median(t_tol))}


def gpu_identity():
    import torch
    out = {"gpu": torch.cuda.get_device_name(0)}
    try:
        out["power_limit_and_max_sm_clock"] = subprocess.run(
            ["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                                              # noqa: BLE001
        out["power_limit_and_max_sm_clock"] = f"unavailable: {e}"
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    res = {**gpu_identity(), "variant": "pr", "repeats": args.repeats, "overhead": [], "time_to_solution": []}
    probs = problems()
    sessions = {}
    try:
        for name, path, iters in OVERHEAD:
            A, dinv, b, x0, _ = probs[name]
            sess = sessions.setdefault(name, Session(A, dinv=dinv))
            rec = {"case": name, "path": path, **overhead(sess, b, x0, path, iters, args.repeats)}
            res["overhead"].append(rec)
            print(json.dumps(rec), flush=True)
        for name, path, reps in SOLUTION:
            A, dinv, b, x0, max_iter = probs[name]
            rec = {"case": name, "path": path, **solution(sessions[name], b, x0, path, max_iter, reps or args.repeats)}
            res["time_to_solution"].append(rec)
            print(json.dumps(rec), flush=True)
    finally:
        for s in sessions.values():
            s.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
