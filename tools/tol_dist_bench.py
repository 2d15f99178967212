"""Cost and benefit of stopping a PARTITIONED solve at a relative tolerance (GroupSession.solve(..., tol=)).

    python tools/tol_dist_bench.py [--repeats 5] [--out profiles/tol_dist_bench_b200.json]

The ranks are emulated on one GPU (GroupSession: every rank a context on device 0, the same kernels and
the same peer-to-peer protocol as one process per GPU).  These numbers say nothing about NVLink: they
measure the device-side stop test and the host's chunked polling on the partitioned kernels.

1. Overhead: µs per iteration (rank 0's loop_ms / iterations) with no tolerance against the same run
   with a tolerance that is not reached (tol = 1e-150), same iterations on both sides, on the stream path
   (two-kernel PR-CG, single-launch PR-CG), the persistent path on slabs, and a CSR row partition.
   One warm-up of each, then `repeats` alternating pairs; median / min / max.
2. Benefit: wall time of a solve (host copies in and out included, no histories) with tol = 1e-8
   against a fixed max_iter.
The GPU name, power limit and clocks are read in the same process as the measurements."""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

from new_cg_variants_b200 import PoissonStencil                         # noqa: E402
from new_cg_variants_b200.dist import GroupSession                      # noqa: E402
from new_cg_variants_b200.experiments import banded_model_problem       # noqa: E402
from tol_bench import gpu_identity, stat                                # noqa: E402

NEVER, REACHED = 1e-150, 1e-8


def problems():
    """name -> (operator, dinv, b, x0)."""
    out = {}
    for name, S in (("poisson3d_128", PoissonStencil(128, 128, 128, dim=3)),
                    ("poisson3d_64x64x16", PoissonStencil(64, 64, 16, dim=3))):
        rng = np.random.default_rng(0)
        out[name] = (S, np.full(S.shape[0], 1.0 / S.diag), rng.standard_normal(S.shape[0]), np.zeros(S.shape[0]))
    A = banded_model_problem(n=400000, k=7)[0]
    rng = np.random.default_rng(0)
    out["banded_400k"] = (A, None, rng.standard_normal(A.shape[0]), np.zeros(A.shape[0]))
    return out


# (label, problem, variant, path, options, iterations of the overhead runs, fixed max_iter)
CASES = [
    ("stream two-kernel PR", "poisson3d_128", "pr", "stream", {"pr_fused": 0}, 1000, 2000),
    ("stream fused PR", "poisson3d_128", "pr", "stream", {"pr_fused": 1, "fused_min_slab": 1}, 1000, 2000),
    ("stream CG", "poisson3d_128", "cg", "stream", {}, 1000, 2000),
    ("persistent PR", "poisson3d_64x64x16", "pr", "persistent", {}, 2000, 2000),
    ("CSR row partition CG", "banded_400k", "cg", "stream", {}, 1000, 5000),
]


def overhead(grp, tag, b, x0, path, iters, repeats):
    def run(tol):
        infos = grp.solve(tag, b, x0, iters, histories=(), path=path, tol=tol)[2]
        assert infos[0]["path"] == (1 if path == "stream" else 2)
        return infos[0]

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


def solution(grp, tag, b, x0, path, max_iter, repeats):
    def run(tol):
        t0 = time.perf_counter()
        infos = grp.solve(tag, b, x0, max_iter, histories=(), path=path, tol=tol)[2]
        return time.perf_counter() - t0, infos[0]
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--worlds", default="2,4")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    res = {**gpu_identity(), "emulation": "all ranks on one GPU (GroupSession): no NVLink traffic is measured",
           "repeats": args.repeats, "overhead": [], "time_to_solution": []}
    probs = problems()
    for world in map(int, args.worlds.split(",")):
        for label, name, tag, path, opts, iters, max_iter in CASES:
            A, dinv, b, x0 = probs[name]
            grp = GroupSession(A, world, dinv=dinv)
            try:
                for m in grp.members:
                    for k, v in opts.items():
                        m.set_option(k, v)
                head = {"case": label, "problem": name, "variant": tag, "path": path, "world": world,
                        "emulated": True, "options": opts}
                rec = {**head, **overhead(grp, tag, b, x0, path, iters, args.repeats)}
                res["overhead"].append(rec)
                print(json.dumps(rec), flush=True)
                rec = {**head, **solution(grp, tag, b, x0, path, max_iter, args.repeats)}
                res["time_to_solution"].append(rec)
                print(json.dumps(rec), flush=True)
            finally:
                grp.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
