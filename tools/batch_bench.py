"""Nine variants of a case one after another (Session.solve, persistent path, default CTA shape on all
SMs) against the same nine in one cooperative launch (session.solve_batch, 1/9 of the SMs each).

    python tools/batch_bench.py [--repeats 5] [--out profiles/batch_bench.json]

Wall clock around work that ends in a device synchronise (both sides include the host copies of b, x0,
x_true in and x, histories out), one warm-up of each, then alternating repeats; median / min / max.
Per batch entry: µs per iteration of the shared launch and its CTA shape (threads T, CTAs nb, row
chunks per CTA R).  The batch's CTA width is fixed the way the library picks it first for a nine-way
share (256 threads up to 16 x 256 rows, else 512) so that the shape printed is the shape run."""
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
from new_cg_variants_b200 import PoissonStencil, Session, _lib          # noqa: E402
from new_cg_variants_b200.session import solve_batch                    # noqa: E402

TAGS = list(orc.VARIANTS)


def cases():
    out = []
    for case, iters in (("bcsstk18_None", 20000), ("bcsstk15_jacobi", None), ("nos2_None", None)):
        A, b, x0, xt, dinv, max_iter = helpers.case_problem(case)
        out.append((case, A, b, x0, xt, dinv, iters or max_iter))
    S = PoissonStencil(64, 64, 64, dim=3)
    xt, b, x0 = orc.setup_problem(S.tocsr())
    out.append(("poisson3d_64_jacobi", S, b, x0, xt, np.full(S.shape[0], 1.0 / S.diag), 2000))
    return out


def shape(n, sms, count=9):
    share = max(1, sms // count)
    T = 256 if n <= share * 256 else 512
    chunks = -(-n // T)
    R = -(-chunks // share)
    return T, -(-chunks // R), R


def bench_case(name, A, b, x0, xt, dinv, max_iter, hists, repeats, sms):
    n = A.shape[0]
    solo = Session(A, dinv=dinv)
    T, nb, R = shape(n, sms)
    batch = []
    for _ in TAGS:
        s = Session(A, dinv=dinv)
        s.set_option("pers_threads", T)
        batch.append(s)
    items = [(s, t, b, x0, max_iter, xt) for s, t in zip(batch, TAGS)]
    rec = {"case": name, "n": n, "max_iter": max_iter, "histories": list(hists)}

    def run_seq():
        return [solo.solve(t, b, x0, max_iter, x_true=xt, histories=hists, path="persistent")[2] for t in TAGS]

    def run_batch():
        return solve_batch(items, histories=hists)

    try:
        try:
            run_batch()
        except _lib.CgxError as e:
            rec["batch_refused"] = str(e)
        run_seq()
        seq, bat, infos = [], [], None
        for _ in range(repeats):
            t0 = time.perf_counter()
            seq_infos = run_seq()
            seq.append(time.perf_counter() - t0)
            if "batch_refused" not in rec:
                t0 = time.perf_counter()
                infos = [r[2] for r in run_batch()]
                bat.append(time.perf_counter() - t0)
        stat = lambda v: {"median_s": float(np.median(v)), "min_s": float(min(v)), "max_s": float(max(v))}   # noqa: E731
        rec["sequential"] = stat(seq)
        rec["sequential"]["us_per_iter"] = {t: 1e3 * i["loop_ms"] / max(1, i["iterations"]) for t, i in zip(TAGS, seq_infos)}
        if bat:
            rec["batch"] = stat(bat)
            rec["batch"]["cta_shape"] = {"T": T, "nb": nb, "R": R}
            rec["batch"]["us_per_iter"] = {t: 1e3 * i["loop_ms"] / max(1, i["iterations"]) for t, i in zip(TAGS, infos)}
            rec["speedup_median"] = rec["sequential"]["median_s"] / rec["batch"]["median_s"]
    finally:
        solo.close()
        for s in batch:
            s.close()
    return rec


def gpu_identity():
    import torch
    out = {"gpu": torch.cuda.get_device_name(0), "sms": torch.cuda.get_device_properties(0).multi_processor_count}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        out["power_limit_and_max_sm_clock"] = q
    except Exception as e:                                              # noqa: BLE001
        out["power_limit_and_max_sm_clock"] = f"unavailable: {e}"
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    ident = gpu_identity()
    res = {**ident, "repeats": args.repeats, "results": []}
    for name, A, b, x0, xt, dinv, max_iter in cases():
        for hists in (_lib.HIST_NAMES, ()):
            rec = bench_case(name, A, b, x0, xt, dinv, max_iter, hists, args.repeats, ident["sms"])
            res["results"].append(rec)
            print(json.dumps(rec), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
