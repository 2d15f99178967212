"""Variable-coefficient stencil (VariableStencil) against the same matrix as CSR, on one GPU.

    python tools/varstencil_bench.py [--repeats 5] [--iters 300] [--out profiles/varstencil_bench_b200.json]

1. µs per iteration (info loop_ms / iterations, stream path, no histories, Jacobi vector) at 256^3 and
   4096^2 for HS, CG, PR, GV and pipe-PR.  Operators: VariableStencil, Session(S.tocsr()), and the
   constant-coefficient PoissonStencil of the same grid with its Jacobi vector (the ceiling: no matrix
   bytes).  One warm-up run of every (operator, variant), then `repeats` rounds that alternate the three
   operators; median / min / max.
2. SpMV roofline of the VariableStencil pass (and of the PoissonStencil pass for comparison): event-timed
   duration per launch of the variant's SpMV class (Session.set_profile) against its algorithmic bytes,
   8 n (vector words + coefficient words: diag, cx, cy [, cz] = 4 in 3-D, 3 in 2-D; 0 for PoissonStencil),
   as a fraction of the HBM peak bench.py uses (MEASURED_PEAKS.json hbm_gbs, or its stated fallback).
The coefficients: a diffusion operator -div(k grad u) with a log-normal k, so every coupling differs.
The GPU name and power limit are read in the same process as the measurements."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from new_cg_variants_b200 import PoissonStencil, Session, VariableStencil      # noqa: E402

VARIANTS = ("hs", "cg", "pr", "gv", "pipe_pr")
# vector words the variant's SpMV pass moves per row with a Jacobi vector (cgx_varstencil.cuh epilogues)
SP_CLASS = {"hs": ("sp_hs", 2), "cg": ("sp_cg", 3), "pr": ("sp_pr", 4), "gv": ("sp_gv", 2), "pipe_pr": ("sp_pipe_r", 4)}
GRIDS = {"3d_256": (256, 256, 256, 3), "2d_4096": (4096, 4096, 1, 2)}


def diffusion(nx, ny, nz, dim, seed=0):
    """Cell-centred -div(k grad u) with a log-normal k per point: the coupling between neighbours i and
    j is -2 k_i k_j / (k_i + k_j), the diagonal the sum of the couplings' magnitudes (Dirichlet: a
    neighbour outside the grid still adds its face, with k of the point itself)."""
    rng = np.random.default_rng(seed)
    k = np.exp(rng.standard_normal((nz, ny, nx)))
    coefs, diag = [], np.zeros_like(k)
    for axis in ((2, 1, 0) if dim == 3 else (2, 1)):
        a = np.moveaxis(k, axis, -1)
        c = np.zeros_like(a)
        c[..., :-1] = -2.0 * a[..., :-1] * a[..., 1:] / (a[..., :-1] + a[..., 1:])
        d = -c
        d[..., 1:] += -c[..., :-1]
        d[..., 0] += a[..., 0]
        d[..., -1] += a[..., -1]
        coefs.append(np.moveaxis(c, -1, axis).reshape(-1))
        diag += np.moveaxis(d, -1, axis)
    cz = coefs[2] if dim == 3 else None
    return VariableStencil(nx, ny, nz, diag.reshape(-1), coefs[0], coefs[1], cz)


def stat(v):
    return {"median": float(np.median(v)), "min": float(min(v)), "max": float(max(v)), "n": len(v)}


def us_per_iter(sess, tag, b, x0, iters):
    info = sess.solve(tag, b, x0, iters, histories=(), path="stream", return_x=False)[2]
    assert info["path"] == 1 and info["iterations"] == iters - 1
    return 1e3 * info["loop_ms"] / info["iterations"]


def sp_duration_ms(sess, tag, b, x0, iters):
    sess.set_profile(True)
    try:
        sess.solve(tag, b, x0, iters, histories=(), path="stream", return_x=False)
        prof = sess.get_profile()
    finally:
        sess.set_profile(False)
    if SP_CLASS[tag][0] not in prof:           # (PoissonStencil PR: one fused launch per iteration, no SpMV pass)
        return None
    ms, cnt = prof[SP_CLASS[tag][0]]
    return ms / cnt


def peak_gbs():
    """The HBM peak bench.py divides by (MEASURED_PEAKS.json hbm_gbs when the machine has one), and its source."""
    import bench
    return bench.measured_peak()


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
    ap.add_argument("--iters", type=int, default=300)
    ap.add_argument("--grids", default=",".join(GRIDS))
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    peak, peak_note = peak_gbs()
    res = {**gpu_identity(), "repeats": args.repeats, "iterations": args.iters - 1, "path": "stream",
           "preconditioner": "Jacobi vector", "peak_gbs": peak, "peak_source": peak_note, "cases": []}
    for gname in args.grids.split(","):
        nx, ny, nz, dim = GRIDS[gname]
        S = diffusion(nx, ny, nz, dim)
        n = S.shape[0]
        rng = np.random.default_rng(1)
        b, x0 = rng.standard_normal(n), np.zeros(n)
        P = PoissonStencil(nx, ny, nz, dim=dim)
        ops = {"varstencil": (S, 1.0 / S.diag), "csr": (S.tocsr(), 1.0 / S.diag), "poisson": (P, np.full(n, 1.0 / P.diag))}
        sessions = {}
        try:
            for name, (A, dinv) in ops.items():
                sessions[name] = Session(A, dinv=dinv)
            for tag in VARIANTS:
                for s in sessions.values():
                    us_per_iter(s, tag, b, x0, args.iters)                 # warm-up
                t = {name: [] for name in sessions}
                for _ in range(args.repeats):
                    for name, s in sessions.items():
                        t[name].append(us_per_iter(s, tag, b, x0, args.iters))
                rec = {"grid": gname, "n": n, "variant": tag, **{f"us_per_iter_{k}": stat(v) for k, v in t.items()}}
                rec["speedup_vs_csr_median"] = rec["us_per_iter_csr"]["median"] / rec["us_per_iter_varstencil"]["median"]
                cls, vw = SP_CLASS[tag]
                for name, cw in (("varstencil", dim + 1), ("poisson", 0)):
                    ms = sp_duration_ms(sessions[name], tag, b, x0, min(args.iters, 100))
                    if ms is None:
                        continue
                    bytes_ = 8.0 * n * (vw + cw)
                    rec[f"spmv_{name}"] = {"class": cls, "us_per_launch": 1e3 * ms, "algorithmic_bytes": bytes_,
                                           "gbs": bytes_ / (ms * 1e6),
                                           "fraction_of_peak": bytes_ / (ms * 1e6) / peak}
                res["cases"].append(rec)
                print(json.dumps(rec), flush=True)
        finally:
            for s in sessions.values():
                s.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
