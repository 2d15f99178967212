#!/usr/bin/env python3
"""bench.py -- headline benchmark of the B200 CG path (contract: see DESIGN.md "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--variant pr] [--grid 256] [--dim 3] [--iters 200] [--dump-outputs DIR]

Workload (BASELINE.json configs[3], the one the metric is quoted on): 3-D Poisson 7-point,
256^3 grid (16.8 M unknowns), Jacobi-preconditioned, x_true = 1/sqrt(n), b = A x_true,
x0 = 0, fp64.  A "step" is one solve of `iters` CG iterations from x0 (initialisation
included).  N GPUs shard the grid into z-slabs (strong scaling, one problem).

  value  : iterations/s with b, x0 resident in HBM, timed with CUDA events on the library's
           launch stream (max over ranks), instrumentation off (the reference's
           callbacks=[] timing protocol, BASELINE.md section 2)
  e2e    : the same through the C-ABI call with HOST buffers (cgx_solve_host): pinned
           b/x0 copied in, x copied out (into a pinned buffer), inside the timed region
           (wall clock + sync)
  roofline / cpu_baseline : see DESIGN.md
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W_V = {"hs": 13, "cg": 14, "pr": 14, "m": 14, "gv": 21, "pipe_pr": 23, "pipe_p": 23,
       "pipe_pr_m": 23, "pipe_p_m": 23}          # SURVEY.md section 8d: fp64 words/row/iteration
# algorithmic fp64 words per row per launch of each kernel class (reads + writes; "+d" = one
# more when a Jacobi vector is read) -- DESIGN.md "Kernels"
CLASS_WORDS = {"ew_hs1": (3, 1), "ew_hs2": (5, 1), "ew_cg": (11, 1), "ew_gv": (19, 1), "ew_pr": (9, 1),
               "ew_pipe_r": (14, 1), "ew_pipe_n": (18, 1), "sp_hs": (2, 0), "sp_cg": (3, 0), "sp_gv": (2, 0),
               "sp_pr": (3, 1), "sp_pipe_r": (4, 0), "sp_pipe_n": (2, 0),
               "pr_fused": (10, 0)}        # one launch per PR-CG iteration: R x,r,p,s,rt  W x,r,p,s,rt
# with a constant Jacobi diagonal (or none) on the TMA stencil path CG-CG does not stream r~ and
# GV does not stream w~ (DESIGN.md "Kernels"): their kernels then move fewer words
CLASS_WORDS_ELIDED = {"ew_cg": (9, 0), "sp_cg": (2, 0), "ew_gv": (17, 0)}
REF_FUN = {"hs": "hs_pcg", "cg": "cg_pcg", "gv": "gv_pcg", "pr": "pr_pcg", "m": "m_pcg",
           "pipe_pr": "pipe_pr_pcg"}


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled every 200 ms during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "200", "-i", str(self.gpu)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [l.strip().split(",") for l in open(self.f.name) if l.strip()]
        os.unlink(self.f.name)
        sm, smmax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[1])); smmax.append(float(r[2]))
                for nm, v in zip(names, r[5:9]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None,
                "sm_max_mhz": max(smmax) if smmax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def build_problem(grid, dim=3):
    from new_cg_variants_b200 import PoissonStencil
    S = PoissonStencil(grid, grid, grid, dim=3) if dim == 3 else PoissonStencil(grid, grid, 1, dim=2)
    n = S.shape[0]
    x_true = np.ones(n) / np.sqrt(n)           # figure_gen.py:31-34
    b = S @ x_true
    x0 = np.zeros(n)
    dinv = 1 / S.diagonal()                    # figure_gen.py:43
    return S, b, x0, x_true, dinv


def pinned(a):
    import torch
    t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    return t, t.numpy()


DUMP_MAX_ENTRIES = 1 << 22        # 32 MB of float64


def dump_outputs(out_dir, x):
    """--dump-outputs: the solution x of the last timed step as out_dir/x.npy (float64).  Above
    DUMP_MAX_ENTRIES entries it holds x at the sorted indices
    np.random.default_rng(0).choice(n, DUMP_MAX_ENTRIES, replace=False): the same entries for
    the same arguments, so that two builds can be compared output for output."""
    if x.shape[0] > DUMP_MAX_ENTRIES:
        x = x[np.sort(np.random.default_rng(0).choice(x.shape[0], DUMP_MAX_ENTRIES, replace=False))]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "x.npy"), np.ascontiguousarray(x, dtype=np.float64))


# ------------------------------------------------------------------------------ reference arm
def _cpu_threads():
    """Use every host core for the BLAS part whatever the launcher exported (torchrun sets
    OMP_NUM_THREADS=1): returns (context manager, threads actually in use)."""
    from threadpoolctl import threadpool_info, threadpool_limits
    want = max(1, len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1))
    ctl = threadpool_limits(limits=want)
    blas = max([p.get("num_threads", 1) for p in threadpool_info()] or [1])
    return ctl, blas


def _timed_oracle(orc, variant, A, b, x0, dinv, its, repeats):
    """Seconds per `its` loop iterations of the oracle, initialisation excluded: each repeat times
    solve(max_iter = its + 1) minus the initialisation alone (solve(max_iter = 1), best of 2)."""
    t_init = None
    for _ in range(2):
        t0 = time.perf_counter()
        orc.solve(variant, A, b, x0, 1, dinv=dinv, history=False)
        dt = time.perf_counter() - t0
        t_init = dt if t_init is None else min(t_init, dt)
    out = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        orc.solve(variant, A, b, x0, its + 1, dinv=dinv, history=False)
        out.append(max(1e-9, time.perf_counter() - t0 - t_init))
    return out, t_init


def run_reference(args, rank, world):
    """The reference's CPU path: its algorithm restated in numpy/scipy (oracle/cg_oracle.py,
    bit-identical to the reference's *_pcg on the same machine) on the same workload.  The
    reference is pure Python and /root/reference does not travel to the GPU box, so this is
    the "port" kind.  Each step is a bounded sample: `ref_iters` loop iterations from x0
    (BASELINE.md section 2: 6 iterations, callbacks=[], precomputed dinv), initialisation
    excluded, all host cores."""
    if rank != 0:
        return
    from oracle import cg_oracle as orc
    ctl, blas = _cpu_threads()
    t0 = time.time()
    A = orc.poisson3d(args.grid) if args.dim == 3 else orc.poisson2d(args.grid)
    x_true, b, x0 = orc.setup_problem(A)
    dinv = orc.jacobi_dinv(A)
    build_s = time.time() - t0
    its = args.ref_iters
    for _ in range(min(args.warmup, 1)):       # one warm-up solve (BASELINE.md section 2)
        orc.solve(args.variant, A, b, x0, its + 1, dinv=dinv, history=False)
    times, t_init = _timed_oracle(orc, args.variant, A, b, x0, dinv, its, args.steps)
    dt = sum(times)
    value = its * args.steps / dt
    n = A.shape[0]
    line = {
        "impl": "reference", "metric": f"CG iterations/s ({REF_FUN.get(args.variant, args.variant)}, Jacobi, {args.dim}-D Poisson {args.grid}^{args.dim})",
        "value": value, "unit": "iterations/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"poisson{args.dim}d_{args.grid} {REF_FUN.get(args.variant, args.variant)} jacobi (scipy CSR, nnz={A.nnz})",
                   "iters_per_step": its, "n": n},
        "cpu_baseline": {"value": value, "unit": "iterations/s", "cores": blas, "kind": "port",
                         "best_step_value": its / min(times),
                         "sample": f"{args.steps} x {its} loop iterations of the numpy/scipy restatement on the full {args.grid}^{args.dim} CSR matrix, "
                                   f"initialisation ({t_init:.2f}s) excluded (scipy SpMV single-threaded, OpenBLAS dots {blas} threads set explicitly, "
                                   f"host has {os.cpu_count()} cpus; matrix build {build_s:.1f}s untimed)"},
        "e2e": {"value": value, "unit": "iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "hbm_gbs_model": value * (8 * n * W_V[args.variant] + 12 * A.nnz + 4 * (n + 1)) / 1e9,
    }
    emit(line)


# ------------------------------------------------------------------------------------ our arm
def cpu_baseline_sample(args, dev_hist=None):
    """Bounded CPU sample of the same workload (min of 3 runs of `cpu_iters` loop iterations,
    initialisation excluded) and -- the oracle being the checker -- the agreement of the device's
    first iterations with it (`parity`)."""
    from oracle import cg_oracle as orc
    ctl, blas = _cpu_threads()
    A = orc.poisson3d(args.grid) if args.dim == 3 else orc.poisson2d(args.grid)
    x_true, b, x0 = orc.setup_problem(A)
    dinv = orc.jacobi_dinv(A)
    its = args.cpu_iters
    orc.solve(args.variant, A, b, x0, 2, dinv=dinv, history=False)      # warm-up
    times, t_init = _timed_oracle(orc, args.variant, A, b, x0, dinv, its, 3)
    best = min(times)
    out = {"value": its / best, "unit": "iterations/s", "cores": blas, "kind": "port",
           "sample": f"min of 3 runs of {its} loop iterations of oracle/cg_oracle.py ({REF_FUN.get(args.variant, args.variant)}, callbacks=[], "
                     f"precomputed dinv, initialisation excluded) on the full {args.grid}^{args.dim} scipy CSR matrix; scipy SpMV single-threaded, "
                     f"OpenBLAS {blas} threads, host {os.cpu_count()} cpus"}
    parity = None
    if dev_hist is not None:
        k = args.parity_iters
        ref = orc.solve(args.variant, A, b, x0, k, dinv=dinv, x_true=x_true)
        worst = 0.0
        for h in ("updated_residual_2_norm", "residual_2_norm", "error_A_norm"):
            rel = np.abs(dev_hist[h][:k] - ref[h][:k]) / np.abs(ref[h][:k])
            worst = max(worst, float(rel.max()))
        parity = {"iterations": k, "max_rel": worst, "tolerance": 1e-10, "ok": bool(worst <= 1e-10),
                  "what": "device histories (updated/true residual norm, A-norm error) vs the oracle on the same problem, k < %d" % k}
    return out, parity


def read_traffic(kernel_class):
    """ncu-measured DRAM bytes per launch of `kernel_class` from profiles/traffic.json -- only when
    the file was recorded for the library that is loaded now (kernel-source fingerprint), so a
    stale capture is never echoed."""
    try:
        from new_cg_variants_b200 import build as _b
        t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        ent = t.get(kernel_class)
        if not isinstance(ent, dict):
            return None, "no ncu capture recorded for this kernel"
        if ent.get("kernel_sources_sha") != _b.kernel_fingerprint(kernel_class):
            return None, "stale: profiles/traffic.json was captured for other kernel sources"
        return ent["dram_bytes_per_launch"], ent.get("source", "profiles/traffic.json")
    except Exception as e:                                    # noqa: BLE001
        return None, f"unavailable ({type(e).__name__})"


def check_partitioned_answer(args, sess, S, b, x0, x_true, dinv, rank, world, local_rank):
    """N > 1: verify the answer of the path that was timed.
      (1) side problem 64^3, 25 iterations: the N-process run (x and all four histories) is
          BIT-IDENTICAL to the same partition emulated as N contexts on rank 0's GPU;
      (2) the full problem, 40 iterations with instrumentation: the partitioned histories agree
          with the single-GPU run on rank 0 to 1e-10 (another summation order of the dots)."""
    import torch.distributed as dist
    from new_cg_variants_b200 import PoissonStencil, Session
    from new_cg_variants_b200.dist import DistSession, GroupSession
    out = {"ok": True}
    hn = ("error_A_norm", "residual_2_norm", "error_2_norm", "updated_residual_2_norm")
    # (1)
    g = 64
    S2 = PoissonStencil(g, g, g, dim=3)
    n2 = S2.shape[0]
    xt2 = np.ones(n2) / np.sqrt(n2)
    b2, x02, d2 = S2 @ xt2, np.zeros(n2), 1 / S2.diagonal()
    ds = DistSession(S2, dinv=d2, device=local_rank, rank=rank, world=world)
    xl, hl, _ = ds.solve(args.variant, b2, x02, 26, x_true=xt2, histories=hn, path="stream")
    xg = ds.gather_x(xl)
    ds.close()
    if rank == 0:
        gs = GroupSession(S2, world, dinv=d2, devices=[local_rank] * world)
        xe, he, _ = gs.solve(args.variant, b2, x02, 26, x_true=xt2, histories=hn, path="stream")
        gs.close()
        same = bool(np.array_equal(xg, xe)) and all(np.array_equal(hl[h], he[h]) for h in hn)
        out["side_problem_bitwise_equal_to_emulation"] = same
        out["ok"] &= same
    # (2)
    k = 41
    sess.load_problem(b, x0, x_true)
    sess.run(args.variant, k, histories=hn, path=args.path)
    _, hist = sess.fetch_local(want_x=False, want_hist=True)
    sess.load_problem(b, x0, None)
    if rank == 0:
        one = Session(S, dinv=dinv, device=local_rank)
        _, h1, _ = one.solve(args.variant, b, x0, k, x_true=x_true, path="stream")
        one.close()
        worst = 0.0
        for i, h in enumerate(hn):
            rel = np.abs(hist[i] - h1[h]) / np.abs(h1[h])
            worst = max(worst, float(rel.max()))
        out["full_problem_vs_1gpu_max_rel"] = worst
        out["full_problem_iterations"] = k - 1
        out["ok"] &= bool(worst <= 1e-10)
    flag = __import__("torch").tensor([1 if out["ok"] else 0], device="cuda")
    dist.broadcast(flag, 0)
    out["ok"] = bool(flag.item())
    return out


def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from new_cg_variants_b200 import Session

    torch.cuda.set_device(local_rank)
    if world > 1:
        from new_cg_variants_b200.dist import DistSession      # row-partitioned multi-GPU path
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    S, b, x0, x_true, dinv = build_problem(args.grid, args.dim)
    n = S.shape[0]
    its = args.iters
    variant = args.variant
    if world > 1:
        sess = DistSession(S, dinv=dinv, device=local_rank, rank=rank, world=world)
    else:
        sess = Session(S, dinv=dinv, device=local_rank)
    sess.load_problem(b, x0, None)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_resident():
        info = sess.run(variant, its + 1, histories=(), path=args.path)
        return info["setup_ms"] + info["loop_ms"], info["loop_ms"], info["kernel_launches"]

    for _ in range(args.warmup):
        step_resident()
    sampler = ClockSampler(local_rank)
    barrier()
    if rank == 0:
        sampler.start()
    t0 = time.perf_counter()
    dev_ms = loop_ms = 0.0
    launches = 0
    for _ in range(args.steps):
        a, l, k = step_resident()
        dev_ms += a; loop_ms += l; launches += k
    barrier()
    wall_ms = 1e3 * (time.perf_counter() - t0)
    clocks = sampler.stop() if rank == 0 else None
    if world > 1:
        t = torch.tensor([dev_ms, loop_ms, wall_ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms, loop_ms, wall_ms = t.tolist()
    value = its * args.steps / (dev_ms / 1e3)
    if args.dump_outputs:              # before the e2e pass below overwrites x
        x = sess.fetch(want_hist=False)[0] if world == 1 else sess.gather_x(sess.fetch_local(want_hist=False)[0])
        if rank == 0:
            dump_outputs(args.dump_outputs, x)

    # ---- e2e through the C-ABI call with host buffers (pinned), copies inside the timing
    e2e = None
    if world == 1:
        tb, hb = pinned(b)
        tx0, hx0 = pinned(x0)
        txo, hxo = pinned(np.empty(n))          # the result lands in pinned host memory too
        for _ in range(2):
            sess.solve(variant, hb, hx0, its + 1, histories=(), path=args.path, x_out=hxo)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            x, _, info = sess.solve(variant, hb, hx0, its + 1, histories=(), path=args.path, x_out=hxo)
        barrier()
        e_dt = time.perf_counter() - t0
        e2e = {"value": its * args.steps / e_dt, "unit": "iterations/s",
               "h2d_bytes_per_step": info["h2d_bytes"], "d2h_bytes_per_step": info["d2h_bytes"],
               "ms_per_step": 1e3 * e_dt / args.steps,
               "api": "cgx_solve_host (Session.solve): pinned host b,x0 in, x out (pinned)"}
    else:
        tb, hb = pinned(sess.local(b))
        tx0, hx0 = pinned(sess.local(x0))
        txo, hxo = pinned(np.empty(sess.n))
        e2e = sess.e2e_bench(variant, hb, hx0, its + 1, args.steps, barrier, x_out=hxo)
        t = torch.tensor([e2e["ms_per_step"]], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e["ms_per_step"] = t.item()
        e2e["value"] = its / (t.item() / 1e3)

    # ---- per-kernel timing for the roofline (separate, untimed pass with event pairs; on
    #      N > 1 the rows are this rank's slab and the times include waiting for the peers)
    n_loc = n if world == 1 else sess.n
    peak, peak_src = measured_peak()
    sess.set_profile(True)
    sess.run(variant, its + 1, histories=(), path="stream")
    prof = sess.get_profile()
    sess.set_profile(False)
    top = max(prof, key=lambda c: prof[c][0])
    ms, cnt = prof[top]
    # a constant Jacobi diagonal (every Poisson stencil) travels as a scalar: no dinv stream
    dinv_stream = 0 if np.all(dinv == dinv[0]) else 1
    words_tab = dict(CLASS_WORDS)
    if not dinv_stream:
        words_tab.update(CLASS_WORDS_ELIDED)
    cw = lambda c: words_tab[c][0] + words_tab[c][1] * dinv_stream
    words = cw(top)
    bytes_per_launch = 8.0 * n_loc * words
    achieved = bytes_per_launch / (ms / cnt * 1e-3) / 1e9
    traffic, traffic_note = read_traffic(top)
    roofline = {"bound": "hbm", "kernel": top, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic if world == 1 else None, "traffic_source": traffic_note,
                "peak_source": peak_src,
                "algorithmic_bytes_per_launch": bytes_per_launch, "avg_launch_ms": ms / cnt,
                "rows_per_launch": n_loc,
                "share_of_loop": ms / sum(v[0] for v in prof.values()),
                "kernels": {c: {"avg_ms": v[0] / v[1], "launches": v[1],
                                "words_per_row": cw(c),
                                "actual_us": 1e3 * v[0] / v[1],
                                "ideal_us": 8.0 * n_loc * cw(c) / (peak * 1e9) * 1e6,
                                "GBps": 8.0 * n_loc * cw(c) / (v[0] / v[1] * 1e-3) / 1e9}
                            for c, v in prof.items() if c in CLASS_WORDS}}
    # ---- the other variants on the same problem (2 solves each, resident inputs)
    variants = {}
    for v in ("hs", "cg", "m", "gv", "pr", "pipe_pr"):
        sess.run(v, its + 1, histories=(), path=args.path)
        info = sess.run(v, its + 1, histories=(), path=args.path)
        lm = info["loop_ms"]
        if world > 1:
            t = torch.tensor([lm], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            lm = t.item()
        ips = its / (lm / 1e3)
        variants[v] = {"iterations_per_s_loop": ips, "ms_per_iteration": lm / its,
                       "hbm_gbs_model": ips * 8 * n * W_V[v] / 1e9,
                       "pct_of_8TBs_per_gpu": 100 * ips * 8 * n * W_V[v] / 8e12 / world}

    # ---- correctness of what was timed
    dist_check = None
    if world > 1:
        dist_check = check_partitioned_answer(args, sess, S, b, x0, x_true, dinv, rank, world, local_rank)
    cpu = parity = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        _, dev_hist, _ = sess.solve(variant, b, x0, args.parity_iters, x_true=x_true, path=args.path)
        cpu, parity = cpu_baseline_sample(args, dev_hist)

    if rank == 0:
        b_iter = 8.0 * n * W_V[variant]
        line = {
            "metric": f"CG iterations/s ({REF_FUN.get(variant, variant)}, Jacobi, {args.dim}-D Poisson {args.grid}^{args.dim})",
            "value": value, "unit": "iterations/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"poisson{args.dim}d_{args.grid} {REF_FUN.get(variant, variant)} jacobi (matrix-free {2 * args.dim + 1}-point stencil)",
                       "n": n, "iters_per_step": its, "path": args.path, "partition": f"z-slabs x{world}",
                       "l2": "no flush needed: one iteration streams %.2f GB >> 126 MB L2" % (b_iter / 1e9)},
            "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
            "wall_ms_per_step": wall_ms / args.steps, "loop_ms_per_iteration": loop_ms / (its * args.steps),
            "hbm_gbs_model": value * b_iter / 1e9, "pct_of_8TBs": 100 * value * b_iter / 8e12 / world,
            "pct_of_measured_peak": 100 * value * b_iter / 1e9 / measured_peak()[0] / world,
            "roofline": roofline, "cpu_baseline": cpu, "variants": variants,
        }
        if parity is not None:
            line["parity"] = parity
            line["parity_max_rel"] = parity["max_rel"]
        if dist_check is not None:
            line["dist_check"] = "ok" if dist_check["ok"] else "FAILED"
            line["dist_check_detail"] = dist_check
        emit(line)
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------- latency-bound tail (configs[4])
def run_tail(args, rank, world, local_rank):
    """BASELINE.json configs[4] / SURVEY.md section 8d "allreduce-hiding metric": 3-D Poisson 64^3,
    fixed 2000 iterations, HS-CG vs PR-CG vs pipe-PR-CG (+ GV, CG-CG).  Per variant, exchange mode
    (peer-to-peer LL records | ncclAllReduce on a side stream) and path (stream kernels |
    persistent cooperative kernel): loop time per iteration with the scalar exchange LIVE and
    STUBBED to a local stand-in, `--tail-reps` repeats each (median, min, max; CUDA events, max
    over ranks).   exposed = live - stub ;  hidden(v) = 1 - exposed(v) / exposed(base)."""
    import torch
    import torch.distributed as dist
    from new_cg_variants_b200 import PoissonStencil, Session
    torch.cuda.set_device(local_rank)
    g = args.tail_grid
    S = PoissonStencil(g, g, g, dim=3)
    n = S.shape[0]
    x_true = np.ones(n) / np.sqrt(n)
    b, x0, dinv = S @ x_true, np.zeros(n), 1 / S.diagonal()
    its, reps = args.tail_iters, max(5, args.tail_reps)
    variants = ("hs", "cg", "pr", "gv", "pipe_pr")
    stats = lambda v: {"median": statistics.median(v), "min": min(v), "max": max(v)}     # noqa: E731
    out = {}
    if world > 1:
        from new_cg_variants_b200.dist import DistSession
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def timed(sess, v, path):
        ts = []
        for rep in range(reps + 1):
            if world > 1:
                dist.barrier()
            info = sess.run(v, its + 1, path=path)
            t = info["loop_ms"]
            if world > 1:
                tt = torch.tensor([t], dtype=torch.float64, device="cuda")
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                t = tt.item()
            if rep > 0:
                ts.append(1e3 * t / its)
        return ts

    combos = [("p2p", "stream"), ("p2p", "persistent"), ("nccl", "stream")] if world > 1 else [("none", "stream"), ("none", "persistent")]
    for mode, path in combos:
        if world > 1:
            sess = DistSession(S, dinv=dinv, device=local_rank, rank=rank, world=world, mode=mode)
        else:
            sess = Session(S, dinv=dinv, device=local_rank)
        sess.load_problem(b, x0, None)
        m = {}
        for v in variants:
            live = timed(sess, v, path)
            ent = {"live": stats(live)}
            if world > 1:
                sess.set_option("stub_allreduce", 1)
                stub = timed(sess, v, path)
                sess.set_option("stub_allreduce", 0)
                ent["stub"] = stats(stub)
                ent["exposed"] = ent["live"]["median"] - ent["stub"]["median"]
                ent["exposed_per_repeat"] = [a - c for a, c in zip(sorted(live), sorted(stub))]
            m[v] = ent
        if world > 1:
            for v in m:
                for base in ("hs", "pr"):
                    if m[base]["exposed"] > 0:
                        m[v][f"hidden_vs_{base}"] = 1 - m[v]["exposed"] / m[base]["exposed"]
                        m[v][f"hidden_vs_{base}_per_repeat"] = [1 - e / f if f > 0 else None for e, f in
                                                                zip(m[v]["exposed_per_repeat"], m[base]["exposed_per_repeat"])]
        out[f"{mode}/{path}"] = m
        sess.close()
        if world > 1:
            dist.barrier()
    if rank == 0:
        key = min(out, key=lambda k: out[k]["pipe_pr"]["live"]["median"])
        best = out[key]
        line = {"metric": f"latency-bound tail: us/iteration (pipe_pr_pcg, Jacobi, 3-D Poisson {g}^3, {its} iterations)",
                "value": best["pipe_pr"]["live"]["median"], "unit": "us/iteration", "n_gpus": world, "steps": reps,
                "warmup": 1, "higher_is_better": False, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
                "data": "synthetic", "config": {"workload": f"poisson3d_{g} tail (BASELINE.json configs[4])", "n": n,
                                                "iters_per_step": its, "best_mode_path": key},
                "hs_us_per_iteration": best["hs"]["live"]["median"], "pr_us_per_iteration": best["pr"]["live"]["median"],
                "hidden_fraction": ({"pipe_pr_vs_pr": best["pipe_pr"].get("hidden_vs_pr"), "pipe_pr_vs_hs": best["pipe_pr"].get("hidden_vs_hs"),
                                     "gv_vs_pr": best["gv"].get("hidden_vs_pr")} if world > 1 else None),
                "tail": out}
        emit(line)
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------- banded model problem (SURVEY 8f rank 3)
SP_CSR_WORDS = {"sp_hs": 2, "sp_cg": 3, "sp_gv": 2, "sp_pr": 3, "sp_pipe_r": 4, "sp_pipe_n": 2}    # vector words per row


def run_banded(args, rank, world, local_rank):
    """The PETSc driver's model problem (ex2b.c:86-97; n = 650 000, k = 32, 65 non-zeros per row,
    un-preconditioned, 4000 fixed iterations, strong_scaling_tests.py:49-56,121-126) on the CSR
    kernels: us/iteration per variant, final error ||x - 1||_2 next to the reference's printed value
    (slurm-864568.out), and the roofline of the fused CSR SpMV pass on its algorithmic bytes
    12 nnz + 4 (n+1) + 8 n W.  N > 1: rows are block-partitioned (general-CSR halo lists)."""
    import torch
    from new_cg_variants_b200 import Session
    from new_cg_variants_b200.experiments import BANDED_KAT, banded_model_problem
    torch.cuda.set_device(local_rank)
    if world > 1:
        import torch.distributed as dist
        from new_cg_variants_b200.dist import CsrDistSession
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    A, b, x_true = banded_model_problem(args.banded_n, args.banded_k)
    n, nnz = A.shape[0], A.nnz
    x0 = np.zeros(n)
    its = args.banded_iters
    peak, peak_src = measured_peak()
    sess = CsrDistSession(A, device=local_rank, rank=rank, world=world) if world > 1 else Session(A, device=local_rank)
    n_loc, nnz_loc = (sess.n, sess.nnz) if world > 1 else (n, nnz)
    if world > 1:
        sess.load_problem(b, x0, None)
    else:
        sess.load_problem(b, x0, None)
    rows = {}
    for v in ("hs", "cg", "gv", "pr", "pipe_pr", "pipe_p"):
        best = None
        for _ in range(max(1, args.steps // 3)):
            if world > 1:
                dist.barrier()
            info = sess.run(v, its + 1, histories=(), path="stream")
            t = info["loop_ms"]
            if world > 1:
                tt = torch.tensor([t], dtype=torch.float64, device="cuda")
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                t = tt.item()
            best = t if best is None else min(best, t)
        x = sess.fetch(want_hist=False)[0] if world == 1 else sess.gather_x(sess.fetch_local(want_hist=False)[0])
        err = float(np.linalg.norm(x - x_true))
        sess.set_profile(True)
        sess.run(v, min(its, 300) + 1, histories=(), path="stream")
        prof = sess.get_profile()
        sess.set_profile(False)
        row = {"us_per_iteration": 1e3 * best / its, "iterations_per_s": its / (best / 1e3), "error_2_norm": err,
               "reference_error_2_norm": BANDED_KAT.get(v), "kernels": {}}
        for kname, (ms, cnt) in prof.items():
            us = 1e3 * ms / cnt
            row["kernels"][kname] = {"us": us}
            if kname in SP_CSR_WORDS:
                by = 12.0 * nnz_loc + 4.0 * (n_loc + 1) + 8.0 * n_loc * SP_CSR_WORDS[kname]
                row["kernels"][kname].update(GBps=by / (us * 1e-6) / 1e9, algorithmic_bytes=by, frac=by / (us * 1e-6) / 1e9 / peak)
        rows[v] = row
    if rank == 0:
        v = args.variant if args.variant in rows else "pr"
        spk = max((k for k in rows[v]["kernels"] if k in SP_CSR_WORDS), key=lambda k: rows[v]["kernels"][k]["us"])
        kk = rows[v]["kernels"][spk]
        traffic, traffic_note = read_traffic("csr_" + spk)
        line = {"metric": f"CG iterations/s ({REF_FUN.get(v, v)}, un-preconditioned, banded model problem n={n} k={args.banded_k})",
                "value": rows[v]["iterations_per_s"], "unit": "iterations/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": rows[v]["us_per_iteration"] * its / 1e3, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": f"banded model problem (ex2b.c:86-97) n={n} k={args.banded_k} nnz={nnz}, {its} iterations",
                           "l2": "matrix + vectors = %.2f GB per iteration >> 126 MB L2" % ((12.0 * nnz + 8.0 * n * 12) / 1e9)},
                "roofline": {"bound": "hbm", "kernel": ("csr_stream<%s>" if spk == "sp_pipe_r" else "csr_bulk<%s>") % spk, "achieved": kk["GBps"], "peak": peak, "unit": "GB/s",
                             "frac": kk["frac"], "traffic": traffic if world == 1 else None, "traffic_source": traffic_note,
                             "peak_source": peak_src,
                             "algorithmic_bytes_per_launch": kk["algorithmic_bytes"], "avg_launch_ms": kk["us"] / 1e3},
                "variants": rows}
        emit(line)
    sess.close()
    if world > 1:
        dist.destroy_process_group()


_REAL_STDOUT = None


def emit(line):
    """The ONE JSON line of the contract goes to the real stdout; everything else any library
    prints (e.g. NCCL's version banner) was redirected to stderr in main()."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)                      # fd 1 -> stderr for the duration of the run
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--variant", default="pr", choices=sorted(W_V))
    ap.add_argument("--grid", type=int, default=256)
    ap.add_argument("--dim", type=int, default=3, choices=[2, 3],
                    help="3: BASELINE configs[3] (default, the headline); 2 with --grid 4096: configs[2]")
    ap.add_argument("--iters", type=int, default=200, help="CG iterations per step (our arm)")
    ap.add_argument("--ref-iters", type=int, default=6, help="CG iterations per step (reference arm; BASELINE.md section 2)")
    ap.add_argument("--parity-iters", type=int, default=8, help="history entries compared with the oracle (cpu_baseline leg)")
    ap.add_argument("--cpu-iters", type=int, default=10, help="iterations of the cpu_baseline sample")
    ap.add_argument("--path", default="auto", choices=["auto", "stream", "persistent"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--config", default="headline", choices=["headline", "tail", "banded"],
                    help="headline: configs[3] (default, the driver's contract); tail: configs[4] latency-bound 64^3 "
                         "allreduce-hiding experiment; banded: the PETSc driver's banded model problem as a CSR benchmark")
    ap.add_argument("--banded-n", type=int, default=650000)
    ap.add_argument("--banded-k", type=int, default=32)
    ap.add_argument("--banded-iters", type=int, default=4000)
    ap.add_argument("--tail-grid", type=int, default=64)
    ap.add_argument("--tail-iters", type=int, default=2000)
    ap.add_argument("--tail-reps", type=int, default=5)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps write the solution x of the last one to DIR/x.npy "
                         "(float64; a fixed seeded sample above %d entries)" % DUMP_MAX_ENTRIES)
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.steps < 1 or args.warmup < 0:
        ap.error("steps >= 1, warmup >= 0")
    if args.dump_outputs and (args.impl != "ours" or args.config != "headline"):
        ap.error("--dump-outputs writes the outputs of the headline workload (--impl ours --config headline)")
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        ap.error("--gpus N > 1 must be launched with torchrun (one rank per GPU)")
    if args.config == "tail":
        run_tail(args, rank, world, local_rank)
        return
    if args.config == "banded":
        run_banded(args, rank, world, local_rank)
        return
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
