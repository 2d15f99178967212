"""torchrun worker: one rank per GPU runs partitioned solves with a tolerance (DistSession, CUDA IPC
windows).  Every rank must stop at the same k, and rank 0 compares x and the histories with the
single-GPU emulation of the same partition (GroupSession) with the same tolerance: same bits.  A
tolerance under the NCCL scalar exchange is refused.  Also the mpi4py-shaped solvers with tol=."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(ROOT))
sys.path.insert(0, ROOT)


def main():
    import torch
    import torch.distributed as dist
    import helpers
    from new_cg_variants_b200 import PoissonStencil, _lib, cg_variants_mpi4py as mp
    from new_cg_variants_b200.dist import DistSession, GroupSession

    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dist.init_process_group("gloo")          # plumbing only: window handles and barriers
    hist = _lib.HIST_NAMES
    ok = True

    def stops_agree(stop):
        out = [None] * world
        dist.all_gather_object(out, stop)
        return len(set(out)) == 1 and stop > 0

    S = PoissonStencil(64, 20, 24, dim=3)
    n = S.shape[0]
    xt = np.ones(n) / np.sqrt(n)
    b, x0 = S @ xt, np.zeros(n)
    A = helpers.load_matrix("bcsstk16")
    xtA, bA, x0A = helpers.orc.setup_problem(A)
    cases = (("slabs", S, 1 / S.diagonal(), b, x0, xt, 1e-6, ("stream", "persistent")),
             ("csr", A, 1 / A.diagonal(), bA, x0A, xtA, 1e-5, ("stream",)))
    for label, op, dinv, bb, xx0, xxt, tol, paths in cases:
        sess = DistSession(op, dinv=dinv, device=local)
        res = {}
        for path in paths:
            for tag in ("hs", "cg", "gv", "pr", "m", "pipe_pr", "pipe_p"):
                x_loc, h, info = sess.solve(tag, bb, xx0, 600, x_true=xxt, histories=hist, path=path, tol=tol)
                good = stops_agree(info["stop_iter"])
                if not good:
                    print(f"[{label}/{path}] {tag}: ranks disagree on the stop", flush=True)
                ok = ok and good
                res[(tag, path)] = (sess.gather_x(x_loc), h, info["stop_iter"])
        sess.close()
        if rank == 0:
            grp = GroupSession(op, world, dinv=dinv, devices=[local] * world)
            for (tag, path), (x, h, stop) in res.items():
                xg, hg, ig = grp.solve(tag, bb, xx0, 600, x_true=xxt, path=path, tol=tol)
                same = ig[0]["stop_iter"] == stop and np.array_equal(x, xg) and \
                    all(np.array_equal(h[k], hg[k], equal_nan=True) for k in hg)
                print(f"[{label}/{path}] {tag}: stop {stop} {'match' if same else 'MISMATCH'}", flush=True)
                ok = ok and same
            grp.close()
        dist.barrier()

    # NCCL scalar exchange: refused with a tolerance, before anything is enqueued
    sess = DistSession(S, dinv=1 / S.diagonal(), device=local, mode="nccl")
    try:
        sess.solve("cg", b, x0, 40, tol=1e-6)
        refused = False
    except _lib.CgxError as e:
        refused = e.code == _lib.ERR_UNSUPPORTED
    print(f"[nccl] tolerance {'refused' if refused else 'NOT refused'}", flush=True)
    ok = ok and refused
    sess.close()
    dist.barrier()

    # the mpi4py-shaped solvers: the same stop on every rank, reported on rank 0
    comm = mp.GpuComm()
    r0, r1 = rank * (n // world), (rank + 1) * (n // world)
    for fn in (mp.hs_cg, mp.pr_cg, mp.pipe_pr_cg):
        _, times = fn(comm, S, b[r0:r1], 20)
        good = rank != 0 or "stop_iter" not in times
        _, times = mp.solve_to_tol(fn.__name__, comm, S, b[r0:r1], 2000, 1e-6)
        good = good and (rank != 0 or times["stop_iter"] > 0)
        print(f"[mpi4py-shaped] {fn.__name__}: {'ok' if good else 'MISMATCH'}", flush=True)
        ok = ok and good
    mp.clear_sessions()

    flag = torch.tensor([1 if ok else 0])
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    dist.destroy_process_group()
    if rank == 0 and flag.item():
        print("dist_tol_worker ok", flush=True)
    sys.exit(0 if flag.item() else 1)


if __name__ == "__main__":
    main()
