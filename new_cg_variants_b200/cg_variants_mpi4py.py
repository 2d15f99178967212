"""The reference's distributed solver signature (scaling_experiments_mpi4py/cg_variants/*.py):

    x_local, times = f(comm, A, b, max_iter)        f in {hs_cg, cg_cg, gv_cg, pr_cg, pipe_pr_cg}

un-preconditioned, x0 = 0, exactly `max_iter` loop trips (`for k in range(max_iter)`,
hs_cg.py:36, pr_cg.py:49), no convergence test, no history; `times` is a dict with the wall
time under 'tot' on rank 0 and None elsewhere (hs_cg.py:13-16,66).

An extension: `solve_to_tol("pr_cg", comm, A, b, max_iter, tol)` (any of the five names) stops every
rank at the first k >= 1 with nu_k <= tol^2 nu_0 (nu_k = ||r_k||^2 here, the all-rank total;
include/cgx.h cgx_set_tolerance), and rank 0's `times` then also holds 'stop_iter' (-1 when `max_iter`
trips ran first).  Every rank must pass the same `tol`.  The five solvers keep the reference's signature
and outputs.

Here `comm` is a `GpuComm` (one rank per GPU; `Get_size/Get_rank/Barrier` as mpi4py's) -- or
anything with those three methods, e.g. a real `MPI.COMM_WORLD` -- and the rows are
partitioned in contiguous blocks as in the reference (rank r owns rows r*m .. (r+1)*m-1).

`A` may be
  * the reference's own operand: a dense `(n, n/P)` ndarray, this rank's COLUMN block of a symmetric
    matrix (scaling_tests.py:44-50) -- its transpose is this rank's row block, which is what is
    uploaded (general CSR row partition, ghost entries gathered through index lists);
  * a square scipy sparse / dense matrix: the global operator, held by every rank (row blocks are cut
    here; e.g. `model_problem(n)` or `experiments.banded_model_problem`);
  * a `PoissonStencil` (the global operator; partitioned into z-slabs over the ranks).
`b` is this rank's slice `(n/P,)`.  The reference's solvers count `max_iter` updates of x; the
numerical-experiment functions count `max_iter - 1`, hence the `+ 1` below.
"""
from __future__ import annotations

import time

import numpy as np
import scipy.sparse as sps

from . import _lib
from .operators import PoissonStencil, VariableStencil
from .session import Session


class GpuComm:
    """mpi4py-shaped communicator over torch.distributed (or a single process)."""

    def __init__(self, group=None):
        try:
            import torch.distributed as dist
            self._dist = dist if dist.is_available() and dist.is_initialized() else None
        except Exception:
            self._dist = None
        self.group = group

    def Get_size(self):
        return self._dist.get_world_size(self.group) if self._dist else 1

    def Get_rank(self):
        return self._dist.get_rank(self.group) if self._dist else 0

    def Barrier(self):
        if self._dist:
            self._dist.barrier(self.group)

    # the two collectives scaling_tests.py uses around the solvers (numpy buffers, mpi4py semantics)
    def Scatter(self, sendbuf, recvbuf, root=0):
        if not self._dist:
            recvbuf[...] = np.asarray(sendbuf).reshape(recvbuf.shape)
            return
        size, rank = self.Get_size(), self.Get_rank()
        parts = [np.ascontiguousarray(p) for p in np.asarray(sendbuf).reshape(size, -1)] if rank == root else None
        out = [None]
        self._dist.scatter_object_list(out, parts, src=root, group=self.group)
        recvbuf[...] = out[0].reshape(recvbuf.shape)

    def Gather(self, sendbuf, recvbuf, root=0):
        if not self._dist:
            recvbuf[...] = np.asarray(sendbuf).reshape(recvbuf.shape)
            return
        size, rank = self.Get_size(), self.Get_rank()
        parts = [None] * size if rank == root else None
        self._dist.gather_object(np.ascontiguousarray(sendbuf), parts, dst=root, group=self.group)
        if rank == root:
            recvbuf[...] = np.stack(parts).reshape(recvbuf.shape)


_SESSIONS = {}          # (id(A), size, rank) -> (A, session); holding A keeps its id from being reused
_MAX_SESSIONS = 4


def _operator_session(comm, A, m):
    """One resident operator per (operator, partition) -- the reference builds A once and runs
    five variants on it (scaling_tests.py:60-66).  The cache entry keeps a strong reference to A
    (so `id(A)` cannot be recycled by another matrix while the entry lives) and is bounded."""
    size, rank = comm.Get_size(), comm.Get_rank()
    key = (id(A), size, rank)
    if key in _SESSIONS and _SESSIONS[key][0] is A:
        return _SESSIONS[key][1]
    while len(_SESSIONS) >= _MAX_SESSIONS:
        _SESSIONS.pop(next(iter(_SESSIONS)))[1].close()
    shape = getattr(A, "shape", None)
    column_block = (not isinstance(A, PoissonStencil)) and shape is not None and len(shape) == 2 and shape[0] != shape[1]
    if column_block:                                   # (n, n/P): the reference's operand (scaling_tests.py:44-50)
        n = shape[0]
        if shape[1] != m or n != m * size:
            raise ValueError(f"column block of shape {shape} does not match b of length {m} on {size} ranks")
        rows = sps.csr_matrix(np.ascontiguousarray(np.asarray(A).T) if not sps.issparse(A) else A.T)
        if size == 1:
            sess = Session(rows)
        else:
            from .dist import DistSession
            sess = DistSession(rows, dinv=None, rank=rank, world=size, group=getattr(comm, "group", None),
                               row_block=(rank * m, (rank + 1) * m), n_global=n)
    elif size == 1:
        sess = Session(A)
    else:
        from .dist import DistSession
        sess = DistSession(A, dinv=None, rank=rank, world=size, group=getattr(comm, "group", None))
        if sess.n != m:
            raise ValueError(f"b has {m} entries on rank {rank}, the row block of A has {sess.n}")
    _SESSIONS[key] = (A, sess)
    return sess


def _run(tag, comm, A, b, max_iter, tol=None):
    if isinstance(A, VariableStencil):
        raise NotImplementedError("cg_variants_mpi4py: a VariableStencil runs on one GPU (Session, cg_variants)")
    size, rank = comm.Get_size(), comm.Get_rank()
    if tol is not None:
        _lib.check_tol(tol)
    b = np.ascontiguousarray(np.asarray(b, dtype=np.float64))
    m = len(b)
    times = {'tot': 0., 'c_ip': 0., 'c_mv': 0., 'w_mv': 0., 'w_ip': 0., 'w_vec': 0.} if rank == 0 else None
    sess = _operator_session(comm, A, m)
    x0 = np.zeros(m)
    if size == 1:
        sess.load_problem(b, x0, None)
    else:
        sess.load_problem_local(b, x0, None)
    comm.Barrier()                                     # hs_cg.py:30-33: timing starts after a barrier
    t0 = time.perf_counter()
    info = sess.run(tag, int(max_iter) + 1, histories=(), tol=tol)
    comm.Barrier()
    if rank == 0:
        times['tot'] += time.perf_counter() - t0
        if tol is not None:
            times['stop_iter'] = int(info["stop_iter"])
    x = sess.fetch(want_hist=False)[0] if size == 1 else sess.fetch_local(want_hist=False)[0]
    return x, times


def hs_cg(comm, A, b, max_iter):
    return _run("hs", comm, A, b, max_iter)


def cg_cg(comm, A, b, max_iter):
    return _run("cg", comm, A, b, max_iter)


def gv_cg(comm, A, b, max_iter):
    return _run("gv", comm, A, b, max_iter)


def pr_cg(comm, A, b, max_iter):
    return _run("pr", comm, A, b, max_iter)


def pipe_pr_cg(comm, A, b, max_iter):
    return _run("pipe_pr", comm, A, b, max_iter)


SOLVERS = {"hs_cg": "hs", "cg_cg": "cg", "gv_cg": "gv", "pr_cg": "pr", "pipe_pr_cg": "pipe_pr"}


def solve_to_tol(name, comm, A, b, max_iter, tol):
    """`name(comm, A, b, max_iter)` (a key of SOLVERS) that stops every rank at the first k >= 1 with
    nu_k <= tol^2 nu_0; rank 0's `times` also holds 'stop_iter'.  The five solvers keep the reference's
    exact signature."""
    if name not in SOLVERS:
        raise ValueError(f"unknown solver {name!r}; one of {sorted(SOLVERS)}")
    if tol is None:
        raise ValueError("tol is required (the solvers themselves run max_iter trips)")
    return _run(SOLVERS[name], comm, A, b, max_iter, tol)


def model_problem(n, kappa=1e6, rho=0.9):
    """scaling_tests.py:31-36,53: diagonal matrix of the model spectrum and b with x* = ones/sqrt(n)."""
    lam = 1 / kappa + (1 - 1 / kappa) * np.arange(n) / (n - 1) * rho ** np.arange(n - 1, -1, -1, dtype='float')
    return sps.diags(lam).tocsr(), lam / np.sqrt(n)


def clear_sessions():
    for _, s in _SESSIONS.values():
        s.close()
    _SESSIONS.clear()
