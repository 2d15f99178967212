"""Row-partitioned multi-GPU runs (SURVEY.md section 8e): z-slabs of the Poisson grid, one
rank per GPU, halo planes by peer-to-peer stores over NVLink, the fused scalars summed in
rank order on every GPU.

Operators: a ``PoissonStencil`` is cut into z-slabs (halo = boundary planes); any scipy sparse or
dense matrix is cut into contiguous row blocks whose ghost entries are gathered through per-neighbour
index lists (the layout of the reference's PETSc driver, ex2b.c:71; the reference's mpi4py column
blocks of a symmetric matrix transpose to exactly these row blocks).

``DistSession``  one rank of a torchrun job (one process per GPU); ``torch.distributed`` is
                 used only to hand the 64-byte window handles (and the NCCL id) around and
                 for barriers -- never on the data path.
``GroupSession`` the same partition driven from one process (all ranks on one GPU sharing a
                 stream, or one context per visible GPU): how the protocol is tested on a
                 single GPU, bit-identical to the multi-process run.

The reference's distributed solvers are ``scaling_experiments_mpi4py/cg_variants/*.py``
(column blocks + an Allreduce of the whole vector, hs_cg.py:49-51); the row/slab layout
follows its PETSc driver (ex2b.c:71).
"""
from __future__ import annotations

import ctypes as C
import os
from pickle import dumps as pickle_dumps, loads as pickle_loads

import numpy as np

from . import _lib
from .operators import PoissonStencil, VariableStencil
from .session import _f64

MODES = {"p2p": 1, "nccl": 2}


# ---------------------------------------------------------------------------------------
# host-side partition logic (pure Python; covered by the CPU tests)
# ---------------------------------------------------------------------------------------
def _refuse_variable_stencil(S, who):
    if isinstance(S, VariableStencil):
        raise NotImplementedError(f"{who}: a VariableStencil runs on one GPU (Session); partitions are not supported")


def slab_grid(S: PoissonStencil):
    """(nx, ny, nz) of the 3-D slab view of a stencil operator: a 2-D nx x ny grid is the
    3-D grid nx x 1 x ny (same canonical term order: y-1, x-1, c, x+1, y+1)."""
    if S.dim == 3:
        return S.nx, S.ny, S.nz
    return S.nx, 1, S.ny


def partition_planes(nz: int, world: int):
    """Contiguous plane ranges [z0, z1) per rank, sizes differing by at most one."""
    if world < 1 or nz < world:
        raise ValueError(f"cannot cut {nz} planes into {world} non-empty slabs")
    base, extra = divmod(nz, world)
    out, z = [], 0
    for r in range(world):
        m = base + (1 if r < extra else 0)
        out.append((z, z + m))
        z += m
    return out


def row_range(S: PoissonStencil, world: int, rank: int):
    nx, ny, nz = slab_grid(S)
    z0, z1 = partition_planes(nz, world)[rank]
    return z0 * nx * ny, z1 * nx * ny


# ---- general CSR row partition (SURVEY.md section 8e "General CSR") ------------------------------
def block_rows(n: int, world: int):
    """Contiguous row ranges [r0, r1) per rank, sizes differing by at most one (the reference's
    mpi4py drivers use n/P rows per rank, scaling_tests.py:44-50; PETSc's default split likewise)."""
    if world < 1 or n < world:
        raise ValueError(f"cannot cut {n} rows into {world} non-empty blocks")
    base, extra = divmod(n, world)
    out, r = [], 0
    for k in range(world):
        m = base + (1 if k < extra else 0)
        out.append((r, r + m))
        r += m
    return out


def csr_local_block(A_rows, row0, row1):
    """Rows [row0, row1) of a global matrix given as a CSR block with GLOBAL column indices
    (shape (row1-row0, n)) -> (local CSR arrays with columns remapped, sorted ghost column list).
    A column owned by this rank becomes its local row number, any other column becomes
    n_local + (its position in the ghost list); the stored order inside a row is untouched."""
    import scipy.sparse as sps
    A_rows = sps.csr_matrix(A_rows)
    A_rows.sort_indices()
    n_loc = row1 - row0
    cols = A_rows.indices.astype(np.int64)
    owned = (cols >= row0) & (cols < row1)
    ghost = np.unique(cols[~owned])
    new = np.where(owned, cols - row0, n_loc + np.searchsorted(ghost, cols))
    return (A_rows.indptr.astype(np.int32), new.astype(np.int32), np.ascontiguousarray(A_rows.data, dtype=np.float64),
            ghost.astype(np.int64))


def csr_exchange_lists(ghosts, ranges, rank):
    """From every rank's sorted ghost list: what `rank` receives and sends.
    -> recv_count[r], send_count[r], send_idx (local rows, concatenated per destination),
       send_off[r] (start of this rank's segment in r's ghost list), nghost_of[r]."""
    world = len(ranges)
    row0, row1 = ranges[rank]
    mine = ghosts[rank]
    recv = [int(np.count_nonzero((mine >= a) & (mine < b))) for a, b in ranges]
    send_count, send_off, send_idx = [], [], []
    for q in range(world):
        g = ghosts[q]
        lo, hi = int(np.searchsorted(g, row0)), int(np.searchsorted(g, row1))
        if q == rank:
            lo = hi = 0
        send_count.append(hi - lo)
        send_off.append(lo)
        send_idx.append((g[lo:hi] - row0).astype(np.int32))
    i32 = lambda v: np.ascontiguousarray(np.asarray(v, dtype=np.int32))          # noqa: E731
    return (i32(recv), i32(send_count), i32(np.concatenate(send_idx) if send_idx else []), i32(send_off),
            i32([len(g) for g in ghosts]))


def nccl_library_path():
    """libnccl.so.2 bundled with torch (the library this process already has loaded)."""
    try:
        import nvidia.nccl
        base = os.path.dirname(nvidia.nccl.__file__) if getattr(nvidia.nccl, "__file__", None) \
            else list(nvidia.nccl.__path__)[0]
        p = os.path.join(base, "lib", "libnccl.so.2")
        if os.path.exists(p):
            return p
    except Exception:
        pass
    return "libnccl.so.2"


def exchange_bytes(payload: bytes, group=None):
    """all-gather one bytes object per rank through torch.distributed (any backend)."""
    import torch.distributed as dist
    world = dist.get_world_size(group)
    out = [None] * world
    dist.all_gather_object(out, payload, group=group)
    return out


def _mask(histories):
    m = 0
    for h in histories:
        m |= _lib.HIST_BITS[h]
    return m


class _RankBase:
    """Shared by DistSession / the members of a GroupSession."""

    def _create(self, S, world, rank, device):
        self._lib = _lib.load()
        self.S, self.world, self.rank, self.device = S, int(world), int(rank), int(device)
        self.n_global = S.shape[0]
        nx, ny, nz = slab_grid(S)
        z0, z1 = partition_planes(nz, self.world)[self.rank]
        self.row0, self.row1 = z0 * nx * ny, z1 * nx * ny
        self.n = self.row1 - self.row0
        self._ctx = C.c_void_p()
        _lib.check(self._lib.cgx_ctx_create(self.device, C.byref(self._ctx)))
        _lib.check(self._lib.cgx_set_stencil_slab(self._ctx, nx, ny, z1 - z0, self.world, self.rank,
                                                  S.diag, S.off))
        self.info = None
        self._max_iter = 0

    def _create_csr(self, blk, ghosts, ranges, world, rank, device, n_global):
        """blk = csr_local_block(...) of this rank; ghosts = every rank's ghost list."""
        self._lib = _lib.load()
        self.S, self.world, self.rank, self.device = None, int(world), int(rank), int(device)
        self.n_global = int(n_global)
        self.row0, self.row1 = ranges[rank]
        self.n = self.row1 - self.row0
        indptr, indices, data, ghost = blk
        self.nnz = int(indptr[-1])
        recv, send_count, send_idx, send_off, nghost_of = csr_exchange_lists(ghosts, ranges, rank)
        self._ctx = C.c_void_p()
        _lib.check(self._lib.cgx_ctx_create(self.device, C.byref(self._ctx)))
        _lib.check(self._lib.cgx_set_csr_part_host(
            self._ctx, self.n, len(ghost), self.nnz, _lib.iptr(indptr), _lib.iptr(indices), _lib.dptr(data),
            self.world, self.rank, _lib.iptr(recv), _lib.iptr(send_count),
            _lib.iptr(send_idx) if len(send_idx) else None, _lib.iptr(send_off), _lib.iptr(nghost_of)))
        self.info = None
        self._max_iter = 0

    def _set_jacobi(self, dinv):
        if dinv is None:
            _lib.check(self._lib.cgx_set_jacobi_host(self._ctx, None, self.n))
        else:
            d = _f64(dinv, self.n_global, "dinv")[self.row0:self.row1].copy()
            _lib.check(self._lib.cgx_set_jacobi_host(self._ctx, _lib.dptr(d), self.n))

    def local(self, v):
        return None if v is None else np.ascontiguousarray(_f64(v, self.n_global)[self.row0:self.row1])

    def close(self):
        if getattr(self, "_ctx", None) is not None and self._ctx:
            self._lib.cgx_ctx_destroy(self._ctx)
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def get_info(self):
        info = _lib.CgxInfo()
        _lib.check(self._lib.cgx_get_info(self._ctx, C.byref(info)))
        self.info = info.as_dict()
        return self.info

    def fetch_local(self, want_x=True, want_hist=True):
        x = np.empty(self.n) if want_x else None
        hist = np.empty((len(_lib.HIST_NAMES), self._max_iter)) if want_hist else None
        _lib.check(self._lib.cgx_fetch_host(self._ctx, _lib.dptr(x), _lib.dptr(hist)))
        return x, hist

    def scalars(self):
        out = np.zeros(9)
        _lib.check(self._lib.cgx_get_scalars(self._ctx, _lib.dptr(out)))
        return dict(zip(("a", "a1", "b", "nu", "nu1", "mu", "eta", "delta", "gamma"), out.tolist()))

    def set_option(self, name, value):
        _lib.check(self._lib.cgx_set_option(self._ctx, name.encode(), int(value)))

    def _set_tol(self, tol):
        """This rank's relative tolerance for the next begin / run (None or 0: off).  Collective in
        effect: every rank of a partition must set the same value (include/cgx.h cgx_set_tolerance)."""
        _lib.check(self._lib.cgx_set_tolerance(self._ctx, 0.0 if tol is None else _lib.check_tol(tol)))

    def set_profile(self, on=True):
        _lib.check(self._lib.cgx_set_profile(self._ctx, 1 if on else 0))

    def get_profile(self):
        out = {}
        for cls in range(self._lib.cgx_profile_class_count()):
            ms, cnt = C.c_double(), C.c_int64()
            _lib.check(self._lib.cgx_get_profile(self._ctx, cls, C.byref(ms), C.byref(cnt)))
            if cnt.value:
                out[self._lib.cgx_profile_class_name(cls).decode()] = (ms.value, cnt.value)
        return out


class DistSession(_RankBase):
    """This process's rank of a partitioned operator (``torch.distributed`` must be
    initialised; any backend).  Every method is collective."""

    def __init__(self, S, dinv=None, device=None, rank=None, world=None, mode="p2p", group=None, row_block=None,
                 n_global=None):
        """S: a PoissonStencil (z-slab partition), or a scipy sparse / dense matrix (general CSR row
        partition: contiguous row blocks, ghost entries gathered through index lists).  A matrix is
        either the GLOBAL one, held by every rank, or -- with ``row_block=(row0, row1)`` and
        ``n_global`` -- only this rank's rows (shape (row1-row0, n_global), global column indices);
        the ghost lists are then exchanged through torch.distributed."""
        _refuse_variable_stencil(S, "DistSession")
        import torch.distributed as dist
        self.group = group
        rank = dist.get_rank(group) if rank is None else rank
        world = dist.get_world_size(group) if world is None else world
        device = int(os.environ.get("LOCAL_RANK", rank)) if device is None else device
        if isinstance(S, PoissonStencil):
            self._create(S, world, rank, device)
        else:
            import scipy.sparse as sps
            if row_block is None:
                A = sps.csr_matrix(S)
                n_global = A.shape[0]
                ranges = block_rows(n_global, world)
                blk = csr_local_block(A[ranges[rank][0]:ranges[rank][1]], *ranges[rank])
            else:
                ranges = [tuple(r) for r in (pickle_loads(x) for x in exchange_bytes(pickle_dumps(tuple(row_block)), group))] \
                    if world > 1 else [tuple(row_block)]
                blk = csr_local_block(S, *ranges[rank])
            ghosts = [np.frombuffer(x, dtype=np.int64) for x in exchange_bytes(blk[3].tobytes(), group)] if world > 1 else [blk[3]]
            self._create_csr(blk, ghosts, ranges, world, rank, device, n_global)
        self.mode = mode
        if self.world > 1:
            handle = (C.c_ubyte * 64)()
            _lib.check(self._lib.cgx_dist_ipc_handle(self._ctx, handle))
            handles = exchange_bytes(bytes(handle), group)
            for r, h in enumerate(handles):
                if r != self.rank:
                    buf = (C.c_ubyte * 64).from_buffer_copy(h)
                    _lib.check(self._lib.cgx_dist_attach_ipc(self._ctx, r, buf))
            nid, libpath = None, None
            if mode == "nccl":
                libpath = nccl_library_path().encode()
                raw = (C.c_ubyte * 128)()
                if self.rank == 0:
                    _lib.check(self._lib.cgx_dist_nccl_unique_id(libpath, raw))
                ids = exchange_bytes(bytes(raw), group)
                nid = (C.c_ubyte * 128).from_buffer_copy(ids[0])
            _lib.check(self._lib.cgx_dist_commit(self._ctx, MODES[mode], libpath, nid))
            dist.barrier(group)       # every window is mapped and zeroed before anyone stores into it
        self._set_jacobi(dinv)

    def barrier(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier(self.group)

    def load_problem(self, b, x0, x_true=None):
        """GLOBAL host vectors; each rank copies its own rows."""
        self.load_problem_local(self.local(b), self.local(x0), self.local(x_true))

    def load_problem_local(self, b, x0, x_true=None):
        _lib.check(self._lib.cgx_load_problem_host(self._ctx, _lib.dptr(b), _lib.dptr(x0),
                                                   _lib.dptr(x_true), self.n))

    def run(self, variant, max_iter, histories=(), path="auto", tol=None):
        """``tol``: stop every rank at the first k >= 1 with nu_k <= tol^2 nu_0 (nu: the all-rank total,
        so every rank stops at the same ``info["stop_iter"]``); every rank must pass the same value."""
        if tol is not None:
            _lib.check_tol(tol)
        self._set_tol(tol)
        info = _lib.CgxInfo()
        p = _lib.PATHS[path]
        rc = self._lib.cgx_run(self._ctx, _lib.VARIANT_IDS[variant], int(max_iter), _mask(histories), p,
                               C.byref(info))
        _lib.check(rc, allow_breakdown=True)
        self.info = info.as_dict()
        self._max_iter = int(max_iter)
        return self.info

    def solve_local(self, variant, b_loc, x0_loc, max_iter, x_true_loc=None, histories=(), return_x=True,
                    path="auto", x_out=None, tol=None):
        """The C-ABI round trip with this rank's HOST slices (cgx_solve_host).  ``tol`` as in ``run``;
        the histories then hold ``info["stop_iter"] + 1`` entries."""
        if tol is not None:
            _lib.check_tol(tol)
        self._set_tol(tol)
        mask = _mask(histories)
        x = x_out if x_out is not None else (np.empty(self.n) if return_x else None)
        hist = np.zeros((len(_lib.HIST_NAMES), int(max_iter))) if mask else None
        info = _lib.CgxInfo()
        rc = self._lib.cgx_solve_host(self._ctx, _lib.VARIANT_IDS[variant], _lib.dptr(b_loc), _lib.dptr(x0_loc),
                                      _lib.dptr(x_true_loc), self.n, int(max_iter), mask, _lib.PATHS[path],
                                      _lib.dptr(x), _lib.dptr(hist), C.byref(info))
        _lib.check(rc, allow_breakdown=True)
        self.info = info.as_dict()
        self._max_iter = int(max_iter)
        stop = self.info["stop_iter"]
        end = stop + 1 if stop >= 0 else None
        out = {}
        for i, name in enumerate(_lib.HIST_NAMES):
            if name in histories and (x_true_loc is not None or "error" not in name):
                out[name] = hist[i][:end].copy()
        return x, out, self.info

    def solve(self, variant, b, x0, max_iter, x_true=None, histories=_lib.HIST_NAMES, return_x=True, path="auto",
              tol=None):
        if tol is not None:
            _lib.check_tol(tol)
        return self.solve_local(variant, self.local(b), self.local(x0), max_iter, self.local(x_true),
                                histories, return_x, path, tol=tol)

    def gather_x(self, x_local):
        """Global x on every rank (host side, through torch.distributed objects)."""
        if self.world == 1:
            return x_local
        parts = exchange_bytes(x_local.tobytes(), self.group)
        return np.concatenate([np.frombuffer(p, dtype=np.float64) for p in parts])

    def e2e_bench(self, variant, b_loc, x0_loc, max_iter, steps, barrier, x_out=None):
        """End-to-end timing through cgx_solve_host with (pinned) host slices: wall clock
        between two barriers, max over ranks taken by the caller's barrier."""
        import time
        for _ in range(2):
            self.solve_local(variant, b_loc, x0_loc, max_iter, return_x=True, x_out=x_out)
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            _, _, info = self.solve_local(variant, b_loc, x0_loc, max_iter, return_x=True, x_out=x_out)
        barrier()
        dt = time.perf_counter() - t0
        return {"value": (max_iter - 1) * steps / dt, "unit": "iterations/s",
                "h2d_bytes_per_step": info["h2d_bytes"] * self.world,
                "d2h_bytes_per_step": info["d2h_bytes"] * self.world, "ms_per_step": 1e3 * dt / steps,
                "api": "cgx_solve_host on every rank: pinned host slices of b,x0 in, slice of x out"}


class GroupSession:
    """All ranks of a partition inside this process.  ``devices``: one device index per rank
    (default: every rank on device 0 -- the single-GPU emulation of the protocol)."""

    class _Member(_RankBase):
        pass

    def __init__(self, S, world, dinv=None, devices=None, mode="p2p"):
        _refuse_variable_stencil(S, "GroupSession")
        if mode != "p2p":
            raise NotImplementedError("GroupSession drives the peer-to-peer scalar exchange only")
        self._lib = _lib.load()
        self.S, self.world = S, int(world)
        self.n = S.shape[0]
        devices = [0] * self.world if devices is None else list(devices)
        self.members = []
        if not isinstance(S, PoissonStencil):          # general CSR row partition
            import scipy.sparse as sps
            A = sps.csr_matrix(S)
            ranges = block_rows(self.n, self.world)
            blks = [csr_local_block(A[a:b], a, b) for a, b in ranges]
            ghosts = [blk[3] for blk in blks]
        for r in range(self.world):
            m = GroupSession._Member()
            if isinstance(S, PoissonStencil):
                m._create(S, self.world, r, devices[r])
            else:
                m._create_csr(blks[r], ghosts, ranges, self.world, r, devices[r], self.n)
            self.members.append(m)
        if self.world > 1:
            for a in self.members:
                for b in self.members:
                    if a is not b:
                        _lib.check(self._lib.cgx_dist_attach_ctx(a._ctx, b.rank, b._ctx))
            for m in self.members:
                _lib.check(self._lib.cgx_dist_commit(m._ctx, 1, None, None))
        for m in self.members:
            m._set_jacobi(dinv)
        self._arr = (C.c_void_p * self.world)(*[m._ctx for m in self.members])
        self._max_iter = 0

    def close(self):
        for m in self.members:
            m.close()

    def load_problem(self, b, x0, x_true=None):
        b, x0 = _f64(b, self.n, "b"), _f64(x0, self.n, "x0")
        xt = None if x_true is None else _f64(x_true, self.n, "x_true")
        if self.world == 1:
            m = self.members[0]
            _lib.check(self._lib.cgx_load_problem_host(m._ctx, _lib.dptr(b), _lib.dptr(x0), _lib.dptr(xt), self.n))
        else:
            _lib.check(self._lib.cgx_group_load_problem_host(self._arr, self.world, _lib.dptr(b), _lib.dptr(x0),
                                                             _lib.dptr(xt), self.n))

    def begin(self, variant, max_iter, histories=(), path="stream", tol=None):
        """``tol``: stop all ranks at the first k >= 1 with nu_k <= tol^2 nu_0 (nu: the all-rank total);
        ``advance`` after the stop does nothing.  None: no tolerance."""
        if tol is not None:
            _lib.check_tol(tol)
        for m in self.members:
            m._set_tol(tol)
        if self.world == 1:
            _lib.check(self._lib.cgx_begin(self.members[0]._ctx, _lib.VARIANT_IDS[variant], int(max_iter),
                                           _mask(histories), _lib.PATHS[path]))
        else:
            _lib.check(self._lib.cgx_group_begin(self._arr, self.world, _lib.VARIANT_IDS[variant], int(max_iter),
                                                 _mask(histories), _lib.PATHS[path]))
        self._max_iter = int(max_iter)
        for m in self.members:
            m._max_iter = int(max_iter)

    def advance(self, niter):
        if self.world == 1:
            _lib.check(self._lib.cgx_advance(self.members[0]._ctx, int(niter)))
        else:
            _lib.check(self._lib.cgx_group_advance(self._arr, self.world, int(niter)))

    def solve(self, variant, b, x0, max_iter, x_true=None, histories=_lib.HIST_NAMES, path="stream", tol=None):
        """-> (global x, {history: array}, [per-rank info]).  ``tol`` as in ``begin``: the histories then
        hold ``info["stop_iter"] + 1`` entries."""
        if tol is not None:
            _lib.check_tol(tol)
        self.load_problem(b, x0, x_true)
        self.begin(variant, max_iter, histories, path, tol=tol)
        self.advance(max_iter - 1)
        xs, hists = [], []
        for m in self.members:
            x, h = m.fetch_local()
            xs.append(x)
            hists.append(h)
        for h in hists[1:]:          # every rank holds the same global histories, bit for bit
            if not np.array_equal(h, hists[0]):
                raise AssertionError("ranks disagree on the histories")
        infos = [m.get_info() for m in self.members]
        stop = infos[0]["stop_iter"]
        end = stop + 1 if stop >= 0 else None
        out = {}
        for i, name in enumerate(_lib.HIST_NAMES):
            if name in histories and (x_true is not None or "error" not in name):
                out[name] = hists[0][i][:end].copy()
        return np.concatenate(xs), out, infos


CsrDistSession = DistSession      # (a DistSession given a matrix instead of a PoissonStencil)
