"""Host-side driver: a ``Session`` owns one GPU context of libcgx_b200 with an operator
(and optional Jacobi vector) resident in HBM, and runs the CG variants on it.

Everything numerical happens in the CUDA library; this module only marshals arguments.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import scipy.sparse as sps

from . import _lib
from .operators import PoissonStencil, canonical_csr


def _f64(a, n=None, name="array"):
    a = np.ascontiguousarray(np.asarray(a, dtype=np.float64)).reshape(-1)
    if n is not None and a.shape[0] != n:
        raise ValueError(f"{name} has length {a.shape[0]}, expected {n}")
    return a


class Session:
    """One operator on one GPU.

    >>> s = Session(A, dinv=1/A.diagonal())
    >>> out = s.solve("pr", b, x0, max_iter, x_true=x_true)
    """

    def __init__(self, A, dinv=None, device=0):
        self._lib = _lib.load()
        self._ctx = C.c_void_p()
        _lib.check(self._lib.cgx_ctx_create(int(device), C.byref(self._ctx)))
        self.device = int(device)
        self.info = None
        self._tol = 0.0
        if isinstance(A, PoissonStencil):
            self.kind = "stencil"
            self.n = A.shape[0]
            self.nnz = A.nnz
            _lib.check(self._lib.cgx_set_stencil(self._ctx, A.dim, A.nx, A.ny, A.nz, A.diag, A.off))
        else:
            A = canonical_csr(A)
            self.kind = "csr"
            self.n = A.shape[0]
            self.nnz = A.nnz
            _lib.check(self._lib.cgx_set_csr_host(self._ctx, self.n, A.nnz, _lib.iptr(A.indptr),
                                                  _lib.iptr(A.indices), _lib.dptr(A.data)))
        self.set_jacobi(dinv)

    # -- lifecycle -------------------------------------------------------------------
    def close(self):
        if getattr(self, "_ctx", None) is not None and self._ctx:
            self._lib.cgx_ctx_destroy(self._ctx)
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # -- configuration ---------------------------------------------------------------
    def set_jacobi(self, dinv):
        """dinv = None -> identity preconditioner; else z = dinv * v."""
        if dinv is None:
            _lib.check(self._lib.cgx_set_jacobi_host(self._ctx, None, self.n))
            self.prec = False
        else:
            d = _f64(dinv, self.n, "dinv")
            _lib.check(self._lib.cgx_set_jacobi_host(self._ctx, _lib.dptr(d), self.n))
            self.prec = True

    def set_tolerance(self, tol):
        """Stop every later run once nu_k <= tol^2 nu_0 (nu_k = r~_k . r_k); 0 switches it off.
        Takes effect at the next begin / run / solve (include/cgx.h cgx_set_tolerance)."""
        t = _lib.check_tol(tol)
        _lib.check(self._lib.cgx_set_tolerance(self._ctx, t))
        self._tol = t

    def _with_tol(self, tol, call):
        """Run `call()` with tolerance `tol` (None: the session's own), then restore the session's."""
        if tol is None:
            return call()
        prev = self._tol
        self.set_tolerance(tol)
        try:
            return call()
        finally:
            self.set_tolerance(prev)

    def _stop(self):
        """stop_iter of the last run (-1: it ran to max_iter)."""
        return self.get_info()["stop_iter"]

    def load_problem(self, b, x0, x_true=None):
        b = _f64(b, self.n, "b")
        x0 = _f64(x0, self.n, "x0")
        xt = None if x_true is None else _f64(x_true, self.n, "x_true")
        _lib.check(self._lib.cgx_load_problem_host(self._ctx, _lib.dptr(b), _lib.dptr(x0),
                                                   _lib.dptr(xt), self.n))

    def load_problem_device(self, b_ptr, x0_ptr, x_true_ptr=None):
        """Device pointers (e.g. ``tensor.data_ptr()``) on this session's GPU."""
        _lib.check(self._lib.cgx_load_problem_dev(self._ctx, b_ptr, x0_ptr, x_true_ptr, self.n))

    # -- running ---------------------------------------------------------------------
    def run(self, variant, max_iter, histories=(), path="auto", tol=None):
        """Iterate on the loaded problem; returns the info dict (device timings etc.).
        ``tol``: relative tolerance for this run (see ``set_tolerance``); ``info["stop_iter"]``
        is the iteration it stopped at, or -1."""
        if tol is not None:
            _lib.check_tol(tol)
        mask = 0
        for h in histories:
            mask |= _lib.HIST_BITS[h]
        info = _lib.CgxInfo()
        rc = self._with_tol(tol, lambda: self._lib.cgx_run(self._ctx, _lib.VARIANT_IDS[variant], int(max_iter), mask,
                                                           _lib.PATHS[path], C.byref(info)))
        _lib.check(rc, allow_breakdown=True)
        self.info = info.as_dict()
        self._max_iter = int(max_iter)
        return self.info

    def begin(self, variant, max_iter, histories=(), path="auto", tol=None):
        """Initialise a stepwise solve (``advance``); ``tol`` as in ``run``.  ``advance`` after the
        tolerance stop does nothing."""
        if tol is not None:
            _lib.check_tol(tol)
        mask = 0
        for h in histories:
            mask |= _lib.HIST_BITS[h]
        _lib.check(self._with_tol(tol, lambda: self._lib.cgx_begin(self._ctx, _lib.VARIANT_IDS[variant], int(max_iter),
                                                                   mask, _lib.PATHS[path])))
        self._max_iter = int(max_iter)

    def advance(self, niter=1):
        _lib.check(self._lib.cgx_advance(self._ctx, int(niter)))

    def get_info(self):
        info = _lib.CgxInfo()
        _lib.check(self._lib.cgx_get_info(self._ctx, C.byref(info)))
        self.info = info.as_dict()
        return self.info

    def set_option(self, name, value):
        """Library switches, e.g. ("tma", 0) forces the generic stencil kernel."""
        _lib.check(self._lib.cgx_set_option(self._ctx, name.encode(), int(value)))

    def set_profile(self, on=True):
        """Per-kernel-class device timing of the iteration loop (event pair per launch)."""
        _lib.check(self._lib.cgx_set_profile(self._ctx, 1 if on else 0))

    def get_profile(self):
        """{class name: (total ms, launches)} accumulated since set_profile(True)."""
        out = {}
        for cls in range(self._lib.cgx_profile_class_count()):
            ms, cnt = C.c_double(), C.c_int64()
            _lib.check(self._lib.cgx_get_profile(self._ctx, cls, C.byref(ms), C.byref(cnt)))
            if cnt.value:
                out[self._lib.cgx_profile_class_name(cls).decode()] = (ms.value, cnt.value)
        return out

    # -- on-device support for save_x / save_r / lanczos_recurrence / GV w_replace ----------
    def set_capture(self, x=False, r=False, scalars=False):
        """Record x_k / r_k / (a, b) after every iteration in device memory (next begin/run)."""
        _lib.check(self._lib.cgx_set_capture(self._ctx, (1 if x else 0) | (2 if r else 0) | (4 if scalars else 0)))

    def fetch_capture(self, which):
        """which: "x" | "r" -> (max_iter, n) array; "scalars" -> (2, max_iter): rows a, b.
        After a tolerance stop at k: stop + 1 rows / columns."""
        sel = {"x": 0, "r": 1, "scalars": 2}[which]
        out = np.empty((2, self._max_iter)) if sel == 2 else np.empty((self._max_iter, self.n))
        _lib.check(self._lib.cgx_fetch_capture_host(self._ctx, sel, _lib.dptr(out)))
        stop = self._stop()
        if stop >= 0:
            out = (out[:, :stop + 1] if sel == 2 else out[:stop + 1]).copy()
        return out

    def set_gv_replace(self, flags=None):
        """GV-CG residual replacement schedule (gv_cg.py:156-158): flags[k] truthy -> w_k = A r_k."""
        if flags is None:
            _lib.check(self._lib.cgx_set_gv_replace(self._ctx, None, 0))
        else:
            f = np.ascontiguousarray(np.asarray(flags, dtype=np.uint8))
            _lib.check(self._lib.cgx_set_gv_replace(self._ctx, f.ctypes.data_as(C.POINTER(C.c_uint8)), int(f.shape[0])))

    def advance_stages(self, nstages=1):
        _lib.check(self._lib.cgx_advance_stages(self._ctx, int(nstages)))

    def gv_replace_now(self):
        _lib.check(self._lib.cgx_gv_replace_now(self._ctx))

    def scalars(self):
        out = np.zeros(9)
        _lib.check(self._lib.cgx_get_scalars(self._ctx, _lib.dptr(out)))
        return dict(zip(("a", "a1", "b", "nu", "nu1", "mu", "eta", "delta", "gamma"), out.tolist()))

    def fetch(self, want_x=True, want_hist=True):
        """x and the (4, max_iter) history rows; (4, stop + 1) after a tolerance stop."""
        x = np.empty(self.n) if want_x else None
        hist = np.empty((len(_lib.HIST_NAMES), self._max_iter)) if want_hist else None
        _lib.check(self._lib.cgx_fetch_host(self._ctx, _lib.dptr(x), _lib.dptr(hist)))
        if hist is not None:
            stop = self._stop()
            if stop >= 0:
                hist = hist[:, :stop + 1].copy()
        return x, hist

    def vector(self, name):
        out = np.empty(self.n)
        _lib.check(self._lib.cgx_fetch_vector_host(self._ctx, name.encode(), _lib.dptr(out)))
        return out

    def solve(self, variant, b, x0, max_iter, x_true=None, histories=_lib.HIST_NAMES, path="auto",
              return_x=True, x_out=None, tol=None):
        """The reference call in one C-ABI round trip (host buffers in, host buffers out).

        ``x_out``: optional caller-owned (e.g. pinned) float64 array that receives x.
        ``tol``: stop once nu_k <= tol^2 nu_0 (``set_tolerance``; None: the session's own); the
        histories then hold ``info["stop_iter"] + 1`` entries.
        Returns (x, {history name: (max_iter,) array}, info)."""
        if tol is not None:
            _lib.check_tol(tol)
        b = _f64(b, self.n, "b")
        x0 = _f64(x0, self.n, "x0")
        xt = None if x_true is None else _f64(x_true, self.n, "x_true")
        mask = 0
        for h in histories:
            mask |= _lib.HIST_BITS[h]
        if x_out is not None:
            assert x_out.dtype == np.float64 and x_out.flags.c_contiguous and x_out.shape == (self.n,)
            x = x_out
        else:
            x = np.empty(self.n) if return_x else None
        hist = np.zeros((len(_lib.HIST_NAMES), int(max_iter))) if mask else None
        info = _lib.CgxInfo()
        rc = self._with_tol(tol, lambda: self._lib.cgx_solve_host(
            self._ctx, _lib.VARIANT_IDS[variant], _lib.dptr(b), _lib.dptr(x0), _lib.dptr(xt), self.n, int(max_iter),
            mask, _lib.PATHS[path], _lib.dptr(x), _lib.dptr(hist), C.byref(info)))
        _lib.check(rc, allow_breakdown=True)
        self.info = info.as_dict()
        self._max_iter = int(max_iter)
        return x, _hist_dict(hist, histories, xt is not None, self.info["stop_iter"]), self.info

    # -- primitives (unit tests) -------------------------------------------------------
    def spmv(self, v):
        v = _f64(v, self.n, "v")
        y = np.empty(self.n)
        _lib.check(self._lib.cgx_spmv_host(self._ctx, _lib.dptr(v), _lib.dptr(y), self.n))
        return y

    def dot(self, u, v):
        u = _f64(u)
        v = _f64(v, u.shape[0], "v")
        out = C.c_double()
        _lib.check(self._lib.cgx_dot_host(self._ctx, _lib.dptr(u), _lib.dptr(v), u.shape[0], C.byref(out)))
        return out.value


def _hist_dict(hist, histories, has_xt, stop):
    """{name: row} of the selected histories, cut to stop + 1 entries after a tolerance stop."""
    out = {}
    end = stop + 1 if stop >= 0 else None
    for i, name in enumerate(_lib.HIST_NAMES):
        if name in histories and (has_xt or "error" not in name):
            out[name] = hist[i][:end].copy()
    return out


def solve_batch(items, histories=_lib.HIST_NAMES, return_x=True, tol=None):
    """Independent solves side by side on one GPU, in ONE cooperative launch (cgx_batch_run).

    ``items``: sequence of ``(session, variant, b, x0, max_iter[, x_true])``, one distinct Session
    per entry (same device, same operator kind, same preconditioner mode).  Each entry gets a
    1/len(items) share of the SMs; its results are bitwise those of ``session.solve(...,
    path="persistent")`` with the same CTA shape (options ``pers_threads`` / ``pers_ctas``), and
    ``info["loop_ms"]`` is the duration of the shared launch.
    ``tol``: one relative tolerance for every entry (None: each session's own); entries stop
    independently, and each entry's histories are cut at its own ``info["stop_iter"]``.
    Returns ``[(x, {history name: (max_iter,) array}, info), ...]`` as ``Session.solve``."""
    if tol is not None:
        _lib.check_tol(tol)
    items = [tuple(it) for it in items]
    if not items:
        raise ValueError("solve_batch: no items")
    sessions, xts = [], []
    for it in items:
        if len(it) not in (5, 6):
            raise ValueError("solve_batch: items are (session, variant, b, x0, max_iter[, x_true])")
        sess, variant, b, x0, max_iter = it[:5]
        xt = it[5] if len(it) == 6 else None
        if variant not in _lib.VARIANT_IDS:
            raise ValueError(f"solve_batch: unknown variant {variant!r}")
        sess.load_problem(b, x0, xt)
        sessions.append(sess)
        xts.append(xt)
    mask = 0
    for h in histories:
        mask |= _lib.HIST_BITS[h]
    lib = sessions[0]._lib
    count = len(items)
    ctxs = (C.c_void_p * count)(*[s._ctx for s in sessions])
    variants = np.array([_lib.VARIANT_IDS[it[1]] for it in items], dtype=np.int32)
    iters = np.array([int(it[4]) for it in items], dtype=np.int32)
    infos = (_lib.CgxInfo * count)()
    prev = [s._tol for s in sessions]
    try:
        if tol is not None:
            for s in sessions:
                s.set_tolerance(tol)
        rc = lib.cgx_batch_run(ctxs, count, _lib.iptr(variants), _lib.iptr(iters), mask, infos)
    finally:
        if tol is not None:
            for s, t in zip(sessions, prev):
                s.set_tolerance(t)
    _lib.check(rc, allow_breakdown=True)
    results = []
    for sess, it, xt, info in zip(sessions, items, xts, infos):
        sess.info = info.as_dict()
        sess._max_iter = int(it[4])
        x, hist = sess.fetch(want_x=return_x, want_hist=bool(mask))
        results.append((x, _hist_dict(hist, histories, xt is not None, -1) if mask else {}, sess.info))
    return results


def diagonal_of(A):
    if isinstance(A, PoissonStencil) or sps.issparse(A):
        return np.asarray(A.diagonal(), dtype=np.float64)
    return np.asarray(np.diag(A), dtype=np.float64)
