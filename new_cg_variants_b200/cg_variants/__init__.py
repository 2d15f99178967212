"""Drop-in solver functions with the reference's names and signatures
(numerical_experiments/cg_variants/__init__.py:19-44,64-74):

    f(A, b, x0, max_iter, preconditioner=lambda x: x, callbacks=[], **kwargs) -> output dict

for ``hs_pcg, cg_pcg, gv_pcg, pr_pcg, m_pcg, pipe_pr_pcg, pipe_p_pcg, pipe_pr_m_pcg,
pipe_p_m_pcg`` and the un-preconditioned twins ``*_cg`` (no ``preconditioner`` argument).
``gv_*`` also accept ``w_replace`` (gv_cg.py:89,156-158): a predicate that depends only on ``k``
becomes a replacement schedule executed on the GPU; one that reads vectors is evaluated on the
host every iteration against the device state (the replacement ``w = A r`` itself always runs on
the GPU).

Every iteration runs in libcgx_b200 on the GPU (there is no CPU solve path).  ``A`` may be
a scipy sparse matrix, a dense ndarray, or a ``PoissonStencil``.  ``preconditioner`` stays an
opaque callable as in the reference; it is probed once and must act as a fixed diagonal
scaling (identity or Jacobi, figure_gen.py:40-44), otherwise ``NotImplementedError``.

Extra keyword arguments understood here (all optional, ignored by the reference):
``device=0``, ``path="auto"|"stream"|"persistent"``, ``session=Session`` (reuse an operator
already resident on the GPU), ``return_info=True`` (adds ``output['_info']``), ``tol=`` (stop on the
GPU at the first k with nu_k <= tol^2 nu_0, nu_k = r~_k . r_k; the histories then have
``output['stop_iter'] + 1`` entries, and ``output['stop_iter']`` is None when the run went to
``max_iter``).

``solve_concurrently(methods, A, b, x0, max_iter, ...)`` runs several of these solvers on the same
problem in one cooperative launch (figure_gen.py:50-60 runs the nine variants one after another).
"""
from __future__ import annotations

import weakref

import numpy as np
import scipy.sparse as sps

from .. import _lib
from .. import callbacks as _cbk
from ..callbacks import CAPTURE_CALLBACKS, DEVICE_HISTORIES
from ..operators import PoissonStencil, canonical_csr
from ..session import Session

_OWN_KEYS = ("device", "path", "session", "return_info", "w_replace", "tol")

# ---------------------------------------------------------------------------------------
# preconditioner probe (SURVEY.md section 8b)
# ---------------------------------------------------------------------------------------
def probe_preconditioner(preconditioner, n):
    """Return None if ``preconditioner`` is the identity, the vector ``d`` if it is the
    diagonal scaling ``v -> d*v`` (bit for bit on a random probe); raise otherwise."""
    if preconditioner is None:
        return None
    ones = np.ones(n)
    d = np.asarray(preconditioner(ones), dtype=np.float64)
    if d.shape != (n,):
        raise NotImplementedError("preconditioner must map (n,) -> (n,)")
    v = np.random.default_rng(0).standard_normal(n)
    pv = np.asarray(preconditioner(v), dtype=np.float64)
    if not np.array_equal(pv, d * v):
        raise NotImplementedError(
            "only diagonal (identity / Jacobi) preconditioners run on the GPU path; "
            "preconditioner(v) != preconditioner(ones) * v and there is no CPU fallback")
    if np.array_equal(d, ones):
        return None
    return d


# ---------------------------------------------------------------------------------------
# operator cache: keep the last few matrices resident in HBM between calls, as a
# figure_gen-style driver runs nine variants on the same A (figure_gen.py:50-60)
# ---------------------------------------------------------------------------------------
_CACHE: list = []          # entries: [weakref(A) | None, fingerprint, device, Session, dinv]
_CACHE_SIZE = 2


def _fingerprint(A):
    if isinstance(A, PoissonStencil):
        return ("stencil", A.dim, A.nx, A.ny, A.nz, A.diag, A.off)
    if sps.issparse(A):
        if A.format not in ("csr", "csc", "coo", "bsr", "dia"):
            A = A.tocsr()                      # e.g. LIL keeps object-dtype rows
        d = A.data
        step = max(1, d.shape[0] // 4096)
        return ("sparse", A.shape, A.nnz, A.format, float(d.sum()), float(d[::step].sum()))
    a = np.asarray(A)
    return ("dense", a.shape, float(a.sum()), float(a.reshape(-1)[:: max(1, a.size // 4096)].sum()))


def _session_for(A, dinv, device):
    fp = _fingerprint(A)
    for ent in _CACHE:
        ref, efp, edev, sess, edinv = ent
        same = ref is not None and ref() is A
        if isinstance(A, PoissonStencil):
            same = efp == fp
        if same and efp == fp and edev == device and sess._ctx:
            if (dinv is None) != (edinv is None) or (dinv is not None and not np.array_equal(dinv, edinv)):
                sess.set_jacobi(dinv)
                ent[4] = None if dinv is None else dinv.copy()
            _CACHE.remove(ent)
            _CACHE.insert(0, ent)
            return sess
    sess = Session(A, dinv=dinv, device=device)
    try:
        ref = weakref.ref(A)
    except TypeError:
        ref = None
    _CACHE.insert(0, [ref, fp, device, sess, None if dinv is None else dinv.copy()])
    while len(_CACHE) > _CACHE_SIZE:
        _CACHE.pop().__getitem__(3).close()
    return sess


def clear_cache():
    while _CACHE:
        _CACHE.pop()[3].close()


# ---------------------------------------------------------------------------------------
# the driver behind every exported function
# ---------------------------------------------------------------------------------------
def _is_package_callback(cb, name):
    mod = getattr(cb, "__module__", "") or ""
    return cb is getattr(_cbk, name, None) or mod.split(".")[0] == "callbacks" or mod.endswith("callbacks." + name)


def _split_capture(generic):
    """(callbacks served from the device capture buffers, the rest)."""
    cap = [cb for cb in generic if getattr(cb, "__name__", "") in CAPTURE_CALLBACKS
           and _is_package_callback(cb, cb.__name__)]
    return cap, [cb for cb in generic if cb not in cap]


def _split_callbacks(callbacks):
    device, ticks, generic = [], [], []
    for cb in callbacks:
        name = getattr(cb, "__name__", "")
        # the four standard callbacks: this package's objects, or the reference's own (module
        # `callbacks.<name>` of numerical_experiments) -- a user callable that merely shares the name
        # is called like any other
        mod = getattr(cb, "__module__", "") or ""
        std = name in DEVICE_HISTORIES and (cb is getattr(_cbk, name, None) or mod.split(".")[0] == "callbacks"
                                            or mod.endswith("callbacks." + name))
        if std:
            device.append(name)
        elif hasattr(cb, "_cgx_print_every") or name == "pk":
            ticks.append(cb)          # print_k(K): progress only
        else:
            generic.append(cb)
    return device, ticks, generic


def _ensure_x_true(A, b, extra, needed):
    """error_* histories need x_true; if the caller gave none, solve for it once on the
    host exactly as the reference callbacks do (error_A_norm.py:36-39)."""
    if not needed or "x_true" in extra:
        return
    import scipy.sparse.linalg as spla
    if isinstance(A, PoissonStencil):
        A = A.tocsr()
    solver = spla.spsolve if sps.issparse(A) else np.linalg.solve
    extra["x_true"] = solver(A.astype(np.double), np.asarray(b, dtype=np.double))


def _solve(name, tag, A, b, x0, max_iter, preconditioner, callbacks, kwargs):
    own = {k: kwargs.pop(k) for k in _OWN_KEYS if k in kwargs}
    tol = _lib.check_tol(own["tol"]) if own.get("tol") is not None else 0.0
    device = own.get("device", 0)
    path = own.get("path", "auto")
    n = len(b)
    output = {"name": name, "max_iter": max_iter}
    dev_hist, ticks, generic = _split_callbacks(list(callbacks))
    _ensure_x_true(A, b, kwargs, any("error" in h for h in dev_hist))
    x_true = kwargs.get("x_true")

    sess = own.get("session")
    dinv = probe_preconditioner(preconditioner, n)
    if sess is None:
        sess = _session_for(A, dinv, device)
    else:
        sess.set_jacobi(dinv)                  # an explicit session still honours `preconditioner`

    w_replace = own.get("w_replace")
    plan = _plan_w_replace(w_replace, max_iter) if tag == "gv" else None
    capture, other = _split_capture(generic)
    if not other and not isinstance(plan, str):
        if capture and isinstance(A, PoissonStencil):
            A = A.tocsr()                      # the callback bodies multiply / factor A on the host
        sess.set_gv_replace(plan)
        names = {cb.__name__ for cb in capture}
        sess.set_capture(x="save_x" in names, r=bool(names - {"save_x"}), scalars="lanczos_recurrence" in names)
        try:
            _, hist, info = sess.solve(tag, b, x0, max_iter, x_true=x_true, histories=tuple(dev_hist),
                                       path=path, return_x=False, tol=tol)
            for h in dev_hist:
                output[h] = hist[h]
            if capture:
                _replay_captured(sess, tag, A, b, x0, max_iter, capture, output, kwargs, info["stop_iter"])
        finally:
            sess.set_capture()
            sess.set_gv_replace(None)
    else:
        info = _solve_stepwise(sess, tag, A, b, x0, max_iter, x_true, dev_hist, generic, output,
                               kwargs, path, w_replace if isinstance(plan, str) else None, plan, tol)
    stop = info["stop_iter"]
    if own.get("tol") is not None:     # (without tol= the output keeps the reference's keys)
        output["stop_iter"] = stop if stop >= 0 else None
    for cb in ticks:   # leave the terminal as print_k would after the last iteration
        try:
            cb(output=output, k=stop if stop >= 0 else max_iter - 1, max_iter=max_iter)
        except Exception:
            pass
    if own.get("return_info"):
        output["_info"] = info
    return output


def _replay_captured(sess, tag, A, b, x0, max_iter, capture, output, extra, stop=-1):
    """Run the capture-served callbacks once, on the host, from what the GPU recorded during the
    solve: x_k / r_k rows and the (a, b) the recurrences held after every iteration (k = 0 .. stop
    after a tolerance stop).  Same keyword protocol as the reference's `callback(**locals())`."""
    names = {cb.__name__ for cb in capture}
    X = sess.fetch_capture("x") if "save_x" in names else None
    R = sess.fetch_capture("r") if names - {"save_x"} else None
    sc = sess.fetch_capture("scalars") if "lanczos_recurrence" in names else None
    predicted = tag in ("pr", "m") or tag.startswith("pipe")
    b_arr = np.asarray(b, dtype=np.float64)
    a_k1 = a_k2 = b_k = b_k1 = 0.0
    for k in range(stop + 1 if stop >= 0 else max_iter):
        if k > 0 and sc is not None:
            a_k2, a_k1 = a_k1, sc[0][k - 1]
            b_k1, b_k = b_k, (sc[1][k - 1] if predicted else sc[1][k])
        loc = dict(output=output, A=A, b=b_arr, x0=x0, k=k, max_iter=max_iter, n=len(b_arr), kwargs=extra,
                   x_k=None if X is None else X[k], r_k=None if R is None else R[k],
                   x_k1=None if X is None or k == 0 else X[k - 1], r_k1=None if R is None or k == 0 else R[k - 1],
                   a_k=None if sc is None else sc[0][k], a_k1=a_k1, a_k2=a_k2, b_k=b_k, b_k1=b_k1)
        for cb in capture:
            cb(**loc)


def _plan_w_replace(w_replace, max_iter):
    """None: never (the reference's default); a uint8 schedule when the predicate depends only on k
    (it is then evaluated up front, in order, with the reference's `wk_replace_flags` dict);
    "host" when it reads vectors -> evaluated every iteration against the device state."""
    if w_replace is None or w_replace is _never:
        return None
    flags = {}
    sched = np.zeros(max_iter, dtype=np.uint8)
    try:
        for k in range(1, max_iter):
            sched[k] = 1 if w_replace(k=k, A=None, b=None, x=None, w=None, r=None, r_=None, u=None, s=None, p=None,
                                      wk_replace_flags=flags) else 0
    except Exception:                                   # noqa: BLE001 -- it looked at a vector
        return "host"
    return sched if sched.any() else None


def _solve_stepwise(sess, tag, A, b, x0, max_iter, x_true, dev_hist, generic, output, extra, path,
                    w_replace=None, plan=None, tol=0.0):
    """Arbitrary callbacks (and vector-reading GV `w_replace` predicates): step the GPU one
    iteration at a time and hand each callable the reference's keyword set (hs_cg.py:97-98,128-129;
    gv_cg.py:156).  Slow (a device round trip per iteration) but still no CPU arithmetic on the
    solve itself."""
    sess.load_problem(b, x0, x_true)
    host_pred = w_replace is not None
    sess.set_gv_replace(None if host_pred else plan)
    sess.set_option("gv_manual", 1 if host_pred else 0)
    if host_pred:
        path = "stream"
    try:
        sess.begin(tag, max_iter, histories=tuple(dev_hist), path=path, tol=tol)
    finally:
        sess.set_option("gv_manual", 0)
        sess.set_gv_replace(None)
    wk_flags = {}
    import inspect
    state_names = {"rt_k", "p_k", "s_k", "st_k", "w_k", "wt_k", "u_k", "t_k"}
    extra_vectors = set()
    for cb in generic:
        try:
            extra_vectors |= state_names & set(inspect.signature(cb).parameters)
        except (TypeError, ValueError):
            pass
    predicted = tag in ("pr", "m") or tag.startswith("pipe")
    b_arr = np.asarray(b, dtype=np.float64)
    a_k1 = a_k2 = 0.0
    b_k = b_k1 = 0.0
    x_k1 = r_k1 = None
    sc = sess.scalars()
    next_b = sc["b"]
    for k in range(max_iter):
        if k > 0:
            if host_pred:
                # gv_cg.py:151-158: the vector pass forms x_k, r_k, w_k; the predicate sees them (and the
                # previous r, u, s, p) and decides whether w_k is replaced by A r_k before t = A wt
                sess.advance_stages(1)
                if w_replace(k=k, A=A, b=b_arr, x=sess.vector("x"), w=sess.vector("w"), r=sess.vector("r"), r_=r_k1,
                             u=sess.vector("u"), s=sess.vector("s"), p=sess.vector("p"), wk_replace_flags=wk_flags):
                    sess.gv_replace_now()
                sess.advance_stages(1 + (1 if dev_hist else 0))
            else:
                sess.advance(1)
            sc_new = sess.scalars()
            a_k2, a_k1 = a_k1, sc["a"]
            b_k1 = b_k
            b_k = next_b if predicted else sc_new["b"]
            sc = sc_new
            next_b = sc["b"]
        x_k = sess.vector("x")
        r_k = sess.vector("r")
        loc = dict(output=output, A=A, b=b_arr, x0=x0, x_k=x_k, r_k=r_k, k=k, max_iter=max_iter,
                   n=len(b_arr), kwargs=extra, a_k=sc["a"], a_k1=a_k1, a_k2=a_k2, b_k=b_k, b_k1=b_k1,
                   nu_k=sc["nu"], mu_k=sc["mu"], x_k1=x_k1, r_k1=r_k1)
        # the reference hands every local to a callback (`callback(**locals())`); the other state vectors
        # are copied off the device only for callables that NAME them as parameters (p_k, s_k, rt_k, ...)
        for name in extra_vectors:
            loc[name] = sess.vector(name[:-2])
        for cb in generic:
            cb(**loc)
        x_k1, r_k1 = x_k, r_k
        if tol and k > 0 and sess.get_info()["stop_iter"] == k:
            break                                          # the tolerance was met at this iteration
    _, hist = sess.fetch(want_x=False, want_hist=True)
    for h in dev_hist:
        output[h] = hist[_lib.HIST_NAMES.index(h)].copy()
    return sess.get_info()


def _never(**kwargs):
    return False


def _make(name, tag, preconditioned, gv=False):
    if preconditioned and gv:
        def f(A, b, x0, max_iter, w_replace=_never, preconditioner=lambda x: x, callbacks=[], **kwargs):
            kwargs["w_replace"] = w_replace
            return _solve(name, tag, A, b, x0, max_iter, preconditioner, callbacks, kwargs)
    elif preconditioned:
        def f(A, b, x0, max_iter, preconditioner=lambda x: x, callbacks=[], **kwargs):
            return _solve(name, tag, A, b, x0, max_iter, preconditioner, callbacks, kwargs)
    elif gv:
        def f(A, b, x0, max_iter, w_replace=_never, callbacks=[], **kwargs):
            kwargs["w_replace"] = w_replace
            return _solve(name, tag, A, b, x0, max_iter, None, callbacks, kwargs)
    else:
        def f(A, b, x0, max_iter, callbacks=[], **kwargs):
            return _solve(name, tag, A, b, x0, max_iter, None, callbacks, kwargs)
    f.__name__ = f.__qualname__ = name
    f.__doc__ = f"{name}: GPU implementation of the reference's `{name}` (variant tag {tag!r})."
    return f


def solve_concurrently(methods, A, b, x0, max_iter, preconditioner=lambda x: x, callbacks=[], **kwargs):
    """Run several of this module's solvers on the same problem side by side: ONE cooperative launch
    on one GPU (``session.solve_batch``), each method on a 1/len(methods) share of the SMs.

    ``methods``: distinct functions of this module (e.g. ``experiments.ALL_METHODS``), preconditioned
    or all un-preconditioned.  Returns ``{method name: output}``, each output with the keys, names and
    shapes ``method(A, b, x0, max_iter, preconditioner=..., callbacks=..., **kwargs)`` returns.  The
    histories are bitwise those of a solo persistent-path run with the same CTA shape (not
    necessarily of a default solo run, whose CTA shape takes all the SMs).

    Only the four standard callbacks and ``print_k`` are served; any other callback, ``w_replace``,
    ``path=`` or ``session=`` raises ``NotImplementedError`` before the GPU is touched.  One Session
    per method, closed afterwards (the operator cache of the single-method functions is not used).
    Extra keyword arguments: ``x_true``, ``device=0``, ``return_info=True``, ``tol=`` (as for the
    single-method functions; every method stops on its own)."""
    from ..session import solve_batch
    methods = list(methods)
    for key in ("path", "w_replace", "session"):
        if key in kwargs:
            raise NotImplementedError(f"solve_concurrently: `{key}=` is not supported (persistent batch only)")
    tags = []
    for m in methods:
        name = getattr(m, "__name__", "")
        stem, _, suffix = name.rpartition("_")
        if globals().get(name) is not m or suffix not in ("cg", "pcg"):
            raise NotImplementedError(f"solve_concurrently: {name or m!r} is not a GPU solver of this module")
        tags.append((name, stem, suffix == "pcg"))
    if len({t[0] for t in tags}) != len(tags):
        raise ValueError("solve_concurrently: a method is listed twice")
    dev_hist, ticks, generic = _split_callbacks(list(callbacks))
    if generic:
        raise NotImplementedError("solve_concurrently: only the four standard callbacks and print_k run in a batch; "
                                  f"got {[getattr(cb, '__name__', cb) for cb in generic]}")
    device = kwargs.pop("device", 0)
    return_info = kwargs.pop("return_info", False)
    tol_arg = kwargs.pop("tol", None)
    tol = _lib.check_tol(tol_arg) if tol_arg is not None else 0.0
    n = len(b)
    _ensure_x_true(A, b, kwargs, any("error" in h for h in dev_hist))
    x_true = kwargs.get("x_true")
    dinv = probe_preconditioner(preconditioner, n) if any(t[2] for t in tags) else None
    sessions = []
    try:
        for _, _, pre in tags:
            sessions.append(Session(A, dinv=dinv if pre else None, device=device))
        res = solve_batch([(s, tag, b, x0, max_iter, x_true) for s, (_, tag, _) in zip(sessions, tags)],
                          histories=tuple(dev_hist), return_x=False, tol=tol)
    finally:
        for s in sessions:
            s.close()
    outputs = {}
    for (name, _, _), (_, hist, info) in zip(tags, res):
        output = {"name": name, "max_iter": max_iter}
        for h in dev_hist:
            output[h] = hist[h]
        stop = info["stop_iter"]
        if tol_arg is not None:
            output["stop_iter"] = stop if stop >= 0 else None
        for cb in ticks:
            try:
                cb(output=output, k=stop if stop >= 0 else max_iter - 1, max_iter=max_iter)
            except Exception:
                pass
        if return_info:
            output["_info"] = info
        outputs[name] = output
    return outputs


_TAGS = [("hs", "hs"), ("cg", "cg"), ("gv", "gv"), ("pr", "pr"), ("m", "m"), ("pipe_pr", "pipe_pr"),
         ("pipe_p", "pipe_p"), ("pipe_pr_m", "pipe_pr_m"), ("pipe_p_m", "pipe_p_m")]
__all__ = ["probe_preconditioner", "clear_cache", "solve_concurrently"]
for _stem, _tag in _TAGS:
    for _suffix, _pre in (("_pcg", True), ("_cg", False)):
        _fname = _stem + _suffix
        globals()[_fname] = _make(_fname, _tag, _pre, gv=(_tag == "gv"))
        __all__.append(_fname)
del _stem, _tag, _suffix, _pre, _fname
