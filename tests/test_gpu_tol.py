"""GPU: stopping a single-GPU solve on the device at a relative tolerance (cgx_set_tolerance / tol=).

The contract: a run that stops at k = stop returns, bit for bit, what the same run without a tolerance
and with max_iter = stop + 1 returns (x, the state vectors, the scalars, history entries 0 .. stop),
and stop is the first k with nu_k <= tol^2 nu_0."""
import ctypes as C

import numpy as np
import pytest

import helpers
from helpers import orc
from new_cg_variants_b200 import PoissonStencil, Session, _lib, callbacks as cbk, cg_variants
from new_cg_variants_b200.dist import GroupSession
from new_cg_variants_b200.session import solve_batch

pytestmark = pytest.mark.gpu

ALL_TAGS = list(orc.VARIANTS)
TOL = 1e-5
VECS = ("x", "r", "rt", "p", "s")


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def _same(a, b, label):
    assert np.array_equal(_bits(a), _bits(b)), label


# (name, operator factory, preconditioned, max_iter large enough for TOL)
CASES = {
    "nos4": (lambda: helpers.load_matrix("nos4"), False, 1000),
    "bcsstk15_jacobi": (lambda: helpers.load_matrix("bcsstk15"), True, 3000),
    "poisson2d": (lambda: PoissonStencil(64, 64, 1, dim=2), False, 1000),
    "poisson3d_jacobi": (lambda: PoissonStencil(24, 24, 24, dim=3), True, 500),
}
_SESS = {}


def _case(name):
    """(session, b, x0, x_true, max_iter), one session per case for the whole module."""
    if name not in _SESS:
        make, prec, max_iter = CASES[name]
        A = make()
        x_true, b, x0 = orc.setup_problem(A.tocsr() if isinstance(A, PoissonStencil) else A)
        dinv = (1.0 / A.diagonal()) if prec else None
        _SESS[name] = (Session(A, dinv=dinv), b, x0, x_true, max_iter)
    return _SESS[name]


@pytest.fixture(scope="module", autouse=True)
def _close_sessions():
    yield
    for s, *_ in _SESS.values():
        s.close()
    _SESS.clear()


def _nu0(s, tag, b, x0, xt, path):
    s.load_problem(b, x0, xt)
    s.begin(tag, 2, path=path)
    return s.scalars()["nu"]


def _state(s):
    return {v: s.vector(v) for v in VECS}


def check_contract(s, tag, b, x0, xt, max_iter, path, tol=TOL):
    """Runs the three solves of the contract; returns stop."""
    nu0 = _nu0(s, tag, b, x0, xt, path)
    thr = tol * tol * nu0
    x, hist, info = s.solve(tag, b, x0, max_iter, x_true=xt, path=path, tol=tol)
    sc, st = s.scalars(), _state(s)
    stop = info["stop_iter"]
    label = f"{tag}/{path}"
    assert 1 <= stop < max_iter - 1, f"{label}: tol {tol} not reached in {max_iter} iterations"
    assert info["iterations"] == stop and info["path"] == (1 if path == "stream" else 2), label
    assert sc["nu"] <= thr, label
    x1, hist1, _ = s.solve(tag, b, x0, stop + 1, x_true=xt, path=path)
    sc1, st1 = s.scalars(), _state(s)
    _same(x, x1, f"{label}: x")
    assert set(hist) == set(hist1)
    for h in hist1:
        assert hist[h].shape == (stop + 1,), label
        _same(hist[h], hist1[h], f"{label}: {h}")
    _same(list(sc.values()), list(sc1.values()), f"{label}: scalars")
    for v in VECS:
        _same(st[v], st1[v], f"{label}: vector {v}")
    # stop is the FIRST crossing
    s.solve(tag, b, x0, stop, x_true=xt, path=path, histories=())
    assert s.scalars()["nu"] > thr, f"{label}: nu already below the threshold at k = {stop - 1}"
    return stop


@pytest.mark.parametrize("path", ["stream", "persistent"])
@pytest.mark.parametrize("case", list(CASES))
@pytest.mark.parametrize("tag", ALL_TAGS)
def test_contract_all_variants(tag, case, path):
    s, b, x0, xt, max_iter = _case(case)
    check_contract(s, tag, b, x0, xt, max_iter, path)


# each SpMV / pass kernel of the stream path
KERNELS = [
    ("poisson3d_jacobi", {}, ("pr", "m")),                                   # pr_fused_kernel
    ("poisson3d_jacobi", {"pr_fused": 0}, ("pr", "pipe_pr", "hs")),           # stencil_tma_kernel
    ("poisson3d_jacobi", {"tma": 0}, ("hs", "cg", "gv", "pr", "pipe_pr")),    # generic spmv_kernel
    ("poisson2d", {"cg_elide": 0}, ("cg", "gv")),
    ("bcsstk15_jacobi", {"csr_bulk": 0}, ("pr", "pipe_pr", "cg")),            # csr_stream_kernel
    ("bcsstk15_jacobi", {"csr_bulk": 1}, ("pr", "pipe_pr", "gv")),            # csr_bulk_kernel, 1 RHS
    ("bcsstk15_jacobi", {"csr_bulk": 2}, ("pipe_pr", "pipe_pr_m")),           # csr_bulk_kernel, 2 RHS
    ("nos4", {"csr_stream": 0}, ("hs", "pr", "pipe_p")),                      # spmv_kernel<CsrOp>
]
_DEFAULTS = {"pr_fused": 1, "tma": 1, "cg_elide": 1, "csr_bulk": 1, "csr_stream": 1}


@pytest.mark.parametrize("case,opts,tags", KERNELS, ids=[f"{c}-{o}" for c, o, _ in KERNELS])
def test_contract_each_stream_kernel(case, opts, tags):
    s, b, x0, xt, max_iter = _case(case)
    try:
        for k, v in opts.items():
            s.set_option(k, v)
        for tag in tags:
            check_contract(s, tag, b, x0, xt, max_iter, "stream")
    finally:
        for k in opts:
            s.set_option(k, _DEFAULTS[k])


@pytest.mark.parametrize("path", ["stream", "persistent"])
@pytest.mark.parametrize("tag", ["hs", "gv", "pr", "pipe_p_m"])
def test_tolerance_never_reached(tag, path):
    s, b, x0, xt, _ = _case("bcsstk15_jacobi")
    x, hist, info = s.solve(tag, b, x0, 60, x_true=xt, path=path, tol=1e-12)
    sc = s.scalars()
    x1, hist1, info1 = s.solve(tag, b, x0, 60, x_true=xt, path=path)
    assert info["stop_iter"] == -1 and info1["stop_iter"] == -1 and info["iterations"] == 59
    _same(x, x1, "x")
    for h in hist1:
        assert hist[h].shape == (60,)
        _same(hist[h], hist1[h], h)
    _same(list(sc.values()), list(s.scalars().values()), "scalars")


@pytest.mark.parametrize("path", ["stream", "persistent"])
@pytest.mark.parametrize("tag", ["cg", "pipe_pr"])
def test_stepping(tag, path):
    s, b, x0, xt, max_iter = _case("nos4")
    x, hist, info = s.solve(tag, b, x0, max_iter, x_true=xt, path=path, tol=TOL)
    stop = info["stop_iter"]
    assert stop > 7
    s.load_problem(b, x0, xt)
    s.begin(tag, max_iter, histories=orc.HISTORIES, path=path, tol=TOL)
    for _ in range(max_iter // 7 + 1):
        s.advance(7)
    got = s.get_info()
    assert got["stop_iter"] == stop and got["iterations"] == stop
    x2, h2 = s.fetch()
    _same(x2, x, "stepped x")
    assert h2.shape == (4, stop + 1)
    for i, name in enumerate(_lib.HIST_NAMES):
        if name in hist:
            _same(h2[i], hist[name], name)
    sc = s.scalars()
    s.advance(7)                                    # after the stop: nothing happens
    assert s.get_info()["iterations"] == stop
    _same(s.fetch()[0], x, "x after a further advance")
    _same(list(s.scalars().values()), list(sc.values()), "scalars after a further advance")


def test_generic_callback_sees_k_up_to_the_stop():
    A = helpers.load_matrix("nos4")
    x_true, b, x0 = orc.setup_problem(A)
    seen = []

    def cb(k, **kw):
        assert "tol" not in kw["kwargs"]
        seen.append(k)

    ticks = []

    def pk(output, k, max_iter):
        ticks.append(k)

    pk._cgx_print_every = 1
    out = cg_variants.pr_cg(A, b, x0, 1000, callbacks=[cb, pk, cbk.updated_residual_2_norm], x_true=x_true, tol=TOL)
    stop = out["stop_iter"]
    assert stop is not None and seen == list(range(stop + 1)) and ticks == [stop]
    assert out["updated_residual_2_norm"].shape == (stop + 1,)
    ref = cg_variants.pr_cg(A, b, x0, stop + 1, callbacks=[cbk.updated_residual_2_norm], x_true=x_true)
    _same(out["updated_residual_2_norm"], ref["updated_residual_2_norm"], "history")
    assert "stop_iter" not in ref
    never = cg_variants.pr_cg(A, b, x0, 20, callbacks=[cbk.updated_residual_2_norm], tol=1e-12)
    assert never["stop_iter"] is None and never["updated_residual_2_norm"].shape == (20,)


@pytest.mark.parametrize("tag", ["gv", "pr"])
def test_capture_and_gv_replacement(tag):
    s, b, x0, xt, max_iter = _case("nos4")
    sched = np.zeros(max_iter, dtype=np.uint8)
    sched[5::9] = 1
    outs = []
    try:
        for it, tol in ((max_iter, TOL), (None, None)):
            s.set_capture(x=True, r=True, scalars=True)
            if tag == "gv":
                s.set_gv_replace(sched)
            if it is None:
                it = outs[0][2]["stop_iter"] + 1
            x, hist, info = s.solve(tag, b, x0, it, x_true=xt, path="stream", tol=tol)
            outs.append((x, hist, info, [s.fetch_capture(w) for w in ("x", "r", "scalars")], s.scalars()))
    finally:
        s.set_capture()
        s.set_gv_replace(None)
    (x, hist, info, cap, sc), (x1, hist1, info1, cap1, sc1) = outs
    stop = info["stop_iter"]
    assert stop > 5 and info1["stop_iter"] == -1
    _same(x, x1, "x")
    for h in hist1:
        _same(hist[h], hist1[h], h)
    for w, a, a1 in zip(("x", "r", "scalars"), cap, cap1):
        assert a.shape == a1.shape, w
        _same(a, a1, f"capture {w}")
    _same(list(sc.values()), list(sc1.values()), "scalars")
    if tag == "pr":               # the drop-in functions replay the capture-served callbacks up to the stop
        out = cg_variants.pr_cg(helpers.load_matrix("nos4"), b, x0, max_iter, callbacks=[cbk.save_x], tol=TOL, session=s)
        assert out["stop_iter"] == stop
        _same(out["x"][:stop + 1], cap[0], "save_x rows")
        assert not out["x"][stop + 1:].any()


SHAPE = (128, 16)


def _shaped(A, dinv):
    s = Session(A, dinv=dinv)
    s.set_option("pers_threads", SHAPE[0])
    s.set_option("pers_ctas", SHAPE[1])
    return s


def test_batch_entries_stop_independently():
    A = helpers.load_matrix("bcsstk15")
    dinv = orc.jacobi_dinv(A)
    x_true, b, x0 = orc.setup_problem(A)
    rng = np.random.default_rng(3)
    b2 = A @ rng.standard_normal(A.shape[0])
    entries = [("pr", b, x0, 3000, x_true), ("hs", b2, x0, 3000, None), ("pipe_pr", b, x0, 40, x_true),
               ("cg", b2, x0, 3000, None)]
    sess = [_shaped(A, dinv) for _ in entries]
    try:
        res = solve_batch([(s, *e) for s, e in zip(sess, entries)], tol=TOL)
        stops = [r[2]["stop_iter"] for r in res]
        assert stops[2] == -1 and all(st > 0 for i, st in enumerate(stops) if i != 2)
        assert len(set(stops)) > 2
        for i, (s, (tag, bb, xx, it, xt)) in enumerate(zip(sess, entries)):
            solo = s.solve(tag, bb, xx, it, x_true=xt, path="persistent", tol=TOL)
            xb, hb, ib = res[i]
            assert ib["stop_iter"] == solo[2]["stop_iter"] and ib["iterations"] == solo[2]["iterations"]
            _same(xb, solo[0], f"entry {i}: x")
            assert set(hb) == set(solo[1])
            for h in hb:
                _same(hb[h], solo[1][h], f"entry {i}: {h}")
        plain = solve_batch([(s, *e) for s, e in zip(sess, entries)])
        assert all(r[2]["stop_iter"] == -1 for r in plain)
        for i, (s, (tag, bb, xx, it, xt)) in enumerate(zip(sess, entries)):
            _same(plain[i][0], s.solve(tag, bb, xx, it, x_true=xt, path="persistent")[0], f"entry {i} without tol")
    finally:
        for s in sess:
            s.close()


def test_solve_concurrently_with_tol():
    A = helpers.load_matrix("bcsstk15")
    dinv = orc.jacobi_dinv(A)
    x_true, b, x0 = orc.setup_problem(A)
    prec = lambda v: dinv * v
    std = [cbk.error_A_norm, cbk.residual_2_norm, cbk.error_2_norm, cbk.updated_residual_2_norm]
    out = cg_variants.solve_concurrently([cg_variants.pr_pcg], A, b, x0, 3000, preconditioner=prec, callbacks=std,
                                         x_true=x_true, tol=TOL)["pr_pcg"]
    solo = cg_variants.pr_pcg(A, b, x0, 3000, preconditioner=prec, callbacks=std, x_true=x_true, path="persistent",
                              tol=TOL)
    assert out["stop_iter"] is not None and out["stop_iter"] == solo["stop_iter"]
    for h in orc.HISTORIES:
        assert out[h].shape == (out["stop_iter"] + 1,)
        _same(out[h], solo[h], h)


def test_partition_rank_with_a_tolerance_is_refused():
    S = PoissonStencil(32, 32, 32, dim=3)
    x_true, b, x0 = orc.setup_problem(S.tocsr())
    grp = GroupSession(S, 2, dinv=1 / S.diagonal())
    lib = _lib.load()
    try:
        x, hist, _ = grp.solve("pr", b, x0, 40, x_true=x_true)
        assert lib.cgx_set_tolerance(grp.members[1]._ctx, 1e-6) == _lib.OK
        grp.load_problem(b, x0, x_true)
        assert lib.cgx_group_begin(grp._arr, 2, _lib.VARIANT_IDS["pr"], 40, 0, _lib.PATHS["stream"]) == _lib.ERR_UNSUPPORTED
        assert b"partition" in lib.cgx_last_error()
        assert lib.cgx_begin(grp.members[1]._ctx, _lib.VARIANT_IDS["pr"], 40, 0, _lib.PATHS["stream"]) == _lib.ERR_UNSUPPORTED
        assert lib.cgx_set_tolerance(grp.members[1]._ctx, 0.0) == _lib.OK
        x2, hist2, _ = grp.solve("pr", b, x0, 40, x_true=x_true)
        _same(x2, x, "x after the tolerance was cleared")
        for h in hist:
            _same(hist2[h], hist[h], h)
    finally:
        grp.close()
