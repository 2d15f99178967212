"""GPU: independent solves in one cooperative launch (cgx_batch_run / session.solve_batch /
cg_variants.solve_concurrently / experiments.test_matrix(concurrent=True)).

The batch's promise is bitwise equality with a solo persistent-path run of the same CTA shape, so the
bitwise tests force that shape (options pers_threads / pers_ctas) on both sides."""
import ctypes as C
import json
import os
import time

import numpy as np
import pytest

import helpers
from helpers import orc
from new_cg_variants_b200 import PoissonStencil, Session, _lib, callbacks as cbk, cg_variants, experiments as ex
from new_cg_variants_b200.session import solve_batch

pytestmark = pytest.mark.gpu

STD_CALLBACKS = [cbk.error_A_norm, cbk.residual_2_norm, cbk.error_2_norm, cbk.updated_residual_2_norm]
ALL_TAGS = list(orc.VARIANTS)
SHAPE = (128, 16)            # pers_threads, pers_ctas: nine entries x 16 CTAs fit 148 SMs


def _session(A, dinv, shape=SHAPE, slab=None):
    s = Session(A, dinv=dinv)
    s.set_option("pers_threads", shape[0])
    s.set_option("pers_ctas", shape[1])
    if slab is not None:
        s.set_option("csr_slab", slab)
    return s


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def _assert_same(batch_out, solo_out, label):
    """Bit patterns, so that a run that breaks down (NaN from the breakdown on) compares too."""
    xb, hb, ib = batch_out
    xs, hs, _ = solo_out
    assert ib["path"] == 2, label
    assert np.array_equal(_bits(xb), _bits(xs)), f"{label}: x differs from the solo run"
    assert set(hb) == set(hs), label
    for h in hs:
        assert np.array_equal(_bits(hb[h]), _bits(hs[h])), f"{label}/{h}: history differs from the solo run"


def _batch_vs_solo(A, dinv, entries, slab=None, shape=SHAPE):
    """entries: [(variant, b, x0, max_iter, x_true)].  Every batch entry bitwise == its solo run."""
    sess = [_session(A if not callable(A) else A(i), dinv, shape, slab) for i in range(len(entries))]
    try:
        res = solve_batch([(s, *e) for s, e in zip(sess, entries)])
        for i, (s, (tag, b, x0, it, xt)) in enumerate(zip(sess, entries)):
            solo = s.solve(tag, b, x0, it, x_true=xt, path="persistent")
            _assert_same(res[i], solo, f"entry {i} ({tag}, max_iter {it})")
        return res
    finally:
        for s in sess:
            s.close()


def _problem(A, prec):
    x_true, b, x0 = orc.setup_problem(A)
    dinv = orc.jacobi_dinv(A) if prec == "jacobi" else None
    return b, x0, x_true, dinv


BITWISE = [("nos4", "jacobi", 120), ("nos4", None, 150), ("bcsstk15", "jacobi", 830), ("bcsstk18", None, 3000),
           ("model_48_8_3", None, 110), ("1138_bus", "jacobi", 1300)]


@pytest.mark.parametrize("slab", [0, 1])
@pytest.mark.parametrize("name,prec,max_iter", BITWISE)
def test_nine_variants_bitwise_equal_solo_runs_csr(name, prec, max_iter, slab):
    A = helpers.load_matrix(name)
    b, x0, x_true, dinv = _problem(A, prec)
    _batch_vs_solo(A, dinv, [(t, b, x0, max_iter, x_true) for t in ALL_TAGS], slab=slab)


@pytest.mark.parametrize("prec", [None, "jacobi"])
@pytest.mark.parametrize("shape", [(24, 24, 24), (64, 64, 1)])
def test_nine_variants_bitwise_equal_solo_runs_stencil(shape, prec):
    S = PoissonStencil(*shape, dim=3 if shape[2] > 1 else 2)
    b, x0, x_true, dinv = _problem(S.tocsr(), prec)
    _batch_vs_solo(S, dinv, [(t, b, x0, 300, x_true) for t in ALL_TAGS])


def test_heterogeneous_batches():
    A = helpers.load_matrix("bcsstk03")
    n = A.shape[0]
    rng = np.random.default_rng(1)
    _, b0, x0, x_true, dinv, _ = helpers.case_problem("bcsstk03_jacobi")
    b1, b2 = rng.standard_normal(n), A @ rng.standard_normal(n)
    # one matrix, three right-hand sides, different lengths, with and without x_true
    res = _batch_vs_solo(A, dinv, [("pr", b0, x0, 50, x_true), ("pipe_pr", b1, x0, 400, None), ("hs", b2, x0, 1200, None)])
    assert res[1][1].keys() == {"residual_2_norm", "updated_residual_2_norm"}
    assert [r[1]["residual_2_norm"].shape for r in res] == [(50,), (400,), (1200,)]
    # different operators of one kind (CSR, no preconditioner)
    mats = [helpers.load_matrix(m) for m in ("nos4", "bcsstk03", "1138_bus")]
    probs = [orc.setup_problem(M) for M in mats]
    sess = [_session(M, None) for M in mats]
    try:
        items = [(s, tag, p[1], p[2], it, p[0]) for s, tag, p, it in zip(sess, ("cg", "gv", "m"), probs, (150, 300, 500))]
        res = solve_batch(items)
        again = solve_batch(items)
        for i, (s, tag, b, x0_, it, xt) in enumerate(items):
            _assert_same(res[i], s.solve(tag, b, x0_, it, x_true=xt, path="persistent"), f"mixed entry {i}")
            _assert_same(again[i], res[i], f"repeat entry {i}")
    finally:
        for s in sess:
            s.close()
    # a batch of one is cgx_run on the persistent path with the same shape
    _batch_vs_solo(A, dinv, [("gv", b0, x0, 250, x_true)])


def _metrics_ok(case, tag, dev):
    """The checks of test_long_runs_match_reference_metrics for one variant."""
    meta = helpers.cases()[case]
    table = json.load(open(os.path.join(helpers.GOLDEN, "table.json"))).get(case)
    cols = ["hs", "cg", "m", "pr", "gv", "pipe_pr_m", "pipe_pr"]
    it, acc = orc.convergence_metrics(dev["error_A_norm"])
    band = meta["kstar"][tag] if meta["kstar"] else None
    stored = (meta.get("stored_metrics") or {}).get(tag)
    pub = (table["iters"][cols.index(tag)], table["acc"][cols.index(tag)]) if table and tag in cols else None
    if band:
        helpers.check_metrics(dev, band, f"{case}/{tag}")
    aw = (band["acc_band"][1] - band["acc_band"][0]) if band else 0.0
    iw = (band["iters_band"][1] - band["iters_band"][0]) if band and min(band["iters_band"]) > 0 else 0
    for src, ref in (("stored .npy", stored), ("published table", pub)):
        if ref is None:
            continue
        assert abs(acc - ref[1]) <= 1.0 + aw, (case, tag, src, acc, ref)
        if ref[0] and it:
            assert abs(it - ref[0]) <= max(3, 0.05 * ref[0]) + iw, (case, tag, src, it, ref)
    return it, acc


def _concurrent(case, **kw):
    A, b, x0, x_true, dinv, max_iter = helpers.case_problem(case)
    prec = (lambda v: v) if dinv is None else (lambda v: dinv * v)
    methods = [getattr(cg_variants, orc.VARIANTS[t]) for t in ALL_TAGS]
    out = cg_variants.solve_concurrently(methods, A, b, x0, max_iter, preconditioner=prec, callbacks=STD_CALLBACKS,
                                         x_true=x_true, return_info=True, **kw)
    return A, b, x0, x_true, dinv, max_iter, out


@pytest.mark.parametrize("case", helpers.cases_of("full", "prefix"))
def test_solve_concurrently_parity(case):
    """Default geometry: the criteria of test_variants_match_oracle_and_goldens."""
    A, b, x0, x_true, dinv, max_iter, out = _concurrent(case)
    bands = helpers.cases()[case]["kstar"]
    full = helpers.tier(case) == "full"
    assert list(out) == [orc.VARIANTS[t] for t in ALL_TAGS]
    for tag in ALL_TAGS:
        dev = out[orc.VARIANTS[tag]]
        assert dev["name"] == orc.VARIANTS[tag] and dev["max_iter"] == max_iter and dev["_info"]["path"] == 2
        live = orc.solve(tag, A, b, x0, max_iter, dinv=dinv, x_true=x_true)
        for h in orc.HISTORIES:
            assert dev[h].shape == (max_iter,)
        helpers.check_parity(dev, live, bands[tag], f"{case}/{tag} batch vs live oracle")
        gold = {h: helpers.golden_history(case, tag, h) for h in (orc.HISTORIES if full else helpers.RESIDUAL_HISTS)}
        helpers.check_window(dev, gold, bands[tag], f"{case}/{tag} batch vs golden")


@pytest.mark.parametrize("case", helpers.cases_of("metrics"))
def test_long_runs_all_nine_variants_in_one_batch(case):
    t0 = time.perf_counter()
    *_, max_iter, out = _concurrent(case)
    wall = time.perf_counter() - t0
    report = []
    for tag in ALL_TAGS:
        it, acc = _metrics_ok(case, tag, out[orc.VARIANTS[tag]])
        report.append(f"{tag}: it={it} acc={acc:.2f}")
    print(f"\n[{case}] nine variants, {max_iter} iterations, one batch: {wall:.1f} s wall | " + " | ".join(report))


def _run_batch(sessions, variants, max_iter=30):
    lib = sessions[0]._lib
    count = len(sessions)
    ctxs = (C.c_void_p * count)(*[s._ctx for s in sessions])
    v = np.array([_lib.VARIANT_IDS[t] for t in variants], dtype=np.int32)
    it = np.full(count, max_iter, dtype=np.int32)
    infos = (_lib.CgxInfo * count)()
    return lib.cgx_batch_run(ctxs, count, _lib.iptr(v), _lib.iptr(it), 15, infos)


@pytest.mark.parametrize("how", ["mixed_pm", "stencil_and_csr", "capture", "gv_schedule", "too_large"])
def test_refusals_launch_nothing_and_leave_contexts_usable(how):
    A = helpers.load_matrix("nos4")
    x_true, b, x0 = orc.setup_problem(A)
    dinv = orc.jacobi_dinv(A)
    sess = [Session(A), Session(A)]
    tags = ["pr", "gv"]
    if how == "mixed_pm":
        sess[1].set_jacobi(dinv)
    elif how == "stencil_and_csr":
        sess[1].close()
        S = PoissonStencil(10, 10, 1, dim=2)
        sess[1] = Session(S)
    elif how == "capture":
        sess[1].set_capture(x=True)
    elif how == "gv_schedule":
        sess[1].set_gv_replace(np.array([0, 0, 1, 0], dtype=np.uint8))
    elif how == "too_large":
        for s in sess:
            s.close()
        S = PoissonStencil(128, 128, 128, dim=3)
        sess = [Session(S) for _ in range(9)]
        tags = ALL_TAGS
    try:
        for s in sess:
            n = s.n
            s.load_problem(np.ones(n), np.zeros(n), np.ones(n) / np.sqrt(n))
        rc = _run_batch(sess, tags)
        assert rc == _lib.ERR_UNSUPPORTED, (how, rc)
        msg = sess[0]._lib.cgx_last_error().decode()
        assert "cgx_batch_run" in msg, msg
        if how == "capture":
            sess[1].set_capture()
        if how == "gv_schedule":
            sess[1].set_gv_replace(None)
        # the contexts still solve normally
        for s, tag in zip(sess, tags):
            n = s.n
            _, hist, info = s.solve(tag, np.ones(n), np.zeros(n), 20, path="auto")
            assert np.isfinite(hist["updated_residual_2_norm"]).all() and info["iterations"] == 19
    finally:
        for s in sess:
            s.close()


def test_rank_contexts_are_refused():
    """A rank of a partition (world > 1) is refused with CGX_ERR_UNSUPPORTED."""
    lib = _lib.load()
    ctxs = []
    try:
        for r in range(2):
            c = C.c_void_p()
            _lib.check(lib.cgx_ctx_create(0, C.byref(c)))
            ctxs.append(c)
            _lib.check(lib.cgx_set_stencil_slab(c, 8, 8, 4, 2, r, 6.0, -1.0))
        for r in range(2):
            _lib.check(lib.cgx_dist_attach_ctx(ctxs[r], 1 - r, ctxs[1 - r]))
        for r in range(2):
            _lib.check(lib.cgx_dist_commit(ctxs[r], 1, None, None))
        arr = (C.c_void_p * 2)(*ctxs)
        b = np.ones(512)
        _lib.check(lib.cgx_group_load_problem_host(arr, 2, _lib.dptr(b), _lib.dptr(np.zeros(512)), None, 512))
        v = np.array([3, 3], dtype=np.int32)
        it = np.full(2, 30, dtype=np.int32)
        infos = (_lib.CgxInfo * 2)()
        assert lib.cgx_batch_run(arr, 2, _lib.iptr(v), _lib.iptr(it), 0, infos) == _lib.ERR_UNSUPPORTED
        assert b"partition" in lib.cgx_last_error()
        # the partition still solves
        _lib.check(lib.cgx_group_begin(arr, 2, 3, 30, 0, 2))
        _lib.check(lib.cgx_group_advance(arr, 2, 29))
    finally:
        for c in ctxs:
            lib.cgx_ctx_destroy(c)


def test_test_matrix_concurrent_writes_what_the_sequential_driver_writes(tmp_path):
    for name, prec, max_iter in (("bcsstk03", "jacobi", 250), ("nos4", None, 150)):
        A = helpers.load_matrix(name)
        seq = ex.test_matrix(A, max_iter, name, preconditioner=prec, variants=ex.ALL_METHODS, data_dir=str(tmp_path / "seq"))
        con = ex.test_matrix(A, max_iter, name, preconditioner=prec, variants=ex.ALL_METHODS, data_dir=str(tmp_path / "con"),
                             concurrent=True)
        assert list(con) == list(seq)
        d_seq, d_con = tmp_path / "seq" / f"{name}_{prec}", tmp_path / "con" / f"{name}_{prec}"
        assert sorted(os.listdir(d_seq)) == sorted(os.listdir(d_con))
        bands = helpers.cases()[f"{name}_{prec}"]["kstar"]
        for m in ex.ALL_METHODS:
            s = np.load(d_seq / f"{m.__name__}.npy", allow_pickle=True).item()
            c = np.load(d_con / f"{m.__name__}.npy", allow_pickle=True).item()
            assert set(s) == set(c) and c["name"] == m.__name__ and c["max_iter"] == max_iter
            for k in orc.HISTORIES:
                assert c[k].shape == s[k].shape == (max_iter,)
        for fn, tag in zip(ex.TABLE_METHODS, ("hs", "cg", "m", "pr", "gv", "pipe_pr_m", "pipe_pr")):
            helpers.check_metrics(con[fn], bands[tag], f"{name}_{prec}/{fn} concurrent")
        rows = [ex.parse_convergence_data(name, prec, ex.TABLE_METHODS, A=A, data_dir=str(d))[0]
                for d in (tmp_path / "seq", tmp_path / "con")]
        head = lambda r: r.split("&")[:4]                                           # noqa: E731
        assert head(rows[0]) == head(rows[1]) and rows[0].count("&") == rows[1].count("&")
        assert (d_con / "convergence.txt").read_text() == rows[1]
