"""CPU: the tolerance stop's ABI and argument checks, before any device work."""
import ctypes as C
import math
import re

import numpy as np
import pytest

import helpers
from new_cg_variants_b200 import _lib, cg_variants
from new_cg_variants_b200.session import Session, solve_batch


def test_set_tolerance_is_declared_and_exported():
    with open(f"{helpers.ROOT}/include/cgx.h") as f:
        assert re.search(r"int cgx_set_tolerance\(cgx_ctx\* ctx, double rtol\);", f.read())
    assert _lib.PROTOTYPES["cgx_set_tolerance"] == (C.c_int, [C.c_void_p, C.c_double])
    lib = _lib.load()
    assert lib.cgx_set_tolerance(None, 0.5) == _lib.ERR_ARG
    assert b"cgx_set_tolerance" in lib.cgx_last_error()


def test_info_keeps_its_size_and_reports_stop_iter():
    assert C.sizeof(_lib.CgxInfo) == 56
    names = [f for f, _ in _lib.CgxInfo._fields_]
    assert names[-1] == "stop_iter" and "reserved" not in names
    info = _lib.CgxInfo()
    info.stop_iter = 17
    assert info.as_dict()["stop_iter"] == 17


@pytest.mark.parametrize("tol", [-1.0, 1.0, 2.0, math.nan, math.inf])
def test_check_tol_rejects(tol):
    with pytest.raises(ValueError):
        _lib.check_tol(tol)


@pytest.mark.parametrize("tol", [0, 0.0, 1e-300, 0.5, np.float64(1e-8)])
def test_check_tol_accepts(tol):
    assert _lib.check_tol(tol) == float(tol)


def _problem():
    A = helpers.load_matrix("nos4")
    return A, A @ np.ones(A.shape[0]), np.zeros(A.shape[0])


@pytest.mark.parametrize("tol", [-1, 1.0, math.nan])
def test_solvers_validate_tol_before_the_device(tol, monkeypatch):
    A, b, x0 = _problem()

    def no_device(*a, **k):
        raise AssertionError("a context was requested before tol was checked")

    monkeypatch.setattr(cg_variants, "_session_for", no_device)
    monkeypatch.setattr(cg_variants, "Session", no_device)
    with pytest.raises(ValueError):
        cg_variants.pr_pcg(A, b, x0, 20, tol=tol)
    with pytest.raises(ValueError):
        cg_variants.hs_cg(A, b, x0, 20, tol=tol)
    with pytest.raises(ValueError):
        cg_variants.solve_concurrently([cg_variants.pr_pcg], A, b, x0, 20, tol=tol)


def test_session_methods_validate_tol_before_the_device():
    s = object.__new__(Session)          # no context: any use of it would fail differently
    A, b, x0 = _problem()
    with pytest.raises(ValueError):
        s.solve("pr", b, x0, 20, tol=2)
    with pytest.raises(ValueError):
        s.run("pr", 20, tol=-0.5)
    with pytest.raises(ValueError):
        s.begin("pr", 20, tol=math.nan)
    with pytest.raises(ValueError):
        solve_batch([(s, "pr", b, x0, 20)], tol=1.5)


def test_tol_never_reaches_a_callback(monkeypatch):
    A, b, x0 = _problem()
    seen = {}

    class FakeSession:
        def set_jacobi(self, dinv):
            pass

    def fake_stepwise(sess, tag, A, b, x0, max_iter, x_true, dev_hist, generic, output, extra, path,
                      w_replace=None, plan=None, tol=0.0):
        seen["extra"] = dict(extra)
        seen["tol"] = tol
        return {"stop_iter": 4}

    monkeypatch.setattr(cg_variants, "_session_for", lambda *a: FakeSession())
    monkeypatch.setattr(cg_variants, "_solve_stepwise", fake_stepwise)
    out = cg_variants.pr_pcg(A, b, x0, 20, callbacks=[lambda **kw: None], tol=1e-6, other=3)
    assert "tol" not in seen["extra"] and seen["extra"]["other"] == 3
    assert seen["tol"] == 1e-6
    assert out["stop_iter"] == 4
