"""CPU: argument checks of the batch entry point and of its Python wrappers, before any device work."""
import ctypes as C

import numpy as np
import pytest

import helpers
from new_cg_variants_b200 import _lib, callbacks as cbk, cg_variants, experiments as ex

STD = [cbk.error_A_norm, cbk.residual_2_norm, cbk.error_2_norm, cbk.updated_residual_2_norm]


def test_batch_run_rejects_bad_arguments():
    lib = _lib.load()
    info = (_lib.CgxInfo * 1)()
    v = np.zeros(1, dtype=np.int32)
    it = np.full(1, 10, dtype=np.int32)
    assert lib.cgx_batch_run(None, 0, None, None, 0, None) == _lib.ERR_ARG
    assert lib.cgx_batch_run(None, 1, _lib.iptr(v), _lib.iptr(it), 0, info) == _lib.ERR_ARG
    ctxs = (C.c_void_p * 1)(None)
    assert lib.cgx_batch_run(ctxs, 1, _lib.iptr(v), _lib.iptr(it), 0, info) == _lib.ERR_ARG
    assert b"cgx_batch_run" in lib.cgx_last_error()


def _problem():
    A = helpers.load_matrix("nos4")
    x_true = np.ones(A.shape[0]) / np.sqrt(A.shape[0])
    return A, A @ x_true, np.zeros(A.shape[0]), x_true


def _user_callback(**kw):
    pass


@pytest.mark.parametrize("how", ["generic", "capture", "w_replace", "path", "session", "foreign_method"])
def test_solve_concurrently_refuses_what_a_batch_cannot_serve(how):
    A, b, x0, x_true = _problem()
    methods = [cg_variants.hs_pcg, cg_variants.gv_pcg]
    callbacks, kw = list(STD), {}
    if how == "generic":
        callbacks.append(_user_callback)
    elif how == "capture":
        callbacks.append(cbk.save_x)
    elif how == "w_replace":
        kw["w_replace"] = lambda **k: k["k"] == 3
    elif how == "path":
        kw["path"] = "stream"
    elif how == "session":
        kw["session"] = object()
    else:
        methods.append(_user_callback)
    with pytest.raises(NotImplementedError):
        cg_variants.solve_concurrently(methods, A, b, x0, 20, callbacks=callbacks, x_true=x_true, **kw)


def test_test_matrix_concurrent_refuses_the_same_way(tmp_path):
    A, _, _, _ = _problem()
    with pytest.raises(NotImplementedError):
        ex.test_matrix(A, 20, "nos4", variants=[cg_variants.hs_pcg, _user_callback], data_dir=str(tmp_path),
                       concurrent=True)
    with pytest.raises(NotImplementedError):
        ex.test_matrix(A, 20, "nos4", variants=ex.ALL_METHODS, data_dir=str(tmp_path), concurrent=True, path="stream")
