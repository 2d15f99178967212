"""CPU: the tolerance arguments of the partitioned sessions and of the mpi4py-shaped solvers, checked
before any device work."""
import inspect
import math

import numpy as np
import pytest

from new_cg_variants_b200 import cg_variants_mpi4py as mp
from new_cg_variants_b200.dist import DistSession, GroupSession

BAD = [-1.0, 1.0, 2, math.nan, math.inf]


@pytest.mark.parametrize("tol", BAD)
def test_group_session_validates_tol_before_the_device(tol):
    g = object.__new__(GroupSession)      # no contexts: any use of them would fail differently
    b = np.ones(8)
    with pytest.raises(ValueError):
        g.begin("pr", 20, tol=tol)
    with pytest.raises(ValueError):
        g.solve("cg", b, np.zeros(8), 20, tol=tol)


@pytest.mark.parametrize("tol", BAD)
def test_dist_session_validates_tol_before_the_device(tol):
    d = object.__new__(DistSession)
    b = np.ones(8)
    with pytest.raises(ValueError):
        d.run("pr", 20, tol=tol)
    with pytest.raises(ValueError):
        d.solve_local("hs", b, np.zeros(8), 20, tol=tol)
    with pytest.raises(ValueError):
        d.solve("pipe_pr", b, np.zeros(8), 20, tol=tol)


def test_partition_sessions_take_tol():
    for fn in (GroupSession.begin, GroupSession.solve, DistSession.run, DistSession.solve, DistSession.solve_local):
        p = inspect.signature(fn).parameters["tol"]
        assert p.default is None and p.kind == p.POSITIONAL_OR_KEYWORD, fn.__qualname__


@pytest.mark.parametrize("name", ["hs_cg", "cg_cg", "gv_cg", "pr_cg", "pipe_pr_cg"])
def test_mpi4py_signatures(name):
    assert list(inspect.signature(getattr(mp, name)).parameters) == ["comm", "A", "b", "max_iter"]
    assert list(inspect.signature(mp.solve_to_tol).parameters) == ["name", "comm", "A", "b", "max_iter", "tol"]
    assert name in mp.SOLVERS


class _Comm:
    def Get_size(self):
        return 1

    def Get_rank(self):
        return 0

    def Barrier(self):
        pass


class _FakeSession:
    def __init__(self):
        self.tols = []

    def load_problem(self, b, x0, xt):
        pass

    def run(self, tag, max_iter, histories=(), tol=None):
        self.tols.append(tol)
        return {"stop_iter": 7 if tol is not None else -1}

    def fetch(self, want_hist=True):
        return np.zeros(4), None


@pytest.mark.parametrize("name", ["hs_cg", "cg_cg", "gv_cg", "pr_cg", "pipe_pr_cg"])
def test_mpi4py_times_gain_stop_iter_only_with_tol(name, monkeypatch):
    fake = _FakeSession()
    monkeypatch.setattr(mp, "_operator_session", lambda comm, A, m: fake)
    _, times = getattr(mp, name)(_Comm(), None, np.ones(4), 10)
    assert set(times) == {'tot', 'c_ip', 'c_mv', 'w_mv', 'w_ip', 'w_vec'}
    _, times = mp.solve_to_tol(name, _Comm(), None, np.ones(4), 10, 1e-8)
    assert times["stop_iter"] == 7
    assert fake.tols == [None, 1e-8]


@pytest.mark.parametrize("tol", BAD + [None])
def test_mpi4py_validates_tol_before_the_device(tol, monkeypatch):
    def no_device(*a, **k):
        raise AssertionError("a session was requested before tol was checked")

    monkeypatch.setattr(mp, "_operator_session", no_device)
    with pytest.raises(ValueError):
        mp.solve_to_tol("pr_cg", _Comm(), None, np.ones(4), 10, tol)
    with pytest.raises(ValueError):
        mp.solve_to_tol("exact_cg", _Comm(), None, np.ones(4), 10, 1e-8)
