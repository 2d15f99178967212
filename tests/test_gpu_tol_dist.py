"""GPU: stopping a partitioned solve at a relative tolerance (z-slabs and CSR row partitions), exercised
with the single-GPU emulation of the protocol (GroupSession: the ranks are contexts on one device).

The contract: every rank stops at the same k = stop, the first k >= 1 with nu_k <= tol^2 nu_0 (nu: the
all-rank total), and then holds, bit for bit, what the same partition (same world, path and options)
run without a tolerance and with max_iter = stop + 1 holds: its slice of x, its state vectors, its
scalars, and history entries 0 .. stop (later entries are zero)."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import helpers
from helpers import orc
from new_cg_variants_b200 import PoissonStencil, _lib
from new_cg_variants_b200.dist import GroupSession

pytestmark = pytest.mark.gpu

ALL_TAGS = list(orc.VARIANTS)
VECS = ("x", "r", "rt", "p", "s")


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def _same(a, b, label):
    assert np.array_equal(_bits(a), _bits(b)), label


def _problem(A):
    n = A.shape[0]
    x_true = np.ones(n) / np.sqrt(n)
    return x_true, A @ x_true, np.zeros(n)


def _state(m):
    out = {}
    for v in VECS:
        a = np.empty(m.n)
        _lib.check(m._lib.cgx_fetch_vector_host(m._ctx, v.encode(), _lib.dptr(a)))
        out[v] = a
    return out


def _full_hist(grp, max_iter):
    """every rank's (4, max_iter) history rows of the last run (not cut at the stop)"""
    out = []
    for m in grp.members:
        m._max_iter = max_iter
        out.append(m.fetch_local(want_x=False)[1])
    return out


# the scalars a variant's recurrences keep (the others hold initialisation scratch of earlier runs)
USED = {"hs": ("a", "a1", "b", "nu", "nu1", "mu"), "cg": ("a", "a1", "b", "nu", "nu1", "mu", "eta")}
USED["gv"] = USED["cg"]


def _scalars(m, tag):
    s = m.scalars()
    return {k: s[k] for k in USED.get(tag, ("a", "a1", "b", "nu", "nu1", "mu", "delta", "gamma"))}


def check_contract(grp, tag, b, x0, xt, max_iter, path, tol, label):
    """Tolerance run against the same group without one at max_iter = stop + 1; returns stop."""
    x, hist, infos = grp.solve(tag, b, x0, max_iter, x_true=xt, path=path, tol=tol)
    stops = {i["stop_iter"] for i in infos}
    assert len(stops) == 1, f"{label}: ranks disagree on the stop: {stops}"
    stop = stops.pop()
    assert 1 <= stop < max_iter - 1, f"{label}: tol {tol} not reached in {max_iter} iterations"
    assert all(i["iterations"] == stop for i in infos), label
    assert all(i["path"] == (1 if path == "stream" else 2) for i in infos), label
    full = _full_hist(grp, max_iter)
    for h in full:
        assert not np.any(h[:, stop + 1:]), f"{label}: history entries after the stop"
    sc = [_scalars(m, tag) for m in grp.members]
    st = [_state(m) for m in grp.members]
    assert all(s == sc[0] for s in sc), label
    # the reference: the same partition, no tolerance, max_iter = stop + 1
    xr, hr, infr = grp.solve(tag, b, x0, stop + 1, x_true=xt, path=path)
    assert all(i["stop_iter"] == -1 and i["iterations"] == stop for i in infr), label
    _same(x, xr, f"{label}: x")
    for r, m in enumerate(grp.members):
        assert _scalars(m, tag) == sc[r], f"{label}: scalars of rank {r}"
        for v, a in _state(m).items():
            _same(st[r][v], a, f"{label}: {v} of rank {r}")
    assert set(hist) == set(hr), label
    for h in hr:
        assert len(hist[h]) == stop + 1, label
        _same(hist[h], hr[h], f"{label}: {h}")
    return stop


SLAB_CASES = [((16, 12, 8), 2), ((130, 10, 9), 3), ((64, 1, 40), 4)]


def _dinvs(S):
    n = S.shape[0]
    return {"jacobi": 1 / (S.diagonal() + np.arange(n) % 3), "const": 1 / S.diagonal(), "none": None}


@pytest.mark.parametrize("tma", [1, 0])
@pytest.mark.parametrize("shape,world", SLAB_CASES)
def test_slab_partition_stops_at_the_prefix(shape, world, tma):
    """All nine variants on z-slabs (TMA stencil and generic stencil kernels), three preconditioners."""
    S = PoissonStencil(*shape, dim=3)
    xt, b, x0 = _problem(S)
    for pname, dinv in _dinvs(S).items():
        grp = GroupSession(S, world, dinv=dinv)
        try:
            for m in grp.members:
                m.set_option("tma", tma)
            for tag in ALL_TAGS:
                check_contract(grp, tag, b, x0, xt, 400, "stream", 1e-6, f"{shape}x{world}/{pname}/tma{tma}/{tag}")
        finally:
            grp.close()


def _csr_cases():
    from new_cg_variants_b200.experiments import banded_model_problem
    return {
        "bcsstk16": (lambda: helpers.load_matrix("bcsstk16"), True, 1e-5, 3000),
        "1138_bus": (lambda: helpers.load_matrix("1138_bus"), True, 1e-4, 4000),
        "banded": (lambda: banded_model_problem(n=3000, k=7)[0], False, 1e-6, 3000),
    }


@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("name", ["bcsstk16", "1138_bus", "banded"])
def test_csr_partition_stops_at_the_prefix(name, world):
    make, prec, tol, max_iter = _csr_cases()[name]
    A = make()
    xt, b, x0 = _problem(A)
    grp = GroupSession(A, world, dinv=(1 / A.diagonal()) if prec else None)
    try:
        for tag in ALL_TAGS:
            check_contract(grp, tag, b, x0, xt, max_iter, "stream", tol, f"{name}x{world}/{tag}")
    finally:
        grp.close()


@pytest.mark.parametrize("dinv_kind", ["const", "none"])
def test_fused_pr_kernel_on_a_partition_stops_at_the_prefix(dinv_kind):
    """PR-CG / M-CG through pr_fused_kernel<..., DIST>: its producer warp waits for the stop decision."""
    S = PoissonStencil(256, 16, 24, dim=3)
    xt, b, x0 = _problem(S)
    grp = GroupSession(S, 2, dinv=_dinvs(S)[dinv_kind])
    try:
        for m in grp.members:
            m.set_option("fused_min_slab", 1)
            m.set_profile(True)
        for tag in ("pr", "m"):
            check_contract(grp, tag, b, x0, xt, 600, "stream", 1e-6, f"fused/{dinv_kind}/{tag}")
            assert all("pr_fused" in m.get_profile() for m in grp.members), "the fused kernel did not run"
    finally:
        grp.close()


@pytest.mark.parametrize("shape,world", [((16, 12, 8), 2), ((64, 64, 16), 4)])
def test_persistent_path_on_slabs_stops_at_the_prefix(shape, world):
    S = PoissonStencil(*shape, dim=3)
    xt, b, x0 = _problem(S)
    for pname, dinv in _dinvs(S).items():
        grp = GroupSession(S, world, dinv=dinv)
        try:
            for tag in ALL_TAGS:
                check_contract(grp, tag, b, x0, xt, 400, "persistent", 1e-6, f"pers/{shape}x{world}/{pname}/{tag}")
        finally:
            grp.close()


@pytest.mark.parametrize("path", ["stream", "persistent"])
def test_stop_is_the_first_crossing_on_every_rank(path):
    """Step the no-tolerance group one iteration at a time and find the first k >= 1 with
    nu_k <= tol^2 nu_0 from the scalars: the tolerance run stops exactly there, on every rank."""
    S = PoissonStencil(16, 12, 8, dim=3)
    xt, b, x0 = _problem(S)
    tol = 1e-6
    grp = GroupSession(S, 2, dinv=1 / S.diagonal())
    try:
        for tag in ALL_TAGS:
            _, _, infos = grp.solve(tag, b, x0, 400, path=path, tol=tol)
            stop = infos[0]["stop_iter"]
            assert all(i["stop_iter"] == stop for i in infos)
            grp.load_problem(b, x0)
            grp.begin(tag, 400, path=path)
            nu0 = grp.members[0].scalars()["nu"]
            thr = (tol * tol) * nu0
            first = -1
            for k in range(1, 399):
                grp.advance(1)
                nus = [m.scalars()["nu"] for m in grp.members]
                assert all(v == nus[0] for v in nus)
                if nus[0] <= thr:
                    first = k
                    break
            assert first == stop, f"{tag}/{path}: stopped at {stop}, first crossing at {first}"
    finally:
        grp.close()


def test_tolerance_never_met_gives_the_run_without_one():
    S = PoissonStencil(130, 10, 9, dim=3)
    xt, b, x0 = _problem(S)
    grp = GroupSession(S, 3, dinv=1 / S.diagonal())
    try:
        for path in ("stream", "persistent"):
            for tag in ALL_TAGS:
                x1, h1, i1 = grp.solve(tag, b, x0, 40, x_true=xt, path=path, tol=1e-150)
                sc1 = [_scalars(m, tag) for m in grp.members]
                x2, h2, i2 = grp.solve(tag, b, x0, 40, x_true=xt, path=path)
                assert all(i["stop_iter"] == -1 and i["iterations"] == 39 for i in i1 + i2)
                _same(x1, x2, f"{tag}/{path}")
                assert [_scalars(m, tag) for m in grp.members] == sc1
                for h in h2:
                    _same(h1[h], h2[h], f"{tag}/{path}/{h}")
    finally:
        grp.close()


@pytest.mark.parametrize("path", ["stream", "persistent"])
def test_stepping_across_the_stop_and_reuse(path):
    """begin + advance in pieces across the stop, advances after it, then solves without a tolerance on
    the same group equal a fresh group bit for bit (no epoch or scalar-parity drift)."""
    S = PoissonStencil(64, 64, 16, dim=3) if path == "persistent" else PoissonStencil(130, 10, 9, dim=3)
    world = 4 if path == "persistent" else 3
    xt, b, x0 = _problem(S)
    tol = 1e-6
    grp = GroupSession(S, world, dinv=1 / S.diagonal())
    try:
        for tag in ALL_TAGS:
            xs, hs, infos = grp.solve(tag, b, x0, 400, x_true=xt, path=path, tol=tol)
            stop = infos[0]["stop_iter"]
            assert stop > 40, f"{tag}: the pieces below should cross chunk boundaries before the stop"
            sc = [_scalars(m, tag) for m in grp.members]
            grp.load_problem(b, x0, xt)
            grp.begin(tag, 400, orc.HISTORIES, path=path, tol=tol)
            done = 0
            for chunk in (1, 5, 33, 7, 100, 300, 50, 1):
                grp.advance(chunk)
                done = min(done + chunk, stop)
                infos = [m.get_info() for m in grp.members]
                assert all(i["iterations"] == done for i in infos), (tag, chunk)
                assert all(i["stop_iter"] == (stop if done == stop else -1) for i in infos), (tag, chunk)
            x = np.concatenate([m.fetch_local(want_hist=False)[0] for m in grp.members])
            _same(x, xs, f"{tag}: x after stepping")
            assert [_scalars(m, tag) for m in grp.members] == sc, tag
            hh = _full_hist(grp, 400)[0]
            for i, h in enumerate(orc.HISTORIES):
                _same(hh[i][:stop + 1], hs[h], f"{tag}: {h} after stepping")
            # a later solve without a tolerance on these contexts: the bits of fresh contexts
            xa, ha, _ = grp.solve(tag, b, x0, 60, x_true=xt, path=path)
            fresh = GroupSession(S, world, dinv=1 / S.diagonal())
            try:
                xf, hf, _ = fresh.solve(tag, b, x0, 60, x_true=xt, path=path)
                scf = [_scalars(m, tag) for m in fresh.members]
            finally:
                fresh.close()
            _same(xa, xf, f"{tag}: reuse after a stop")
            assert [_scalars(m, tag) for m in grp.members] == scf, tag
            for h in hf:
                _same(ha[h], hf[h], f"{tag}: {h} on reuse")
    finally:
        grp.close()


def test_refusals():
    lib = _lib.load()
    A = helpers.load_matrix("bcsstk16")
    xt, b, x0 = _problem(A)
    grp = GroupSession(A, 3, dinv=1 / A.diagonal())
    try:
        grp.load_problem(b, x0, xt)
        # tolerances that differ between the ranks of one group
        for r, t in enumerate((1e-6, 1e-6, 1e-5)):
            assert lib.cgx_set_tolerance(grp.members[r]._ctx, t) == _lib.OK
        assert lib.cgx_group_begin(grp._arr, 3, _lib.VARIANT_IDS["cg"], 50, 0, _lib.PATHS["stream"]) == _lib.ERR_UNSUPPORTED
        assert b"partition" in lib.cgx_last_error()
        # the timing stand-in for the allreduce: the ranks' nu differ by construction
        for m in grp.members:
            m.set_option("stub_allreduce", 1)
        with pytest.raises(_lib.CgxError) as e:
            grp.begin("cg", 50, tol=1e-6)
        assert e.value.code == _lib.ERR_UNSUPPORTED
        for m in grp.members:
            m.set_option("stub_allreduce", 0)
        # the same group then runs, with and without a tolerance
        _, _, infos = grp.solve("cg", b, x0, 3000, tol=1e-5)
        assert infos[0]["stop_iter"] > 0
        _, _, infos = grp.solve("cg", b, x0, 20)
        assert all(i["stop_iter"] == -1 for i in infos)
    finally:
        grp.close()


def test_two_processes_two_gpus_match_emulation_with_a_tolerance():
    """torchrun, one rank per GPU (CUDA IPC windows): the same stop and the same bits as the emulation,
    on slabs and on a CSR row partition; NCCL exchange with a tolerance is refused."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two visible GPUs: one GPU runs the emulation only")
    worker = os.path.join(os.path.dirname(__file__), "dist_tol_worker.py")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                          "--master-addr", "127.0.0.1", "--master-port", "29573", worker],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "dist_tol_worker ok" in out.stdout
