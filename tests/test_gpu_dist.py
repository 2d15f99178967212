"""GPU (-m gpu): the row-partitioned multi-GPU protocol (z-slabs, peer-to-peer halo planes,
rank-ordered scalar exchange) exercised on ONE GPU with `GroupSession`: the ranks are
contexts sharing a stream and run the very kernels of a multi-process run, stage by stage.
A real 2-GPU run of the same partition (tests/dist_worker.py under torchrun) must return
the same bits; it runs when two devices are visible."""
import os
import subprocess
import sys

import numpy as np
import pytest

import helpers
from helpers import orc
from new_cg_variants_b200 import PoissonStencil, Session
from new_cg_variants_b200.dist import GroupSession

pytestmark = pytest.mark.gpu
ALL_TAGS = list(orc.VARIANTS)


def _problem(S):
    n = S.shape[0]
    x_true = np.ones(n) / np.sqrt(n)
    return x_true, S @ x_true, np.zeros(n)


@pytest.mark.parametrize("shape,world", [((16, 12, 8), 2), ((130, 10, 9), 3), ((258, 9, 12), 4),
                                         ((20, 18, 16), 8), ((64, 1, 40), 4), ((7, 6, 10), 2),
                                         ((32, 6, 3), 3), ((128, 8, 5), 4)])       # one-plane slabs too
def test_partitioned_run_matches_single_gpu(shape, world):
    """Every variant, Jacobi and identity: histories of the G-slab run agree with the
    single-context run to rounding over the first iterations (only the summation order of
    the dots differs: per-rank partials added in rank order), x likewise; all ranks hold
    identical histories (checked inside GroupSession.solve); runs are bitwise repeatable."""
    nx, ny, nz = shape
    S = PoissonStencil(nx, ny, nz, dim=3)
    x_true, b, x0 = _problem(S)
    n = S.shape[0]
    for dinv in (1 / S.diagonal(), None, 1 / (S.diagonal() + np.arange(n) % 3)):
        grp = GroupSession(S, world, dinv=dinv)
        one = Session(S, dinv=dinv)
        try:
            for tag in ALL_TAGS:
                xg, hg, infos = grp.solve(tag, b, x0, 14, x_true=x_true)
                xg2, hg2, _ = grp.solve(tag, b, x0, 14, x_true=x_true)
                x1, h1, _ = one.solve(tag, b, x0, 14, x_true=x_true, path="stream")
                assert all(i["kernel_launches"] > 0 for i in infos)
                np.testing.assert_allclose(xg, x1, rtol=1e-9, atol=1e-13, err_msg=f"{shape}x{world}/{tag}")
                assert np.array_equal(xg, xg2)
                for h in orc.HISTORIES:
                    np.testing.assert_allclose(hg[h][:10], h1[h][:10], rtol=1e-10, err_msg=f"{shape}x{world}/{tag}/{h}")
                    assert np.array_equal(hg[h], hg2[h], equal_nan=True)
        finally:
            grp.close()
            one.close()


def test_partitioned_run_parity_with_oracle():
    """The parity rule of tests/helpers.py on a partitioned run (poisson3d_12 fixture, 3 slabs)."""
    case = "poisson3d_12_jacobi"
    A, b, x0, x_true, dinv, max_iter = helpers.case_problem(case)
    S = PoissonStencil(12, 12, 12, dim=3)
    assert (S.tocsr() != A).nnz == 0
    bands = helpers.cases()[case]["kstar"]
    grp = GroupSession(S, 3, dinv=dinv)
    try:
        for tag in ALL_TAGS:
            _, dev, _ = grp.solve(tag, b, x0, max_iter, x_true=x_true)
            live = orc.solve(tag, A, b, x0, max_iter, dinv=dinv, x_true=x_true)
            helpers.check_parity(dev, live, bands[tag], f"{case}/{tag} x3 slabs")
    finally:
        grp.close()


def test_resume_and_scalars_in_partitioned_run():
    S = PoissonStencil(16, 16, 16, dim=3)
    x_true, b, x0 = _problem(S)
    grp = GroupSession(S, 4, dinv=1 / S.diagonal())
    try:
        _, h_one, _ = grp.solve("pipe_pr", b, x0, 30, x_true=x_true)
        grp.load_problem(b, x0, x_true)
        grp.begin("pipe_pr", 30, orc.HISTORIES)
        for chunk in (1, 2, 9, 100):
            grp.advance(chunk)
        sc = [m.scalars() for m in grp.members]
        assert all(s == sc[0] for s in sc)           # identical bits on every rank
        _, hh = grp.members[0].fetch_local()
        for i, h in enumerate(orc.HISTORIES):
            assert np.array_equal(hh[i], h_one[h], equal_nan=True)
    finally:
        grp.close()


def test_two_processes_two_gpus_match_emulation():
    """torchrun, one rank per GPU (CUDA IPC windows, NVLink stores): same bits as the
    single-GPU emulation.  Needs two visible devices; otherwise only the emulation ran."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two visible GPUs: one GPU runs the emulation only")
    worker = os.path.join(os.path.dirname(__file__), "dist_worker.py")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                          "--master-addr", "127.0.0.1", "--master-port", "29571", worker, "--check"],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "dist_worker ok" in out.stdout


@pytest.mark.parametrize("shape,world", [((16, 12, 8), 2), ((64, 10, 9), 3), ((20, 18, 16), 8), ((64, 64, 16), 4),
                                         ((32, 6, 3), 3)])
def test_partitioned_persistent_kernel(shape, world):
    """The persistent kernel on a partition: all ranks inside ONE cooperative launch (CTA range
    r*nb..(r+1)*nb-1 acts as rank r; windows, ghost planes and flags as between GPUs).  Against
    the stream path of the same partition: rounding-level agreement; bitwise repeatable;
    resumable; histories identical on every rank."""
    nx, ny, nz = shape
    S = PoissonStencil(nx, ny, nz, dim=3)
    x_true, b, x0 = _problem(S)
    n = S.shape[0]
    for dinv in (1 / S.diagonal(), 1 / (S.diagonal() + np.arange(n) % 3), None):
        grp = GroupSession(S, world, dinv=dinv)
        try:
            for tag in ALL_TAGS:
                xs, hs, _ = grp.solve(tag, b, x0, 14, x_true=x_true, path="stream")
                xp, hp, infos = grp.solve(tag, b, x0, 14, x_true=x_true, path="persistent")
                xp2, hp2, _ = grp.solve(tag, b, x0, 14, x_true=x_true, path="persistent")
                assert infos[0]["path"] == 2
                np.testing.assert_allclose(xp, xs, rtol=1e-9, atol=1e-13, err_msg=f"{shape}x{world}/{tag}")
                assert np.array_equal(xp, xp2)
                for h in orc.HISTORIES:
                    np.testing.assert_allclose(hp[h][:10], hs[h][:10], rtol=1e-10, err_msg=f"{shape}x{world}/{tag}/{h}")
                    assert np.array_equal(hp[h], hp2[h], equal_nan=True)
            # no instrumentation (the timed configuration) and a run cut into pieces
            grp.load_problem(b, x0, x_true)
            grp.begin("pipe_pr", 40, (), path="persistent")
            grp.advance(39)
            x_one = np.concatenate([m.fetch_local(want_hist=False)[0] for m in grp.members])
            grp.begin("pipe_pr", 40, (), path="persistent")
            for chunk in (1, 5, 33):
                grp.advance(chunk)
            x_cut = np.concatenate([m.fetch_local(want_hist=False)[0] for m in grp.members])
            assert np.array_equal(x_one, x_cut)
            sc = [m.scalars() for m in grp.members]
            assert all(s == sc[0] for s in sc)
        finally:
            grp.close()


@pytest.mark.parametrize("shape,world", [((16, 12, 8), 2), ((130, 10, 9), 3), ((258, 9, 12), 4), ((20, 18, 16), 8),
                                         ((32, 6, 3), 3), ((128, 8, 5), 4), ((256, 16, 24), 2)])
def test_partitioned_pr_fused_equals_two_kernel_path(shape, world):
    """PR-CG / M-CG on a partition run the single-launch kernel too (ghost planes of p, s, r~ as LL
    words, polled by the compute warps; boundary planes pushed the moment they are computed).
    After one loop trip x equals the partitioned two-kernel path BIT FOR BIT; afterwards only the
    summation order of the dots differs."""
    nx, ny, nz = shape
    S = PoissonStencil(nx, ny, nz, dim=3)
    x_true, b, x0 = _problem(S)
    for dinv in (1 / S.diagonal(), None):
        res = {}
        for fused in (1, 0):
            grp = GroupSession(S, world, dinv=dinv)
            try:
                for m in grp.members:
                    m.set_option("pr_fused", fused)
                    m.set_option("fused_min_slab", 1)          # (thin test slabs: force the fused kernel)
                for tag in ("pr", "m"):
                    x1, _, infos = grp.solve(tag, b, x0, 2, x_true=x_true)
                    xk, hk, infos = grp.solve(tag, b, x0, 16, x_true=x_true)
                    xk2, hk2, _ = grp.solve(tag, b, x0, 16, x_true=x_true)
                    assert np.array_equal(xk, xk2)
                    res[(fused, tag)] = (x1, xk, hk, sum(i["kernel_launches"] for i in infos))
            finally:
                grp.close()
        for tag in ("pr", "m"):
            f, t = res[(1, tag)], res[(0, tag)]
            assert f[3] < t[3], "the fused kernel did not run"
            assert np.array_equal(f[0], t[0]), (shape, world, tag)
            np.testing.assert_allclose(f[1], t[1], rtol=1e-9, atol=1e-13)
            for h in orc.HISTORIES:
                np.testing.assert_allclose(f[2][h][:12], t[2][h][:12], rtol=1e-10, err_msg=f"{shape}x{world}/{tag}/{h}")


def _csr_cases():
    import scipy.sparse as sps
    from new_cg_variants_b200.experiments import banded_model_problem
    from new_cg_variants_b200.cg_variants_mpi4py import model_problem
    return {
        "bcsstk16": helpers.load_matrix("bcsstk16"),                       # ghost entries from several ranks
        "1138_bus": helpers.load_matrix("1138_bus"),
        "banded": banded_model_problem(n=3000, k=7)[0],                    # the PETSc driver's matrix, small
        "model_diag": model_problem(1536)[0],                              # scaling_tests.py:31-53: no ghosts at all
        "poisson2d_24": orc.poisson2d(24),
    }


@pytest.mark.parametrize("name", ["bcsstk16", "1138_bus", "banded", "model_diag", "poisson2d_24"])
@pytest.mark.parametrize("world", [2, 3, 8])
def test_general_csr_row_partition_matches_single_gpu(name, world):
    """SURVEY.md section 8e "General CSR": contiguous row blocks, ghost entries gathered through
    per-neighbour index lists into staging arrays, rank-ordered scalar exchange.  Every variant
    against the single-context run: the row sums are bit-identical (same stored order), the dots
    are summed per rank then in rank order -> agreement to rounding; all ranks hold identical
    histories; bitwise repeatable."""
    A = _csr_cases()[name]
    x_true, b, x0 = orc.setup_problem(A)
    for dinv in (orc.jacobi_dinv(A), None):
        grp = GroupSession(A, world, dinv=dinv)
        one = Session(A, dinv=dinv)
        try:
            for tag in ALL_TAGS:
                xg, hg, infos = grp.solve(tag, b, x0, 12, x_true=x_true)
                xg2, hg2, _ = grp.solve(tag, b, x0, 12, x_true=x_true)
                x1, h1, _ = one.solve(tag, b, x0, 12, x_true=x_true, path="stream")
                assert all(i["kernel_launches"] > 0 and i["path"] == 1 for i in infos)
                np.testing.assert_allclose(xg, x1, rtol=1e-8, atol=1e-12 * np.abs(x1).max(), err_msg=f"{name}x{world}/{tag}")
                assert np.array_equal(xg, xg2)
                for h in orc.HISTORIES:
                    # (the banded / diagonal model problems converge to rounding level within a few
                    # iterations: absolute floor relative to the k = 0 entry)
                    np.testing.assert_allclose(hg[h][:8], h1[h][:8], rtol=1e-10, atol=1e-12 * h1[h][0],
                                               err_msg=f"{name}x{world}/{tag}/{h}")
                    assert np.array_equal(hg[h], hg2[h], equal_nan=True)
        finally:
            grp.close()
            one.close()


def test_csr_partition_parity_with_oracle():
    """The parity rule on a CSR row partition (bcsstk15 + Jacobi fixture, 4 row blocks)."""
    case = "bcsstk15_jacobi"
    A, b, x0, x_true, dinv, max_iter = helpers.case_problem(case)
    bands = helpers.cases()[case]["kstar"]
    grp = GroupSession(A, 4, dinv=dinv)
    try:
        for tag in ("hs", "pr", "pipe_pr", "gv"):
            _, dev, _ = grp.solve(tag, b, x0, max_iter, x_true=x_true)
            live = orc.solve(tag, A, b, x0, max_iter, dinv=dinv, x_true=x_true)
            helpers.check_parity(dev, live, bands[tag], f"{case}/{tag} x4 row blocks")
    finally:
        grp.close()
