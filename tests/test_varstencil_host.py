"""CPU: VariableStencil's host surface (matvec, tocsr, validation) and the refusals raised
before any device work (partitions, batches, concurrent solves)."""
import ctypes as C
import re

import numpy as np
import pytest
import scipy.sparse as sps

import helpers
from new_cg_variants_b200 import PoissonStencil, VariableStencil, _lib, cg_variants, cg_variants_mpi4py
from new_cg_variants_b200 import session as session_mod


def random_coefs(nx, ny, nz, dim, seed=0, zero_frac=0.1):
    """Random positive / negative couplings with some interior zeros; off-grid couplings 0."""
    rng = np.random.default_rng(seed)
    n = nx * ny * nz
    shape = (nz, ny, nx)

    def coupling(last_axis):
        c = rng.standard_normal(shape)
        c[rng.random(shape) < zero_frac] = 0.0
        idx = [slice(None)] * 3
        idx[last_axis] = -1
        c[tuple(idx)] = 0.0
        return c.reshape(-1)

    cx, cy = coupling(2), coupling(1)
    cz = coupling(0) if dim == 3 else None
    diag = 6.0 + rng.random(n)
    return diag, cx, cy, cz


SHAPES = [(2, 7, 5, 1), (2, 1, 9, 1), (2, 13, 1, 1), (2, 1, 1, 1),
          (3, 5, 4, 3), (3, 7, 1, 4), (3, 1, 6, 5), (3, 9, 3, 1), (3, 6, 6, 6)]


@pytest.mark.parametrize("dim,nx,ny,nz", SHAPES)
def test_matvec_is_bitwise_tocsr(dim, nx, ny, nz):
    diag, cx, cy, cz = random_coefs(nx, ny, nz, dim, seed=nx * 100 + ny * 10 + nz)
    S = VariableStencil(nx, ny, nz, diag, cx, cy, cz)
    assert S.dim == dim and S.shape == (nx * ny * nz,) * 2
    A = S.tocsr()
    assert A.has_canonical_format and A.nnz == S.nnz
    assert A.indices.dtype == np.int32 and A.indptr.dtype == np.int32
    assert (abs(A - A.T)).nnz == 0                       # symmetric
    assert np.array_equal(A.diagonal(), S.diagonal())
    rng = np.random.default_rng(1)
    for v in (rng.standard_normal(S.shape[0]), np.ones(S.shape[0]), rng.integers(-3, 4, S.shape[0]).astype(float)):
        assert np.array_equal(S @ v, A @ v)
        assert np.array_equal(S.matvec(v), A @ v)


def test_tocsr_keeps_the_full_pattern_and_places_couplings():
    nx, ny, nz = 4, 3, 2
    diag, cx, cy, cz = random_coefs(nx, ny, nz, 3, seed=5, zero_frac=0.5)
    S = VariableStencil(nx, ny, nz, diag, cx, cy, cz)
    A = S.tocsr().toarray()
    P = PoissonStencil(nx, ny, nz, dim=3).tocsr()
    assert S.tocsr().nnz == P.nnz                         # explicit zeros inside the grid are stored
    for i in range(nx * ny * nz):
        x, y, z = i % nx, (i // nx) % ny, i // (nx * ny)
        if x < nx - 1:
            assert A[i, i + 1] == cx[i] and A[i + 1, i] == cx[i]
        if y < ny - 1:
            assert A[i, i + nx] == cy[i] and A[i + nx, i] == cy[i]
        if z < nz - 1:
            assert A[i, i + nx * ny] == cz[i] and A[i + nx * ny, i] == cz[i]


@pytest.mark.parametrize("dim,nx,ny,nz", [(2, 6, 5, 1), (3, 4, 5, 3), (3, 5, 1, 2)])
@pytest.mark.parametrize("d,off", [(4.0, -1.0), (6.0, -1.0), (2.5, 0.75)])
def test_constant_coefficients_equal_poisson(dim, nx, ny, nz, d, off):
    n = nx * ny * nz
    g = lambda a: a.reshape(nz, ny, nx)
    cx, cy = np.full(n, off), np.full(n, off)
    g(cx)[:, :, -1] = 0.0
    g(cy)[:, -1, :] = 0.0
    cz = None
    if dim == 3:
        cz = np.full(n, off)
        g(cz)[-1] = 0.0
    S = VariableStencil(nx, ny, nz, np.full(n, d), cx, cy, cz)
    P = PoissonStencil(nx, ny, nz, dim=dim, diag=d, off=off)
    A, B = S.tocsr(), P.tocsr()
    assert np.array_equal(A.indptr, B.indptr) and np.array_equal(A.indices, B.indices)
    assert np.array_equal(A.data, B.data)
    v = np.random.default_rng(2).standard_normal(n)
    assert np.array_equal(S @ v, P @ v)


def _ok(nx=4, ny=3, nz=2, dim=3):
    return random_coefs(nx, ny, nz, dim, seed=9)


def test_arrays_are_copied_and_read_only():
    diag, cx, cy, cz = _ok()
    S = VariableStencil(4, 3, 2, diag, cx, cy, cz)
    diag[0] = 123.0
    assert S.diag[0] != 123.0
    with pytest.raises(ValueError):
        S.cx[0] = 1.0


@pytest.mark.parametrize("case", ["short_diag", "long_cx", "short_cz", "nan_diag", "inf_cy", "nan_cz",
                                  "cx_off_grid", "cy_off_grid", "cz_off_grid", "dim2_with_cz", "dim2_nz2",
                                  "dim3_without_cz", "dim4", "zero_size"])
def test_validation_errors(case):
    nx, ny, nz = 4, 3, 2
    diag, cx, cy, cz = _ok()
    kw = dict(nx=nx, ny=ny, nz=nz, diag=diag.copy(), cx=cx.copy(), cy=cy.copy(), cz=cz.copy())
    g = lambda a: a.reshape(nz, ny, nx)
    if case == "short_diag":
        kw["diag"] = diag[:-1]
    elif case == "long_cx":
        kw["cx"] = np.concatenate([cx, [0.0]])
    elif case == "short_cz":
        kw["cz"] = cz[:5]
    elif case == "nan_diag":
        kw["diag"][3] = np.nan
    elif case == "inf_cy":
        kw["cy"][0] = np.inf
    elif case == "nan_cz":
        kw["cz"][0] = np.nan
    elif case == "cx_off_grid":
        g(kw["cx"])[1, 2, -1] = 0.5
    elif case == "cy_off_grid":
        g(kw["cy"])[0, -1, 1] = -0.5
    elif case == "cz_off_grid":
        g(kw["cz"])[-1, 0, 0] = 1.0
    elif case == "dim2_with_cz":
        kw.update(nz=1, diag=diag[:12], cx=g(cx)[0].reshape(-1), cy=g(cy)[0].reshape(-1), cz=cz[:12], dim=2)
    elif case == "dim2_nz2":
        kw.update(cz=None, dim=2)
    elif case == "dim3_without_cz":
        kw.update(cz=None, dim=3)
    elif case == "dim4":
        kw["dim"] = 4
    elif case == "zero_size":
        kw.update(nx=0, diag=np.zeros(0), cx=np.zeros(0), cy=np.zeros(0), cz=np.zeros(0))
    with pytest.raises(ValueError):
        VariableStencil(**kw)


def test_c_entry_point_is_declared_and_exported():
    with open(f"{helpers.ROOT}/include/cgx.h") as f:
        assert re.search(r"int cgx_set_stencil_coef_host\(cgx_ctx\* ctx, int dim, int64_t nx, int64_t ny, int64_t nz,\s*"
                         r"const double\* diag, const double\* cx, const double\* cy,\s*const double\* cz\);", f.read())
    lib = _lib.load()
    one = np.zeros(1)
    p = _lib.dptr(one)
    assert lib.cgx_set_stencil_coef_host(None, 2, 1, 1, 1, p, p, p, None) == _lib.ERR_ARG
    assert b"cgx_set_stencil_coef_host" in lib.cgx_last_error()


def _no_device(monkeypatch):
    def boom(*a, **k):
        raise AssertionError("a GPU context was requested before the refusal")
    monkeypatch.setattr(_lib, "load", boom)
    monkeypatch.setattr(cg_variants, "Session", boom)
    monkeypatch.setattr(cg_variants, "_session_for", boom)


def _small():
    diag, cx, cy, cz = _ok()
    S = VariableStencil(4, 3, 2, diag, cx, cy, cz)
    return S, S @ np.ones(S.shape[0]), np.zeros(S.shape[0])


def test_partitions_refuse_a_variable_stencil(monkeypatch):
    from new_cg_variants_b200 import dist
    S, b, _ = _small()
    _no_device(monkeypatch)
    with pytest.raises(NotImplementedError, match="VariableStencil"):
        dist.GroupSession(S, 2)
    with pytest.raises(NotImplementedError, match="VariableStencil"):
        dist.DistSession(S, rank=0, world=2)
    with pytest.raises(NotImplementedError, match="VariableStencil"):
        dist.CsrDistSession(S, rank=0, world=2)

    class Comm:
        def Get_size(self):
            return 1

        def Get_rank(self):
            return 0

        def Barrier(self):
            raise AssertionError("reached the communicator")

    for f in (cg_variants_mpi4py.hs_cg, cg_variants_mpi4py.pr_cg, cg_variants_mpi4py.pipe_pr_cg):
        with pytest.raises(NotImplementedError, match="VariableStencil"):
            f(Comm(), S, b, 10)
    with pytest.raises(NotImplementedError, match="VariableStencil"):
        cg_variants_mpi4py.solve_to_tol("pr_cg", Comm(), S, b, 10, 1e-6)


def test_batch_and_concurrent_refuse_a_variable_stencil(monkeypatch):
    S, b, x0 = _small()
    _no_device(monkeypatch)
    with pytest.raises(NotImplementedError, match="VariableStencil"):
        cg_variants.solve_concurrently([cg_variants.pr_cg, cg_variants.hs_cg], S, b, x0, 10)

    class FakeSession:                                   # what Session(VariableStencil) reports as its kind
        kind = "varstencil"
    with pytest.raises(NotImplementedError, match="VariableStencil"):
        session_mod.solve_batch([(FakeSession(), "pr", b, x0, 10)])


def test_operator_cache_keys_on_identity(monkeypatch):
    """Two operators of one shape with different coefficients never share a cached session."""
    made = []

    class FakeSession:
        def __init__(self, A, dinv=None, device=0):
            self.A, self._ctx = A, 1
            made.append(self)

        def set_jacobi(self, dinv):
            pass

        def close(self):
            self._ctx = None

    monkeypatch.setattr(cg_variants, "Session", FakeSession)
    cg_variants.clear_cache()
    try:
        d1, cx, cy, cz = _ok()
        S1 = VariableStencil(4, 3, 2, d1, cx, cy, cz)
        S2 = VariableStencil(4, 3, 2, d1 + 1.0, cx, cy, cz)
        a = cg_variants._session_for(S1, None, 0)
        b = cg_variants._session_for(S2, None, 0)
        assert a is not b and a.A is S1 and b.A is S2
        assert cg_variants._session_for(S1, None, 0) is a
        assert cg_variants._fingerprint(S1) == cg_variants._fingerprint(S2)   # same shape: identity decides
    finally:
        cg_variants._CACHE.clear()


def test_x_true_is_solved_on_tocsr():
    S, b, _ = _small()
    extra = {}
    cg_variants._ensure_x_true(S, b, extra, True)
    assert np.allclose(S @ extra["x_true"], b)
    assert np.array_equal(session_mod.diagonal_of(S), S.diag)
