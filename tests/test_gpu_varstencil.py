"""GPU (-m gpu): the variable-coefficient stencil (VariableStencil, cgx_set_stencil_coef_host).

SpMV bits against scipy on tocsr() for the TMA-staged and the generic kernel, all nine variants on
both execution paths against the oracle and against the CSR-path solve of the same matrix, the
tolerance contract, the drop-in surface with capture, the operator cache and the refusals."""
import ctypes as C

import numpy as np
import pytest

import helpers
from helpers import orc
from new_cg_variants_b200 import PoissonStencil, Session, VariableStencil, _lib, callbacks as cbk, cg_variants
from new_cg_variants_b200.session import solve_batch

pytestmark = pytest.mark.gpu

STD_CALLBACKS = [cbk.error_A_norm, cbk.residual_2_norm, cbk.error_2_norm, cbk.updated_residual_2_norm]
ALL_TAGS = list(orc.VARIANTS)


def make_var(nx, ny, nz, dim, seed=0, zero_frac=0.1, signed=True):
    """A symmetric, strictly diagonally dominant (so SPD) operator with random couplings -- negative and,
    with `signed`, positive ones -- some interior zeros, and 0 on the couplings that leave the grid."""
    rng = np.random.default_rng(seed)
    shape = (nz, ny, nx)

    def coupling(axis):
        c = -(0.5 + rng.random(shape))
        if signed:
            c[rng.random(shape) < 0.2] *= -1.0
        c[rng.random(shape) < zero_frac] = 0.0
        idx = [slice(None)] * 3
        idx[axis] = -1
        c[tuple(idx)] = 0.0
        return c

    cs = [coupling(2), coupling(1)] + ([coupling(0)] if dim == 3 else [])
    row = np.zeros(shape)
    for axis, c in zip((2, 1, 0), cs):
        row += np.abs(c)
        back = np.zeros(shape)
        sl_dst = [slice(None)] * 3
        sl_src = [slice(None)] * 3
        sl_dst[axis], sl_src[axis] = slice(1, None), slice(None, -1)
        back[tuple(sl_dst)] = np.abs(c[tuple(sl_src)])
        row += back
    diag = row + 0.1 + rng.random(shape)
    cz = cs[2].reshape(-1) if dim == 3 else None
    return VariableStencil(nx, ny, nz, diag.reshape(-1), cs[0].reshape(-1), cs[1].reshape(-1), cz)


# ------------------------------------------------------------------------------- SpMV
# the shapes of test_stencil_spmv_bitwise_csr (partial x-tiles: 130, 258), plus 3-D grids with nz = 1
SHAPES = [(16, 16, 1), (33, 7, 1), (6, 5, 4), (12, 12, 12), (64, 3, 5), (1, 1, 9),
          (256, 20, 1), (130, 9, 3), (258, 17, 9), (2, 3, 70), (128, 8, 33)]


@pytest.mark.parametrize("shape", SHAPES + [(20, 12, "3d1"), (130, 5, "3d1")])
def test_spmv_bitwise_csr(shape):
    nx, ny, nz = shape
    dim = 3 if nz == "3d1" or nz > 1 else 2
    nz = 1 if nz == "3d1" else nz
    S = make_var(nx, ny, nz, dim, seed=nx + 7 * ny + 31 * nz)
    A = S.tocsr()
    rng = np.random.default_rng(3)
    for v in (rng.standard_normal(S.shape[0]), np.ones(S.shape[0])):
        ref = A @ v
        assert np.array_equal(S @ v, ref)
        for tma in (1, 0):
            with Session(S) as s:
                s.set_option("tma", tma)
                assert np.array_equal(s.spmv(v), ref), (shape, tma)


@pytest.mark.parametrize("dim,shape", [(2, (64, 40, 1)), (3, (18, 10, 7)), (3, (7, 6, 5))])
def test_constant_coefficients_equal_poisson_spmv(dim, shape):
    nx, ny, nz = shape
    n = nx * ny * nz
    g = lambda a: a.reshape(nz, ny, nx)
    cx, cy = np.full(n, -1.0), np.full(n, -1.0)
    g(cx)[:, :, -1] = 0.0
    g(cy)[:, -1, :] = 0.0
    cz = None
    if dim == 3:
        cz = np.full(n, -1.0)
        g(cz)[-1] = 0.0
    S = VariableStencil(nx, ny, nz, np.full(n, 2.0 * dim), cx, cy, cz)
    P = PoissonStencil(nx, ny, nz, dim=dim)
    v = np.random.default_rng(4).standard_normal(n)
    for tma in (1, 0):
        with Session(S) as s, Session(P) as p:
            s.set_option("tma", tma)
            p.set_option("tma", tma)
            assert np.array_equal(s.spmv(v), p.spmv(v)), tma


# ------------------------------------------------------------------------------- solves
OPS = {
    "2d": lambda: make_var(24, 20, 1, 2, seed=1),
    "3d": lambda: make_var(10, 9, 8, 3, seed=2),
    "3d_odd": lambda: make_var(9, 8, 7, 3, seed=3, signed=False),   # odd nx: generic kernel
}
_PROB = {}


def _problem(name):
    if name not in _PROB:
        S = OPS[name]()
        A = S.tocsr()
        x_true, b, x0 = orc.setup_problem(A)
        assert np.array_equal(S @ x_true, b)
        _PROB[name] = (S, A, b, x0, x_true, 1.0 / A.diagonal())
    return _PROB[name]


def _device_solve(tag, A, b, x0, max_iter, dinv, x_true, **kw):
    f = getattr(cg_variants, orc.VARIANTS[tag])
    prec = (lambda v: v) if dinv is None else (lambda v: dinv * v)
    return f(A, b, x0, max_iter, preconditioner=prec, callbacks=STD_CALLBACKS, x_true=x_true, **kw)


@pytest.mark.parametrize("path", ["stream", "persistent"])
@pytest.mark.parametrize("prec", [True, False])
@pytest.mark.parametrize("name", list(OPS))
def test_variants_match_oracle_and_csr(name, prec, path):
    S, A, b, x0, x_true, dinv = _problem(name)
    d = dinv if prec else None
    for tag in ALL_TAGS:
        out = _device_solve(tag, S, b, x0, 40, d, x_true, path=path, return_info=True)
        assert out["_info"]["path"] == (1 if path == "stream" else 2)
        ref = orc.solve(tag, A, b, x0, 40, dinv=d, x_true=x_true)
        for h in helpers.RESIDUAL_HISTS:
            np.testing.assert_allclose(out[h][:12], ref[h][:12], rtol=helpers.RTOL, err_msg=f"{tag}/{h} vs oracle")
        csr = _device_solve(tag, A, b, x0, 40, d, x_true, path=path)
        for h in orc.HISTORIES:
            np.testing.assert_allclose(out[h][:12], csr[h][:12], rtol=1e-10, err_msg=f"{tag}/{h} vs CSR")
            np.testing.assert_allclose(out[h], csr[h], rtol=1e-6, atol=1e-11 * csr[h][0], err_msg=f"{tag}/{h} vs CSR")
    cg_variants.clear_cache()


def test_generic_kernel_solves_match_the_oracle():
    """tma forced off on an even grid: the generic kernel's solves meet P1 as the TMA kernel's do (its fused
    dots are summed in another order, so the two agree to rounding, not bitwise)."""
    S, A, b, x0, x_true, dinv = _problem("3d")
    for tag in ("hs", "cg", "gv", "pr", "pipe_pr"):
        with Session(S, dinv=dinv) as s:
            s.set_option("tma", 0)
            _, hist, _ = s.solve(tag, b, x0, 30, x_true=x_true, path="stream")
        ref = orc.solve(tag, A, b, x0, 30, dinv=dinv, x_true=x_true)
        for h in helpers.RESIDUAL_HISTS:
            np.testing.assert_allclose(hist[h][:12], ref[h][:12], rtol=helpers.RTOL, err_msg=f"{tag}/{h}")


def test_runs_are_bitwise_repeatable():
    S, A, b, x0, x_true, dinv = _problem("3d")
    for path in ("stream", "persistent"):
        for tag in ("hs", "pr", "pipe_pr", "gv"):
            o1 = _device_solve(tag, S, b, x0, 60, dinv, x_true, path=path)
            o2 = _device_solve(tag, S, b, x0, 60, dinv, x_true, path=path)
            for h in orc.HISTORIES:
                assert np.array_equal(o1[h], o2[h], equal_nan=True), (path, tag, h)
    cg_variants.clear_cache()


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


@pytest.mark.parametrize("path", ["stream", "persistent"])
@pytest.mark.parametrize("tag", ALL_TAGS)
def test_tolerance_contract(tag, path):
    """DESIGN.md section 5b: a run stopped at stop_k holds the bits of the run with max_iter = stop_k + 1."""
    S, A, b, x0, x_true, dinv = _problem("3d")
    tol = 1e-6
    with Session(S, dinv=dinv) as s:
        x, hist, info = s.solve(tag, b, x0, 500, x_true=x_true, path=path, tol=tol)
        stop = info["stop_iter"]
        assert 1 <= stop < 499 and info["iterations"] == stop
        sc = s.scalars()
        vec = {v: s.vector(v) for v in ("x", "r", "rt", "p", "s")}
        x1, hist1, _ = s.solve(tag, b, x0, stop + 1, x_true=x_true, path=path)
        assert np.array_equal(_bits(x), _bits(x1))
        for h in hist1:
            assert hist[h].shape == (stop + 1,) and np.array_equal(_bits(hist[h]), _bits(hist1[h])), h
        assert np.array_equal(_bits(list(sc.values())), _bits(list(s.scalars().values())))
        for v, a in vec.items():
            assert np.array_equal(_bits(a), _bits(s.vector(v))), v


def test_drop_in_with_jacobi_callbacks_and_capture():
    S, A, b, x0, x_true, dinv = _problem("2d")
    out = cg_variants.pr_pcg(S, b, x0, 30, preconditioner=lambda v: dinv * v,
                             callbacks=[cbk.updated_residual_2_norm, cbk.save_x], x_true=x_true)
    ref = orc.solve("pr", A, b, x0, 30, dinv=dinv, x_true=x_true)
    np.testing.assert_allclose(out["updated_residual_2_norm"][:12], ref["updated_residual_2_norm"][:12], rtol=1e-10)
    assert out["x"].shape == (30, S.shape[0])
    assert np.array_equal(out["x"][0], x0)
    with Session(S, dinv=dinv) as s:                     # the captured rows are the solve's own x_k
        x29, _, _ = s.solve("pr", b, x0, 30, path="stream", histories=())
        x9, _, _ = s.solve("pr", b, x0, 10, path="stream", histories=())
    assert np.array_equal(out["x"][29], x29) and np.array_equal(out["x"][9], x9)
    # a user callback (stepwise protocol) sees the operator itself
    seen = []
    cg_variants.pr_pcg(S, b, x0, 5, preconditioner=lambda v: dinv * v,
                       callbacks=[lambda **kw: seen.append(np.linalg.norm(kw["b"] - kw["A"] @ kw["x_k"]))])
    assert len(seen) == 5 and np.isclose(seen[0], np.linalg.norm(b - A @ x0))
    # error histories without x_true: solved for on the host (tocsr)
    e = cg_variants.hs_pcg(S, b, x0, 10, preconditioner=lambda v: dinv * v, callbacks=[cbk.error_A_norm])
    np.testing.assert_allclose(e["error_A_norm"][0], ref["error_A_norm"][0], rtol=1e-6)
    cg_variants.clear_cache()


def test_same_shape_different_coefficients_never_share_a_session():
    S1 = make_var(16, 12, 6, 3, seed=10)
    S2 = make_var(16, 12, 6, 3, seed=11)
    b = np.ones(S1.shape[0])
    x0 = np.zeros_like(b)
    cg_variants.clear_cache()
    o1 = cg_variants.pr_cg(S1, b, x0, 20, callbacks=[cbk.residual_2_norm])
    o2 = cg_variants.pr_cg(S2, b, x0, 20, callbacks=[cbk.residual_2_norm])
    r1 = orc.solve("pr", S1.tocsr(), b, x0, 20)
    r2 = orc.solve("pr", S2.tocsr(), b, x0, 20)
    np.testing.assert_allclose(o1["residual_2_norm"][:10], r1["residual_2_norm"][:10], rtol=1e-10)
    np.testing.assert_allclose(o2["residual_2_norm"][:10], r2["residual_2_norm"][:10], rtol=1e-10)
    assert not np.array_equal(o1["residual_2_norm"], o2["residual_2_norm"])
    assert len(cg_variants._CACHE) == 2 and cg_variants._CACHE[0][3] is not cg_variants._CACHE[1][3]
    cg_variants.clear_cache()


# ------------------------------------------------------------------------------- refusals and validation
def test_c_entry_point_validates():
    lib = _lib.load()
    nx, ny, nz = 4, 3, 2
    S = make_var(nx, ny, nz, 3, seed=5)
    p = _lib.dptr
    with Session(S) as s:
        ctx = s._ctx
        assert lib.cgx_set_stencil_coef_host(ctx, 3, nx, ny, nz, p(S.diag), p(S.cx), p(S.cy), p(S.cz)) == _lib.OK
        assert lib.cgx_set_stencil_coef_host(ctx, 3, nx, ny, nz, p(S.diag), p(S.cx), p(S.cy), None) == _lib.ERR_ARG
        assert lib.cgx_set_stencil_coef_host(ctx, 2, nx, ny, 1, p(S.diag[:12]), p(S.cx[:12]), p(S.cy[:12]),
                                             p(S.cz[:12])) == _lib.ERR_ARG
        for name in ("diag", "cx", "cy", "cz"):
            arrs = {k: getattr(S, k).copy() for k in ("diag", "cx", "cy", "cz")}
            arrs[name][0] = np.nan
            assert lib.cgx_set_stencil_coef_host(ctx, 3, nx, ny, nz, *(p(arrs[k]) for k in ("diag", "cx", "cy", "cz"))) \
                == _lib.ERR_ARG, name
        for name, i in (("cx", nx - 1), ("cy", nx * (ny - 1)), ("cz", nx * ny * (nz - 1))):
            arrs = {k: getattr(S, k).copy() for k in ("diag", "cx", "cy", "cz")}
            arrs[name][i] = 1.0
            assert lib.cgx_set_stencil_coef_host(ctx, 3, nx, ny, nz, *(p(arrs[k]) for k in ("diag", "cx", "cy", "cz"))) \
                == _lib.ERR_ARG, name
        assert lib.cgx_set_stencil_coef_host(ctx, 3, 1 << 11, 1 << 11, 1 << 10, p(S.diag), p(S.cx), p(S.cy),
                                             p(S.cz)) == _lib.ERR_UNSUPPORTED


def test_batch_and_partition_rank_refuse_in_c():
    lib = _lib.load()
    S = make_var(8, 6, 4, 3, seed=6)
    b = np.ones(S.shape[0])
    with Session(S) as s1, Session(S) as s2:
        for s in (s1, s2):
            s.load_problem(b, np.zeros_like(b))
        ctxs = (C.c_void_p * 2)(s1._ctx, s2._ctx)
        variants = np.array([3, 0], dtype=np.int32)
        iters = np.array([5, 5], dtype=np.int32)
        infos = (_lib.CgxInfo * 2)()
        assert lib.cgx_batch_run(ctxs, 2, _lib.iptr(variants), _lib.iptr(iters), 0, infos) == _lib.ERR_UNSUPPORTED
        with pytest.raises(NotImplementedError):
            solve_batch([(s1, "pr", b, np.zeros_like(b), 5)])
        s1.run("pr", 5)                                  # a refused batch leaves the context usable
    with Session(PoissonStencil(8, 6, 4, dim=3)) as r:
        assert lib.cgx_set_stencil_slab(r._ctx, 8, 6, 2, 2, 0, 6.0, -1.0) == _lib.OK
        p = _lib.dptr
        assert lib.cgx_set_stencil_coef_host(r._ctx, 3, 8, 6, 4, p(S.diag), p(S.cx), p(S.cy), p(S.cz)) \
            == _lib.ERR_UNSUPPORTED
