"""Operator objects accepted as ``A`` by the solvers.

The reference passes a scipy CSR matrix (``figure_gen.py:350``); that still works.  For
the synthetic Poisson configurations of BASELINE.json a matrix-free operator is added:
it never materialises the 84-117 M non-zeros, and its host-side ``@`` (used only by the
caller to form ``b = A @ x_true``, figure_gen.py:33) reproduces scipy's CSR product of the
equivalent matrix bit for bit (same term order, separately rounded multiply/add).
"""
from __future__ import annotations

import numpy as np
import scipy.sparse as sps


def canonical_csr(A) -> sps.csr_matrix:
    """Anything scipy can turn into CSR -> canonical fp64/int32 CSR (sorted, no duplicates),
    the form ``csr_matrix(mmread(...))`` has in the reference."""
    if isinstance(A, np.ndarray):
        A = sps.csr_matrix(A)
    elif not sps.issparse(A):
        raise TypeError(f"cannot interpret {type(A).__name__} as a matrix")
    A = A.tocsr()
    if A.dtype != np.float64:
        A = A.astype(np.float64)
    if not A.has_canonical_format:
        A = A.copy()
        A.sum_duplicates()
        A.sort_indices()
    if A.shape[0] != A.shape[1]:
        raise ValueError("A must be square")
    if A.indices.dtype != np.int32 or A.indptr.dtype != np.int32:
        if A.nnz >= 2**31 or A.shape[0] >= 2**31:
            raise ValueError("matrix too large for int32 indices")
        A = sps.csr_matrix((A.data, A.indices.astype(np.int32), A.indptr.astype(np.int32)),
                           shape=A.shape)
    return A


class PoissonStencil:
    """Matrix-free Dirichlet Laplacian, natural ordering ``i = x + nx*(y + ny*z)``.

    dim=2: 5-point (diag 4, off -1) == ``kron(I,T)+kron(T,I)``; dim=3: 7-point (diag 6).
    """

    def __init__(self, nx, ny=None, nz=None, dim=None, diag=None, off=-1.0):
        if dim is None:
            dim = 2 if nz is None else 3
        ny = nx if ny is None else ny
        nz = (nx if dim == 3 else 1) if nz is None else nz
        if dim == 2 and nz != 1:
            raise ValueError("2-D stencil needs nz == 1")
        self.dim, self.nx, self.ny, self.nz = int(dim), int(nx), int(ny), int(nz)
        self.diag = float(2 * dim if diag is None else diag)
        self.off = float(off)
        n = self.nx * self.ny * self.nz
        self.shape = (n, n)
        self.dtype = np.dtype(np.float64)

    # scipy-like surface used by figure_gen-style callers
    def get_shape(self):
        return self.shape

    @property
    def nnz(self):
        nx, ny, nz = self.nx, self.ny, self.nz
        n = nx * ny * nz
        return n + 2 * ((nx - 1) * ny * nz + nx * (ny - 1) * nz + (nx * ny * (nz - 1) if self.dim == 3 else 0))

    def diagonal(self):
        return np.full(self.shape[0], self.diag)

    def matvec(self, v):
        """Host product in canonical-CSR term order (z-1, y-1, x-1, centre, x+1, y+1, z+1)."""
        v = np.asarray(v, dtype=np.float64)
        nx, ny, nz = self.nx, self.ny, self.nz
        g = v.reshape(nz, ny, nx)
        y = np.zeros_like(g)
        if nz > 1:
            y[1:] += self.off * g[:-1]
        if ny > 1:
            y[:, 1:] += self.off * g[:, :-1]
        if nx > 1:
            y[:, :, 1:] += self.off * g[:, :, :-1]
        y += self.diag * g
        if nx > 1:
            y[:, :, :-1] += self.off * g[:, :, 1:]
        if ny > 1:
            y[:, :-1] += self.off * g[:, 1:]
        if nz > 1:
            y[:-1] += self.off * g[1:]
        return y.reshape(-1)

    def __matmul__(self, v):
        return self.matvec(v)

    def tocsr(self):
        t = lambda m: sps.diags([1.0, 0.0, 1.0], [-1, 0, 1], shape=(m, m))
        eye = sps.identity
        nx, ny, nz = self.nx, self.ny, self.nz
        off = (sps.kron(eye(nz), sps.kron(eye(ny), t(nx))) + sps.kron(eye(nz), sps.kron(t(ny), eye(nx))))
        if nz > 1:
            off = off + sps.kron(t(nz), sps.kron(eye(ny), eye(nx)))
        A = sps.csr_matrix(self.off * off + self.diag * eye(nx * ny * nz))
        A.eliminate_zeros()
        A.sort_indices()
        return A

    def __repr__(self):
        return f"PoissonStencil(dim={self.dim}, nx={self.nx}, ny={self.ny}, nz={self.nz}, diag={self.diag}, off={self.off})"


class VariableStencil:
    """Matrix-free symmetric Dirichlet 5-point (dim 2) or 7-point (dim 3) operator with a coefficient
    per row and direction, natural ordering ``i = x + nx*(y + ny*z)`` as ``PoissonStencil``.

    ``diag[i] = A[i, i]``, ``cx[i] = A[i, i+1]``, ``cy[i] = A[i, i+nx]``, ``cz[i] = A[i, i+nx*ny]``
    (float64, length n each; ``cz`` only in 3-D).  The backward couplings follow by symmetry:
    ``A[i, i-1] = cx[i-1]``, and likewise for y and z.  A coupling that leaves the grid (``cx`` at
    x = nx-1, ``cy`` at y = ny-1, ``cz`` at z = nz-1) must be 0.  ``dim`` defaults to 3 when ``cz``
    is given, else 2.  The arrays are copied and kept read-only.
    """

    def __init__(self, nx, ny, nz, diag, cx, cy, cz=None, dim=None):
        if dim is None:
            dim = 2 if cz is None else 3
        dim, nx, ny, nz = int(dim), int(nx), int(ny), int(nz)
        if dim not in (2, 3):
            raise ValueError("dim must be 2 or 3")
        if min(nx, ny, nz) < 1:
            raise ValueError("nx, ny and nz must be >= 1")
        if dim == 2 and (nz != 1 or cz is not None):
            raise ValueError("a 2-D stencil needs nz == 1 and no cz")
        if dim == 3 and cz is None:
            raise ValueError("a 3-D stencil needs cz")
        n = nx * ny * nz
        self.dim, self.nx, self.ny, self.nz = dim, nx, ny, nz
        arrs = {}
        for name, a in (("diag", diag), ("cx", cx), ("cy", cy), ("cz", cz)):
            if a is None:
                arrs[name] = None
                continue
            a = np.array(a, dtype=np.float64, copy=True).reshape(-1)
            if a.shape[0] != n:
                raise ValueError(f"{name} has length {a.shape[0]}, expected n = {n}")
            if not np.all(np.isfinite(a)):
                raise ValueError(f"{name} has a non-finite entry")
            a.flags.writeable = False
            arrs[name] = a
        g = lambda a: a.reshape(nz, ny, nx)
        if np.any(g(arrs["cx"])[:, :, -1] != 0.0):
            raise ValueError("cx must be 0 at x = nx-1 (the coupling leaves the grid)")
        if np.any(g(arrs["cy"])[:, -1, :] != 0.0):
            raise ValueError("cy must be 0 at y = ny-1 (the coupling leaves the grid)")
        if arrs["cz"] is not None and np.any(g(arrs["cz"])[-1] != 0.0):
            raise ValueError("cz must be 0 at z = nz-1 (the coupling leaves the grid)")
        self.diag, self.cx, self.cy, self.cz = arrs["diag"], arrs["cx"], arrs["cy"], arrs["cz"]
        self.shape = (n, n)
        self.dtype = np.dtype(np.float64)

    def get_shape(self):
        return self.shape

    @property
    def nnz(self):
        """Entries of the full 5/7-point pattern (zero couplings inside the grid included)."""
        nx, ny, nz = self.nx, self.ny, self.nz
        return nx * ny * nz + 2 * ((nx - 1) * ny * nz + nx * (ny - 1) * nz + nx * ny * (nz - 1))

    def diagonal(self):
        return self.diag.copy()

    def matvec(self, v):
        """Host product in canonical-CSR term order (z-1, y-1, x-1, centre, x+1, y+1, z+1), bit for bit
        ``self.tocsr() @ v``."""
        v = np.asarray(v, dtype=np.float64)
        nx, ny, nz = self.nx, self.ny, self.nz
        g = v.reshape(nz, ny, nx)
        cx, cy = self.cx.reshape(nz, ny, nx), self.cy.reshape(nz, ny, nx)
        y = np.zeros_like(g)
        if nz > 1:
            cz = self.cz.reshape(nz, ny, nx)
            y[1:] += cz[:-1] * g[:-1]
        if ny > 1:
            y[:, 1:] += cy[:, :-1] * g[:, :-1]
        if nx > 1:
            y[:, :, 1:] += cx[:, :, :-1] * g[:, :, :-1]
        y += self.diag.reshape(nz, ny, nx) * g
        if nx > 1:
            y[:, :, :-1] += cx[:, :, :-1] * g[:, :, 1:]
        if ny > 1:
            y[:, :-1] += cy[:, :-1] * g[:, 1:]
        if nz > 1:
            y[:-1] += cz[:-1] * g[1:]
        return y.reshape(-1)

    def __matmul__(self, v):
        return self.matvec(v)

    def tocsr(self):
        """Canonical CSR with the full 5/7-point pattern: zero couplings inside the grid are stored."""
        nx, ny, nz = self.nx, self.ny, self.nz
        n, plane = nx * ny * nz, nx * ny
        if self.nnz >= 2**31:
            raise ValueError("matrix too large for int32 indices")
        idx = np.arange(n, dtype=np.int64)
        x, y, z = idx % nx, (idx // nx) % ny, idx // plane
        cz = self.cz if self.cz is not None else np.zeros(n)
        # one slot per neighbour, in ascending column order: a row's stored entries come out sorted
        slots = ((-plane, z > 0, cz, -plane), (-nx, y > 0, self.cy, -nx), (-1, x > 0, self.cx, -1),
                 (0, None, self.diag, 0), (1, x < nx - 1, self.cx, 0), (nx, y < ny - 1, self.cy, 0),
                 (plane, z < nz - 1, cz, 0))
        cols = np.empty((n, 7), dtype=np.int32)
        vals = np.empty((n, 7))
        mask = np.empty((n, 7), dtype=bool)
        for s, (off, ok, coef, shift) in enumerate(slots):
            mask[:, s] = True if ok is None else ok
            cols[:, s] = np.clip(idx + off, 0, n - 1)
            vals[:, s] = coef[np.clip(idx + shift, 0, n - 1)]
        indptr = np.zeros(n + 1, dtype=np.int32)
        np.cumsum(mask.sum(axis=1), out=indptr[1:])
        A = sps.csr_matrix((vals[mask], cols[mask], indptr), shape=(n, n))
        A.has_sorted_indices = True
        return A

    def __repr__(self):
        return f"VariableStencil(dim={self.dim}, nx={self.nx}, ny={self.ny}, nz={self.nz})"


def poisson2d(nx, ny=None):
    return PoissonStencil(nx, ny, 1, dim=2)


def poisson3d(nx, ny=None, nz=None):
    return PoissonStencil(nx, ny, nx if nz is None else nz, dim=3)
