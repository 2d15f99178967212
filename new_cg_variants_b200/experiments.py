"""Matplotlib-free restatement of the reference's numerical-experiment driver
(numerical_experiments/figure_gen.py:21-124), running every solve on the GPU path:

    test_matrix(A, max_iter, title, preconditioner=None|'jacobi', variants=[...], data_dir=...)
    parse_convergence_data(matrix_name, preconditioner, variants, A=..., data_dir=...)
    gen_convergence_table(data_dir, out_path)

The `.npy` dictionaries and the `convergence.txt` rows have the reference's format, so they
can be diffed against `numerical_experiments/data/*` and `figures/convergence_table_data.tex`.
`exact_pcg` (extended precision, figure_gen.py:53-56) is not part of the GPU path: pass the
reference's function in `variants` if it is wanted; it is then called exactly as there.
"""
from __future__ import annotations

import glob
import os

import numpy as np

from . import callbacks as _cb
from . import cg_variants as _cg

# figure_gen.py:347-348 (method list) and :360 (table columns)
ALL_METHODS = [_cg.hs_pcg, _cg.cg_pcg, _cg.m_pcg, _cg.pr_pcg, _cg.gv_pcg, _cg.pipe_pr_m_pcg, _cg.pipe_pr_pcg,
               _cg.pipe_p_pcg, _cg.pipe_p_m_pcg]
TABLE_METHODS = ["hs_pcg", "cg_pcg", "m_pcg", "pr_pcg", "gv_pcg", "pipe_pr_m_pcg", "pipe_pr_pcg"]


def setup_problem(A):
    """figure_gen.py:31-34: x_true = ones/sqrt(N), b = A x_true, x0 = 0."""
    N = A.get_shape()[0] if hasattr(A, "get_shape") else A.shape[0]
    x_true = np.ones(N) / np.sqrt(N)
    b = A @ x_true
    x0 = np.zeros(N)
    return x_true, b, x0


def test_matrix(A, max_iter, title, preconditioner=None, variants=(), data_dir="./data", save=True, concurrent=False,
                **solver_kwargs):
    """figure_gen.py:21-60.  Returns {method name: output dict}.

    ``concurrent=True``: the GPU methods run side by side in one launch (cg_variants.solve_concurrently;
    bitwise equal to solo runs with the same CTA shape, not to default solo runs); ``exact_pcg``, if listed,
    is still the reference's own call.  The files written are the same."""
    N = A.get_shape()[0] if hasattr(A, "get_shape") else A.shape[0]
    x_true, b, x0 = setup_problem(A)
    callbacks = [_cb.error_A_norm, _cb.residual_2_norm, _cb.error_2_norm, _cb.updated_residual_2_norm]
    prec = lambda x: x                                            # noqa: E731
    prec_long = lambda x: x                                       # noqa: E731
    if preconditioner == "jacobi":
        dinv = 1 / A.diagonal()                                   # figure_gen.py:43 (hoisted: same products)
        prec = lambda x: dinv * x                                 # noqa: E731
        prec_long = lambda x: (1 / A.diagonal().astype(np.longdouble)) * x    # noqa: E731
    out_dir = os.path.join(data_dir, f"{title}_{preconditioner}")
    if save:
        os.makedirs(out_dir, exist_ok=True)
    trials = {}
    batch = {}
    if concurrent:
        gpu = [m for m in variants if m.__name__ != "exact_pcg"]
        if gpu:
            batch = _cg.solve_concurrently(gpu, A, b, x0, max_iter, preconditioner=prec, callbacks=callbacks,
                                           x_true=x_true, **solver_kwargs)
    for method in variants:
        if method.__name__ in batch:
            trial = batch[method.__name__]
        elif method.__name__ == "exact_pcg":                        # the reference's own function, its own call
            trial = method(A.astype(np.longdouble), b.astype(np.longdouble), x0.astype(np.longdouble),
                           min(max_iter, N), callbacks=callbacks, x_true=x_true.astype(np.longdouble),
                           preconditioner=prec_long)
        else:
            trial = method(A, b, x0, max_iter, callbacks=callbacks, x_true=x_true, preconditioner=prec,
                           **solver_kwargs)
        trials[method.__name__] = trial
        if save:
            np.save(os.path.join(out_dir, method.__name__), trial, allow_pickle=True)
    return trials


def convergence_metrics(error_A_norm, error_tol=1e-5):
    """figure_gen.py:80-89: (first k with relative A-norm error <= tol, 0 = never;
    log10 of the smallest relative A-norm error)."""
    rel = np.asarray(error_A_norm) / error_A_norm[0]
    with np.errstate(divide="ignore", invalid="ignore"):
        return int(np.argmin(rel > error_tol)), float(np.log10(np.nanmin(rel)))


def format_table_row(matrix_name, preconditioner, n, nnz, iters, accuracies):
    r"""One row of figures/convergence_table_data.tex, written from the row format

        \texttt{name} & prec & n & nnz & {it_1} ... & {it_m} &{acc_1} ... &{acc_m}\\

    name with escaped underscores; prec "Jac." or "-"; an iteration count of 0 ("never reached
    1e-5") prints as "-"; accuracies with two decimals.  A cell is wrapped in \tableemph when the
    variant is visibly worse than the first column (HS-CG): more than 10 % more iterations or no
    convergence; attainable accuracy (a negative log10) above 0.9 of the first column's."""
    head = ["\\texttt{%s}" % matrix_name.replace("_", "\\_"), "Jac." if preconditioner == "jacobi" else "-", str(n), str(nnz)]
    it_cells, acc_cells = [], []
    for it, acc in zip(iters, accuracies):
        slow = it == 0 or it > 1.1 * iters[0]
        it_cells.append("& %s{%s}" % ("\\tableemph" if slow else "", it if it else "-"))
        acc_cells.append("&%s{%.2f}" % ("\\tableemph" if acc > 0.9 * accuracies[0] else "", acc))
    return " & ".join(head) + "".join(it_cells) + "".join(acc_cells) + "\\\\ \n"


def banded_model_problem(n=650000, k=32, kappa=1e6, rho=0.95, off=1e-4):
    """The PETSc driver's model problem (scaling_experiments_petsc/ex2b.c:86-97,
    strong_scaling_tests.py:49-56) as a scipy CSR matrix: half-bandwidth k (2k+1 non-zeros per
    interior row), off-diagonals `off`, diagonal 1 + (i/(n-1)) (kappa-1) rho^(n-1-i); the driver
    solves A x = A 1 from x0 = 0 without preconditioner and prints ||x - 1||_2
    (ex2b.c:138-139,192-200).  Returns (A, b, x_true)."""
    import scipy.sparse as sps
    i = np.arange(n, dtype=np.float64)
    diag = 1.0 + (i / (n - 1)) * (kappa - 1) * rho ** (n - 1 - i)
    offs = [o for o in range(-k, k + 1) if o != 0]
    A = sps.diags([np.full(n - abs(o), off) for o in offs], offs, shape=(n, n), format="csr") + sps.diags(diag)
    A = sps.csr_matrix(A)
    A.sort_indices()
    x_true = np.ones(n)
    return A, A @ x_true, x_true


# final errors ||x - 1||_2 after 4000 iterations printed by the reference's run on 336 / 280 MPI ranks
# (scaling_experiments_petsc/config_info/slurm-864568.out:129,148,167,186,205 and :224-300); PETSc KSP
# names -> ours (strong_scaling_plots.py:72-79): cg = HS, chcg = CG-CG, pipecg = GV, pipeprcg = pipe-PR,
# pipeprcg_0 (-recompute_q 0) = pipe-P
BANDED_KAT = {"hs": (1.60099e-07, 1.88385e-07), "cg": (2.46479e-07, 2.17013e-07), "gv": (0.000135586, 0.000125243),
              "pipe_pr": (3.24332e-07, 3.10494e-07), "pipe_p": (8.94408e-05, 8.74067e-05)}


def parse_convergence_data(matrix_name, preconditioner=None, variants=TABLE_METHODS, A=None, n=None, nnz=None,
                           data_dir="./data", trials=None, write=True):
    """figure_gen.py:62-124: one LaTeX table row (also written to <dir>/convergence.txt)."""
    if A is not None:
        n, nnz = A.shape[0], A.nnz
    out_dir = os.path.join(data_dir, f"{matrix_name}_{preconditioner}")
    min_iters, min_errors = [], []
    for method in variants:
        name = method if isinstance(method, str) else method.__name__
        trial = trials[name] if trials is not None else \
            np.load(os.path.join(out_dir, name + ".npy"), allow_pickle=True).item()
        it, acc = convergence_metrics(trial["error_A_norm"])
        min_iters.append(it)
        min_errors.append(acc)
    data = format_table_row(matrix_name, preconditioner, n, nnz, min_iters, min_errors)
    if write:
        os.makedirs(out_dir, exist_ok=True)
        with open(os.path.join(out_dir, "convergence.txt"), "w") as fh:
            fh.write(data)
    return data, min_iters, min_errors


def gen_convergence_table(data_dir="./data", out_path="./figures/convergence_table_data.tex"):
    """figure_gen.py:117-124: concatenate the rows, un-preconditioned cases first."""
    rows = []
    for suffix in ("None", "jacobi"):
        for path in sorted(glob.glob(os.path.join(data_dir, f"*{suffix}", "convergence.txt"))):
            rows.append(open(path).read())
    os.makedirs(os.path.dirname(out_path) or ".", exist_ok=True)
    with open(out_path, "w") as fh:
        fh.write("".join(rows))
    return rows
