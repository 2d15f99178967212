"""new_cg_variants_b200 -- the predict-and-recompute CG inner loop of
tchen-research/new_cg_variants on NVIDIA B200 (sm_100a).

    from new_cg_variants_b200.cg_variants import hs_pcg, pr_pcg, pipe_pr_pcg, ...
    from new_cg_variants_b200.callbacks import error_A_norm, residual_2_norm, ...

keep the reference's Python signatures; the arithmetic runs in ``libcgx_b200.so``
(hand-written CUDA behind the C ABI of ``include/cgx.h``).  No CPU fallback.
"""
from .operators import PoissonStencil, VariableStencil, canonical_csr, poisson2d, poisson3d   # noqa: F401
from .session import Session                                                  # noqa: F401
from . import callbacks, cg_variants, cg_variants_mpi4py, experiments              # noqa: F401

__version__ = "0.1.0"
