"""scilmm_b200: B200-native estimation engine behind SciLMM's SparseCholesky path.

Mirrors the reference package facade (scilmm/__init__.py:1-2 star-imports SparseCholesky), so
`from scilmm_b200 import HE, REML, SparseCholesky, run_estimates` works like `from scilmm import ...`.
"""
from .SparseCholesky import (HE, MINQUE, REML, B200Factor, association, NotPositiveDefiniteError, SlmmError,  # noqa: F401
                             SparseCholesky, bolt_gradient_estimation, compute_gradients, compute_hess,
                             compute_varcomp_stderr, estimate_fixed_effects, estimate_var_comps,
                             matrices_weighted_sum, negative_log_likelihood, run_estimates,
                             run_estimates_from_paths, simulate_vector)

from .legacy import LMM, compute_HE  # noqa: F401,E402  (reference scilmm/Estimation/LMM.py:154, HE.py:22)
from .matrices import load_sparse_csr, pairwise_epistasis, save_sparse_csr  # noqa: F401,E402  (Matrices/*.py)

__version__ = "0.1.0"
