"""scde_b200 -- B200 (sm_100a) implementation of scde's differential-expression posterior path.

Public API mirrors the reference's R functions (see ``api``); all numeric work runs in ``libscde_b200.so``
(hand-written CUDA, C ABI in ``include/scde_b200.h``).  There is no CPU fallback.
"""
from .api import (DifferenceJob, DifferenceSession, calculate_ratio_posterior, expand_contrasts, jpmat_log_batch_boot,
                  jpmat_log_boot, mat_slide_mult, quick_distribution_summary, scde_expression_difference,
                  scde_expression_difference_contrasts, scde_expression_magnitude, scde_posteriors,
                  scde_test_gene_expression_difference)
from ._lib import Context, ScdeB200Error, default_context

__all__ = ["scde_expression_difference", "scde_posteriors", "scde_expression_magnitude", "calculate_ratio_posterior",
           "quick_distribution_summary", "scde_test_gene_expression_difference", "mat_slide_mult", "jpmat_log_boot", "jpmat_log_batch_boot", "DifferenceJob",
           "scde_expression_difference_contrasts", "DifferenceSession", "expand_contrasts",
           "Context", "ScdeB200Error", "default_context"]
