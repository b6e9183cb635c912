"""icikendalltau_b200 -- B200-native (sm_100a) all-pairs ICI-Kendall-tau.

Host-side mirror of the reference's R interface (`ici_kendalltau`, `ici_kt`, `kt_fast`,
`pairwise_completeness`) over the C ABI of libicikt_b200.so.  No CPU fallback.
"""
from ._lib import (IciktError, Plan, load, p_adjust, pnorm_device, run_cross, run_cross_edges,  # noqa: F401
                   run_cross_topk, run_edges, run_pairs, run_topk)
from .reshaping import cor_matrix_2_long_df, long_df_2_cor_matrix  # noqa: F401
from .api import (IciKtResult, ici_kendalltau, ici_kendalltau_cross, ici_kendalltau_cross_topk,  # noqa: F401
                  ici_kendalltau_topk, ici_kt, kt_fast,
                  pairwise_completeness,
                  setup_comparisons, setup_missing_matrix)

__all__ = ["cor_matrix_2_long_df", "long_df_2_cor_matrix", "ici_kendalltau", "ici_kendalltau_cross", "ici_kendalltau_cross_topk", "ici_kendalltau_topk", "ici_kt", "kt_fast", "pairwise_completeness", "run_pairs", "run_edges", "run_topk", "run_cross", "run_cross_edges", "run_cross_topk", "p_adjust", "Plan",
           "IciktError", "IciKtResult", "load", "pnorm_device", "setup_comparisons",
           "setup_missing_matrix"]
