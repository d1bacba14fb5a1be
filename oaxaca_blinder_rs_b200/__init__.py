"""obboot: B200-native bootstrap inference for the Oaxaca-Blinder decomposition.

Drop-in for the bootstrap hot path of dot-comma-hyphen/oaxaca-blinder-rs (OaxacaBuilder::run /
decompose_quantile).  The compute path is hand-written sm_100a CUDA behind the C ABI in
include/obboot.h; this package is the host-side mirror of the reference's interface.
"""
from .core import (CACHE_FILLED, CACHE_NONE, CACHE_OUTCOME_ONLY, CACHE_SOLVE_ONLY, REF_GROUP_A, REF_GROUP_B, REF_POOLED,
                   REF_WEIGHTED, Context, Design, GramCache, NormVar,
                   OaxacaError, PinnedBuffer, bootstrap, machado_mata, num_stats, pin_in_place, reduce_stats, replicate_shard, unpin)

from .builder import (ComponentResult, OaxacaBlinder, OaxacaBuilder, OaxacaResults, QuantileDecompositionBuilder,
                      QuantileDecompositionDetail, QuantileDecompositionResults, ReferenceCoefficients, read_csv)

__all__ = ["QuantileDecompositionBuilder", "QuantileDecompositionDetail", "QuantileDecompositionResults", "ComponentResult", "OaxacaBlinder", "OaxacaBuilder", "OaxacaResults", "ReferenceCoefficients", "REF_GROUP_A", "REF_GROUP_B", "REF_POOLED", "REF_WEIGHTED", "Context", "Design", "GramCache", "CACHE_NONE", "CACHE_FILLED", "CACHE_OUTCOME_ONLY", "CACHE_SOLVE_ONLY", "NormVar",
           "OaxacaError", "PinnedBuffer", "pin_in_place", "unpin", "replicate_shard", "bootstrap", "machado_mata", "num_stats", "reduce_stats", "read_csv"]
