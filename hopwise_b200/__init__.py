"""hopwise_b200: B200-native (sm_100a) drop-in for hopwise's knowledge-graph-embedding hot path.

Public surface (mirrors the reference names so a hopwise user can switch imports):
  TransE, DistMult, RotatE, ComplEx      KnowledgeRecommender-compatible models (recommender.py)
  KGSampler, RecSampler                  bit-exact GPU negative samplers (sampler.py)
  FusedCollector, evaluate_full_sort     fused full-sort top-k and GAUC evaluation (evaluator.py)
  enable_row_sparse_data_parallel        row-sparse / dense gradient exchange over NCCL (distributed.py)
  DevicePrefetcher                       host->device batch staging one step ahead (loader.py)
"""

from .recommender import (  # noqa: F401
    MODELS, ComplEx, DistMult, FusedKGEModel, KnowledgeRecommender, RotatE, TorusE, TransD, TransE, TransH,
)

__all__ = ["TransE", "DistMult", "RotatE", "ComplEx", "TorusE", "TransH", "TransD", "FusedKGEModel",
           "KnowledgeRecommender", "MODELS"]
__version__ = "0.1.0"
