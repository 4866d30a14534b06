"""pps_b200 — B200-native retrieval hot path of PPS (part-power-set pooling + re-ID ranking).

Python here is the thin host layer over ``libpps_b200.so`` (hand-written sm_100a CUDA behind
the C ABI of ``include/pps_b200.h``); PyTorch only hands tensors and streams across.
"""
from .pooling import (ReIDPoolCfg, add_pps_part_head, add_pps_part_head_, blob_names, comb_to_mask, mask_to_comb,
                      pps_pool, pps_pool_autograd, pps_pool_backward, pyramid_combs, uniform_partition_split)
from .evaluator import (PairLists, RankEngine, RankResult, cmc, compute_dist, evaluate, evaluate_arrays, evaluate_host, mean_ap,
                        rank_distmat, rank_eval, reid_results)
from .index import GalleryIndex
from .embedding import ReidEmbedHead, add_reid_outputs, embed_maps, fold_bn, l2_normalize_rows
from .rerank import re_ranking, re_ranking_from_features

__all__ = [
    "ReIDPoolCfg", "add_pps_part_head", "add_pps_part_head_", "blob_names", "comb_to_mask", "mask_to_comb",
    "pps_pool", "pps_pool_autograd", "pps_pool_backward", "pyramid_combs", "uniform_partition_split",
    "GalleryIndex", "PairLists", "RankEngine", "RankResult", "cmc", "compute_dist", "evaluate", "evaluate_arrays", "evaluate_host", "mean_ap",
    "rank_distmat", "rank_eval", "reid_results",
    "ReidEmbedHead", "add_reid_outputs", "embed_maps", "fold_bn", "l2_normalize_rows",
    "re_ranking", "re_ranking_from_features",
]
__version__ = "0.1.0"
