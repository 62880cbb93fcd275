"""rustsolver_b200 — B200-native vectorized CFR engine behind RustSolver's solver loop.

The product is rustsolver_b200/libb200cfr.so (hand-written sm_100a CUDA + C++ host, C ABI in
include/b200cfr.h).  This package is the thin Python face used by the tests and bench.py.
"""
from .solver import (sample_runouts, kmeans_init_pp, kmeans_init_random, ActionAbstraction, CardAbstraction, Engine, EngineError, GameTree, HandIndexer,
                     MCCFRTrainer, Options, Plan, build_game_tree, default_flop, evaluate,
                     get_card_mask, nccl_unique_id, range_from_string)
from .solver import (RS_ABS_BUCKET_TABLE, RS_ABS_CLUSTER_ARR, RS_ABS_ISOMORPHIC, RS_ABS_NONE,
                     RS_FLAG_NO_GRAPH, RS_FLAG_NO_CHAIN_SPLIT, RS_FLAG_STREET_KERNEL, RS_FLAG_SHARD_ISOLATED, RS_DIST_EMD_1D, RS_DIST_L2,
                     RS_RULE_VANILLA, RS_RULE_DCFR, RS_RULE_LCFR, RS_RULE_CFR_PLUS)
from .solver import generate_histograms, histogram_distances, kmeans_assign, kmeans_fit_growbatch, kmeans_fit_regular, kmeans_update_min_dists

__all__ = ["sample_runouts", "kmeans_init_pp", "kmeans_init_random", "ActionAbstraction", "CardAbstraction", "Engine", "EngineError", "GameTree", "HandIndexer",
           "MCCFRTrainer", "Options", "Plan", "build_game_tree", "default_flop", "evaluate",
           "get_card_mask", "nccl_unique_id", "range_from_string", "RS_ABS_BUCKET_TABLE",
           "RS_ABS_CLUSTER_ARR", "RS_ABS_ISOMORPHIC", "RS_ABS_NONE", "RS_FLAG_NO_GRAPH", "RS_FLAG_NO_CHAIN_SPLIT", "RS_FLAG_STREET_KERNEL", "RS_FLAG_SHARD_ISOLATED", "RS_DIST_EMD_1D", "RS_DIST_L2",
           "RS_RULE_VANILLA", "RS_RULE_DCFR", "RS_RULE_LCFR", "RS_RULE_CFR_PLUS",
           "generate_histograms", "histogram_distances", "kmeans_assign", "kmeans_fit_growbatch", "kmeans_fit_regular", "kmeans_update_min_dists"]
