"""ctypes declarations for libb200cfr.so (include/b200cfr.h + include/b200cfr_host.h)."""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_HERE = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ.get("RS_ENGINE_LIB", str(_HERE / "libb200cfr.so")))

u8p = C.POINTER(C.c_uint8)
u16p = C.POINTER(C.c_uint16)
u32p = C.POINTER(C.c_uint32)
u64p = C.POINTER(C.c_uint64)
i32p = C.POINTER(C.c_int32)
f32p = C.POINTER(C.c_float)
f64p = C.POINTER(C.c_double)

RS_NCCL_ID_BYTES = 128
RS_EXCHANGE_HANDLE_BYTES = 64


class rs_tree(C.Structure):
    _fields_ = [("n_nodes", C.c_uint32), ("type", u8p), ("parent", i32p), ("child_offset", u32p),
                ("children", u32p), ("player", u8p), ("an_index", u32p), ("round_idx", u8p),
                ("value", u32p), ("ttype", u8p), ("last_to_act", u8p)]


class rs_ranges(C.Structure):
    _fields_ = [("n_hands", C.c_uint32 * 2), ("hands", u8p * 2)]


class rs_round_abstraction(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("cluster_arr", u32p), ("cluster_arr_len", C.c_uint64),
                ("bucket_table", u32p * 2)]


class rs_abstraction(C.Structure):
    _fields_ = [("n_rounds", C.c_uint32), ("rounds", rs_round_abstraction * 3)]


class rs_config(C.Structure):
    _fields_ = [("board_mask", C.c_uint64), ("device", C.c_int32), ("rank", C.c_int32),
                ("world_size", C.c_int32), ("nccl_id", C.c_uint8 * RS_NCCL_ID_BYTES),
                ("flags", C.c_uint32), ("threads_per_block", C.c_uint32),
                ("discount_interval", C.c_uint64), ("discount_cap", C.c_uint64)]


class rs_stats(C.Structure):
    _fields_ = [("iterations", C.c_uint64), ("updates_per_iteration", C.c_uint64),
                ("updates_per_iteration_global", C.c_uint64), ("device_ms", C.c_double),
                ("kernel_launches", C.c_uint64), ("table_bytes", C.c_uint64), ("n_rounds", C.c_uint32),
                ("n_boards", C.c_uint32 * 3), ("n_boards_local", C.c_uint32 * 3),
                ("n_hands", C.c_uint32 * 2), ("n_combos", C.c_uint64)]


class rs_update_rule(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("alpha", C.c_float), ("beta", C.c_float), ("gamma", C.c_float)]


class rs_kernel_time(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("phase", C.c_uint32), ("traverser", C.c_uint32), ("grid", C.c_uint32),
                ("ms", C.c_float), ("table_bytes", C.c_uint64), ("vector_bytes", C.c_uint64)]


# every symbol the two headers declare: name -> (restype, argtypes)
VP = C.c_void_p
ENGINE_API = {
    "rs_last_error": (C.c_char_p, []),
    "rs_version": (C.c_int, []),
    "rs_device_count": (C.c_int, []),
    "rs_nccl_unique_id": (C.c_int, [u8p]),
    "rs_kmeans_assign": (C.c_int, [f32p, C.c_size_t, C.c_uint32, f32p, C.c_uint32, C.c_uint32, u32p, f32p, f64p, f32p]),
    "rs_kmeans_fit_regular": (C.c_int, [f32p, C.c_size_t, C.c_uint32, f32p, C.c_uint32, C.c_uint32, C.c_uint32, u32p, f32p]),
    "rs_histogram_distances": (C.c_int, [f32p, f32p, C.c_size_t, C.c_uint32, C.c_uint32, f32p]),
    "rs_kmeans_update_min_dists": (C.c_int, [f32p, C.c_size_t, C.c_uint32, f32p, C.c_uint32, f32p]),
    "rs_kmeans_init_pp": (C.c_int, [f32p, C.c_size_t, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint64, u32p, f32p]),
    "rs_generate_histograms": (C.c_int, [C.c_uint32, C.c_uint64, C.c_size_t, C.c_uint32, C.c_uint32, C.c_uint64, f32p, u8p, f32p]),
    "rs_kmeans_fit_growbatch": (C.c_int, [f32p, C.c_size_t, C.c_uint32, f32p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint64, u32p, u32p, f32p]),
    "rs_kmeans_init_random": (C.c_int, [f32p, C.c_size_t, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint64, u32p, f32p]),
    "rs_gpu_index_hands": (C.c_int, [C.c_uint32, u8p, C.c_size_t, u64p, f32p]),
    "rs_exchange_export": (C.c_int, [VP, u8p]),
    "rs_exchange_import": (C.c_int, [VP, u8p, C.c_uint32]),
    "rs_exchange_disable": (C.c_int, [VP]),
    "rs_create": (C.c_int, [C.POINTER(rs_tree), C.POINTER(rs_ranges), C.POINTER(rs_abstraction),
                            C.POINTER(rs_config), C.POINTER(VP)]),
    "rs_create_batch": (C.c_int, [C.POINTER(rs_tree), C.POINTER(rs_ranges), C.POINTER(rs_abstraction),
                                  C.POINTER(rs_config), u64p, C.c_uint32, C.POINTER(VP)]),
    "rs_destroy": (None, [VP]),
    "rs_iterate": (C.c_int, [VP, C.c_uint64]),
    "rs_iterate_sampled": (C.c_int, [VP, u8p, C.c_uint32]),
    "rs_discount": (C.c_int, [VP, C.c_float]),
    "rs_set_prune_threshold": (C.c_int, [VP, C.c_float]),
    "rs_set_opponent_sampling": (C.c_int, [VP, C.c_uint32, C.c_uint64]),
    "rs_set_wait_timeout_ms": (C.c_int, [VP, C.c_uint64]),
    "rs_abort": (C.c_int, [VP]),
    "rs_sample_runouts": (C.c_int, [C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32, C.c_int, u8p]),
    "rs_set_update_rule": (C.c_int, [VP, C.POINTER(rs_update_rule)]),
    "rs_get_update_rule": (C.c_int, [VP, C.POINTER(rs_update_rule), u64p]),
    "rs_reset": (C.c_int, [VP]),
    "rs_read_infoset": (C.c_int, [VP, C.c_uint32, C.c_uint32, f32p, f32p, C.c_size_t, u32p, u32p]),
    "rs_write_infoset": (C.c_int, [VP, C.c_uint32, C.c_uint32, f32p, f32p, C.c_size_t]),
    "rs_average_strategy": (C.c_int, [VP, C.c_uint32, C.c_uint32, f32p, C.c_size_t, u32p, u32p]),
    "rs_dump_average_strategy": (C.c_int, [VP, C.c_char_p, u64p]),
    "rs_current_strategy": (C.c_int, [VP, C.c_uint32, C.c_uint32, f32p, C.c_size_t, u32p, u32p]),
    "rs_board_id": (C.c_int, [VP, C.c_uint32, u8p, C.c_uint32, u32p]),
    "rs_card_table": (C.c_int, [VP, C.c_uint32, C.c_uint32, C.c_uint32, u16p, C.c_size_t, u32p]),
    "rs_best_response": (C.c_int, [VP, f64p]),
    "rs_average_value": (C.c_int, [VP, f64p]),
    "rs_root_values": (C.c_int, [VP, C.c_uint32, f32p, C.c_size_t]),
    "rs_stats_get": (C.c_int, [VP, C.POINTER(rs_stats)]),
    "rs_set_range_weights": (C.c_int, [VP, C.c_uint32, f32p, C.c_size_t]),
    "rs_profile_iteration": (C.c_int, [VP, C.POINTER(rs_kernel_time), C.c_size_t, u32p]),
    "rs_debug_task_timing": (C.c_int, [VP, u64p, C.c_int]),
    "rs_plan_create": (C.c_int, [C.POINTER(rs_tree), C.POINTER(rs_ranges), C.POINTER(rs_abstraction),
                                 C.POINTER(rs_config), u64p, C.c_uint32, C.POINTER(VP)]),
    "rs_plan_destroy": (None, [VP]),
    "rs_plan_stats": (C.c_int, [VP, C.POINTER(rs_stats)]),
    "rs_plan_board_id": (C.c_int, [VP, C.c_uint32, u8p, C.c_uint32, u32p]),
    "rs_plan_card_table": (C.c_int, [VP, C.c_uint32, C.c_uint32, C.c_uint32, u16p, C.c_size_t, u32p]),
    "rs_plan_infoset_offset": (C.c_int, [VP, C.c_uint32, C.c_uint32, u64p, u32p, u32p]),
    "rs_plan_showdown_order": (C.c_int, [VP, C.c_uint32, C.c_uint32, u16p, u32p, C.c_size_t, u32p]),
    "rs_plan_local_tables": (C.c_int, [VP, C.c_uint32, C.c_uint32, C.c_uint32, u32p, u16p, u16p, u32p]),
    "rs_plan_check_execution_order": (C.c_int, [VP, C.c_uint32, C.c_int, u32p, u32p]),
    "rs_plan_street_info": (C.c_int, [VP, C.c_uint32, u32p]),
    "rs_plan_street_program": (C.c_int, [VP, C.c_uint32, C.c_uint32, u32p, C.c_size_t, u32p, u32p, C.c_size_t, u32p]),
}
HOST_API = {
    "rsh_options_default_flop": (VP, []),
    "rsh_options_new": (VP, [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32]),
    "rsh_options_free": (None, [VP]),
    "rsh_options_set_sizes": (C.c_int, [VP, C.c_uint32, u32p, f64p, u32p, f64p]),
    "rsh_options_set_range": (C.c_int, [VP, C.c_uint32, C.c_char_p]),
    "rsh_options_set_range_hands": (C.c_int, [VP, C.c_uint32, u8p, C.c_uint32]),
    "rsh_options_board_mask": (C.c_uint64, [VP]),
    "rsh_options_range": (C.c_int, [VP, C.c_uint32, u8p, C.c_size_t]),
    "rsh_build_game_tree": (C.c_int, [VP, C.POINTER(VP)]),
    "rsh_tree_free": (None, [VP]),
    "rsh_tree_n_nodes": (C.c_uint32, [VP]),
    "rsh_tree_n_actions": (C.c_uint32, [VP]),
    "rsh_tree_n_edges": (C.c_uint32, [VP]),
    "rsh_tree_view": (C.c_int, [VP, C.POINTER(rs_tree)]),
    "rsh_tree_round": (u8p, [VP]),
    "rsh_tree_action_kind": (u8p, [VP]),
    "rsh_tree_action_amount": (f64p, [VP]),
    "rsh_evaluate": (C.c_uint32, [u8p, C.c_uint32]),
    "rsh_get_card_mask": (C.c_int, [C.c_char_p, u64p]),
    "rsh_range_from_string": (C.c_int, [C.c_char_p, C.c_uint64, u8p, C.c_size_t]),
    "rsh_indexer_new": (VP, [C.c_uint32, u8p]),
    "rsh_indexer_free": (None, [VP]),
    "rsh_indexer_size": (C.c_uint64, [VP, C.c_uint32]),
    "rsh_indexer_index": (C.c_uint64, [VP, u8p]),
    "rsh_indexer_index_many": (None, [VP, u8p, C.c_size_t, u64p]),
    "rsh_indexer_get_hand": (C.c_int, [VP, C.c_uint32, C.c_uint64, u8p]),
}

_lib = None


def load():
    """Load libb200cfr.so; raises (never falls back) when the extension is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -m rustsolver_b200.build` "
            "(there is no CPU/Python fallback for the engine)")
    # torch bundles the NCCL the engine dlopens for board-sharded runs; point at it if present
    if "RS_NCCL_LIB" not in os.environ:
        try:
            import importlib.util
            spec = importlib.util.find_spec("nvidia.nccl")
            if spec and spec.submodule_search_locations:
                cand = Path(list(spec.submodule_search_locations)[0]) / "lib" / "libnccl.so.2"
                if cand.exists():
                    os.environ["RS_NCCL_LIB"] = str(cand)
        except Exception:
            pass
    lib = C.CDLL(str(LIB_PATH))
    for table in (ENGINE_API, HOST_API):
        for name, (res, args) in table.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
    _lib = lib
    return lib


class EngineError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"b200cfr error {code}: {msg}")
        self.code = code


def check(rc: int):
    if rc != 0:
        raise EngineError(rc, load().rs_last_error().decode())
