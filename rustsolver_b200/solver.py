"""Python face of the host-side mirror: the names a user of RustSolver's `src/solver` knows.

    Options / ActionAbstraction / default_flop()        options.rs, action_abstraction.rs
    build_game_tree(options) -> (n_actions, GameTree)   tree_builder.rs:9-14
    MCCFRTrainer.init(options) / .train(iterations)     cfr.rs:159-297
    trainer.get_strategy / get_final_strategy           infoset.rs:83-123
    trainer.calc_br()                                   cfr.rs:629-638

Everything heavy happens behind the C ABI of libb200cfr.so (include/b200cfr.h); numpy arrays are
the host buffers.  There is no Python or CPU fallback: without the built library `load()` raises,
and without a B200-class device `MCCFRTrainer.init` raises EngineError.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import List, Optional, Sequence

import numpy as np

from . import _lib
from ._lib import (EngineError, check, f32p, f64p, i32p, rs_abstraction, rs_config, rs_ranges,
                   rs_round_abstraction, rs_stats, rs_tree, rs_update_rule, u8p, u16p, u32p, u64p)

RS_ABS_NONE, RS_ABS_ISOMORPHIC, RS_ABS_CLUSTER_ARR, RS_ABS_BUCKET_TABLE = 0, 1, 2, 3
RS_FLAG_NO_GRAPH = 1
RS_FLAG_NO_CHAIN_SPLIT = 2
RS_FLAG_STREET_KERNEL = 4
RS_FLAG_SHARD_ISOLATED = 8
RS_RULE_VANILLA, RS_RULE_DCFR, RS_RULE_LCFR, RS_RULE_CFR_PLUS = 0, 1, 2, 3
NODE_ACTION, NODE_TERMINAL, NODE_PUBLIC_CHANCE, NODE_PRIVATE_CHANCE = 0, 1, 2, 3
TERM_ALLIN, TERM_SHOWDOWN, TERM_UNCONTESTED = 0, 1, 2
ACTION_NAMES = {0: "Bet", 1: "Raise", 2: "Check", 3: "Call", 4: "Fold"}


def _ptr(a: np.ndarray, t):
    return a.ctypes.data_as(t)


def get_card_mask(s: str) -> int:
    """rust_poker::hand_range::get_card_mask (options.rs:57)."""
    m = C.c_uint64()
    check(_lib.load().rsh_get_card_mask(s.encode(), C.byref(m)))
    return m.value


def range_from_string(s: str, board_mask: int = 0) -> np.ndarray:
    """HandRange::from_string + remove_invalid_combos -> uint8 [n, 2]."""
    lib = _lib.load()
    out = np.zeros((1326, 2), dtype=np.uint8)
    n = lib.rsh_range_from_string(s.encode(), board_mask, _ptr(out, u8p), 1326)
    if n < 0:
        check(n)
    return out[:n].copy()


def evaluate(cards: Sequence[int]) -> int:
    a = np.asarray(cards, dtype=np.uint8)
    return int(_lib.load().rsh_evaluate(_ptr(a, u8p), len(a)))


@dataclass
class ActionAbstraction:
    bet_sizes: List[List[float]] = field(default_factory=list)
    raise_sizes: List[List[float]] = field(default_factory=list)


@dataclass
class Options:
    """options.rs:10-28, field for field (hand_ranges as range strings or uint8 [n,2] arrays)."""
    n_players: int = 2
    hand_ranges: List = field(default_factory=lambda: ["random", "random"])
    stack_sizes: List[int] = field(default_factory=lambda: [500, 500])
    board_mask: int = 0
    starting_pot: int = 0
    all_in_threshold: float = 0.67  # declared, never read by the rules (state.rs uses constants.rs)
    action_abstraction: ActionAbstraction = field(default_factory=ActionAbstraction)
    max_raises: int = 2  # declared, never read

    def _handle(self):
        lib = _lib.load()
        h = lib.rsh_options_new(self.board_mask, self.starting_pot, self.stack_sizes[0], self.stack_sizes[1])
        aa = self.action_abstraction
        nb = np.asarray([len(x) for x in aa.bet_sizes], dtype=np.uint32)
        nr = np.asarray([len(x) for x in aa.raise_sizes], dtype=np.uint32)
        if len(nb) != len(nr):
            lib.rsh_options_free(h)
            raise ValueError("bet_sizes and raise_sizes need one entry per round")
        bets = np.asarray([v for x in aa.bet_sizes for v in x] + [0.0], dtype=np.float64)
        raises = np.asarray([v for x in aa.raise_sizes for v in x] + [0.0], dtype=np.float64)
        check(lib.rsh_options_set_sizes(h, len(nb), _ptr(nb, u32p), _ptr(bets, f64p), _ptr(nr, u32p), _ptr(raises, f64p)))
        try:
            for p in range(2):
                r = self.hand_ranges[p]
                if isinstance(r, str):
                    check(lib.rsh_options_set_range(h, p, r.encode()))
                else:
                    a = np.ascontiguousarray(r, dtype=np.uint8)
                    check(lib.rsh_options_set_range_hands(h, p, _ptr(a, u8p), len(a)))
        except Exception:
            lib.rsh_options_free(h)
            raise
        return h

    def ranges(self) -> List[np.ndarray]:
        """hand_ranges after remove_invalid_combos (cfr.rs:161-163)."""
        lib = _lib.load()
        h = self._handle()
        try:
            out = []
            for p in range(2):
                buf = np.zeros((1326, 2), dtype=np.uint8)
                n = lib.rsh_options_range(h, p, _ptr(buf, u8p), 1326)
                if n < 0:
                    check(n)
                out.append(buf[:n].copy())
            return out
        finally:
            lib.rsh_options_free(h)


def default_flop() -> Options:
    """options::default_flop() (options.rs:52-81) — a river spot despite its name."""
    return Options(n_players=2, stack_sizes=[500, 500], board_mask=get_card_mask("4d5dAs3cKs"), starting_pot=35,
                   all_in_threshold=0.67, max_raises=2, hand_ranges=["random", "random"],
                   action_abstraction=ActionAbstraction(bet_sizes=[[0.5, 1.0]], raise_sizes=[[3.0]]))


class GameTree:
    """Tree<GameTreeNode> (tree.rs:12-24) flattened into numpy arrays; node id = arena index."""

    def __init__(self, type, parent, child_offset, children, player, an_index, round_idx, value, ttype,
                 last_to_act, round=None, action_kind=None, action_amount=None):
        self.type = np.ascontiguousarray(type, dtype=np.uint8)
        self.parent = np.ascontiguousarray(parent, dtype=np.int32)
        self.child_offset = np.ascontiguousarray(child_offset, dtype=np.uint32)
        self.children = np.ascontiguousarray(children, dtype=np.uint32)
        self.player = np.ascontiguousarray(player, dtype=np.uint8)
        self.an_index = np.ascontiguousarray(an_index, dtype=np.uint32)
        self.round_idx = np.ascontiguousarray(round_idx, dtype=np.uint8)
        self.value = np.ascontiguousarray(value, dtype=np.uint32)
        self.ttype = np.ascontiguousarray(ttype, dtype=np.uint8)
        self.last_to_act = np.ascontiguousarray(last_to_act, dtype=np.uint8)
        self.round = None if round is None else np.ascontiguousarray(round, dtype=np.uint8)
        self.action_kind = None if action_kind is None else np.ascontiguousarray(action_kind, dtype=np.uint8)
        self.action_amount = None if action_amount is None else np.ascontiguousarray(action_amount, dtype=np.float64)

    @property
    def n_nodes(self) -> int:
        return len(self.type)

    @property
    def n_actions(self) -> int:
        return int((self.type == NODE_ACTION).sum())

    def children_of(self, i: int) -> np.ndarray:
        return self.children[self.child_offset[i]:self.child_offset[i + 1]]

    def view(self) -> rs_tree:
        t = rs_tree()
        t.n_nodes = self.n_nodes
        t.type = _ptr(self.type, u8p)
        t.parent = _ptr(self.parent, i32p)
        t.child_offset = _ptr(self.child_offset, u32p)
        t.children = _ptr(self.children, u32p)
        t.player = _ptr(self.player, u8p)
        t.an_index = _ptr(self.an_index, u32p)
        t.round_idx = _ptr(self.round_idx, u8p)
        t.value = _ptr(self.value, u32p)
        t.ttype = _ptr(self.ttype, u8p)
        t.last_to_act = _ptr(self.last_to_act, u8p)
        return t

    def dump(self) -> List[str]:
        """One line per node in the notation of SURVEY.md Appendix A."""
        out = []
        for i in range(self.n_nodes):
            ch = [int(c) for c in self.children_of(i)]
            t = self.type[i]
            if t == NODE_PRIVATE_CHANCE:
                out.append(f"{i} P ->{ch}")
            elif t == NODE_PUBLIC_CHANCE:
                out.append(f"{i} C ->{ch}")
            elif t == NODE_TERMINAL:
                k = {TERM_ALLIN: "L", TERM_SHOWDOWN: "S", TERM_UNCONTESTED: "U"}[int(self.ttype[i])]
                out.append(f"{i} {k} {int(self.value[i])}/{int(self.last_to_act[i])}")
            else:
                acts = []
                for e in range(self.child_offset[i], self.child_offset[i + 1]):
                    kind = int(self.action_kind[e])
                    amt = float(self.action_amount[e])
                    acts.append({2: "X", 3: "C", 4: "F"}.get(kind) or (("B" if kind == 0 else "R") + f"{amt:g}"))
                out.append(f"{i} A {int(self.an_index[i])}/P{int(self.player[i])} [{','.join(acts)}] ->{ch}")
        return out


def build_game_tree(options: Options):
    """tree_builder.rs:9-14 -> (n_actions, GameTree).  Raises EngineError where the reference panics."""
    lib = _lib.load()
    h = options._handle()
    th = C.c_void_p()
    try:
        check(lib.rsh_build_game_tree(h, C.byref(th)))
    finally:
        lib.rsh_options_free(h)
    try:
        v = rs_tree()
        check(lib.rsh_tree_view(th, C.byref(v)))
        n = v.n_nodes
        ne = lib.rsh_tree_n_edges(th)

        def arr(p, count, dt):
            return np.ctypeslib.as_array(p, shape=(count,)).astype(dt, copy=True) if count else np.zeros(0, dt)

        tree = GameTree(arr(v.type, n, np.uint8), arr(v.parent, n, np.int32), arr(v.child_offset, n + 1, np.uint32),
                        arr(v.children, ne, np.uint32), arr(v.player, n, np.uint8), arr(v.an_index, n, np.uint32),
                        arr(v.round_idx, n, np.uint8), arr(v.value, n, np.uint32), arr(v.ttype, n, np.uint8),
                        arr(v.last_to_act, n, np.uint8), arr(lib.rsh_tree_round(th), n, np.uint8),
                        arr(lib.rsh_tree_action_kind(th), ne, np.uint8), arr(lib.rsh_tree_action_amount(th), ne, np.float64))
        return int(lib.rsh_tree_n_actions(th)), tree
    finally:
        lib.rsh_tree_free(th)


RS_DIST_EMD_1D, RS_DIST_L2 = 0, 1


def kmeans_assign(points: np.ndarray, centers: np.ndarray, dist: int = RS_DIST_EMD_1D, return_ms: bool = False):
    """Kmeans::predict (gen_abstraction/kmeans.rs:173-211) on the GPU: (cluster[n], min_dist[n], inertia[, kernel ms])."""
    lib = _lib.load()
    x = np.ascontiguousarray(points, dtype=np.float32)
    c = np.ascontiguousarray(centers, dtype=np.float32)
    assert x.ndim == 2 and c.ndim == 2 and x.shape[1] == c.shape[1]
    cl = np.zeros(len(x), dtype=np.uint32)
    md = np.zeros(len(x), dtype=np.float32)
    inertia, ms = C.c_double(0.0), C.c_float(0.0)
    check(lib.rs_kmeans_assign(_ptr(x, f32p), len(x), x.shape[1], _ptr(c, f32p), len(c), dist, _ptr(cl, u32p), _ptr(md, f32p),
                               C.byref(inertia), C.byref(ms)))
    return (cl, md, float(inertia.value), float(ms.value)) if return_ms else (cl, md, float(inertia.value))


def kmeans_fit_regular(points: np.ndarray, centers: np.ndarray, dist: int = RS_DIST_EMD_1D, rounds: int = 10):
    """Kmeans::fit_regular (gen_abstraction/kmeans.rs:497-599) on the GPU: (cluster[n], new centers[k][dim], inertia)."""
    lib = _lib.load()
    x = np.ascontiguousarray(points, dtype=np.float32)
    c = np.array(centers, dtype=np.float32, copy=True, order="C")
    assert x.ndim == 2 and c.ndim == 2 and x.shape[1] == c.shape[1]
    cl = np.zeros(len(x), dtype=np.uint32)
    inertia = C.c_float(0.0)
    check(lib.rs_kmeans_fit_regular(_ptr(x, f32p), len(x), x.shape[1], _ptr(c, f32p), len(c), dist, rounds, _ptr(cl, u32p),
                                    C.byref(inertia)))
    return cl, c, float(inertia.value)


def generate_histograms(round_: int, first_index: int, count: int, samples: int, bins: int, seed: int = 1, return_ms: bool = False):
    """generate_histograms (gen_abstraction/main.rs:79-159) on the GPU with the EHS computed exactly instead of read from
    ehs.dat: (histograms [count][bins], un-indexed hands [count][7])."""
    lib = _lib.load()
    out = np.zeros((count, bins), dtype=np.float32)
    cards = np.zeros((count, 7), dtype=np.uint8)
    ms = C.c_float(0.0)
    check(lib.rs_generate_histograms(round_, first_index, count, samples, bins, seed, _ptr(out, f32p), _ptr(cards, u8p), C.byref(ms)))
    return (out, cards, float(ms.value)) if return_ms else (out, cards)


def kmeans_fit_growbatch(points: np.ndarray, centers: np.ndarray, initial_batch_size: int, dist: int = RS_DIST_EMD_1D, seed: int = 1):
    """Kmeans::fit_growbatch (kmeans.rs:336-494; one pass, its loop ends with `break`) on the GPU:
    (batch indices [batch], cluster [batch], new centers [k][dim], min_change, inertia)."""
    lib = _lib.load()
    x = np.ascontiguousarray(points, dtype=np.float32)
    c = np.array(centers, dtype=np.float32, copy=True, order="C")
    assert x.ndim == 2 and c.ndim == 2 and x.shape[1] == c.shape[1]
    idx = np.zeros(initial_batch_size, dtype=np.uint32)
    cl = np.zeros(initial_batch_size, dtype=np.uint32)
    stats = np.zeros(2, dtype=np.float32)
    check(lib.rs_kmeans_fit_growbatch(_ptr(x, f32p), len(x), x.shape[1], _ptr(c, f32p), len(c), dist, initial_batch_size, seed,
                                      _ptr(idx, u32p), _ptr(cl, u32p), _ptr(stats, f32p)))
    return idx, cl, c, float(stats[0]), float(stats[1])


def histogram_distances(p: np.ndarray, q: np.ndarray, dist: int = RS_DIST_EMD_1D) -> np.ndarray:
    """out[i] = emd_1d(p[i], q[i]) (emd.rs:54-113) or l2_dist (kmeans.rs:622-630) on the GPU."""
    lib = _lib.load()
    a = np.ascontiguousarray(p, dtype=np.float32)
    b = np.ascontiguousarray(q, dtype=np.float32)
    assert a.shape == b.shape and a.ndim == 2
    out = np.zeros(len(a), dtype=np.float32)
    check(lib.rs_histogram_distances(_ptr(a, f32p), _ptr(b, f32p), len(a), a.shape[1], dist, _ptr(out, f32p)))
    return out


def kmeans_update_min_dists(points: np.ndarray, new_center: np.ndarray, min_dists: np.ndarray, dist: int = RS_DIST_EMD_1D) -> np.ndarray:
    """update_min_dists (kmeans.rs:603-619) on the GPU; returns the updated copy."""
    lib = _lib.load()
    x = np.ascontiguousarray(points, dtype=np.float32)
    c = np.ascontiguousarray(new_center, dtype=np.float32)
    md = np.array(min_dists, dtype=np.float32, copy=True)
    check(lib.rs_kmeans_update_min_dists(_ptr(x, f32p), len(x), x.shape[1], _ptr(c, f32p), dist, _ptr(md, f32p)))
    return md


def kmeans_init_pp(points: np.ndarray, k: int, dist: int = RS_DIST_EMD_1D, seed: int = 1):
    """Kmeans::init_pp (kmeans.rs:60-90) on the GPU with the stated splitmix64 stream: (chosen indices [k], centres [k][dim])."""
    lib = _lib.load()
    x = np.ascontiguousarray(points, dtype=np.float32)
    chosen = np.zeros(k, dtype=np.uint32)
    centers = np.zeros((k, x.shape[1]), dtype=np.float32)
    check(lib.rs_kmeans_init_pp(_ptr(x, f32p), len(x), x.shape[1], k, dist, seed, _ptr(chosen, u32p), _ptr(centers, f32p)))
    return chosen, centers


def kmeans_init_random(points: np.ndarray, k: int, n_restarts: int, dist: int = RS_DIST_EMD_1D, seed: int = 1):
    """Kmeans::init_random (kmeans.rs:103-166) on the GPU: (chosen indices [k], centres [k][dim]) of the most spread out set."""
    lib = _lib.load()
    x = np.ascontiguousarray(points, dtype=np.float32)
    chosen = np.zeros(k, dtype=np.uint32)
    centers = np.zeros((k, x.shape[1]), dtype=np.float32)
    check(lib.rs_kmeans_init_random(_ptr(x, f32p), len(x), x.shape[1], k, n_restarts, dist, seed, _ptr(chosen, u32p), _ptr(centers, f32p)))
    return chosen, centers


class HandIndexer:
    """rust_poker::hand_indexer_s (card_abstraction.rs:88-90)."""

    def __init__(self, cards_per_round: Sequence[int]):
        self._lib = _lib.load()
        cpr = np.asarray(cards_per_round, dtype=np.uint8)
        self.cards_per_round = [int(x) for x in cpr]
        self._h = self._lib.rsh_indexer_new(len(cpr), _ptr(cpr, u8p))
        if not self._h:
            raise EngineError(-1, self._lib.rs_last_error().decode())

    def __del__(self):
        if getattr(self, "_h", None):
            self._lib.rsh_indexer_free(self._h)
            self._h = None

    def size(self, round: int) -> int:
        return int(self._lib.rsh_indexer_size(self._h, round))

    def get_index(self, cards: Sequence[int]) -> int:
        a = np.asarray(cards, dtype=np.uint8)
        return int(self._lib.rsh_indexer_index(self._h, _ptr(a, u8p)))

    def index_many(self, cards: np.ndarray) -> np.ndarray:
        a = np.ascontiguousarray(cards, dtype=np.uint8)
        assert a.ndim == 2 and a.shape[1] == sum(self.cards_per_round)
        out = np.zeros(len(a), dtype=np.uint64)
        self._lib.rsh_indexer_index_many(self._h, _ptr(a, u8p), len(a), _ptr(out, u64p))
        return out

    def index_many_gpu(self, cards: np.ndarray, return_ms: bool = False):
        """index_many on the device (rs_gpu_index_hands): indexer must be [2, 3|4|5]; fails without a GPU."""
        assert len(self.cards_per_round) == 2 and self.cards_per_round[0] == 2
        a = np.ascontiguousarray(cards, dtype=np.uint8)
        assert a.ndim == 2 and a.shape[1] == sum(self.cards_per_round)
        out = np.zeros(len(a), dtype=np.uint64)
        ms = C.c_float(0.0)
        check(self._lib.rs_gpu_index_hands(self.cards_per_round[1], _ptr(a, u8p), len(a), _ptr(out, u64p), C.byref(ms)))
        return (out, float(ms.value)) if return_ms else out

    def get_hand(self, round: int, index: int) -> List[int]:
        n = sum(self.cards_per_round[:round + 1])
        out = np.zeros(n, dtype=np.uint8)
        check(self._lib.rsh_indexer_get_hand(self._h, round, index, _ptr(out, u8p)))
        return [int(x) for x in out]


@dataclass
class CardAbstraction:
    """One entry of MCCFRTrainer.card_abs (cfr.rs:167-172; card_abstraction.rs:62-66)."""
    kind: int = RS_ABS_NONE
    cluster_arr: Optional[np.ndarray] = None        # EMD / OCHS: contents of round_N_{emd,ochs}.dat
    bucket_table: Optional[List[np.ndarray]] = None  # explicit keys [n_boards, n_hands] per player

    @staticmethod
    def ISOMORPHIC():
        return CardAbstraction(RS_ABS_ISOMORPHIC)

    @staticmethod
    def NONE():
        return CardAbstraction(RS_ABS_NONE)

    @staticmethod
    def from_file(path: str):
        """EMD::init / OCHS::init: headerless little-endian u32 per canonical index (card_abstraction.rs:227-229)."""
        return CardAbstraction(RS_ABS_CLUSTER_ARR, cluster_arr=np.fromfile(path, dtype="<u4"))


def _abstraction_struct(card_abs: Sequence[CardAbstraction], keep: list) -> rs_abstraction:
    ab = rs_abstraction()
    ab.n_rounds = len(card_abs)
    for k, ca in enumerate(card_abs):
        ra = ab.rounds[k]
        ra.kind = ca.kind
        if ca.kind == RS_ABS_CLUSTER_ARR:
            arr = np.ascontiguousarray(ca.cluster_arr, dtype=np.uint32)
            keep.append(arr)
            ra.cluster_arr = _ptr(arr, u32p)
            ra.cluster_arr_len = len(arr)
        if ca.kind == RS_ABS_BUCKET_TABLE:
            for p in range(2):
                arr = np.ascontiguousarray(ca.bucket_table[p], dtype=np.uint32)
                keep.append(arr)
                ra.bucket_table[p] = _ptr(arr, u32p)
    return ab


def nccl_unique_id() -> bytes:
    buf = (C.c_uint8 * _lib.RS_NCCL_ID_BYTES)()
    check(_lib.load().rs_nccl_unique_id(buf))
    return bytes(buf)


class _PlanOrEngine:
    """Shared accessors of rs_plan (host only) and rs_engine."""
    _prefix = "rs_"

    def _fn(self, name):
        return getattr(self._lib, self._prefix + name)

    def board_id(self, round_idx: int, dealt: Sequence[int]) -> int:
        a = np.asarray(list(dealt) + [0], dtype=np.uint8)
        out = C.c_uint32()
        check(self._fn("board_id")(self._h, round_idx, _ptr(a, u8p), len(dealt), C.byref(out)))
        return out.value

    def card_table(self, round_idx: int, player: int, board_id: int) -> np.ndarray:
        """card table (README.md:36-39): hand slot -> row, 0xFFFF where the hand hits the board."""
        out = np.zeros(self.n_hands[player], dtype=np.uint16)
        nr = C.c_uint32()
        check(self._fn("card_table")(self._h, round_idx, player, board_id, _ptr(out, u16p), len(out), C.byref(nr)))
        return out

    def num_rows(self, round_idx: int, player: int, board_id: int) -> int:
        nr = C.c_uint32()
        check(self._fn("card_table")(self._h, round_idx, player, board_id, None, 0, C.byref(nr)))
        return nr.value


class Plan(_PlanOrEngine):
    """Host-only compile of the engine's integer tables (no GPU): board/card tables, slab offsets."""
    _prefix = "rs_plan_"

    def __init__(self, tree: GameTree, ranges: Sequence[np.ndarray], board_mask: int,
                 card_abs: Sequence[CardAbstraction] = (), board_masks: Optional[Sequence[int]] = None,
                 rank: int = 0, world_size: int = 1, flags: int = 0):
        self._lib = _lib.load()
        self._keep = []
        tv = tree.view()
        rr = rs_ranges()
        hs = [np.ascontiguousarray(r, dtype=np.uint8) for r in ranges]
        for p in range(2):
            rr.n_hands[p] = len(hs[p])
            rr.hands[p] = _ptr(hs[p], u8p)
        ab = _abstraction_struct(card_abs, self._keep)
        cfg = rs_config()
        cfg.board_mask = board_mask
        cfg.rank, cfg.world_size = rank, world_size
        cfg.flags = flags
        h = C.c_void_p()
        if board_masks is not None:
            bm = np.asarray(board_masks, dtype=np.uint64)
            check(self._lib.rs_plan_create(C.byref(tv), C.byref(rr), C.byref(ab), C.byref(cfg), _ptr(bm, u64p), len(bm), C.byref(h)))
        else:
            check(self._lib.rs_plan_create(C.byref(tv), C.byref(rr), C.byref(ab), C.byref(cfg), None, 0, C.byref(h)))
        self._h = h
        self.n_hands = [len(hs[0]), len(hs[1])]

    def __del__(self):
        if getattr(self, "_h", None):
            self._lib.rs_plan_destroy(self._h)
            self._h = None

    def stats(self) -> rs_stats:
        s = rs_stats()
        check(self._lib.rs_plan_stats(self._h, C.byref(s)))
        return s

    def infoset_offset(self, an_index: int, board_id: int):
        off, nr, na = C.c_uint64(), C.c_uint32(), C.c_uint32()
        check(self._lib.rs_plan_infoset_offset(self._h, an_index, board_id, C.byref(off), C.byref(nr), C.byref(na)))
        return off.value, nr.value, na.value

    def showdown_order(self, player: int, board_id: int):
        order = np.zeros(self.n_hands[player], dtype=np.uint16)
        cls = np.zeros(self.n_hands[player], dtype=np.uint32)
        nl = C.c_uint32()
        check(self._lib.rs_plan_showdown_order(self._h, player, board_id, _ptr(order, u16p), _ptr(cls, u32p), len(order), C.byref(nl)))
        return order[:nl.value].copy(), cls[:nl.value].copy()

    def check_execution_order(self, traverser: int, force_board_major: bool = False):
        """(tickets, slots moved off their task-major ticket); raises EngineError if a consumer could run before a producer."""
        n, moved = C.c_uint32(), C.c_uint32()
        check(self._lib.rs_plan_check_execution_order(self._h, traverser, int(force_board_major), C.byref(n), C.byref(moved)))
        return int(n.value), int(moved.value)

    def local_tables(self, round_idx: int, player: int, board_id: int):
        """(hand records [Hpad][4] u32 of `player` as traverser, card-list entries [2 * Hpad] u16 of `player` as opponent,
        slot_of_pos [Hpad], live hands) in the board-local hand order (csrc/tasks.h)."""
        dims = (C.c_uint32 * 2)()
        check(self._lib.rs_plan_local_tables(self._h, round_idx, player, board_id, None, None, None, dims))
        hp, nl = int(dims[0]), int(dims[1])
        rec = np.zeros((hp, 4), dtype=np.uint32)
        cl = np.zeros(2 * hp, dtype=np.uint16)
        sop = np.zeros(hp, dtype=np.uint16)
        check(self._lib.rs_plan_local_tables(self._h, round_idx, player, board_id, _ptr(rec, u32p), _ptr(cl, u16p), _ptr(sop, u16p), dims))
        return rec, cl, sop, nl

    def street_info(self, traverser: int) -> dict:
        """The final round as fused street programs (csrc/street.h); `why` is set when the round is not eligible."""
        out = (C.c_uint32 * 8)()
        check(self._lib.rs_plan_street_info(self._h, traverser, out))
        keys = ("eligible", "segments", "max_rows", "max_slots", "max_q_sd", "max_q_mo", "down_ops", "up_ops")
        d = dict(zip(keys, [int(x) for x in out]))
        d["why"] = "" if d["eligible"] else self._lib.rs_last_error().decode()
        return d

    def street_program(self, traverser: int, board_id: int) -> dict:
        """List programs of one final-round board (street.h): `lists` [l_steps, 52 * 4] and `chunks` [c_steps, 128] program
        words (one column per piece), `hinfo` [Hpad, 2] per traverser position, `HpP` / `HoP` the padded range sizes."""
        n = C.c_uint32()
        dims = (C.c_uint32 * 4)()
        check(self._lib.rs_plan_street_program(self._h, traverser, board_id, None, 0, C.byref(n), None, 0, dims))
        words = np.zeros(max(n.value, 1), dtype=np.uint32)
        hinfo = np.zeros(2 * dims[2], dtype=np.uint32)
        check(self._lib.rs_plan_street_program(self._h, traverser, board_id, _ptr(words, u32p), len(words), C.byref(n),
                                               _ptr(hinfo, u32p), len(hinfo), dims))
        ls, cs = int(dims[0]), int(dims[1])
        return {"lists": words[:ls * 208].reshape(ls, 208), "chunks": words[ls * 208:ls * 208 + cs * 128].reshape(cs, 128),
                "hinfo": hinfo.reshape(-1, 2), "HpP": int(dims[2]), "HoP": int(dims[3])}


def sample_runouts(seed: int, board_mask: int, n_cards: int, n_paths: int, distinct_first: bool = True) -> np.ndarray:
    """generate_hand's board part (cfr.rs:100-122) behind the ABI (rs_sample_runouts): uint8 [n_paths, n_cards]."""
    out = np.zeros((n_paths, n_cards), dtype=np.uint8)
    check(_lib.load().rs_sample_runouts(seed, board_mask, n_cards, n_paths, int(distinct_first), _ptr(out, u8p)))
    return out


class Engine(_PlanOrEngine):
    """rs_engine handle: the device-resident infoset tables plus the iteration graph."""

    def __init__(self, tree: GameTree, ranges: Sequence[np.ndarray], board_mask: int,
                 card_abs: Sequence[CardAbstraction] = (), board_masks: Optional[Sequence[int]] = None,
                 device: int = 0, rank: int = 0, world_size: int = 1, nccl_id: Optional[bytes] = None,
                 flags: int = 0, threads_per_block: int = 0, discount_interval: int = 0, discount_cap: int = 0):
        self._lib = _lib.load()
        self._keep = []
        self.tree = tree
        tv = tree.view()
        rr = rs_ranges()
        hs = [np.ascontiguousarray(r, dtype=np.uint8) for r in ranges]
        for p in range(2):
            rr.n_hands[p] = len(hs[p])
            rr.hands[p] = _ptr(hs[p], u8p)
        ab = _abstraction_struct(card_abs, self._keep)
        cfg = rs_config()
        cfg.board_mask = board_mask
        cfg.device, cfg.rank, cfg.world_size = device, rank, world_size
        if nccl_id is not None:
            C.memmove(cfg.nccl_id, nccl_id, _lib.RS_NCCL_ID_BYTES)
        cfg.flags = flags
        cfg.threads_per_block = threads_per_block
        cfg.discount_interval, cfg.discount_cap = discount_interval, discount_cap
        h = C.c_void_p()
        if board_masks is not None:
            bm = np.asarray(board_masks, dtype=np.uint64)
            check(self._lib.rs_create_batch(C.byref(tv), C.byref(rr), C.byref(ab), C.byref(cfg), _ptr(bm, u64p), len(bm), C.byref(h)))
        else:
            check(self._lib.rs_create(C.byref(tv), C.byref(rr), C.byref(ab), C.byref(cfg), C.byref(h)))
        self._h = h
        self.n_hands = [len(hs[0]), len(hs[1])]
        self.ranges = hs

    def close(self):
        if getattr(self, "_h", None):
            self._lib.rs_destroy(self._h)
            self._h = None

    __del__ = close

    def iterate(self, n: int = 1):
        check(self._lib.rs_iterate(self._h, n))

    def iterate_sampled(self, paths):
        """One MCCFR-style iteration on sampled run-outs: paths = [[turn, river], ...] dealt cards in deal order."""
        a = np.ascontiguousarray(paths, dtype=np.uint8)
        if a.ndim == 1:
            a = a.reshape(1, -1)
        check(self._lib.rs_iterate_sampled(self._h, _ptr(a, u8p), a.shape[0]))

    def discount(self, d: float):
        check(self._lib.rs_discount(self._h, d))

    def reset(self):
        check(self._lib.rs_reset(self._h))

    def stats(self) -> rs_stats:
        s = rs_stats()
        check(self._lib.rs_stats_get(self._h, C.byref(s)))
        return s

    def _shape(self, an_index: int, board_id: int):
        nr, na = C.c_uint32(), C.c_uint32()
        check(self._lib.rs_read_infoset(self._h, an_index, board_id, None, None, 0, C.byref(nr), C.byref(na)))
        return nr.value, na.value

    def read_infoset(self, an_index: int, board_id: int = 0):
        """-> (regrets, strategy_sum), each float32 [rows, n_actions] (README.md:45-47)."""
        nr, na = self._shape(an_index, board_id)
        r = np.zeros((nr, na), dtype=np.float32)
        s = np.zeros((nr, na), dtype=np.float32)
        check(self._lib.rs_read_infoset(self._h, an_index, board_id, _ptr(r, f32p), _ptr(s, f32p), r.size, None, None))
        return r, s

    def write_infoset(self, an_index: int, board_id: int, regrets: np.ndarray, strategy_sum: np.ndarray):
        r = np.ascontiguousarray(regrets, dtype=np.float32)
        s = np.ascontiguousarray(strategy_sum, dtype=np.float32)
        check(self._lib.rs_write_infoset(self._h, an_index, board_id, _ptr(r, f32p), _ptr(s, f32p), r.size))

    def average_strategy(self, an_index: int, board_id: int = 0) -> np.ndarray:
        nr, na = self._shape(an_index, board_id)
        out = np.zeros((nr, na), dtype=np.float32)
        check(self._lib.rs_average_strategy(self._h, an_index, board_id, _ptr(out, f32p), out.size, None, None))
        return out

    def current_strategy(self, an_index: int, board_id: int = 0) -> np.ndarray:
        nr, na = self._shape(an_index, board_id)
        out = np.zeros((nr, na), dtype=np.float32)
        check(self._lib.rs_current_strategy(self._h, an_index, board_id, _ptr(out, f32p), out.size, None, None))
        return out

    def set_range_weights(self, player: int, weights: np.ndarray):
        """Per-hand reach weights of `player`'s range (host buffer -> device, async on the engine stream)."""
        w = np.ascontiguousarray(weights, dtype=np.float32)
        check(self._lib.rs_set_range_weights(self._h, player, _ptr(w, f32p), w.size))

    def profile_iteration(self):
        """One real iteration launched kernel by kernel with CUDA events -> list of dicts."""
        cap = 64
        buf = (_lib.rs_kernel_time * cap)()
        n = C.c_uint32()
        check(self._lib.rs_profile_iteration(self._h, buf, cap, C.byref(n)))
        kinds = {0: "traversal", 1: "street", 3: "allreduce"}
        return [dict(kind=kinds[buf[i].kind], phase=buf[i].phase, traverser=buf[i].traverser, grid=buf[i].grid,
                     ms=buf[i].ms, table_bytes=buf[i].table_bytes, vector_bytes=buf[i].vector_bytes) for i in range(n.value)]

    def dump_average_strategy(self, path: str) -> int:
        """Headerless LE fp32 dump of the average strategy (rs_dump_average_strategy); returns the number of floats."""
        n = C.c_uint64(0)
        check(self._lib.rs_dump_average_strategy(self._h, str(path).encode(), C.byref(n)))
        return int(n.value)

    def set_prune_threshold(self, threshold: float):
        """Traverser actions with regret <= threshold keep their regret (cfr.rs:352,379-386); -inf = off."""
        check(self._lib.rs_set_prune_threshold(self._h, float(threshold)))

    def set_opponent_sampling(self, mode: int, seed: int = 0):
        """mccfr()'s opponent arm for every hand at once (cfr.rs:466-475): 0 = off, 1 = one sampled action per opponent
        hand and node keeps the whole reach, 2 = keeps reach * sigma(sampled action) as the reference's code does."""
        check(self._lib.rs_set_opponent_sampling(self._h, int(mode), int(seed)))

    def set_update_rule(self, kind: int, alpha: float = 1.5, beta: float = 0.0, gamma: float = 2.0):
        """Update rule of the traverser's table update from the next iteration on (rs_set_update_rule): RS_RULE_VANILLA,
        RS_RULE_DCFR(alpha, beta, gamma), RS_RULE_LCFR or RS_RULE_CFR_PLUS.  Restarts the rule's iteration count t."""
        r = rs_update_rule(int(kind), float(alpha), float(beta), float(gamma))
        check(self._lib.rs_set_update_rule(self._h, C.byref(r)))

    def update_rule(self):
        """-> (kind, alpha, beta, gamma, t): the rule and t of the last iteration run under it."""
        r, t = rs_update_rule(), C.c_uint64()
        check(self._lib.rs_get_update_rule(self._h, C.byref(r), C.byref(t)))
        return r.kind, r.alpha, r.beta, r.gamma, int(t.value)

    def set_wait_timeout_ms(self, ms: int):
        """Bound of every wait inside the traversal kernel (default 30 s, 0 = unbounded): see rs_set_wait_timeout_ms."""
        check(self._lib.rs_set_wait_timeout_ms(self._h, int(ms)))

    def abort(self):
        """Make a running traversal give up (rs_abort); callable from another thread."""
        check(self._lib.rs_abort(self._h))

    def exchange_export(self) -> bytes:
        """Handle of this rank's exchange buffer (board-sharded engines): gather one per rank, then exchange_import."""
        buf = (C.c_uint8 * _lib.RS_EXCHANGE_HANDLE_BYTES)()
        check(self._lib.rs_exchange_export(self._h, buf))
        return bytes(buf)

    def exchange_import(self, handles: Sequence[bytes]):
        """Map every rank's exchange buffer: the traversal kernel then exchanges the chance-node sums itself over
        NVLink peer memory (one launch per traversal, no NCCL call).  Collective: every rank, same point."""
        blob = b"".join(handles)
        assert len(blob) == len(handles) * _lib.RS_EXCHANGE_HANDLE_BYTES
        arr = (C.c_uint8 * len(blob)).from_buffer_copy(blob)
        check(self._lib.rs_exchange_import(self._h, arr, len(handles)))

    def enable_fused_exchange(self, dist, device):
        """All-gather the exchange handles over a torch.distributed group and import them (see exchange_import)."""
        import torch
        mine = torch.tensor(list(self.exchange_export()), dtype=torch.uint8, device=device)
        allh = [torch.zeros_like(mine) for _ in range(dist.get_world_size())]
        dist.all_gather(allh, mine)
        ok = 1
        try:
            self.exchange_import([bytes(h.cpu().tolist()) for h in allh])
        except EngineError as e:  # no peer access between some pair of GPUs: every rank stays on the NCCL path
            print(f"[rustsolver_b200] in-kernel exchange unavailable on this rank: {e}", flush=True)
            ok = 0
        flag = torch.tensor([ok], dtype=torch.int32, device=device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if int(flag.item()) == 0:
            check(self._lib.rs_exchange_disable(self._h))
            return False
        return True

    def best_response(self):
        out = (C.c_double * 2)()
        check(self._lib.rs_best_response(self._h, out))
        return [out[0], out[1]]

    def average_value(self):
        out = (C.c_double * 2)()
        check(self._lib.rs_average_value(self._h, out))
        return [out[0], out[1]]

    def root_values(self, player: int) -> np.ndarray:
        st = self.stats()
        out = np.zeros(st.n_boards_local[0] * self.n_hands[player], dtype=np.float32)
        check(self._lib.rs_root_values(self._h, player, _ptr(out, f32p), out.size))
        return out.reshape(st.n_boards_local[0], self.n_hands[player])


class MCCFRTrainer:
    """MCCFRTrainer of src/solver/cfr.rs:150-297 with its hot path on the GPU."""

    def __init__(self):
        self.engine: Optional[Engine] = None
        self.game_tree: Optional[GameTree] = None
        self.hand_ranges: List[np.ndarray] = []
        self.initial_board_mask = 0
        self.card_abs: List[CardAbstraction] = []

    @staticmethod
    def init(options: Options, card_abs: Optional[Sequence[CardAbstraction]] = None, **engine_kwargs) -> "MCCFRTrainer":
        """cfr.rs:159-184: remove_invalid_combos, build_game_tree, card abstraction, create_infosets."""
        t = MCCFRTrainer()
        t.hand_ranges = options.ranges()
        n_actions, t.game_tree = build_game_tree(options)
        t.initial_board_mask = options.board_mask
        n_rounds = int(t.game_tree.round_idx.max()) + 1
        # the reference instantiates ISOMORPHIC for its single round (cfr.rs:171)
        t.card_abs = list(card_abs) if card_abs is not None else [CardAbstraction.ISOMORPHIC() for _ in range(n_rounds)]
        t.engine = Engine(t.game_tree, t.hand_ranges, options.board_mask, t.card_abs, **engine_kwargs)
        return t

    def train(self, iterations: int):
        """cfr.rs:188-297: each iteration traverses and updates player 0 then player 1 (cfr.rs:216-226)."""
        self.engine.iterate(iterations)

    def get_strategy(self, an_index: int, cluster_idx: int, board_id: int = 0) -> np.ndarray:
        """Infoset::get_strategy (infoset.rs:83-102) of infosets[an_index][cluster_idx]."""
        return self.engine.current_strategy(an_index, board_id)[cluster_idx]

    def get_final_strategy(self, an_index: int, cluster_idx: int, board_id: int = 0) -> np.ndarray:
        """Infoset::get_final_strategy (infoset.rs:104-123)."""
        return self.engine.average_strategy(an_index, board_id)[cluster_idx]

    def calc_br(self) -> List[float]:
        """cfr.rs:629-638 (a stub in the reference; a true best response here)."""
        return self.engine.best_response()

    def exploitability(self, bb: float = 1.0) -> dict:
        br = self.engine.best_response()
        chips = 0.5 * (br[0] + br[1])
        return {"chips": chips, "mbb_per_game": 1000.0 * chips / bb, "br": br}
