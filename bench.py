#!/usr/bin/env python
"""bench.py — CFR iterations/s of the B200 engine on BASELINE.json's workloads.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload config4] [--dump-outputs DIR]

Default workload: config 4 (flop-rooted subgame, 49 turn cards x 48 river cards = 2 352 river boards, 29 GB of infoset
tables: the largest configuration that fits one B200 and the one north_star names for board sharding).  The same run
also measures config 2 (turn + river, 48 river boards) and config 5 (512 independent river subgames) and reports them
under "extra", so every N carries all three workloads.

One "step" = one full CFR iteration (both players traversed and updated, cfr.rs:216-226) over the whole public tree of
the workload.  N > 1 is launched by torchrun, one rank per GPU; the first dealt-card level is sharded across ranks and
the counterfactual values at the shared chance nodes are exchanged every traversal inside the traversal kernel over
NVLink peer memory (strong scaling: the job is the same subgame at every N; config 5 shards by subgame, no exchange).

Rank 0 prints ONE JSON line: value = iterations/s with all inputs resident in HBM (CUDA events around each of the K
timed steps, L2 flushed between steps, max over ranks), e2e = the same through the C ABI from host
buffers, roofline = the dominant kernel (one launch per player traversal) from CUDA events on the engine's stream,
cpu_baseline = the literal scalar port of the reference's cfr() on this box's host cores (plus, for context, the
vector-form fp64 oracle and the literal 8-thread mccfr port).
`--impl reference` times that port alone (the reference itself cannot be built: no Rust toolchain); it rebuilds the
workload from tests/golden/workload_*.npz and oracle/tree_oracle.py and never loads the product library.

`--dump-outputs DIR` (one GPU) writes what the engine holds after the last timed step of the main workload, i.e. after
exactly W + K iterations from zero tables, as float .npy files (see collect_outputs).  The inputs are fixed by the
workload, so two builds run with the same arguments can be compared array by array.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

import numpy as np  # noqa: E402

METRIC = "cfr_iterations_per_sec"
UNIT = "iter/s"
BYTES_PER_UPDATE = 20  # SURVEY §8(d): regret R+W (8) + strategy_sum R+W (8) + opponent-side regret read (4)
BB_CHIPS = 1.0         # the reference has no big blind (options.rs:10-28): mbb/g is quoted for a big blind of 1 chip
DUMP_BYTES = 60_000_000  # arrays of --dump-outputs: with their .npy headers below 64 MB
DUMP_SEED = 20240601


def load_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            d = json.loads(p.read_text())
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""

    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device = device
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-i", str(self.device), "-lms", "200"], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------
# workload description shared by both arms (identical `config` dicts: same game, same abstraction)
# ------------------------------------------------------------------------------------------------
def load_fixture(name: str):
    """tests/golden/workload_<name>.npz (scripts/make_workload_fixtures.py): Options fields, ranges, bucket keys."""
    z = np.load(ROOT / "tests" / "golden" / f"workload_{name}.npz")
    meta = json.loads(bytes(z["meta"]).decode())
    return meta, z


def config_dict(name: str, n_gpus: int) -> dict:
    """What the workload IS (both arms print exactly this): built from the committed fixture and the pure-Python tree."""
    from oracle import tree_oracle
    meta, z = load_fixture(name)
    _, nodes = tree_oracle.build_game_tree(meta["stack_sizes"], meta["board_mask"], meta["starting_pot"], meta["bet_sizes"], meta["raise_sizes"])
    st = tree_oracle.tree_stats(nodes)
    n_board = bin(meta["board_mask"]).count("1")
    rounds = len(meta["bet_sizes"])
    boards, left = [1], 52 - n_board
    for _ in range(rounds - 1):
        boards.append(boards[-1] * left)
        left -= 1
    if "board_masks" in z.files:
        boards = [int(len(z["board_masks"]))]
    return {"workload": meta["name"], "nodes": st["nodes"], "action_nodes": st["action_nodes"], "rounds": rounds,
            "boards": boards, "hands": [int(len(z["range0"])), int(len(z["range1"]))],
            "root_round_buckets": (int(z["keys0"].max()) + 1) if "keys0" in z.files else None,
            "starting_pot_chips": meta["starting_pot"], "stack_chips": meta["stack_sizes"],
            "parallelism": ("single GPU" if n_gpus == 1 else f"first dealt-card level (or the subgames of a batch) sharded over {n_gpus} GPUs, one rank per GPU")
                           + " [GPU arm]; all host cores [CPU arm]",
            "l2": "GPU arm: flushed between timed steps (256 MiB device write), each step timed by CUDA events on the launch stream"}


# ------------------------------------------------------------------------------------------------
# reference arm: the literal scalar port of cfr() on the host cores.  No product code on this path.
# ------------------------------------------------------------------------------------------------
def oracle_game_from_fixture(name: str, subgame: int = 0):
    from oracle import OracleGame, tree_oracle
    meta, z = load_fixture(name)
    _, nodes = tree_oracle.build_game_tree(meta["stack_sizes"], meta["board_mask"], meta["starting_pot"], meta["bet_sizes"], meta["raise_sizes"])
    tree = {k: np.asarray(v) for k, v in tree_oracle.flatten(nodes).items()}
    ranges = [z["range0"], z["range1"]]
    rounds = len(meta["bet_sizes"])
    keys = None
    if "keys0" in z.files:
        keys = [[z["keys0"], z["keys1"]]] + [None] * (rounds - 1)
    bm = int(z["board_masks"][subgame]) if "board_masks" in z.files else meta["board_mask"]
    n_sub = len(z["board_masks"]) if "board_masks" in z.files else 1
    return OracleGame(tree, ranges, bm, keys=keys), n_sub


def cpu_port_rate(name: str, target_seconds: float, steps: int = 1, warmup: int = 0):
    """Times oracle.literal_cfr on a bounded sample of the workload.

    One step = cfr(player 0) + cfr(player 1) over every `stride`-th root hole-card combo (cfr.rs:493-499 iterates all of
    them, in parallel over the combos like the reference's rayon loop); a full iteration costs stride x that, so
    iterations/s = 1 / (stride * t_step).  A batch of subgames (config 5) is sampled on its first subgame and costs
    n_subgames x that."""
    og, n_sub = oracle_game_from_fixture(name)
    n_combos = int(og.n_combos)
    # calibrate: grow a thin sample until it runs for half a second, then size the stride for ~target_seconds per step.
    # Every sample is run twice and the second run is timed: the oracle's tables are allocated lazily, and a first touch
    # pays page faults that the reference (tables allocated at init, infoset.rs:63-81) never sees in its steady state.
    n_try = max(1, og.num_threads)
    while True:
        stride = max(1, n_combos // n_try)
        og.literal_cfr(1, stride, 0)
        t0 = time.perf_counter()
        visited, _ = og.literal_cfr(1, stride, 0)
        t_cal = time.perf_counter() - t0
        if t_cal >= 0.5 or stride == 1:
            break
        n_try *= 4
    per_combo = t_cal / max(visited, 1)
    want = max(1, int(target_seconds / max(per_combo, 1e-9)))
    stride = max(1, n_combos // want)
    og.literal_cfr(1, stride, 0)  # touches the sample's pages
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        visited, _ = og.literal_cfr(1, stride, 0)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    t_step = float(np.mean(times))
    iters_per_s = 1.0 / (t_step * stride * n_sub)
    sample = (f"literal cfr() port (i32 x10000 tables, per-hand-pair recursion), every {stride}-th of {n_combos} root hole-card combos per step "
              f"({visited} combos, {t_step:.2f} s/step)" + (f" of 1 of {n_sub} subgames" if n_sub > 1 else "") + f", extrapolated x{stride * n_sub}")
    return iters_per_s, t_step, og.num_threads, sample, int(og.updates_per_iter) * n_sub


def set_host_threads():
    """torchrun exports OMP_NUM_THREADS=1; the reference's rayon loop uses every hardware thread (cfr.rs:493)."""
    n = os.cpu_count() or 1
    os.environ["OMP_NUM_THREADS"] = str(n)
    try:
        ctypes.CDLL("libgomp.so.1").omp_set_num_threads(n)
    except OSError:
        pass
    return n


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    set_host_threads()
    steps, warmup = args.steps, args.warmup
    target = min(8.0, 150.0 / (steps + warmup))  # the whole run stays within a few minutes whatever K and W are
    rate, t_step, cores, sample, upd = cpu_port_rate(args.workload, target, steps, warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": warmup, "ms_per_step": 1000.0 / rate, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "i32 fixed-point x10000 (f32 math)", "data": "synthetic",
        "config": config_dict(args.workload, args.gpus),
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "updates_per_iteration": upd, "updates_per_sec": rate * upd,
        "product_library_loaded": any("libb200cfr" in ln for ln in open("/proc/self/maps")),
    }
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
class Ctx:
    pass


def _dealt_cards(i: int, live, k: int):
    """The i-th deal, in lexicographic order, of k cards one after another from `live`."""
    rest, out = list(live), []
    for j in range(k):
        q, i = divmod(i, int(np.prod([len(rest) - 1 - t for t in range(k - 1 - j)])))
        out.append(rest.pop(q))
    return out


def collect_outputs(eng, w, tree, ranges) -> dict:
    """What a caller of rs_iterate reads back, keyed by what the caller supplies (hand slots of its ranges, dealt
    cards) rather than by the engine's row and board numbering:
      root_values_p0/_p1   [root boards, hands]   rs_root_values: counterfactual values of the last traversal
      regrets/strategy_sum [S, hands, actions]    rs_read_infoset row of each hand slot (card table); 0 where the
                                                  hand hits the board (it has no reach), past the player's range or
                                                  past the node's actions
      slab_keys            [S, 4]                 action node index, its number of actions, then the cards dealt
                                                  beyond the root board (the subgame for a batch); -1 where unused
    The S slabs are a fixed seeded sample of all (action node, board) pairs: as many as DUMP_BYTES leaves room for."""
    st = eng.stats()
    out = {f"root_values_p{p}": eng.root_values(p) for p in range(2)}
    nodes = [i for i in range(tree.n_nodes) if tree.type[i] == 0]
    rounds = [int(tree.round_idx[i]) for i in nodes]
    counts = np.array([st.n_boards[k] for k in rounds], dtype=np.int64)
    first = np.cumsum(counts) - counts
    live = [c for c in range(52) if not (w.options.board_mask >> c) & 1]
    H, A = max(len(r) for r in ranges), max(len(tree.children_of(i)) for i in nodes)
    room = DUMP_BYTES - sum(a.nbytes for a in out.values())
    n = int(min(counts.sum(), room // (2 * 4 * H * A + 4 * 8)))
    pick = np.sort(np.random.default_rng(DUMP_SEED).choice(int(counts.sum()), n, replace=False))
    regrets = np.zeros((n, H, A), dtype=np.float32)
    ssum = np.zeros((n, H, A), dtype=np.float32)
    keys = np.full((n, 4), -1.0)
    for s, flat in enumerate(pick):
        j = int(np.searchsorted(first, flat, side="right")) - 1
        node, k, b = nodes[j], rounds[j], int(flat - first[j])
        if w.board_masks is not None:  # a batch: subgame b is board b of round 0
            keys[s, 2] = b
        else:
            dealt = _dealt_cards(b, live, k)
            keys[s, 2:2 + k] = dealt
            b = eng.board_id(k, dealt)
        rows = eng.card_table(k, int(tree.player[node]), b)
        r, sm = eng.read_infoset(int(tree.an_index[node]), b)
        keys[s, :2] = int(tree.an_index[node]), r.shape[1]
        hands = np.flatnonzero(rows != 0xFFFF)
        regrets[s, hands, :r.shape[1]] = r[rows[hands]]
        ssum[s, hands, :r.shape[1]] = sm[rows[hands]]
    out.update(regrets=regrets, strategy_sum=ssum, slab_keys=keys)
    return out


def write_outputs(d: Path, arrays: dict):
    d.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(d / f"{name}.npy", a)


def measure(cx, name: str, steps: int, warmup: int, with_clocks: bool, dump_dir=None):
    """Device-resident throughput, end-to-end throughput and the per-kernel roofline of one workload; with `dump_dir`,
    the outputs of the last timed step are written there."""
    import torch
    import torch.distributed as dist
    import rustsolver_b200 as rb
    from rustsolver_b200 import configs

    w = getattr(configs, name)()
    n_actions, tree = rb.build_game_tree(w.options)
    ranges = configs.workload_ranges(w)
    nccl_id = None
    if cx.world > 1:
        idt = torch.zeros(128, dtype=torch.uint8, device=cx.dev)
        if cx.rank == 0:
            idt = torch.tensor(list(rb.nccl_unique_id()), dtype=torch.uint8, device=cx.dev)
        dist.broadcast(idt, 0)
        nccl_id = bytes(idt.cpu().tolist())
    t0 = time.perf_counter()
    eng = rb.Engine(tree, ranges, w.options.board_mask, w.card_abs, board_masks=w.board_masks, device=cx.local_rank,
                    rank=cx.rank, world_size=cx.world, nccl_id=nccl_id, flags=int(os.environ.get("RS_ENGINE_FLAGS", "0")))
    fused = False
    if cx.world > 1 and os.environ.get("RS_NO_FUSED", "0") != "1" and eng.stats().n_rounds > 1:
        # the kernel exchanges the chance-node sums itself over NVLink peer memory (False: some rank could not map
        # its peers, every rank stays on the NCCL all-reduce)
        fused = eng.enable_fused_exchange(dist, cx.dev)
    create_s = time.perf_counter() - t0
    st = eng.stats()
    upd_global = int(st.updates_per_iteration_global)

    def barrier():
        if cx.world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        t = torch.tensor([x], dtype=torch.float64, device=cx.dev)
        if cx.world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident throughput: K steps, each bracketed by the engine's own CUDA events ----
    for _ in range(warmup):
        eng.iterate(1)
    sampler = ClockSampler(cx.local_rank) if with_clocks else None
    barrier()
    if sampler:
        sampler.start()
    wall0 = time.perf_counter()
    s0 = eng.stats()
    for _ in range(steps):
        cx.flush_l2()
        barrier()
        eng.iterate(1)  # rs_iterate records events on its launch stream around the graph replay
    barrier()
    s1 = eng.stats()
    wall = time.perf_counter() - wall0
    clocks = sampler.stop() if sampler else None
    launches = int(s1.kernel_launches - s0.kernel_launches)
    ms_per_step = max_over_ranks(s1.device_ms - s0.device_ms) / steps
    value = 1000.0 / ms_per_step
    if dump_dir is not None:
        write_outputs(dump_dir, collect_outputs(eng, w, tree, ranges))

    # ---- end to end through the C ABI with host buffers ----
    # per step: H2D of both players' range weights (the host input of a re-solve step) from pinned memory,
    # rs_iterate(1) (synchronous), D2H of both players' root counterfactual values
    pinned = [torch.ones(len(ranges[p]), dtype=torch.float32).pin_memory() for p in range(2)]
    h2d = sum(x.numel() * 4 for x in pinned)
    d2h = 0
    lib = eng._lib
    e2e_t = 0.0
    for i in range(warmup + steps):
        cx.flush_l2()
        barrier()
        t0 = time.perf_counter()
        for p in range(2):
            rc = lib.rs_set_range_weights(eng._h, p, ctypes.cast(pinned[p].data_ptr(), ctypes.POINTER(ctypes.c_float)), pinned[p].numel())
            assert rc == 0, lib.rs_last_error()
        eng.iterate(1)
        outs = [eng.root_values(p) for p in range(2)]
        dt = time.perf_counter() - t0
        if i >= warmup:
            e2e_t += dt
        d2h = sum(o.nbytes for o in outs)
    e2e_value = steps / max_over_ranks(e2e_t)

    # ---- roofline of the dominant kernel: CUDA events on the engine's stream, launch by launch (rs_profile_iteration
    # launches the same kernels directly, without the captured graph) ----
    peak, peak_src = load_peaks()
    prof_runs = []
    for _ in range(3):
        cx.flush_l2()
        prof_runs.append(eng.profile_iteration())
    dom_kind = "street" if any(k["kind"] == "street" for k in prof_runs[0]) else "traversal"
    dom = [[k for k in run if k["kind"] == dom_kind and k["phase"] == 0] for run in prof_runs]
    dom_ms = float(np.mean([k["ms"] for run in dom for k in run]))
    dom_bytes = float(np.mean([k["table_bytes"] for run in dom for k in run]))
    achieved = dom_bytes / (dom_ms * 1e-3) / 1e9
    shares = {}
    for k in prof_runs[-1]:
        key = f'{k["kind"]}_p{k["traverser"]}_phase{k["phase"]}'
        shares[key] = shares.get(key, 0.0) + k["ms"]
    traffic = None
    tp = ROOT / "profiles" / "traffic.json"
    if tp.exists():
        try:
            traffic = json.loads(tp.read_text()).get(name, {}).get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "peak_source": peak_src,
                "kernel": ("street_kernel<CFR>: the final round of one player's traversal" if dom_kind == "street" else
                           "task_kernel<CFR>: persistent dataflow kernel, one launch = one player's traversal of the whole tree") + " (mean of both players)",
                "algorithmic_bytes_per_launch": dom_bytes, "ms_per_launch": dom_ms,
                "kernel_share_of_iteration": sum(k["ms"] for k in dom[-1]) / sum(k["ms"] for k in prof_runs[-1]),
                "per_kernel_ms": {k: round(v, 5) for k, v in shares.items()},
                "whole_iteration_frac": (upd_global * BYTES_PER_UPDATE / cx.world) / (ms_per_step * 1e-3) / 1e9 / peak}

    # exploitability of the average strategy after everything run so far (rs_best_response: two best-response traversals,
    # same kernel).  Batches report the sum over this rank's subgames.
    st_end = eng.stats()
    br = eng.best_response()
    chips = 0.5 * (br[0] + br[1])
    exploit = {"iterations": int(st_end.iterations), "chips": chips, "mbb_per_game": 1000.0 * chips / BB_CHIPS, "bb_chips": BB_CHIPS,
               "pct_of_starting_pot": 100.0 * chips / float(w.options.starting_pot), "best_response_values": [br[0], br[1]]}
    out = {"value": value, "ms_per_step": ms_per_step, "updates_per_iteration": upd_global, "updates_per_sec": value * upd_global,
           "gpu_launches": launches, "launches_per_step": launches / steps,
           "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                   "what": "per step: rs_set_range_weights x2 from pinned host memory, rs_iterate(1), rs_root_values x2"},
           "roofline": roofline, "exploitability": exploit, "clocks": clocks, "engine_create_s": create_s,
           "wall_s_timed_region": wall, "table_bytes_per_gpu": int(st.table_bytes),
           "exchange": None if cx.world == 1 or st.n_rounds == 1 else ("in-kernel over NVLink peer memory" if fused else "ncclAllReduce between two launches")}
    eng.close()
    return out


def oracle_exploitability_check(name: str, iterations: int):
    """The engine and the fp64 oracle run the same number of iterations from zero tables on the same workload; the two
    exploitabilities (own best response, both sides) must agree to 2 % / 0.02 chips (tests/test_gpu_parity.py bound)."""
    import rustsolver_b200 as rb
    from rustsolver_b200 import configs
    w = getattr(configs, name)()
    n_actions, tree = rb.build_game_tree(w.options)
    eng = rb.Engine(tree, configs.workload_ranges(w), w.options.board_mask, w.card_abs, board_masks=w.board_masks)
    eng.iterate(iterations)
    br = eng.best_response()
    eng.close()
    og, _ = oracle_game_from_fixture(name)
    t0 = time.perf_counter()
    og.iterate(iterations)
    t_it = (time.perf_counter() - t0) / iterations
    obr = og.best_response()
    e, o = 0.5 * (br[0] + br[1]), 0.5 * (obr[0] + obr[1])
    return {"workload": name, "iterations": iterations, "engine_chips": e, "oracle_chips": o, "engine_mbb_per_game": 1000 * e / BB_CHIPS,
            "oracle_mbb_per_game": 1000 * o / BB_CHIPS, "abs_diff_chips": abs(e - o), "bound_chips": max(0.02 * abs(o), 0.02),
            "ok": bool(abs(e - o) <= max(0.02 * abs(o), 0.02))}, t_it, og.num_threads


def other_cpu_baselines(name: str, t_vec_all: float, threads_all: int):
    """BASELINE.md §3: B-vec-CPU (vector-form fp64 oracle, 1 thread and all threads) and B-lit-MCCFR (8 threads)."""
    out = {}
    og, n_sub = oracle_game_from_fixture(name)
    try:
        gomp = ctypes.CDLL("libgomp.so.1")
        gomp.omp_set_num_threads(1)
        t0 = time.perf_counter()
        og.iterate(1)
        t1 = time.perf_counter() - t0
        gomp.omp_set_num_threads(os.cpu_count() or 1)
        out["B-vec-CPU"] = {"what": "vector-form synchronous fp64 CFR over the public tree (the parity oracle), " + name,
                            "iter_per_s_1_thread": 1.0 / (t1 * n_sub), "iter_per_s_all_threads": 1.0 / (t_vec_all * n_sub), "threads_all": threads_all}
    except OSError:
        pass
    t0 = time.perf_counter()
    n_iter = 4000
    og.literal_mccfr(n_iter, n_threads=8, seed=1)
    out["B-lit-MCCFR"] = {"what": "literal port of train()'s external-sampling mccfr worker loop (cfr.rs:188-229,299-479), 8 threads, " + name,
                          "sampled_iter_per_s": n_iter / (time.perf_counter() - t0), "threads": 8,
                          "note": "one sampled iteration visits one deal; not comparable 1:1 with a full iteration"}
    return out


def run_ours(args):
    import torch
    import torch.distributed as dist

    cx = Ctx()
    cx.world = int(os.environ.get("WORLD_SIZE", "1"))
    cx.rank = int(os.environ.get("RANK", "0"))
    cx.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU fallback")
    torch.cuda.set_device(cx.local_rank)
    cx.dev = torch.device("cuda", cx.local_rank)
    if cx.world > 1:
        dist.init_process_group("nccl", device_id=cx.dev)
    flush_buf = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=cx.dev)  # > 126 MB L2

    def flush_l2():
        flush_buf.add_(1)
        torch.cuda.synchronize()

    cx.flush_l2 = flush_l2
    steps, warmup = args.steps, args.warmup
    if warmup < 3 and cx.rank == 0:
        print(f"bench.py: --warmup {warmup} is below the 3 warm-up steps the timing rules ask for", file=sys.stderr)
    main = measure(cx, args.workload, steps, warmup, with_clocks=True, dump_dir=args.dump_outputs)
    extra = {}
    if not args.no_extra:
        for name in ("config2", "config5"):
            if name != args.workload:
                m = measure(cx, name, 20, max(warmup, 3), with_clocks=False)
                extra[name] = {"config": config_dict(name, cx.world), "value": m["value"], "unit": UNIT, "ms_per_step": m["ms_per_step"],
                               "updates_per_sec": m["updates_per_sec"], "e2e": m["e2e"],
                               "roofline": {k: m["roofline"][k] for k in ("frac", "achieved", "peak", "ms_per_launch", "algorithmic_bytes_per_launch", "whole_iteration_frac")},
                               "exploitability": m["exploitability"], "exchange": m["exchange"]}
    parity = None
    if cx.world > 1 and not args.no_parity:
        # the sharded path against the fp64 oracle on the live ranks: turn- and flop-rooted games, both exchange paths
        from tests import mgpu_worker
        cases, worst, all_ok = [], 0.0, True
        for case, fused in (("turn", True), ("flop", True), ("turn", False), ("batch", False)):
            ok, wr, msg, boards = mgpu_worker.check_case(case, cx.rank, cx.world, cx.local_rank, cx.dev, fused)
            t = torch.tensor([wr], dtype=torch.float64, device=cx.dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            cases.append({"case": case, "exchange": "in-kernel" if fused else "nccl", "ok": bool(ok), "worst_ratio": float(t.item())})
            worst = max(worst, float(t.item()))
            all_ok = all_ok and ok
            if msg:
                print(f"[rank {cx.rank}] parity {case} FAILED: {msg}", file=sys.stderr, flush=True)
        parity = {"what": "sharded engine vs the fp64 oracle in lock-step on every rank (tests/mgpu_worker.py), diff / bound", "cases": cases,
                  "worst_ratio": worst, "ok": bool(all_ok)}
    rc = 0 if (parity is None or parity["ok"]) else 1

    if cx.rank == 0:
        cpu = None
        expl_check = None
        if cx.world == 1 and not args.no_cpu_baseline:
            set_host_threads()
            rate, t_step, cores, sample, _ = cpu_port_rate(args.workload, target_seconds=12.0)
            cpu = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample}
            expl_check, t_vec, thr = oracle_exploitability_check("config2", 10)
            cpu["others"] = other_cpu_baselines("config2", t_vec, thr)
            if not expl_check["ok"]:
                rc = 1
        cfg = config_dict(args.workload, cx.world)
        line = {
            "metric": METRIC, "value": main["value"], "unit": UNIT, "n_gpus": cx.world, "steps": steps, "warmup": warmup,
            "ms_per_step": main["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": cfg,
            "updates_per_iteration": main["updates_per_iteration"], "updates_per_sec": main["updates_per_sec"],
            "gpu_launches": main["gpu_launches"], "launches_per_step": main["launches_per_step"],
            "timed_region": {"steps": steps, "statistic": "device time of the K steps summed", "wall_s": main["wall_s_timed_region"]},
            "e2e": main["e2e"], "roofline": main["roofline"], "cpu_baseline": cpu,
            "exploitability": main["exploitability"], "exploitability_vs_oracle": expl_check, "clocks": main["clocks"],
            "exchange": main["exchange"], "table_bytes_per_gpu": main["table_bytes_per_gpu"], "engine_create_s": main["engine_create_s"],
            "extra": extra, "parity": parity,
        }
        print(json.dumps(line), flush=True)
    if cx.world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return rc


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="config4", choices=["config1", "config2", "config3", "config4", "config5"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the config 2 / config 5 lines reported under `extra`")
    ap.add_argument("--no-parity", action="store_true", help="N > 1: skip the sharded-parity cases after the timed region")
    ap.add_argument("--dump-outputs", metavar="DIR", type=Path,
                    help="write the engine's outputs after the last timed step of the main workload to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs is not None and (args.gpus != 1 or args.impl != "ours"):
        ap.error("--dump-outputs needs --gpus 1 and --impl ours")
    if args.impl == "reference":
        return run_reference(args)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.gpus > 1 and world == 1:
        # convenience: re-launch under torchrun the way the driver does
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29531", __file__] + sys.argv[1:]
        return subprocess.call(cmd)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
