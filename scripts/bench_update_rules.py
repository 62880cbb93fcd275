"""Iterations and wall time to a target exploitability under each update rule (rs_set_update_rule), one GPU.

    python scripts/bench_update_rules.py [--configs config2,config4,config5] [--iters 300] [--out FILE.json]

For every workload and rule (vanilla CFR, DCFR(1.5, 0, 2), LCFR, CFR+) one engine trains from zero tables.  The training
is cut at the checkpoints below; at each one the exploitability (rs_best_response, (br0 + br1) / 2 chips per deal) is
taken outside the timed region.  Reported per rule:
  - iter/s: iterations over the summed wall time of the rs_iterate calls (each returns with the device idle);
  - exploitability after 10, 30, 100 and 300 iterations;
  - the target: vanilla CFR's exploitability after --iters iterations (stated in the output), and for every rule the
    first checkpoint at which it is reached, with the rs_iterate wall time up to there.  The checkpoint grid bounds the
    resolution of "iterations to target".
Config 5 (a batch of river subgames) reports what rs_best_response returns for the whole batch.
The GPU's name and power limit are printed with the numbers."""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))

import rustsolver_b200 as rb  # noqa: E402
from rustsolver_b200 import configs  # noqa: E402

RULES = [("vanilla", (rb.RS_RULE_VANILLA,)), ("dcfr_1.5_0_2", (rb.RS_RULE_DCFR, 1.5, 0.0, 2.0)), ("lcfr", (rb.RS_RULE_LCFR,)),
         ("cfr_plus", (rb.RS_RULE_CFR_PLUS,))]
REPORT = (10, 30, 100, 300)


def checkpoints(n: int):
    pts = sorted({*range(1, 11), *range(12, 31, 2), *range(35, 101, 5), *range(110, 301, 10), *[x for x in REPORT if x <= n], n})
    return [p for p in pts if p <= n]


def run(name: str, rule, n: int):
    w = getattr(configs, name)()
    _, tree = rb.build_game_tree(w.options)
    eng = rb.Engine(tree, configs.workload_ranges(w), w.options.board_mask, w.card_abs, board_masks=w.board_masks)
    eng.set_update_rule(*rule)
    eng.iterate(1)  # warm-up: graph capture, first launches; then back to zero tables and t = 0
    eng.reset()
    curve, wall, done = [], 0.0, 0
    for c in checkpoints(n):
        t0 = time.perf_counter()
        eng.iterate(c - done)
        wall += time.perf_counter() - t0
        done = c
        curve.append((c, wall, sum(eng.best_response()) / 2))
    eng.close()
    return curve


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="config2,config4,config5")
    ap.add_argument("--iters", type=int, default=300)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    res = {"gpu": gpu, "iters": a.iters, "workloads": {}}
    print(f"# GPU: {gpu}", flush=True)
    for name in a.configs.split(","):
        curves = {r: run(name, rule, a.iters) for r, rule in RULES}
        target = curves["vanilla"][-1][2]
        rows = {}
        for r, cv in curves.items():
            hit = next(((c, t) for c, t, e in cv if e <= target), None)
            rows[r] = {"iter_per_s": cv[-1][0] / cv[-1][1],
                       "exploitability": {str(c): e for c, _, e in cv if c in REPORT},
                       "iters_to_target": hit[0] if hit else None, "seconds_to_target": hit[1] if hit else None,
                       "curve": [[c, round(t, 6), e] for c, t, e in cv]}
        res["workloads"][name] = {"target_chips": target, "target_is": f"vanilla CFR after {a.iters} iterations", "rules": rows}
        print(f"\n{name}: target = {target:.6g} chips (vanilla CFR after {a.iters} iterations)")
        print(f"{'rule':14s} {'iter/s':>9s} " + " ".join(f"{'ex@' + str(c):>10s}" for c in REPORT if c <= a.iters) +
              f" {'iters->tgt':>10s} {'s->tgt':>8s}")
        for r, d in rows.items():
            ex = " ".join(f"{d['exploitability'].get(str(c), float('nan')):10.4g}" for c in REPORT if c <= a.iters)
            it = d["iters_to_target"] if d["iters_to_target"] is not None else "-"
            sec = f"{d['seconds_to_target']:.3f}" if d["seconds_to_target"] is not None else "-"
            print(f"{r:14s} {d['iter_per_s']:9.2f} {ex} {it!s:>10s} {sec:>8s}", flush=True)
    if a.out:
        Path(a.out).write_text(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
