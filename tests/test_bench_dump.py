"""bench.py --dump-outputs: the files hold what a fresh engine holds after exactly warm-up + timed steps iterations of the
same workload (the engine is bit-reproducible), as finite float arrays below 64 MB in all."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

import bench
import rustsolver_b200 as rb
from rustsolver_b200 import configs

ROOT = Path(__file__).resolve().parent.parent
pytestmark = pytest.mark.gpu


def test_dump_outputs_hold_the_tables_after_warmup_plus_steps(tmp_path):
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--workload", "config2", "--steps", "3", "--warmup", "2",
                        "--no-extra", "--no-cpu-baseline", "--dump-outputs", str(out)],
                       capture_output=True, text=True, cwd=tmp_path, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 3 and line["warmup"] == 2
    files = sorted(out.glob("*.npy"))
    assert sum(f.stat().st_size for f in files) <= 64_000_000
    dumped = {f.stem: np.load(f) for f in files}
    assert all(a.dtype in (np.float32, np.float64) and np.isfinite(a).all() for a in dumped.values())

    w = configs.config2()
    _, tree = rb.build_game_tree(w.options)
    ranges = configs.workload_ranges(w)
    eng = rb.Engine(tree, ranges, w.options.board_mask, w.card_abs, board_masks=w.board_masks)
    eng.iterate(2 + 3)
    want = bench.collect_outputs(eng, w, tree, ranges)
    eng.close()
    assert sorted(want) == sorted(dumped)
    assert len(want["slab_keys"]) > 1000  # a sample of the river slabs, not only the root round
    assert np.abs(want["regrets"]).max() > 0 and np.abs(want["root_values_p0"]).max() > 0
    for name, a in want.items():
        assert np.array_equal(dumped[name], a), name
