#!/usr/bin/env python
"""Compare two `bench.py --dump-outputs` directories array by array.

    python scripts/compare_outputs.py DIR_A DIR_B

Every .npy file of either directory must exist in both and be np.array_equal (same shape, same values; +0 and -0 count
as equal).  For an array that differs, prints how many elements differ and the largest difference in units of the last
place (float32) or the largest absolute difference (other types).  Exit status 0 when every pair is equal, 1 otherwise.
"""
from __future__ import annotations

import sys
from pathlib import Path

import numpy as np


def ulp_distance(a: np.ndarray, b: np.ndarray) -> int:
    """Largest distance between a and b in float32 units of the last place (monotone integer mapping of the bits)."""
    def key(x):
        i = np.ascontiguousarray(x, dtype=np.float32).view(np.int32).astype(np.int64)
        return np.where(i < 0, np.int64(-0x80000000) - i, i)
    return int(np.abs(key(a) - key(b)).max()) if a.size else 0


def main() -> int:
    if len(sys.argv) != 3:
        print(__doc__, file=sys.stderr)
        return 2
    da, db = Path(sys.argv[1]), Path(sys.argv[2])
    names = sorted({p.name for p in da.glob("*.npy")} | {p.name for p in db.glob("*.npy")})
    if not names:
        print(f"no .npy files in {da} or {db}")
        return 1
    bad = 0
    for n in names:
        pa, pb = da / n, db / n
        if not (pa.exists() and pb.exists()):
            print(f"{n}: missing in {db if pa.exists() else da}")
            bad += 1
            continue
        a, b = np.load(pa), np.load(pb)
        if a.shape != b.shape or a.dtype != b.dtype:
            print(f"{n}: shape / dtype {a.shape} {a.dtype} vs {b.shape} {b.dtype}")
            bad += 1
        elif not np.array_equal(a, b):
            nd = int(np.count_nonzero(a != b))
            how = f"{ulp_distance(a, b)} ulp" if a.dtype == np.float32 else f"{float(np.abs(a - b).max()):.3e}"
            print(f"{n}: {nd} of {a.size} elements differ, at most {how}")
            bad += 1
    print(f"{len(names) - bad} of {len(names)} arrays equal ({da} vs {db})")
    return 0 if bad == 0 else 1


if __name__ == "__main__":
    sys.exit(main())
