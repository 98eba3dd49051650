"""
TEST INFRASTRUCTURE ONLY. Writes tests/golden/adaptive_ransac_pins.npz: the adaptive RANSAC oracle's winner, stopping
point, counts and first survivors on fixed seeded match sets (PIN_CASES), so that tests/test_adaptive_ransac_host.py
can hold oracle/adaptive_ransac_oracle.py in place.

    python -m oracle.make_adaptive_ransac_pins
"""

from __future__ import annotations

import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import adaptive_ransac_oracle as oracle  # noqa: E402
from shot_fpfh_b200 import synthetic  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "adaptive_ransac_pins.npz")
THRESHOLD = 0.01
# (name, matches, inlier ratio, noise, synthetic seed, ransac seed, max_draws)
PIN_CASES = (
    ("m300_w30", 300, 0.30, 0.002, 21, 0, 1 << 24),
    ("m2000_w10", 2000, 0.10, 0.002, 22, 9, 1 << 24),
    ("m2000_w1_capped", 2000, 0.01, 0.0, 23, 1, oracle.BATCH + 1000),
)


def case_matches(n: int, w: float, noise: float, seed: int) -> tuple[np.ndarray, np.ndarray]:
    scan, ref, si, ri, _, _ = synthetic.corrupted_matches(n, w, noise=noise, seed=seed)
    return np.ascontiguousarray(scan[si]), np.ascontiguousarray(ref[ri])


def compute() -> dict:
    out = {}
    for name, n, w, noise, seed, ransac_seed, max_draws in PIN_CASES:
        a, b = case_matches(n, w, noise, seed)
        r = oracle.ransac_adaptive(a, b, THRESHOLD, max_draws=max_draws, seed=ransac_seed)
        first = oracle.run_batch(a, b, THRESHOLD, 0.9, ransac_seed, 0, 4096)
        out[f"{name}_counters"] = np.array([r[k] for k in ("best_draw", "best_count", "draws_used", "batches",
                                                           "survivors", "valid")], dtype=np.int64)
        out[f"{name}_transform"] = r["transform"]
        out[f"{name}_mask"] = r["mask"]
        out[f"{name}_first_survivors"] = first["survivors"]
        out[f"{name}_first_valid"] = first["valid_draws"]
        out[f"{name}_first_counts"] = first["counts"]
    return out


def main() -> None:
    out = compute()
    np.savez_compressed(OUT, **out)
    print(f"wrote {OUT}: " + ", ".join(f"{k} {v.tolist()}" for k, v in out.items() if k.endswith("_counters")))


if __name__ == "__main__":
    main()
