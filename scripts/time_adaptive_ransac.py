"""
Times adaptive RANSAC (csrc/registration.cu sf_ransac_adaptive, matching.ransac_on_matches_adaptive) on synthetic
match sets of known quality, and runs the reference's 10 000-draw `ransac_on_matches` on the same inputs:

    python scripts/time_adaptive_ransac.py [--matches 20000,400000] [--ratios 0.27,0.05,0.02] [--repeats 5] [--out DIR]

Inputs: `synthetic.corrupted_matches(m, w, noise=0.2 * threshold)` (a bumpy-sphere pair, match i correct for a share w
of the matches, a random reference point otherwise), threshold 0.01 on a unit-size cloud. Per case: the draws, batches,
edge-check survivors and valid hypotheses of the search; end-to-end time of ransac_on_matches_adaptive from host
arrays (min / median / max of `repeats` runs after one warm-up); the rotation and translation error of its result and
of the reference algorithm's; and, in a separate torch.profiler run of one call, the device time per kernel. The card's
name and power limit are read in the same run. Prints one JSON line (and writes DIR/adaptive_ransac_b200.json).
"""

import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import shot_fpfh_b200.matching.ransac as ransac_module  # noqa: E402
from shot_fpfh_b200 import ops, synthetic  # noqa: E402
from shot_fpfh_b200.device import require_cuda, upload  # noqa: E402
from shot_fpfh_b200.matching import ransac_on_matches, ransac_on_matches_adaptive  # noqa: E402

THRESHOLD = 0.01
BATCH = 1 << 20


def card() -> dict:
    info = {"name": torch.cuda.get_device_name(), "power_limit_w": None}
    try:
        out = subprocess.run(["nvidia-smi", f"--id={torch.cuda.current_device()}", "--query-gpu=power.limit",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout
        info["power_limit_w"] = float(out.strip().splitlines()[0])
    except (OSError, ValueError, IndexError, subprocess.SubprocessError):
        pass
    return info


def errors(transform, rot, trans) -> dict:
    return {"rotation_error": float(np.abs(transform.rotation - rot).max()),
            "translation_error": float(np.abs(transform.translation - trans).max())}


def kernel_times(fn) -> dict:
    """Device time per kernel name over one call of fn, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
        if t > 0:
            out[e.key] = {"calls": int(e.count), "device_ms": t / 1e3}
    return dict(sorted(out.items(), key=lambda kv: -kv[1]["device_ms"]))


def time_case(m: int, w: float, repeats: int) -> dict:
    scan, ref, si, ri, rot, trans = synthetic.corrupted_matches(m, w, noise=0.2 * THRESHOLD, seed=1)
    a, b = upload(scan[si]), upload(ref[ri])
    search = ops.ransac_adaptive(a, b, THRESHOLD, 0.9, 0, 1 << 24, 0.999)
    batches = math.ceil(search["draws_used"] / BATCH)
    survivors = 0
    for k in range(batches):
        n = min(BATCH, search["draws_used"] - k * BATCH)
        survivors += int(ops.ransac_adaptive_batch(a, b, THRESHOLD, 0.9, 0, k * BATCH, n)["survivors"].shape[0])

    def call():
        return ransac_on_matches_adaptive(si, ri, scan, ref, distance_threshold=THRESHOLD)

    call()  # warm-up
    ms = []
    for _ in range(repeats):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ratio, transform = call()
        ms.append(1e3 * (time.perf_counter() - t0))
    ransac_module.rng = np.random.default_rng(seed=72)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ref_ratio, ref_transform = ransac_on_matches(si, ri, scan, ref, n_draws=10_000, distance_threshold=THRESHOLD)
    ref_ms = 1e3 * (time.perf_counter() - t0)
    return {
        "matches": m, "inlier_ratio": w, "threshold": THRESHOLD, "noise": 0.2 * THRESHOLD,
        "draws_used": search["draws_used"], "batches": batches, "survivors": survivors, "valid": search["valid"],
        "best_count": search["best_count"], "found_ratio": ratio,
        "end_to_end_ms": {"min": min(ms), "median": float(np.median(ms)), "max": max(ms)},
        **errors(transform, rot, trans),
        "reference_10000_draws": {"ratio": ref_ratio, "ms": ref_ms, **errors(ref_transform, rot, trans)},
        "kernels": kernel_times(call),
    }


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--matches", default="20000,400000")
    ap.add_argument("--ratios", default="0.27,0.05,0.02")
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    require_cuda()
    cases = [time_case(int(m), float(w), args.repeats) for m in args.matches.split(",") for w in args.ratios.split(",")]
    line = json.dumps({"card": card(), "cases": cases})
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "adaptive_ransac_b200.json"), "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
