"""
Tuning / attribution run for the C2 SHOT step on one B200 (not part of the product, not a benchmark line):
per-stage CUDA-event times of the fused single-scale driver, by default and under each environment of --envs,
the number of queries the float32 descriptor kernel hands to the float64 kernel, and its rows against the float64
kernel's (SF_SHOT_EXACT=1).

    python scripts/tune_shot.py [--envs NAME=VALUE+NAME=VALUE,...] [--steps 12] [--n 1000000]
"""

from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", default="", help="variants besides the default, each a +-joined list of NAME=VALUE, separated by commas")
    ap.add_argument("--no-profile", action="store_true", help="step times only: no CUDA events between the kernels")
    ap.add_argument("--steps", type=int, default=12)
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--out", default=os.path.join(ROOT, "gpurun_out", "tune_shot.json"))
    args = ap.parse_args()

    import torch

    import bench
    from shot_fpfh_b200 import ops, synthetic
    from shot_fpfh_b200.device import Grid, upload

    bench.N_POINTS = args.n
    pts, normals, kp, radius = bench.make_shot_workload(0)
    p_dev, n_dev, k_dev = upload(pts), upload(normals), upload(kp)
    q = kp.shape[0]
    flush_buf = torch.empty(512 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    grid = Grid().set_speculative(builds=True, shot_lists=True)
    results = {"queries": int(q), "points": int(pts.shape[0])}

    def run(tag, env):
        for k in [k for k in os.environ if k.startswith("SF_")]:
            os.environ.pop(k, None)
        os.environ.update(env)
        out = torch.zeros((q, 352), dtype=torch.float32, device="cuda")
        ops.profile_enable(not args.no_profile)
        stage_ms, step_ms, grid_ms = [], [], []
        pairs = deferred = None
        for it in range(3 + args.steps):
            flush_buf.fill_(1)
            e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            e0.record()
            grid.build(p_dev, n_dev, radius)
            e1.record()
            _, _, pr = ops.shot_single_scale(grid, k_dev, radius, bench.MIN_NB, True, out=out, want_pairs=it == 0)
            e2.record()
            if pr is not None:
                pairs, deferred = pr, ops.shot_last_deferred()
            torch.cuda.synchronize()
            if it >= 3:
                stage_ms.append(ops.profile_read() if not args.no_profile else (0.0, 0.0, 0.0))
                step_ms.append(e0.elapsed_time(e2))
                grid_ms.append(e0.elapsed_time(e1))
        ops.profile_enable(False)
        assert grid.poll() == 0, "a speculative call did nothing"
        sm = np.mean(np.array(stage_ms), axis=0)
        res = {"step_ms": float(np.mean(step_ms)), "grid_ms": float(np.mean(grid_ms)), "search_moments_ms": float(sm[0]),
               "eigen_ms": float(sm[1]), "descriptor_ms": float(sm[2]), "pairs": pairs, "deferred": deferred}
        results[tag] = res
        print(tag, json.dumps(res), flush=True)
        return out

    exact = run("exact", {"SF_SHOT_EXACT": "1"})
    exact_norm = exact.double().norm(dim=1).clamp_min(1e-300)
    variants = [("default", {})]
    variants += [(e, dict(kv.split("=") for kv in e.split("+"))) for e in args.envs.split(",") if e]
    for v, env in variants:
        got = run(f"fast_{v}", env)
        err = (got.double() - exact.double()).norm(dim=1) / exact_norm
        zero_mismatch = int(((got.abs().sum(dim=1) == 0) != (exact.abs().sum(dim=1) == 0)).sum().item())
        results[f"fast_{v}"].update({"max_rel_l2_vs_exact": float(err.max().item()), "median_rel_l2_vs_exact": float(err.median().item()),
                                     "rows_above_1e-5": int((err > 1e-5).sum().item()), "rows_above_1e-4": int((err > 1e-4).sum().item()),
                                     "zero_row_mismatch": zero_mismatch})
        print(f"fast_{v} vs exact:", {k: results[f'fast_{v}'][k] for k in ("max_rel_l2_vs_exact", "median_rel_l2_vs_exact", "rows_above_1e-5", "rows_above_1e-4", "zero_row_mismatch")}, flush=True)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
