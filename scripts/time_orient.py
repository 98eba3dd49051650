"""
Times consistent normal orientation (csrc/orient.cu, descriptors.orient_normals) on the bumpy sphere at 1M and 10M
points, k = 10, normals = the true normals with random signs (what PCA normals look like to the orientation):

    python scripts/time_orient.py [--sizes 1000000,10000000] [--repeats 5] [--out DIR]

Inputs are resident on the device and both stages are warmed up. CUDA events per stage: the k-NN lists
(`knn_device(points, points, k + 1)`, which synchronises while it calibrates its reach) and the orientation
(sf_orient_normals, which synchronises once per Borůvka round and pointer-jumping step); then end to end, host float64
arrays in and out. The card's name and power limit are read in the same run. Prints one JSON line (and writes it to
DIR/orient_b200.json with --out).
"""

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from shot_fpfh_b200 import ops, synthetic  # noqa: E402
from shot_fpfh_b200.descriptors import orient_normals  # noqa: E402
from shot_fpfh_b200.descriptors.pca_based_descriptors import knn_device  # noqa: E402
from shot_fpfh_b200.device import require_cuda, upload  # noqa: E402

K = 10


def card() -> dict:
    info = {"name": torch.cuda.get_device_name(), "power_limit_w": None}
    try:
        out = subprocess.run(["nvidia-smi", f"--id={torch.cuda.current_device()}", "--query-gpu=power.limit",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout
        info["power_limit_w"] = float(out.strip().splitlines()[0])
    except (OSError, ValueError, IndexError, subprocess.SubprocessError):
        pass
    return info


def time_size(n: int, repeats: int) -> dict:
    pts_host, dirs = synthetic.bumpy_sphere(n, seed=0)
    true = synthetic.bumpy_sphere_true_normals(dirs)
    nrm_host = true * np.random.default_rng(0).choice([-1.0, 1.0], size=(n, 1))
    pts, nrm = upload(pts_host), upload(nrm_host)
    events = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    knn_ms, orient_ms, trees = [], [], 0
    for r in range(repeats + 1):  # pass 0 warms up
        torch.cuda.synchronize()
        events[0].record()
        nbr = knn_device(pts, pts, K + 1)
        events[1].record()
        out, trees = ops.orient_normals(pts, nrm, nbr)
        events[2].record()
        torch.cuda.synchronize()
        if r:
            knn_ms.append(events[0].elapsed_time(events[1]))
            orient_ms.append(events[1].elapsed_time(events[2]))
    agree = (torch.einsum("ij,ij->i", out, upload(true)) > 0).double().mean().item()
    e2e = []
    for _ in range(max(repeats // 2, 1)):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        orient_normals(pts_host, nrm_host, K)
        e2e.append(1e3 * (time.perf_counter() - t0))
    return {
        "n_points": n, "k": K, "trees": trees, "outward_share": max(agree, 1.0 - agree),
        "knn_ms": float(np.median(knn_ms)), "orient_ms": float(np.median(orient_ms)),
        "orient_ms_min": float(np.min(orient_ms)), "orient_ms_max": float(np.max(orient_ms)),
        "end_to_end_ms": float(np.median(e2e)),
    }


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1000000,10000000")
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    require_cuda()
    result = {"card": card(), "sizes": [time_size(int(s), args.repeats) for s in args.sizes.split(",")]}
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "orient_b200.json"), "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
