"""
Times ISS salient-keypoint detection (csrc/iss.cu, keypoint_selection.select_keypoints_iss) on the bumpy sphere at 1M
and 10M points, r_s = 5 spacings (about 72 neighbours, as in C2/C3) and r_n = 3.75 spacings:

    python scripts/time_iss.py [--sizes 1000000,10000000] [--repeats 10] [--out DIR]

Inputs are resident on the device and every stage is warmed up; a 512 MB buffer is overwritten between passes so that
no pass finds the previous one's data in L2. CUDA events per stage: grid build, saliency, non-maximum suppression +
compaction (sf_iss_select, which ends in a synchronisation); then end to end, host float64 points in -> host int64
keypoints out. Bytes per stage are the algorithmic ones, computed from shapes (what each stage must read and write at
least once). The CPU oracle is timed on a 100k-point decimation of the 1M cloud (every 10th point, radii of that
density), labelled as such. Prints one JSON line (and writes it to DIR/iss_b200.json with --out).
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
from shot_fpfh_b200.device import Grid, require_cuda, upload  # noqa: E402
from shot_fpfh_b200.keypoint_selection import select_keypoints_iss  # noqa: E402

M, G21, G32 = 5, 0.975, 0.975


def card() -> dict:
    info = {"name": torch.cuda.get_device_name(), "power_limit_w": None}
    try:
        out = subprocess.run(["nvidia-smi", f"--id={torch.cuda.current_device()}", "--query-gpu=power.limit",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout
        info["power_limit_w"] = float(out.strip().splitlines()[0])
    except (OSError, ValueError, IndexError, subprocess.SubprocessError):
        pass
    return info


def stage_bytes(n: int, candidates: int, keypoints: int) -> dict:
    """Least bytes each stage moves: every input read once, every output written once."""
    return {
        # xyz read (24) + pts written (32, double4) + float32 side copy (16) + perm and inv_perm (8) + key and slot (8)
        "grid": n * (24 + 32 + 16 + 8 + 8),
        # each point's record read once (32) + saliency written (8)
        "saliency": n * (32 + 8),
        # saliency read by the selection (8) + flags cleared and read (2) + candidates written and read (4 + 4) and
        # their records and saliencies (32 + 8) + keypoints written (4)
        "nms": n * (8 + 2) + candidates * (4 + 4 + 32 + 8) + keypoints * 4,
    }


def time_size(n: int, repeats: int, flush: torch.Tensor) -> dict:
    pts_host, _ = synthetic.bumpy_sphere(n, seed=0)
    s = synthetic.mean_spacing(n)
    rs, rn = 5.0 * s, 3.75 * s
    pts = upload(pts_host)
    grid = Grid()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    ms = {"grid": [], "saliency": [], "nms": []}
    kp = None
    for it in range(repeats + 2):  # two warm-up passes
        flush.fill_(it)
        ev[0].record()
        grid.build(pts, None, max(rs, rn))
        ev[1].record()
        sal, _, _ = ops.iss_saliency(grid, rs, M, G21, G32)
        ev[2].record()
        kp = ops.iss_select(grid, sal, rn, M)
        ev[3].record()
        torch.cuda.synchronize()
        if it >= 2:
            for k, name in enumerate(ms):
                ms[name].append(ev[k].elapsed_time(ev[k + 1]))
    candidates = int((sal > 0).sum())
    grid.close()
    del pts
    e2e = []
    for it in range(max(3, repeats // 2) + 1):
        flush.fill_(it)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = select_keypoints_iss(pts_host, rs, rn)
        e2e.append(1e3 * (time.perf_counter() - t0))
    assert np.array_equal(out, kp.cpu().numpy())
    med = {k: float(np.median(v)) for k, v in ms.items()}
    nbytes = stage_bytes(n, candidates, int(kp.shape[0]))
    return {
        "n_points": n, "salient_radius": rs, "non_max_radius": rn, "keypoints": int(kp.shape[0]),
        "candidates_s_positive": candidates,
        "stage_ms_median": med, "stage_ms_min": {k: float(np.min(v)) for k, v in ms.items()},
        "kernels_ms_median": float(sum(med.values())),
        "end_to_end_ms_median": float(np.median(e2e[1:])), "end_to_end_ms_min": float(np.min(e2e[1:])),
        "algorithmic_bytes": nbytes,
        "algorithmic_GBps": {k: nbytes[k] / (med[k] * 1e-3) / 1e9 for k in nbytes},
    }


def time_oracle_decimation(n_full: int = 1_000_000) -> dict:
    from oracle import iss_oracle

    pts, _ = synthetic.bumpy_sphere(n_full, seed=0)
    dec = np.ascontiguousarray(pts[::10])
    s = synthetic.mean_spacing(dec.shape[0])
    t0 = time.perf_counter()
    kp = iss_oracle.iss(dec, 5.0 * s, 3.75 * s)
    return {"label": f"CPU oracle on a decimation: every 10th point of the {n_full}-point cloud",
            "n_points": int(dec.shape[0]), "keypoints": int(kp.shape[0]), "seconds": time.perf_counter() - t0}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1000000,10000000")
    ap.add_argument("--repeats", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    require_cuda()
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")  # 512 MB > 126 MB of L2
    result = {"what": "ISS keypoints, bumpy sphere, r_s = 5 spacings, r_n = 3.75 spacings, m = 5, gammas 0.975",
              "card": card(), "l2": "overwritten (512 MB) between passes", "sizes": []}
    for n in (int(x) for x in args.sizes.split(",")):
        result["sizes"].append(time_size(n, args.repeats, flush))
    result["oracle_decimated"] = time_oracle_decimation()
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "iss_b200.json"), "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
