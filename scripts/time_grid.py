"""
Times the grid build (csrc/grid.cu, `Grid.build`) kernel by kernel on the C2 cloud — bumpy sphere, 1M points, normals,
radius 5 mean spacings — and on the same sphere at 10M points:

    python scripts/time_grid.py [--sizes 1000000,10000000] [--builds 200] [--out DIR]

The handle runs in its no-synchronisation mode, as in a repeated `bench.py` step: after one synchronising build every
build assumes the previous box (no bounding-box pass). Inputs are resident on the device, and a 512 MB buffer is
overwritten between builds so that no build finds the previous one's data in L2.
- Whole build: a CUDA-event pair around each of `--builds` builds (after 20 warm-up builds).
- Per kernel: the same number of builds again under torch.profiler (CUDA activity, device timestamps), in a pass of
  its own; each kernel's total is divided by the number of builds. The profiler records the flush too: it is listed but
  not counted in the build.
`least_bytes` is what the build must move at least: xyz and normals read once (48 B per point), and pts, nrm, xyzc,
nrm32, perm and inv_perm written once (104 B per point). Prints one JSON line with the card's name and power limit
(and writes it to DIR/grid_b200.json with --out).
"""

import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from shot_fpfh_b200 import synthetic  # noqa: E402
from shot_fpfh_b200.device import Grid, require_cuda, upload  # noqa: E402

WARMUP = 20
# device activities of one build, by a piece of their name
STAGES = (("bbox", "bbox"), ("Memset", "histogram_memset"), ("key_kernel", "key"), ("DeviceScan", "scan"),
          ("DeviceRadixSort", "radix_sort"), ("place_kernel", "place"), ("rank_reorder_kernel", "rank_reorder"),
          ("reorder_kernel", "reorder"), ("Memcpy", "status_copy"))


def card() -> dict:
    info = {"name": torch.cuda.get_device_name(), "power_limit_w": None, "max_sm_clock_mhz": None}
    try:
        out = subprocess.run(["nvidia-smi", f"--id={torch.cuda.current_device()}", "--query-gpu=power.limit,clocks.max.sm",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout
        power, clock = out.strip().splitlines()[0].split(",")
        info["power_limit_w"], info["max_sm_clock_mhz"] = float(power), float(clock)
    except (OSError, ValueError, IndexError, subprocess.SubprocessError):
        pass
    return info


def stage_of(name: str) -> str | None:
    for piece, stage in STAGES:
        if piece in name:
            return stage
    return None


def time_size(n: int, builds: int, flush: torch.Tensor) -> dict:
    pts, nrm = synthetic.bumpy_sphere(n, seed=0)
    radius = 5.0 * synthetic.mean_spacing(n)
    xyz, nrm_dev = upload(pts), upload(nrm)
    grid = Grid().set_speculative(builds=True)
    grid.build(xyz, nrm_dev, radius)  # the synchronising build whose box the others assume
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(builds)]
    for it in range(WARMUP + builds):
        flush.fill_(it & 0xFF)
        if it >= WARMUP:
            ev[it - WARMUP][0].record()
        grid.build(xyz, nrm_dev, radius)
        if it >= WARMUP:
            ev[it - WARMUP][1].record()
    torch.cuda.synchronize()
    ms = np.array([a.elapsed_time(b) for a, b in ev])

    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for it in range(builds):
            flush.fill_(it & 0xFF)
            grid.build(xyz, nrm_dev, radius)
        torch.cuda.synchronize()
    assert grid.poll() == 0, "a build assumed a box its points did not fit"
    kernels_us, other_us = {}, {}
    for a in prof.key_averages():
        us = float(getattr(a, "self_device_time_total", 0.0) or getattr(a, "device_time_total", 0.0))
        if us <= 0.0:
            continue
        stage = stage_of(a.key)
        if stage is None:
            other_us[a.key[:80]] = us / builds
        else:
            kernels_us[stage] = kernels_us.get(stage, 0.0) + us / builds
    info = grid.info()
    grid.close()
    least = 152 * n
    return {
        "n_points": n, "radius": radius, "ncells": info["ncells"], "builds": builds,
        "build_ms_median": float(np.median(ms)), "build_ms_mean": float(ms.mean()), "build_ms_min": float(ms.min()),
        "build_ms_p90": float(np.percentile(ms, 90)),
        "kernel_us_per_build": kernels_us, "kernels_us_sum": float(sum(kernels_us.values())),
        "not_in_build_us_per_build": other_us,
        "least_bytes": least, "least_bytes_GBps_at_median": least / (np.median(ms) * 1e-3) / 1e9,
    }


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1000000,10000000")
    ap.add_argument("--builds", type=int, default=200)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    require_cuda()
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")  # 512 MB > 126 MB of L2
    result = {"what": "grid build (speculative rebuild), bumpy sphere with normals, radius 5 mean spacings",
              "card": card(), "l2": "overwritten (512 MB) between builds",
              "grid_radix": os.environ.get("SF_GRID_RADIX", "0"), "sizes": []}
    for n in (int(x) for x in args.sizes.split(",")):
        result["sizes"].append(time_size(n, args.builds, flush))
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "grid_b200.json"), "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
