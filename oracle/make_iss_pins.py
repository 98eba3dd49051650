"""
TEST INFRASTRUCTURE ONLY. Writes tests/golden/iss_pins.npz: the ISS oracle's keypoints, saliencies and neighbourhood
sizes on fixed seeded inputs (ISS_CASES), so that tests/test_iss_host.py can hold oracle/iss_oracle.py in place.

    python -m oracle.make_iss_pins
"""

from __future__ import annotations

import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import iss_oracle  # noqa: E402
from shot_fpfh_b200 import synthetic  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "iss_pins.npz")
# (name, cloud, salient radius and non-max radius in mean spacings — None: the defaults from the resolution)
ISS_CASES = (
    ("sphere_rn_lt_rs", "sphere", (5.0, 3.75)),
    ("sphere_rn_gt_rs", "sphere", (3.0, 5.0)),
    ("sphere_defaults", "sphere", None),
    ("box_corner_defaults", "box", None),
)


def case_cloud(kind: str) -> tuple[np.ndarray, float]:
    """(points, mean spacing) of the seeded clouds the pins use."""
    if kind == "sphere":
        n = 3000
        return synthetic.bumpy_sphere(n, seed=41)[0], synthetic.mean_spacing(n)
    from conftest import registration_case

    scan = registration_case(n=2000, seed=43)[0]
    return scan, float(np.sqrt(3.0 / 2000))


def compute() -> dict:
    out = {}
    for name, kind, radii in ISS_CASES:
        pts, s = case_cloud(kind)
        rs, rn = (0.0, 0.0) if radii is None else (radii[0] * s, radii[1] * s)
        kp, d = iss_oracle.iss(pts, rs, rn, details=True)
        out[f"{name}_keypoints"] = kp
        out[f"{name}_saliency"] = d["saliency"]
        out[f"{name}_counts"] = d["counts"]
        out[f"{name}_nms_counts"] = d["nms_counts"]
        out[f"{name}_radii"] = np.array([d["salient_radius"], d["non_max_radius"]])
    return out


def main() -> None:
    out = compute()
    np.savez_compressed(OUT, **out)
    print(f"wrote {OUT}: " + ", ".join(f"{k} {v.shape}" for k, v in out.items() if k.endswith("_keypoints")))


if __name__ == "__main__":
    main()
