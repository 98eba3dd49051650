"""
TEST INFRASTRUCTURE ONLY. Writes tests/golden/orient_pins.npz: the orientation oracle's final parities, tree labels
and tree counts on fixed seeded inputs (ORIENT_CASES), so that tests/test_orient_host.py can hold
oracle/orientation_oracle.py in place.

    python -m oracle.make_orient_pins
"""

from __future__ import annotations

import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import orientation_oracle  # noqa: E402
from shot_fpfh_b200 import synthetic  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "orient_pins.npz")
K = 10
# (name, cloud, viewpoint)
ORIENT_CASES = (
    ("sphere_eigh", "sphere", None),
    ("sphere_eigh_inside", "sphere", "centre"),
    ("two_spheres_flipped", "two_spheres", None),
    ("plane_flipped_above", "plane", (0.3, -0.2, 2.0)),
)


def eigh_normals(points: np.ndarray, nbr: np.ndarray) -> np.ndarray:
    """PCA normals with LAPACK's sign, as compute_normals gives them without pre_computed_normals."""
    nb = points[nbr]
    c = nb - nb.mean(axis=1, keepdims=True)
    return np.linalg.eigh(np.einsum("nki,nkj->nij", c, c) / nbr.shape[1])[1][:, :, 0]


def case_inputs(kind: str) -> tuple[np.ndarray, np.ndarray]:
    """(points, normals) of the seeded clouds the pins use."""
    rng = np.random.default_rng(17)
    if kind == "sphere":
        pts, _ = synthetic.bumpy_sphere(3000, seed=23)
        return pts, eigh_normals(pts, orientation_oracle.sklearn_knn(pts, K))
    if kind == "two_spheres":
        a, da = synthetic.bumpy_sphere(1500, seed=24)
        b, db = synthetic.bumpy_sphere(1500, seed=25)
        pts = np.concatenate([a, b + [5.0, 0.0, 0.0]])
        nrm = synthetic.bumpy_sphere_true_normals(np.concatenate([da, db]))
        return pts, nrm * rng.choice([-1.0, 1.0], size=(3000, 1))
    xy = rng.uniform(-1.0, 1.0, size=(2000, 2))
    pts = np.concatenate([xy, 0.01 * rng.normal(size=(2000, 1))], axis=1)
    nrm = np.tile([0.0, 0.0, 1.0], (2000, 1)) + 0.05 * rng.normal(size=(2000, 3))
    return pts, nrm * rng.choice([-1.0, 1.0], size=(2000, 1))


def compute() -> dict:
    out = {}
    for name, kind, view in ORIENT_CASES:
        pts, nrm = case_inputs(kind)
        towards = pts.mean(axis=0) if view == "centre" else view
        _, d = orientation_oracle.orient(pts, nrm, orientation_oracle.sklearn_knn(pts, K), towards, details=True)
        out[f"{name}_parity"] = d["parity"]
        out[f"{name}_low"] = d["low"]
        out[f"{name}_n_trees"] = np.array(d["n_trees"])
    return out


def main() -> None:
    out = compute()
    np.savez_compressed(OUT, **out)
    print(f"wrote {OUT}: " + ", ".join(f"{k} {int(v)}" for k, v in out.items() if k.endswith("_n_trees")))


if __name__ == "__main__":
    main()
