"""
Seeded synthetic point clouds used by the tests and by bench.py.

The "bumpy sphere" surface scan of SURVEY.md §8(d) / BASELINE.md §3: a unit sphere whose radius is
modulated by a smooth function of the direction, so that the local geometry is not degenerate
(distinct principal curvatures almost everywhere) while the sampling density stays uniform enough
that ``radius = 5 x mean spacing`` gives K ~ 72 neighbours per query.

Nothing here touches the GPU; it only builds the float64 host arrays that the reference API takes.
"""

from __future__ import annotations

import numpy as np
import numpy.typing as npt

_PAIR_ROTVEC = 0.5 * np.array([1.0, 2.0, 3.0]) / np.sqrt(14.0)
_PAIR_TRANSLATION = np.array([0.3, -0.2, 0.1])


def bumpy_sphere(
    n_points: int, seed: int = 0
) -> tuple[npt.NDArray[np.float64], npt.NDArray[np.float64]]:
    """
    Returns (points, directions): ``points = d * rho(d)`` with ``d`` uniform on the unit sphere.
    ``directions`` (unit, radial) double as cheap outward normals at the large sizes.
    """
    rng = np.random.default_rng(seed)
    d = rng.normal(size=(n_points, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    rho = 1.0 + 0.15 * np.sin(5.0 * d[:, 0]) * np.cos(3.0 * d[:, 1]) + 0.05 * np.sin(9.0 * d[:, 2])
    return d * rho[:, None], d


def bumpy_sphere_true_normals(directions: npt.NDArray[np.float64]) -> npt.NDArray[np.float64]:
    """
    Outward unit normals of the bumpy sphere itself at the points `bumpy_sphere` returns for `directions`: for a
    star-shaped surface x = rho(d) d the normal is along rho d - (I - d d^T) grad rho. (The radial directions that the
    benchmark uses as cheap normals make point-to-plane ICP degenerate: every cross(p, n) is perpendicular to the
    pair's translation, so the 6x6 system is singular as soon as the residual is not exactly zero.)
    """
    d = directions
    rho = 1.0 + 0.15 * np.sin(5.0 * d[:, 0]) * np.cos(3.0 * d[:, 1]) + 0.05 * np.sin(9.0 * d[:, 2])
    grad = np.stack([
        0.75 * np.cos(5.0 * d[:, 0]) * np.cos(3.0 * d[:, 1]),
        -0.45 * np.sin(5.0 * d[:, 0]) * np.sin(3.0 * d[:, 1]),
        0.45 * np.cos(9.0 * d[:, 2]),
    ], axis=1)
    tangential = grad - np.sum(grad * d, axis=1, keepdims=True) * d
    n = rho[:, None] * d - tangential
    return n / np.linalg.norm(n, axis=1, keepdims=True)


def mean_spacing(n_points: int) -> float:
    """Mean point spacing of n points on (about) a unit sphere: sqrt(4 pi / n)."""
    return float(np.sqrt(4.0 * np.pi / n_points))


def rotation_from_rotvec(rotvec: npt.NDArray[np.float64]) -> npt.NDArray[np.float64]:
    """Rodrigues formula (kept local so that the generator does not depend on scipy)."""
    angle = float(np.linalg.norm(rotvec))
    if angle == 0.0:
        return np.eye(3)
    k = rotvec / angle
    kx = np.array([[0.0, -k[2], k[1]], [k[2], 0.0, -k[0]], [-k[1], k[0], 0.0]])
    return np.eye(3) + np.sin(angle) * kx + (1.0 - np.cos(angle)) * (kx @ kx)


def rigid_pair(
    points: npt.NDArray[np.float64],
    normals: npt.NDArray[np.float64],
    perm_seed: int = 1,
) -> tuple[
    npt.NDArray[np.float64],
    npt.NDArray[np.float64],
    npt.NDArray[np.int64],
    npt.NDArray[np.float64],
    npt.NDArray[np.float64],
]:
    """
    Builds the second cloud of a registration pair: rotate, translate and permute.
    Returns (ref_points, ref_normals, perm, rotation, translation) with
    ``ref_points = (points @ R.T + t)[perm]``.
    """
    rot = rotation_from_rotvec(_PAIR_ROTVEC)
    perm = np.random.default_rng(perm_seed).permutation(points.shape[0])
    ref = np.ascontiguousarray((points @ rot.T + _PAIR_TRANSLATION)[perm])
    ref_normals = np.ascontiguousarray((normals @ rot.T)[perm])
    return ref, ref_normals, perm, rot, _PAIR_TRANSLATION.copy()


def corrupted_matches(
    n: int, inlier_ratio: float, noise: float = 0.0, seed: int = 0
) -> tuple[
    npt.NDArray[np.float64],
    npt.NDArray[np.float64],
    npt.NDArray[np.int64],
    npt.NDArray[np.int64],
    npt.NDArray[np.float64],
    npt.NDArray[np.float64],
]:
    """
    A registration pair with n matches of known quality, for coarse-alignment tests: the bumpy sphere of n points and
    its `rigid_pair` copy, with isotropic Gaussian noise of standard deviation `noise` added to the reference points.
    Match i pairs scan point i with its true counterpart for round(inlier_ratio * n) randomly chosen i and with a
    uniformly drawn reference point otherwise. Returns (scan, ref, scan_idx, ref_idx, rotation, translation), with
    ref ~ (scan @ rotation.T + translation)[perm].
    """
    scan, directions = bumpy_sphere(n, seed=seed)
    ref, _, perm, rot, trans = rigid_pair(scan, directions, perm_seed=seed + 1)
    rng = np.random.default_rng(seed + 2)
    if noise > 0.0:
        ref = ref + rng.normal(scale=noise, size=ref.shape)
    inverse = np.empty(n, dtype=np.int64)
    inverse[perm] = np.arange(n)
    scan_idx = np.arange(n, dtype=np.int64)
    ref_idx = rng.integers(0, n, size=n)
    correct = rng.permutation(n)[: int(round(inlier_ratio * n))]
    ref_idx[correct] = inverse[correct]
    return scan, np.ascontiguousarray(ref), scan_idx, ref_idx, rot, trans


def voxel_first_point_queries(
    points: npt.NDArray[np.float64], voxel_size: float
) -> npt.NDArray[np.int64]:
    """
    Cheap O(N log N) query selector for the large benchmark sizes: one point per occupied voxel
    (the first one in index order). The reference's grid_subsampling picks the point closest to the
    voxel barycentre with a Python loop over voxels (4.4 s at 1M points, SURVEY.md §6); which point of
    the voxel is the query is irrelevant to the descriptor kernels, so the benchmark uses this.
    """
    keys = np.floor((points - points.min(axis=0)) / voxel_size).astype(np.int64)
    dims = keys.max(axis=0) + 1
    flat = (keys[:, 0] * dims[1] + keys[:, 1]) * dims[2] + keys[:, 2]
    _, first = np.unique(flat, return_index=True)
    return np.sort(first).astype(np.int64)


def sparse_unit_rows(
    n_rows: int, dim: int = 352, density: float = 0.14, seed: int = 2
) -> npt.NDArray[np.float32]:
    """
    Random non-negative rows with ~86 % exact zeros and unit L2 norm: the statistics of real SHOT rows
    (SURVEY.md F7), used as the pure-throughput input of the matching benchmark.
    """
    rng = np.random.default_rng(seed)
    rows = rng.random((n_rows, dim), dtype=np.float32)
    rows *= rng.random((n_rows, dim), dtype=np.float32) < density
    rows[:, 0] += 1e-3  # no all-zero rows
    rows /= np.linalg.norm(rows, axis=1, keepdims=True)
    return rows
