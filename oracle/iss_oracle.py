"""
TEST INFRASTRUCTURE — CPU restatement of ISS salient-keypoint detection (Intrinsic Shape Signatures, Zhong 2009) as
shot_fpfh_b200.keypoint_selection.select_keypoints_iss computes it. Only tests/ and oracle/ may import this module.

The reference has no ISS, so this module IS the specification (DESIGN.md §2, "pinned to a documented restatement").
It follows Open3D's definition (defaults, ratio tests, ties kept) with one deliberate difference, the covariance:

  1. N_s(i) = { j : ((dx*dx + dy*dy) + dz*dz) <= r_s^2 }, d = p_j - p_i, float64 without FMA — sklearn's
     `query_radius` predicate (i itself and any duplicates included); n_i = |N_s(i)|. N_n(i) likewise with r_n.
  2. c_j = p_j - p_i, mu = sum c_j / n_i, C_i = sum c_j c_j^T / n_i - mu mu^T: the covariance about the barycentre,
     accumulated about the point (Open3D accumulates about the origin, which loses the digits of a cloud far from it).
  3. e3 <= e2 <= e1 = np.linalg.eigh(C_i)[0] (the dsyevd path; eigvalsh takes dsterf and differs in the last bits).
  4. s_i = e3 if n_i >= m and e2 / e1 < gamma_21 and e3 / e2 < gamma_32 (IEEE divisions; NaN fails), else 0.
  5. i is a keypoint iff s_i > 0, |N_n(i)| >= m and s_i >= s_j for every j in N_n(i) (ties keep both).
  6. Output: original indices, int64, ascending.
  7. Radii 0.0 mean r_s = 6 res, r_n = 4 res, res = mean distance to the nearest OTHER point (a duplicate counts 0).

Sums run sequentially over each neighbourhood in KDTree order (np.add.reduceat), so the result does not depend on the
BLAS the machine has. Pinned by tests/golden/iss_pins.npz (oracle/make_iss_pins.py).
"""

from __future__ import annotations

import numpy as np
from sklearn.neighbors import KDTree

DEFAULT_GAMMA_21 = 0.975
DEFAULT_GAMMA_32 = 0.975
DEFAULT_MIN_NEIGHBORS = 5
SALIENT_MULTIPLIER = 6.0
NON_MAX_MULTIPLIER = 4.0


def neighbourhoods(points: np.ndarray, radius: float, queries: np.ndarray | None = None):
    """CSR (offsets int64[q + 1], flat int64 indices) of the cloud points within `radius` of each query (default: the
    cloud's own points)."""
    q = points if queries is None else queries
    nbh = KDTree(points).query_radius(q, radius)
    counts = np.array([a.shape[0] for a in nbh], dtype=np.int64)
    offsets = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    flat = np.concatenate(list(nbh)).astype(np.int64) if q.shape[0] else np.empty(0, np.int64)
    return offsets, flat


def _segment_sums(values: np.ndarray, offsets: np.ndarray) -> np.ndarray:
    """Sequential sum of values[offsets[q]:offsets[q + 1]] per q (every segment holds at least the point itself)."""
    return np.add.reduceat(values, offsets[:-1], axis=0)


def covariance_eigenvalues(points: np.ndarray, salient_radius: float, idx: np.ndarray | None = None):
    """(n_i int64, eigenvalues (q, 3) ascending, covariances (q, 3, 3)) of the points `idx` (default: all)."""
    idx = np.arange(points.shape[0]) if idx is None else np.asarray(idx, dtype=np.int64)
    offsets, flat = neighbourhoods(points, salient_radius, points[idx])
    counts = np.diff(offsets)
    owner = np.repeat(np.arange(idx.shape[0]), counts)
    c = points[flat] - points[idx][owner]
    n = counts.astype(np.float64)[:, None]
    mu = _segment_sums(c, offsets) / n
    outer = (c[:, :, None] * c[:, None, :]).reshape(-1, 9)
    cov = (_segment_sums(outer, offsets) / n).reshape(-1, 3, 3) - mu[:, :, None] * mu[:, None, :]
    eig = np.linalg.eigh(cov)[0] if idx.shape[0] else np.empty((0, 3))
    return counts, eig, cov


def saliency_of(counts: np.ndarray, eig: np.ndarray, min_neighbors: int, gamma_21: float, gamma_32: float) -> np.ndarray:
    """Step 4: e3 where the ratio tests pass and the neighbourhood is large enough, else 0."""
    with np.errstate(divide="ignore", invalid="ignore"):
        r21 = eig[:, 1] / eig[:, 2]
        r32 = eig[:, 0] / eig[:, 1]
    ok = (counts >= min_neighbors) & (r21 < gamma_21) & (r32 < gamma_32)
    return np.where(ok, eig[:, 0], 0.0)


def resolution(points: np.ndarray) -> float:
    """Mean distance from each point to its nearest other point (a duplicate counts 0)."""
    dist, _ = KDTree(points).query(points, k=2)
    return float(dist[:, 1].mean())


def default_radii(points: np.ndarray) -> tuple[float, float]:
    res = resolution(points)
    return SALIENT_MULTIPLIER * res, NON_MAX_MULTIPLIER * res


def iss(
    points: np.ndarray,
    salient_radius: float = 0.0,
    non_max_radius: float = 0.0,
    gamma_21: float = DEFAULT_GAMMA_21,
    gamma_32: float = DEFAULT_GAMMA_32,
    min_neighbors: int = DEFAULT_MIN_NEIGHBORS,
    details: bool = False,
):
    """Keypoints (int64, ascending); with `details` a dict of everything the tests compare as well."""
    points = np.ascontiguousarray(points, dtype=np.float64).reshape(-1, 3)
    n = points.shape[0]
    empty = np.empty(0, np.int64)
    if salient_radius == 0.0 or non_max_radius == 0.0:
        salient_radius, non_max_radius = default_radii(points) if n >= 2 else (0.0, 0.0)
    if n == 0:
        return (empty, {"keypoints": empty}) if details else empty
    counts, eig, _ = covariance_eigenvalues(points, salient_radius)
    s = saliency_of(counts, eig, min_neighbors, gamma_21, gamma_32)
    offsets, flat = neighbourhoods(points, non_max_radius)
    nms_counts = np.diff(offsets)
    nbr_max = np.maximum.reduceat(s[flat], offsets[:-1])
    keep = (s > 0.0) & (nms_counts >= min_neighbors) & (s >= nbr_max)
    kp = np.flatnonzero(keep).astype(np.int64)
    if not details:
        return kp
    return kp, {
        "keypoints": kp, "saliency": s, "counts": counts, "eigenvalues": eig, "nms_counts": nms_counts,
        "nms_offsets": offsets, "nms_flat": flat, "salient_radius": float(salient_radius),
        "non_max_radius": float(non_max_radius),
    }


def margin_points(eig: np.ndarray, gamma_21: float, gamma_32: float, salient_radius: float) -> np.ndarray:
    """Points whose ratio tests, or the sign of e3, lie within the rounding a reordered float64 sum can move them."""
    tol = 1e-12 * salient_radius**2
    with np.errstate(divide="ignore", invalid="ignore"):
        r21 = eig[:, 1] / eig[:, 2]
        r32 = eig[:, 0] / eig[:, 1]
        m32 = 1e-9 + tol / np.abs(eig[:, 1])
    return (np.abs(r21 - gamma_21) <= 1e-9) | (np.abs(r32 - gamma_32) <= m32) | (np.abs(eig[:, 0]) <= tol)


def excused(d: dict, gamma_21: float, gamma_32: float) -> np.ndarray:
    """
    The points whose keypoint decision an implementation that only reorders the float64 sums may take differently:
    i, or a member of N_n(i), is a margin point, or a member j != i of N_n(i) has |s_i - s_j| <= 1e-12 r_s^2.
    """
    tol = 1e-12 * d["salient_radius"] ** 2
    margin = margin_points(d["eigenvalues"], gamma_21, gamma_32, d["salient_radius"])
    offsets, flat = d["nms_offsets"], d["nms_flat"]
    s = d["saliency"]
    owner = np.repeat(np.arange(s.shape[0]), np.diff(offsets))
    near_tie = (flat != owner) & (np.abs(s[owner] - s[flat]) <= tol)
    out = margin.copy()
    np.logical_or.at(out, owner, margin[flat] | near_tie)
    return out
