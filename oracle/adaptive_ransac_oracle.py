"""
TEST INFRASTRUCTURE — NumPy restatement of adaptive RANSAC on matches as
shot_fpfh_b200.matching.ransac_on_matches_adaptive computes it. Only tests/, oracle/ and scripts/ may import this module.

The reference has no adaptive RANSAC, so this module IS the specification (as iss_oracle.py is for ISS). With m
matches (a_i scan keypoint, b_i reference keypoint, float64):

  1. Draw d (a global index 0, 1, 2, ... independent of batching), slot s = 0, 1, 2:
     u_s = splitmix64(seed * 0x9E3779B97F4A7C15 + 3d + s) >> 32 (uint64, wrapping; splitmix64 = the finaliser only),
     j0 = (u0 m) >> 32; j1 = (u1 (m-1)) >> 32, +1 if >= j0; j2 = (u2 (m-2)) >> 32, +1 if >= min(j0, j1), then +1 if
     >= max(j0, j1). The three indices are distinct and every product fits in 64 bits (u < 2^32, m < 2^32).
  2. Edge check: for every pair (p, q) of the three, min(|a_p-a_q|, |b_p-b_q|) >= edge_similarity * max(...), each
     length sqrt((dx*dx + dy*dy) + dz*dz) without FMA.
  3. Kabsch on the three pairs: centres ((x0 + x1) + x2) / 3, H = sum_k a_c b_c^T, M = H^T H (each entry summed
     k = 0, 1, 2 in that order), eigh(M) (np.linalg.eigh, the dsyevd path); v1, v2 = eigenvectors of the largest and
     middle eigenvalue; degenerate (rejected) if lambda_mid <= 1e-12 lambda_max; u_k = H v_k / |H v_k|,
     u3 = u1 x u2, v3 = v1 x v2, R = [v1 v2 v3][u1 u2 u3]^T, t = b_bar - R a_bar.
  4. Self-check: the draw is valid only if its own three pairs are inliers of (R, t).
  5. Inlier: sqrt(|R a + t - b|^2) <= threshold, i.e. |.|^2 <= T with T the largest double whose sqrt is <= threshold.
  6. Winner: the valid draw with the most inliers, ties to the lowest draw index. Draws run in batches of
     B = 2^20; after batch k stop if k B >= max_draws (the last batch is truncated to max_draws), or if the winner's
     count c > 0 and k B log1p(-(c/m)^3) <= log(1 - confidence).

Pinned by tests/golden/adaptive_ransac_pins.npz (oracle/make_adaptive_ransac_pins.py).
"""

from __future__ import annotations

import math

import numpy as np

BATCH = 1 << 20
GOLDEN_GAMMA = 0x9E3779B97F4A7C15
MASK64 = (1 << 64) - 1
DEGENERATE = 1e-12
PAIRS = ((0, 1), (0, 2), (1, 2))


def splitmix64(z: np.ndarray) -> np.ndarray:
    z = np.asarray(z, dtype=np.uint64).copy()
    with np.errstate(over="ignore"):
        z ^= z >> np.uint64(30)
        z *= np.uint64(0xBF58476D1CE4E5B9)
        z ^= z >> np.uint64(27)
        z *= np.uint64(0x94D049BB133111EB)
        z ^= z >> np.uint64(31)
    return z


def draw_indices(seed: int, draws: np.ndarray, m: int) -> np.ndarray:
    """(D, 3) int64 match indices of the global draw indices `draws`."""
    base = np.uint64((int(seed) * GOLDEN_GAMMA) & MASK64)
    d = np.asarray(draws, dtype=np.uint64)
    with np.errstate(over="ignore"):
        x = base + np.uint64(3) * d
        u = [splitmix64(x + np.uint64(s)) >> np.uint64(32) for s in range(3)]
    m64 = np.uint64(m)
    j0 = (u[0] * m64) >> np.uint64(32)
    j1 = (u[1] * (m64 - np.uint64(1))) >> np.uint64(32)
    j1 = j1 + (j1 >= j0).astype(np.uint64)
    j2 = (u[2] * (m64 - np.uint64(2))) >> np.uint64(32)
    j2 = j2 + (j2 >= np.minimum(j0, j1)).astype(np.uint64)
    j2 = j2 + (j2 >= np.maximum(j0, j1)).astype(np.uint64)
    return np.stack([j0, j1, j2], axis=1).astype(np.int64)


def _length(p: np.ndarray, q: np.ndarray) -> np.ndarray:
    d = p - q
    return np.sqrt((d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2])


def edges_consistent(a3: np.ndarray, b3: np.ndarray, edge_similarity: float) -> np.ndarray:
    """(D,) bool: step 2 on the (D, 3, 3) matched points of each draw."""
    ok = np.ones(a3.shape[0], dtype=bool)
    for p, q in PAIRS:
        la, lb = _length(a3[:, p], a3[:, q]), _length(b3[:, p], b3[:, q])
        ok &= np.minimum(la, lb) >= edge_similarity * np.maximum(la, lb)
    return ok


def _dot3(x: np.ndarray, y: np.ndarray) -> np.ndarray:
    return (x[..., 0] * y[..., 0] + x[..., 1] * y[..., 1]) + x[..., 2] * y[..., 2]


def _cross(x: np.ndarray, y: np.ndarray) -> np.ndarray:
    return np.stack([x[:, 1] * y[:, 2] - x[:, 2] * y[:, 1], x[:, 2] * y[:, 0] - x[:, 0] * y[:, 2],
                     x[:, 0] * y[:, 1] - x[:, 1] * y[:, 0]], axis=1)


def kabsch3(a3: np.ndarray, b3: np.ndarray) -> tuple[np.ndarray, np.ndarray]:
    """Step 3: ((D, 12) rows [R row-major | t], (D,) bool not degenerate)."""
    d = a3.shape[0]
    abar = ((a3[:, 0] + a3[:, 1]) + a3[:, 2]) / 3.0
    bbar = ((b3[:, 0] + b3[:, 1]) + b3[:, 2]) / 3.0
    ac, bc = a3 - abar[:, None], b3 - bbar[:, None]
    h = np.empty((d, 3, 3))
    for i in range(3):
        for j in range(3):
            h[:, i, j] = _dot3(ac[:, :, i], bc[:, :, j])
    mtm = np.empty((d, 3, 3))
    for i in range(3):
        for j in range(3):
            mtm[:, i, j] = _dot3(h[:, :, i], h[:, :, j])
    lam, vec = np.linalg.eigh(mtm) if d else (np.empty((0, 3)), np.empty((0, 3, 3)))
    ok = ~(lam[:, 1] <= DEGENERATE * lam[:, 2])
    v1, v2 = vec[:, :, 2], vec[:, :, 1]
    with np.errstate(divide="ignore", invalid="ignore"):
        hv1 = np.stack([_dot3(h[:, i], v1) for i in range(3)], axis=1)
        hv2 = np.stack([_dot3(h[:, i], v2) for i in range(3)], axis=1)
        u1 = hv1 / np.sqrt(_dot3(hv1, hv1))[:, None]
        u2 = hv2 / np.sqrt(_dot3(hv2, hv2))[:, None]
        u3, v3 = _cross(u1, u2), _cross(v1, v2)
        r = np.empty((d, 3, 3))
        for i in range(3):
            for j in range(3):
                r[:, i, j] = (v1[:, i] * u1[:, j] + v2[:, i] * u2[:, j]) + v3[:, i] * u3[:, j]
        t = bbar - np.stack([_dot3(r[:, i], abar) for i in range(3)], axis=1)
    return np.concatenate([r.reshape(d, 9), t], axis=1), ok


def threshold_sq(threshold: float) -> float:
    """The largest double T with sqrt(T) <= threshold: `d2 <= T` is then exactly `sqrt(d2) <= threshold`."""
    t = float(threshold) * float(threshold)
    while math.sqrt(t) > threshold:
        t = math.nextafter(t, 0.0)
    while math.sqrt(math.nextafter(t, math.inf)) <= threshold:
        t = math.nextafter(t, math.inf)
    return t


def residual_sq(transforms: np.ndarray, a: np.ndarray, b: np.ndarray) -> np.ndarray:
    """|R a + t - b|^2, summed as the device sums it, broadcast over leading axes: transforms (D, 12) against their own
    pairs a, b (D, 3) -> (D,); transforms (D, 1, 12) against all pairs (n, 3) -> (D, n); one (12,) -> (n,)."""
    d = [((transforms[..., 3 * i] * a[..., 0] + transforms[..., 3 * i + 1] * a[..., 1])
          + transforms[..., 3 * i + 2] * a[..., 2]) + transforms[..., 9 + i] - b[..., i] for i in range(3)]
    return (d[0] * d[0] + d[1] * d[1]) + d[2] * d[2]


def count_inliers(transforms: np.ndarray, a: np.ndarray, b: np.ndarray, t_sq: float) -> np.ndarray:
    """(D,) inliers of each transform row, in chunks of about 4M residuals."""
    out = np.zeros(transforms.shape[0], dtype=np.int64)
    chunk = max(1, (1 << 22) // max(1, a.shape[0]))
    for s in range(0, transforms.shape[0], chunk):
        out[s:s + chunk] = (residual_sq(transforms[s:s + chunk, None], a, b) <= t_sq).sum(axis=1)
    return out


def run_batch(a: np.ndarray, b: np.ndarray, threshold: float, edge_similarity: float, seed: int, first: int,
              count: int) -> dict:
    """One batch of draws [first, first + count): the survivors of the edge check, the valid draws, their
    transforms and inlier counts (draw indices ascending)."""
    m = a.shape[0]
    draws = np.arange(first, first + count, dtype=np.int64)
    idx = draw_indices(seed, draws, m)
    passed = edges_consistent(a[idx], b[idx], edge_similarity)
    survivors, idx = draws[passed], idx[passed]
    transforms, ok = kabsch3(a[idx], b[idx])
    t_sq = threshold_sq(threshold)
    own = np.ones(ok.shape[0], dtype=bool)
    for s in range(3):
        own &= residual_sq(transforms, a[idx[:, s]], b[idx[:, s]]) <= t_sq
    valid = ok & own
    return {"survivors": survivors, "valid_draws": survivors[valid], "transforms": transforms[valid],
            "counts": count_inliers(transforms[valid], a, b, t_sq)}


def should_stop(k: int, count: int, m: int, confidence: float) -> bool:
    """The confidence rule after batch k (k >= 1) with the winner's count."""
    if count <= 0:
        return False
    r = count / m
    return float(k * BATCH) * math.log1p(-(r * r * r)) <= math.log(1.0 - confidence)


def ransac_adaptive(a: np.ndarray, b: np.ndarray, threshold: float, confidence: float = 0.999,
                    max_draws: int = 1 << 24, edge_similarity: float = 0.9, seed: int = 0) -> dict:
    """The whole search: winner draw and count (-1 and 0 if no draw is valid), draws used, batches, survivors and
    valid draws over all batches, the winner's transform and the inlier mask of the matches under it."""
    a = np.ascontiguousarray(a, dtype=np.float64)
    b = np.ascontiguousarray(b, dtype=np.float64)
    m = a.shape[0]
    best_key, best_transform = 0, None
    k = survivors = valid = 0
    while True:
        first = k * BATCH
        batch = run_batch(a, b, threshold, edge_similarity, seed, first, min(BATCH, max_draws - first))
        survivors += batch["survivors"].shape[0]
        valid += batch["valid_draws"].shape[0]
        if batch["counts"].shape[0]:
            keys = (batch["counts"].astype(np.uint64) << np.uint64(32)) | (
                np.uint64(0xFFFFFFFF) - batch["valid_draws"].astype(np.uint64))
            top = int(np.argmax(keys))
            if int(keys[top]) > best_key:
                best_key, best_transform = int(keys[top]), batch["transforms"][top]
        k += 1
        if k * BATCH >= max_draws or should_stop(k, best_key >> 32, m, confidence):
            break
    count = best_key >> 32
    out = {"best_draw": 0xFFFFFFFF - (best_key & 0xFFFFFFFF) if count else -1, "best_count": count,
           "draws_used": min(k * BATCH, max_draws), "batches": k, "survivors": survivors, "valid": valid,
           "transform": best_transform}
    if count:
        out["mask"] = residual_sq(best_transform, a, b) <= threshold_sq(threshold)
    return out
