"""
`ransac_on_matches` with the reference's signature and random stream (shot_fpfh/matching/ransac.py:14-82).

What the reference does per draw: pick `draw_size` matches with its module-level `default_rng(72)`, fit a rigid
transform to them (Kabsch), count the matches the transform brings within `distance_threshold`; keep the first draw
with the largest count. The cost is the n_draws x n_matches count: that runs on the device
(`sf_ransac_count_inliers`, csrc/registration.cu). The draws replay NumPy's generator on the host — the same
generator, seeded and advanced the same way, so the same draws, taken from its raw stream in one vectorised pass
(`replay_choices`) — and the n_draws 3x3 SVDs are one batched host call.
The winning transform is then refitted with the scalar solver, i.e. exactly the reference's arithmetic.

`ransac_on_matches_adaptive` is this package's own coarse alignment for match sets with few inliers, where 10 000
draws of 4 matches rarely contain an all-inlier sample (probability w^4 per draw at inlier ratio w): device-drawn
3-match samples, an edge-length check that rejects most outlier triples before any fit, and as many draws as the
confidence asks for (`sf_ransac_adaptive`, csrc/registration.cu; specification: oracle/adaptive_ransac_oracle.py).
"""

from __future__ import annotations

import logging

import numpy as np
import numpy.typing as npt

from ..core import RigidTransform, solver_point_to_point

# the reference's seed and its module-level lifetime (ransac.py:14): successive calls continue the stream
rng = np.random.default_rng(seed=72)


def replay_choices(rng: np.random.Generator, population: int, size: int, n_draws: int) -> npt.NDArray[np.int64]:
    """
    `n_draws` successive `rng.choice(population, size, replace=False, shuffle=False)` (ransac.py:48-53) as ONE
    (n_draws, size) array, leaving `rng` exactly in the state those calls would leave it in — the Python loop of 10 000
    calls was 51 ms of the 83 ms of a RANSAC run. What NumPy does per call, restated on the raw PCG64 stream: Floyd's
    algorithm over j = population - size .. population - 1, each value uniform in [0, j] by Lemire's method on the
    next 32 bits (low half of a 64-bit output first, then its high half, buffered across calls), a value already in
    the sample replaced by j. The rare rejections of Lemire's method shift the stream and are followed one by one;
    anything outside this regime (another bit generator, populations beyond 2^32, NumPy's tail-shuffle regime, a
    run of rejections) falls back to the calls themselves. Bit-identical draws and generator state: checked against
    NumPy on the CPU (tests/test_abi_and_host_logic.py).
    """
    def sequential():
        return np.stack([rng.choice(population, size, replace=False, shuffle=False) for _ in range(n_draws)]) if n_draws else np.zeros((0, size), dtype=np.int64)
    bitgen = rng.bit_generator
    if (type(bitgen).__name__ != "PCG64" or n_draws == 0 or size <= 0 or size > population or population > 0xFFFFFFFF
            or population - size < 1 or (population > 10000 and size > population // 50)):
        return sequential()
    start = bitgen.state
    pending = bool(start["has_uint32"])
    need = n_draws * size
    slack = 64
    words = (need + slack + 1) // 2 + 1
    raw = bitgen.random_raw(words)
    stream = np.empty(2 * words + 1, dtype=np.uint64)
    off = 0
    if pending:
        stream[0] = start["uinteger"]
        off = 1
    stream[off::2][:words] = raw & np.uint64(0xFFFFFFFF)
    stream[off + 1::2][:words] = raw >> np.uint64(32)
    total = off + 2 * words
    # bounds of the `size` Floyd steps: j = population - size + t, value uniform in [0, j]
    j = np.arange(population - size, population, dtype=np.uint64)
    excl = j + np.uint64(1)
    threshold = (np.uint64(1 << 32) - excl) % excl
    vals = np.empty(need, dtype=np.uint64)
    pos = 0          # next stream element
    done = 0         # flat draws completed
    rejections = 0
    while done < need:
        count = need - done
        if pos + count > total:
            bitgen.state = start
            return sequential()
        t = (done + np.arange(count)) % size
        m = stream[pos:pos + count] * excl[t]
        rejected = (m & np.uint64(0xFFFFFFFF)) < threshold[t]
        bad = np.flatnonzero(rejected)
        ok = count if bad.size == 0 else int(bad[0])
        vals[done:done + ok] = m[:ok] >> np.uint64(32)
        done += ok
        pos += ok
        if bad.size:
            rejections += 1
            pos += 1  # the rejected element is consumed; the same draw takes the next one
            if rejections > 64:
                bitgen.state = start
                return sequential()
    vals = vals.reshape(n_draws, size).astype(np.int64)
    out = np.empty_like(vals)
    ji = j.astype(np.int64)
    for t in range(size):  # Floyd: a value already drawn in this sample is replaced by j
        dup = (vals[:, t:t + 1] == out[:, :t]).any(axis=1) if t else np.zeros(n_draws, dtype=bool)
        out[:, t] = np.where(dup, ji[t], vals[:, t])
    # leave the generator where the sequential calls would: `pos` stream elements consumed
    consumed = pos - off  # elements taken from fresh 64-bit outputs
    bitgen.state = start
    bitgen.advance((consumed + 1) // 2)
    after = bitgen.state
    if consumed > 0:  # the high half of the last output is what the buffer holds, used (even count) or not (odd)
        after["has_uint32"] = consumed % 2
        after["uinteger"] = int(stream[off + 2 * ((consumed - 1) // 2) + 1])
    else:  # only the element that was pending at entry, if any, was taken
        after["has_uint32"] = 0 if pos > 0 else start["has_uint32"]
        after["uinteger"] = start["uinteger"]
    bitgen.state = after
    return out


def _batched_kabsch(scan: npt.NDArray[np.float64], ref: npt.NDArray[np.float64]) -> npt.NDArray[np.float64]:
    """(D, k, 3) x2 -> (D, 12) rows [rotation row-major | translation] of the fit of each draw (solvers.py:9-31)."""
    scan_centre, ref_centre = scan.mean(axis=1), ref.mean(axis=1)
    cov = np.einsum("dki,dkj->dij", scan - scan_centre[:, None, :], ref - ref_centre[:, None, :])
    u, _, vt = np.linalg.svd(cov)
    rotation = np.einsum("dki,djk->dij", vt, u)  # V U^T
    reflected = np.linalg.det(rotation) < 0
    if reflected.any():
        u = u.copy()
        u[reflected, :, -1] *= -1  # the reference negates the last row of U^T
        rotation = np.einsum("dki,djk->dij", vt, u)
    translation = ref_centre - np.einsum("dij,dj->di", rotation, scan_centre)
    return np.concatenate([rotation.reshape(-1, 9), translation], axis=1)


def ransac_on_matches(
    scan_descriptors_indices: np.ndarray,
    ref_descriptors_indices: np.ndarray,
    scan_keypoints: npt.NDArray[np.float64],
    ref_keypoints: npt.NDArray[np.float64],
    n_draws: int = 10000,
    draw_size: int = 4,
    distance_threshold: float = 1,
    verbose: bool = False,
    disable_progress_bar: bool = False,
) -> tuple[float, RigidTransform]:
    """Returns (share of the matches that are inliers of the best draw, its rigid transform), as the reference."""
    import torch

    from .. import ops
    from ..device import upload

    n_matches = scan_descriptors_indices.shape[0]
    matched_scan = np.ascontiguousarray(scan_keypoints[scan_descriptors_indices], dtype=np.float64)
    matched_ref = np.ascontiguousarray(ref_keypoints[ref_descriptors_indices], dtype=np.float64)
    # ransac.py:48-53, one call per draw: the generator's stream is what makes the result reproducible
    draws = replay_choices(rng, int(n_matches), int(draw_size), int(n_draws))
    transforms = _batched_kabsch(matched_scan[draws], matched_ref[draws])
    counts = ops.ransac_count_inliers(upload(matched_scan), upload(matched_ref), upload(transforms),
                                      float(distance_threshold))
    best = int(torch.argmax(counts).item())  # first maximum = the reference's strict `>` update (ransac.py:63)
    best_n_inliers = int(counts[best].item())
    if verbose:
        logging.info(f"Best draw: #{best} with {best_n_inliers} inliers out of {n_matches} matches")
    best_transform = solver_point_to_point(matched_scan[draws[best]], matched_ref[draws[best]])
    best_transform.normalize_rotation()
    return best_n_inliers / n_matches, best_transform


def ransac_on_matches_adaptive(
    scan_descriptors_indices: np.ndarray,
    ref_descriptors_indices: np.ndarray,
    scan_keypoints: npt.NDArray[np.float64],
    ref_keypoints: npt.NDArray[np.float64],
    distance_threshold: float = 1,
    confidence: float = 0.999,
    max_draws: int = 1 << 24,
    edge_similarity: float = 0.9,
    seed: int = 0,
    verbose: bool = False,
) -> tuple[float, RigidTransform]:
    """
    Adaptive RANSAC on the matches, on the device. Returns (share of the matches that are inliers of the best
    hypothesis, its transform refitted on all those inliers by `solver_point_to_point`, rotation normalised), as
    `ransac_on_matches` does.

    Draw d takes three distinct matches from a counter-based generator seeded by `seed`; it is fitted only if every
    edge of the triple has the same length in both clouds within `edge_similarity` (shorter >= edge_similarity x
    longer), and kept only if its own three matches are inliers of its fit. A match is an inlier when
    ||R a + t - b|| <= distance_threshold. Draws run in batches of 2^20 until `max_draws`, or until the chance that
    every draw so far missed an all-inlier triple, (1 - (c / m)^3)^draws for the best count c, is at most
    1 - confidence. The best hypothesis has the most inliers; ties go to the earliest draw. The result depends only
    on the inputs and `seed`.

    Raises ValueError on fewer than 3 or more than 2^32 - 1 matches, non-finite matched keypoints,
    distance_threshold <= 0, confidence outside (0, 1), edge_similarity outside (0, 1] or max_draws outside
    [1, 2^32 - 1]; RuntimeError when no draw passes the checks (e.g. every triple collinear).
    """
    from .. import ops
    from ..device import upload

    n_matches = len(scan_descriptors_indices)
    if len(ref_descriptors_indices) != n_matches:
        raise ValueError(f"{n_matches} scan indices but {len(ref_descriptors_indices)} reference indices")
    if not 3 <= n_matches <= 0xFFFFFFFF:
        raise ValueError(f"adaptive RANSAC needs 3 to 2^32 - 1 matches, got {n_matches}")
    if not (np.isfinite(distance_threshold) and distance_threshold > 0):
        raise ValueError(f"distance_threshold must be positive and finite, got {distance_threshold}")
    if not 0.0 < confidence < 1.0:
        raise ValueError(f"confidence must lie in (0, 1), got {confidence}")
    if not 0.0 < edge_similarity <= 1.0:
        raise ValueError(f"edge_similarity must lie in (0, 1], got {edge_similarity}")
    if not 1 <= max_draws <= 0xFFFFFFFF:
        raise ValueError(f"max_draws must lie in [1, 2^32 - 1], got {max_draws}")
    matched_scan = np.ascontiguousarray(scan_keypoints[scan_descriptors_indices], dtype=np.float64)
    matched_ref = np.ascontiguousarray(ref_keypoints[ref_descriptors_indices], dtype=np.float64)
    if not (np.isfinite(matched_scan).all() and np.isfinite(matched_ref).all()):
        raise ValueError("the matched keypoints must be finite")
    out = ops.ransac_adaptive(upload(matched_scan), upload(matched_ref), float(distance_threshold),
                              float(edge_similarity), int(seed), int(max_draws), float(confidence))
    if out["valid"] == 0:
        raise RuntimeError(f"adaptive RANSAC: none of {out['draws_used']} draws passed the edge and fit checks "
                           "(collinear or inconsistent matches)")
    if verbose:
        logging.info(f"Best draw: #{out['best_draw']} with {out['best_count']} inliers out of {n_matches} matches "
                     f"({out['draws_used']} draws, {out['valid']} valid)")
    inliers = out["mask"].cpu().numpy().astype(bool)
    best_transform = solver_point_to_point(matched_scan[inliers], matched_ref[inliers])
    best_transform.normalize_rotation()
    return out["best_count"] / n_matches, best_transform
