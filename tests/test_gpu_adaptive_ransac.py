"""
Adaptive RANSAC on the device (csrc/registration.cu: sf_ransac_adaptive) against its specification,
oracle/adaptive_ransac_oracle.py: the first batch's draws, edge-check survivors, fits and counts; the winner, the
stopping point and the refit; recovery at a low inlier ratio; repeatability, max_draws and the error cases.
"""

import numpy as np
import pytest

from oracle import adaptive_ransac_oracle as oracle
from shot_fpfh_b200 import synthetic

pytestmark = pytest.mark.gpu

THRESHOLD = 0.01
NOISE = 0.2 * THRESHOLD


def case(n, w, seed=5, noise=NOISE):
    scan, ref, si, ri, rot, trans = synthetic.corrupted_matches(n, w, noise=noise, seed=seed)
    return scan, ref, si, ri, rot, trans, np.ascontiguousarray(scan[si]), np.ascontiguousarray(ref[ri])


def device_batch(a, b, first=0, n=oracle.BATCH, seed=0, edge_similarity=0.9):
    from shot_fpfh_b200 import ops
    from shot_fpfh_b200.device import upload

    return ops.ransac_adaptive_batch(upload(a), upload(b), THRESHOLD, edge_similarity, seed, first, n)


@pytest.mark.parametrize("n,w", [(2000, 0.27), (20000, 0.03)])
def test_first_batch_matches_oracle(n, w):
    from shot_fpfh_b200 import ops
    from shot_fpfh_b200.device import upload

    *_, a, b = case(n, w)
    got = device_batch(a, b)
    want = oracle.run_batch(a, b, THRESHOLD, 0.9, 0, 0, oracle.BATCH)
    # the draw indices, edge-check outcomes and valid draws are bit-identical
    assert np.array_equal(got["survivors"].cpu().numpy(), want["survivors"])
    assert np.array_equal(got["valid_draws"].cpu().numpy(), want["valid_draws"])
    # the fits agree to 1e-12 plus the eigenvector perturbation bound eps * lambda_max / lambda_mid of H^T H: the
    # device's eigh3 contracts multiply-adds that LAPACK rounds separately, and a thin triangle (sigma_2 / sigma_1 ~ 0.01,
    # so lambda_max / lambda_mid ~ 1e8) turns those last bits into 1e-8 of its rotation
    diff = np.abs(got["transforms"].cpu().numpy() - want["transforms"]).max(axis=1)
    idx = oracle.draw_indices(0, want["valid_draws"], a.shape[0])
    ac, bc = a[idx] - a[idx].mean(axis=1, keepdims=True), b[idx] - b[idx].mean(axis=1, keepdims=True)
    h = np.einsum("dki,dkj->dij", ac, bc)
    lam = np.linalg.eigvalsh(np.einsum("dki,dkj->dij", h, h))
    assert (diff <= 1e-12 + 1e-15 * lam[:, 2] / lam[:, 1]).all()
    assert (diff[lam[:, 1] >= 1e-2 * lam[:, 2]] <= 1e-12).all()
    assert np.array_equal(got["counts"].cpu().numpy(), want["counts"])
    # the scoring kernel counts what the one-block-per-draw kernel counts on the same transforms
    again = ops.ransac_count_inliers(upload(a), upload(b), got["transforms"], THRESHOLD)
    assert np.array_equal(got["counts"].cpu().numpy(), again.cpu().numpy())


@pytest.mark.parametrize("n,w", [(2000, 0.27), (20000, 0.03)])
def test_winner_matches_oracle(n, w):
    from shot_fpfh_b200 import ops
    from shot_fpfh_b200.core import solver_point_to_point
    from shot_fpfh_b200.device import upload
    from shot_fpfh_b200.matching import ransac_on_matches_adaptive

    scan, ref, si, ri, rot, trans, a, b = case(n, w)
    want = oracle.ransac_adaptive(a, b, THRESHOLD)
    got = ops.ransac_adaptive(upload(a), upload(b), THRESHOLD, 0.9, 0, 1 << 24, 0.999)
    for key in ("best_draw", "best_count", "draws_used", "valid"):
        assert got[key] == want[key], key
    assert np.abs(got["transform"] - want["transform"]).max() <= 1e-12
    mask = got["mask"].cpu().numpy().astype(bool)
    assert np.array_equal(mask, want["mask"])
    ratio, transform = ransac_on_matches_adaptive(si, ri, scan, ref, distance_threshold=THRESHOLD)
    assert ratio == want["best_count"] / n
    refit = solver_point_to_point(a[mask], b[mask])
    refit.normalize_rotation()
    assert np.array_equal(transform.rotation, refit.rotation) and np.array_equal(transform.translation, refit.translation)


def test_recovers_low_inlier_ratio_then_icp():
    from shot_fpfh_b200.core import RigidTransform
    from shot_fpfh_b200.icp import icp_point_to_plane
    from shot_fpfh_b200.matching import ransac_on_matches_adaptive

    n = 20000
    scan, ref, si, ri, rot, trans, a, b = case(n, 0.03, seed=11)
    ratio, coarse = ransac_on_matches_adaptive(si, ri, scan, ref, distance_threshold=THRESHOLD)
    assert 0.025 <= ratio <= 0.035
    # 600 inliers with noise of 0.002 per coordinate on a unit-size cloud: the refit is good to about 1e-4
    assert np.abs(coarse.rotation - rot).max() < NOISE
    assert np.abs(coarse.translation - trans).max() < NOISE
    # ICP on the noise-free pair from there
    directions = scan / np.linalg.norm(scan, axis=1, keepdims=True)
    clean_ref = scan @ rot.T + trans
    ref_normals = synthetic.bumpy_sphere_true_normals(directions) @ rot.T
    s = synthetic.mean_spacing(n)
    fine, _, _ = icp_point_to_plane(scan, clean_ref, ref_normals, RigidTransform(coarse.rotation, coarse.translation),
                                    d_max=2 * s, voxel_size=3.75 * s, max_iter=20, rms_threshold=1e-9)
    assert np.abs(fine.rotation - rot).max() <= 1e-9
    assert np.abs(fine.translation - trans).max() <= 1e-9


def test_repeatable_and_max_draws():
    from shot_fpfh_b200 import ops
    from shot_fpfh_b200.device import upload

    *_, a, b = case(20000, 0.005, seed=7)  # 100 inliers: the confidence rule wants about 53 batches
    da, db = upload(a), upload(b)
    first = ops.ransac_adaptive(da, db, THRESHOLD, 0.9, 3, oracle.BATCH + 5, 0.999)
    second = ops.ransac_adaptive(da, db, THRESHOLD, 0.9, 3, oracle.BATCH + 5, 0.999)
    assert first["transform"].tobytes() == second["transform"].tobytes()
    assert np.array_equal(first["mask"].cpu().numpy(), second["mask"].cpu().numpy())
    assert first["draws_used"] == oracle.BATCH + 5
    want = oracle.ransac_adaptive(a, b, THRESHOLD, max_draws=oracle.BATCH + 5, seed=3)
    for key in ("best_draw", "best_count", "draws_used", "valid"):
        assert first[key] == want[key], key
    few = ops.ransac_adaptive(da, db, THRESHOLD, 0.9, 3, 1000, 0.999)
    assert few["draws_used"] == 1000
    want = oracle.ransac_adaptive(a, b, THRESHOLD, max_draws=1000, seed=3)
    assert (few["best_draw"], few["best_count"], few["valid"]) == (want["best_draw"], want["best_count"], want["valid"])


def test_errors():
    from shot_fpfh_b200.matching import ransac_on_matches_adaptive

    scan, ref, si, ri, *_ = case(2000, 0.27)
    for kwargs in ({"distance_threshold": 0.0}, {"confidence": 1.0}, {"confidence": 0.0}, {"edge_similarity": 0.0},
                   {"edge_similarity": 1.5}, {"max_draws": 0}, {"max_draws": 1 << 32}):
        with pytest.raises(ValueError):
            ransac_on_matches_adaptive(si, ri, scan, ref, **kwargs)
    with pytest.raises(ValueError):
        ransac_on_matches_adaptive(si[:2], ri[:2], scan, ref)
    huge = np.broadcast_to(np.zeros(1, dtype=np.int64), (1 << 32,))
    with pytest.raises(ValueError):
        ransac_on_matches_adaptive(huge, huge, scan, ref)
    bad = scan.copy()
    bad[si[0], 1] = np.nan
    with pytest.raises(ValueError):
        ransac_on_matches_adaptive(si, ri, bad, ref)
    line = np.zeros((50, 3))
    line[:, 0] = np.linspace(0.0, 1.0, 50)
    with pytest.raises(RuntimeError):  # every triple collinear: every fit degenerate
        ransac_on_matches_adaptive(np.arange(50), np.arange(50), line, line + 0.5, distance_threshold=0.01)


def test_c5_match_count():
    """400 000 matches (the C5 registration's count): counts against the one-block-per-draw kernel, and recovery."""
    from shot_fpfh_b200 import ops
    from shot_fpfh_b200.device import upload
    from shot_fpfh_b200.matching import ransac_on_matches_adaptive

    scan, ref, si, ri, rot, trans, a, b = case(400_000, 0.27, seed=13)
    got = device_batch(a, b)
    assert got["valid_draws"].shape[0] > 0
    again = ops.ransac_count_inliers(upload(a), upload(b), got["transforms"], THRESHOLD)
    assert np.array_equal(got["counts"].cpu().numpy(), again.cpu().numpy())
    ratio, coarse = ransac_on_matches_adaptive(si, ri, scan, ref, distance_threshold=THRESHOLD)
    assert 0.26 <= ratio <= 0.28
    assert np.abs(coarse.rotation - rot).max() < 1e-4
