"""
CPU: the ISS oracle (oracle/iss_oracle.py, the specification of select_keypoints_iss) — held to its stored outputs,
checked on hand-built clouds with known answers, measured on the rigid pair for the GPU test's repeatability bar, and
rehearsed end to end (ISS -> SHOT -> matching -> RANSAC) with the CPU oracles so that the GPU end-to-end parameters are
known to register. Also the public function's signature, and its refusal to run without a device.
"""

import inspect

import numpy as np
import pytest
import torch
from conftest import load_golden

from oracle import iss_oracle
from oracle.make_iss_pins import ISS_CASES, case_cloud
from shot_fpfh_b200 import synthetic

# Fraction of the scan's ISS keypoints whose image in the rigidly moved, permuted copy is a keypoint there, measured with
# the oracle on the 30k bumpy sphere below (0.995: 202 of 203). The GPU test holds the device to REPEATABILITY_BAR.
REPEATABILITY_BAR = 0.98


def rigid_pair_30k():
    n = 30_000
    scan, directions = synthetic.bumpy_sphere(n, seed=5)
    normals = synthetic.bumpy_sphere_true_normals(directions)
    ref, ref_normals, perm, rot, trans = synthetic.rigid_pair(scan, normals)
    return scan, normals, ref, ref_normals, perm, rot, trans, synthetic.mean_spacing(n)


def repeatability(scan_kp, ref_kp, perm) -> float:
    """Share of scan keypoints i whose image (ref index k with perm[k] = i) is a ref keypoint."""
    image = np.empty(perm.shape[0], dtype=np.int64)
    image[perm] = np.arange(perm.shape[0])
    return float(np.isin(image[scan_kp], ref_kp).mean())


def test_oracle_reproduces_its_pins():
    g = load_golden("iss_pins")
    for name, kind, radii in ISS_CASES:
        pts, s = case_cloud(kind)
        rs, rn = (0.0, 0.0) if radii is None else (radii[0] * s, radii[1] * s)
        kp, d = iss_oracle.iss(pts, rs, rn, details=True)
        assert np.array_equal(kp, g[f"{name}_keypoints"]), name
        assert np.array_equal(d["saliency"], g[f"{name}_saliency"]), name
        assert np.array_equal(d["counts"], g[f"{name}_counts"]), name
        assert np.array_equal(d["nms_counts"], g[f"{name}_nms_counts"]), name
        assert np.array_equal([d["salient_radius"], d["non_max_radius"]], g[f"{name}_radii"]), name
        assert kp.dtype == np.int64 and kp.shape[0] > 10


def test_duplicates_and_coincident_clusters_have_zero_saliency():
    rng = np.random.default_rng(3)
    cluster = np.tile([[0.5, -0.25, 2.0]], (12, 1))  # all coincident: C = 0, e2 / e1 = 0 / 0
    pair = np.repeat(rng.normal(size=(4, 3)) * 10.0, 2, axis=0)  # far-apart exact duplicates: two positions each
    pts = np.concatenate([cluster, pair])
    counts, eig, _ = iss_oracle.covariance_eigenvalues(pts, 0.1)
    s = iss_oracle.saliency_of(counts, eig, 1, 0.975, 0.975)
    assert np.array_equal(counts, [12] * 12 + [2] * 8)
    assert not s.any()
    assert iss_oracle.iss(pts, 0.1, 0.1, min_neighbors=1).shape == (0,)


def test_fewer_points_than_min_neighbors_gives_empty_int64():
    pts = np.random.default_rng(0).normal(size=(4, 3))
    for rs, rn in ((10.0, 10.0), (0.0, 0.0)):
        kp = iss_oracle.iss(pts, rs, rn, min_neighbors=5)
        assert kp.dtype == np.int64 and kp.shape == (0,)
    assert iss_oracle.iss(np.empty((0, 3))).dtype == np.int64


def mirror_pair_cloud():
    """A cloud symmetric through the origin, p -> -p, on a dyadic lattice (multiples of 1/64): every offset, product
    and sum is exact, c -> -c leaves sum(c c^T) and mu mu^T unchanged, so point i and its mirror i + 40 have
    bit-identical covariances and saliencies."""
    rng = np.random.default_rng(11)
    half = (rng.integers(-12, 13, size=(40, 3)) + [10, 0, 0]) / 64.0
    return np.concatenate([half, -half])


def test_mirror_symmetric_ties_keep_both():
    pts = mirror_pair_cloud()
    kp, d = iss_oracle.iss(pts, 0.3, 1.25, gamma_21=1.0, gamma_32=1.0, details=True)
    s = d["saliency"]
    assert np.array_equal(s[:40], s[40:]) and s.max() > 0.0
    # the non-max radius covers the whole cloud: only the largest saliency survives — held by a point AND its mirror
    assert np.abs(pts).max() * 2 * np.sqrt(3) <= 1.25
    assert kp.shape == (2,) and kp[1] == kp[0] + 40 and s[kp[0]] == s.max()


def test_isolated_points_are_never_keypoints():
    sphere, _ = synthetic.bumpy_sphere(2000, seed=9)
    far = np.array([[5.0, 5.0, 5.0], [-5.0, 4.0, 3.0], [7.0, -6.0, 0.0]])
    pts = np.concatenate([sphere, far])
    s = synthetic.mean_spacing(2000)
    kp, d = iss_oracle.iss(pts, 5 * s, 3.75 * s, min_neighbors=1, details=True)
    assert np.array_equal(d["counts"][-3:], [1, 1, 1]) and not d["saliency"][-3:].any()
    assert not np.isin(np.arange(2000, 2003), kp).any() and kp.shape[0] > 0


def test_default_radii_on_a_lattice():
    h = 0.02
    g = np.arange(12) * h
    lattice = np.stack(np.meshgrid(g, g, g, indexing="ij"), axis=-1).reshape(-1, 3)
    assert iss_oracle.resolution(lattice) == pytest.approx(h, rel=1e-12)
    rs, rn = iss_oracle.default_radii(lattice)
    assert rs == pytest.approx(6 * h, rel=1e-12) and rn == pytest.approx(4 * h, rel=1e-12)
    _, d = iss_oracle.iss(lattice, details=True)
    assert d["salient_radius"] == rs and d["non_max_radius"] == rn
    # a duplicate counts 0 in the mean
    dup = np.concatenate([lattice, lattice[:1]])
    assert iss_oracle.resolution(dup) == pytest.approx(h * (lattice.shape[0] - 1) / dup.shape[0], rel=1e-12)


def test_rigid_pair_repeatability_of_the_oracle():
    scan, _, ref, _, perm, _, _, s = rigid_pair_30k()
    scan_kp = iss_oracle.iss(scan, 5 * s, 3.75 * s)
    ref_kp = iss_oracle.iss(ref, 5 * s, 3.75 * s)
    rate = repeatability(scan_kp, ref_kp, perm)
    print(f"oracle repeatability {rate:.4f} ({scan_kp.shape[0]} / {ref_kp.shape[0]} keypoints)")
    assert scan_kp.shape[0] > 100 and rate >= REPEATABILITY_BAR


def test_end_to_end_rehearsal_with_the_cpu_oracles():
    """The chain the GPU end-to-end test runs (same cloud, radii, SHOT and RANSAC parameters), on the oracles."""
    from oracle import matching_oracle, registration_oracle, shot_oracle

    scan, normals, ref, ref_normals, _, rot, _, s = rigid_pair_30k()
    scan_kp = iss_oracle.iss(scan, 5 * s, 3.75 * s)
    ref_kp = iss_oracle.iss(ref, 5 * s, 3.75 * s)
    d_scan = shot_oracle.shot_single_scale(scan, normals, scan[scan_kp], 5 * s, True, 10)
    d_ref = shot_oracle.shot_single_scale(ref, ref_normals, ref[ref_kp], 5 * s, True, 10)
    a, b = matching_oracle.match_descriptors(d_scan, d_ref, filter_nonreciprocal=True)
    ratio, (r, _) = registration_oracle.ransac_on_matches(
        a, b, scan[scan_kp], ref[ref_kp], np.random.default_rng(72), n_draws=1000, distance_threshold=s)
    print(f"{a.shape[0]} matches, inlier ratio {ratio:.3f}, rotation error {np.abs(r - rot).max():.2e}")
    assert np.abs(r - rot).max() < 0.1


def test_signature_pinned():
    from shot_fpfh_b200.keypoint_selection import select_keypoints_iss

    params = [(p.name, p.default) for p in inspect.signature(select_keypoints_iss).parameters.values()]
    assert params == [
        ("points", inspect.Parameter.empty), ("salient_radius", 0.0), ("non_max_radius", 0.0), ("gamma_21", 0.975),
        ("gamma_32", 0.975), ("min_neighbors", 5),
    ]


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the behaviour without a CUDA device")
def test_no_cpu_fallback():
    from shot_fpfh_b200.keypoint_selection import select_keypoints_iss

    with pytest.raises(RuntimeError, match="no CPU fallback"):
        select_keypoints_iss(np.zeros((10, 3)))
