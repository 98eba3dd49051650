"""
GPU: ISS salient keypoints (csrc/iss.cu, keypoint_selection.select_keypoints_iss) against the oracle
(oracle/iss_oracle.py). Neighbourhood sizes must be identical, eigenvalues within 1e-12 r_s^2 (only the order of the
sums differs), and the keypoint sets may differ only at points the oracle's `excused` set names (a ratio test, the sign
of e3 or a saliency comparison inside that rounding). Also the registration chain through this package's API and
through the unmodified reference pipeline, and a 1M-point cloud checked by sampling.
"""

import importlib

import numpy as np
import pytest
from conftest import ROOT, edge_case_inputs, load_golden, registration_case
from test_iss_host import REPEATABILITY_BAR, repeatability, rigid_pair_30k

from oracle import iss_oracle
from shot_fpfh_b200 import synthetic

pytestmark = pytest.mark.gpu

G21 = G32 = 0.975


def device_details(points, rs, rn, m=5, g21=G21, g32=G32) -> dict:
    """Everything the kernels compute, in ORIGINAL point order."""
    import torch

    from shot_fpfh_b200 import ops
    from shot_fpfh_b200.device import Grid, upload

    pts = upload(points)
    grid = Grid().build(pts, None, max(rs, rn))
    perm = ops.grid_permutation(grid)[0].long()
    sal, counts, eig = ops.iss_saliency(grid, rs, m, g21, g32, want_counts=True, want_eigvals=True)
    _, nms_counts, _ = ops.iss_saliency(grid, rn, m, g21, g32, want_counts=True)
    kp = ops.iss_select(grid, sal, rn, m)

    def original(t):
        out = torch.empty_like(t)
        out[perm] = t
        return out.cpu().numpy()

    d = {"saliency": original(sal), "counts": original(counts), "eigenvalues": original(eig),
         "nms_counts": original(nms_counts), "keypoints": kp.cpu().numpy()}
    grid.close()
    return d


def check_against_oracle(points, rs, rn, m=5, g21=G21, g32=G32, label=""):
    okp, o = iss_oracle.iss(points, rs, rn, g21, g32, m, details=True)
    d = device_details(points, rs, rn, m, g21, g32)
    tol = 1e-12 * rs**2
    assert np.array_equal(d["counts"], o["counts"])
    assert np.array_equal(d["nms_counts"], o["nms_counts"])
    assert np.abs(d["eigenvalues"] - o["eigenvalues"]).max() <= tol
    margin = iss_oracle.margin_points(o["eigenvalues"], g21, g32, rs)
    assert np.abs(d["saliency"] - o["saliency"])[~margin].max(initial=0.0) <= tol
    from shot_fpfh_b200.keypoint_selection import select_keypoints_iss

    kp = select_keypoints_iss(points, rs, rn, g21, g32, m)
    assert kp.dtype == np.int64 and np.array_equal(kp, d["keypoints"])
    excused = iss_oracle.excused(o, g21, g32)
    disagree = np.setxor1d(kp, okp)
    print(f"{label}: {okp.shape[0]} oracle keypoints, |E| = {int(excused.sum())}, {disagree.shape[0]} disagreements")
    assert excused[disagree].all()
    return kp, okp


@pytest.mark.parametrize("radii", [(5.0, 3.75), (3.0, 5.0)], ids=["rn_lt_rs", "rn_gt_rs"])
def test_bumpy_sphere_30k_against_oracle(radii):
    n = 30_000
    pts, _ = synthetic.bumpy_sphere(n, seed=5)
    s = synthetic.mean_spacing(n)
    kp, okp = check_against_oracle(pts, radii[0] * s, radii[1] * s, label=f"sphere {radii}")
    assert okp.shape[0] > 100


def test_box_corner_against_oracle():
    scan = registration_case()[0]
    rs, rn = iss_oracle.default_radii(scan)
    check_against_oracle(scan, rs, rn, label="box corner")


def test_duplicate_laden_edge_cloud_against_oracle():
    pts, _, _, radius = edge_case_inputs(load_golden("edge_cases"))
    check_against_oracle(pts, radius, 0.75 * radius, label="edge cases")
    check_against_oracle(pts, radius, 0.75 * radius, m=1, label="edge cases, m = 1")


def test_defaults_match_the_oracle():
    import torch

    from shot_fpfh_b200.device import upload
    from shot_fpfh_b200.keypoint_selection import _resolution, select_keypoints_iss

    for pts in (synthetic.bumpy_sphere(20_000, seed=8)[0], registration_case()[0]):
        res = _resolution(upload(pts))
        assert res == pytest.approx(iss_oracle.resolution(pts), rel=1e-12)
        torch.cuda.synchronize()
        okp, o = iss_oracle.iss(pts, details=True)
        kp = select_keypoints_iss(pts)
        excused = iss_oracle.excused(o, G21, G32)
        disagree = np.setxor1d(kp, okp)
        print(f"defaults: {okp.shape[0]} oracle keypoints, |E| = {int(excused.sum())}, {disagree.shape[0]} disagreements")
        assert okp.shape[0] > 10 and excused[disagree].all()


def test_tiny_and_degenerate_clouds():
    from shot_fpfh_b200 import ops
    from shot_fpfh_b200.device import Grid
    from shot_fpfh_b200.keypoint_selection import select_keypoints_iss

    rng = np.random.default_rng(4)
    same = np.tile([[0.25, 1.5, -3.0]], (50, 1))
    for pts in (np.empty((0, 3)), rng.normal(size=(1, 3)), rng.normal(size=(4, 3)), same):
        for args in ((), (0.5, 0.5), (0.5, 0.5, G21, G32, 1)):
            kp = select_keypoints_iss(pts, *args)
            okp = iss_oracle.iss(pts, *args)
            assert kp.dtype == np.int64 and kp.shape == (0,) and okp.shape == (0,), (pts.shape, args)
        if pts.shape[0]:
            d = device_details(pts, 0.5, 0.5, m=1)
            assert np.array_equal(d["counts"], iss_oracle.covariance_eigenvalues(pts, 0.5)[0])
            assert not d["saliency"].any() and d["keypoints"].shape == (0,)
    empty = Grid()  # a handle over no points
    sal, _, _ = ops.iss_saliency(empty, 1.0, 5, G21, G32)
    assert sal.shape == (0,) and ops.iss_select(empty, sal, 1.0, 5).shape == (0,)


def test_invalid_arguments_are_refused():
    from shot_fpfh_b200 import ops
    from shot_fpfh_b200._lib import SfError
    from shot_fpfh_b200.device import Grid, upload
    from shot_fpfh_b200.keypoint_selection import select_keypoints_iss

    pts = synthetic.bumpy_sphere(2000, seed=1)[0]
    grid = Grid().build(upload(pts), None, 0.2)
    with pytest.raises(SfError, match="salient radius"):
        ops.iss_saliency(grid, 0.3, 5, G21, G32)
    with pytest.raises(SfError, match="min_neighbors"):
        ops.iss_saliency(grid, 0.2, 0, G21, G32)
    with pytest.raises(SfError, match="gamma"):
        ops.iss_saliency(grid, 0.2, 5, float("nan"), G32)
    sal, _, _ = ops.iss_saliency(grid, 0.2, 5, G21, G32)
    with pytest.raises(SfError, match="non-max radius"):
        ops.iss_select(grid, sal, -1.0, 5)
    grid.close()
    with pytest.raises(ValueError):
        select_keypoints_iss(pts, -1.0, 0.1)
    with pytest.raises(ValueError):
        select_keypoints_iss(pts, 0.1, 0.1, min_neighbors=0)


def test_rigid_pair_repeatability():
    from shot_fpfh_b200.keypoint_selection import select_keypoints_iss

    scan, _, ref, _, perm, _, _, s = rigid_pair_30k()
    scan_kp = select_keypoints_iss(scan, 5 * s, 3.75 * s)
    ref_kp = select_keypoints_iss(ref, 5 * s, 3.75 * s)
    rate = repeatability(scan_kp, ref_kp, perm)
    print(f"device repeatability {rate:.4f} ({scan_kp.shape[0]} / {ref_kp.shape[0]} keypoints)")
    assert rate >= REPEATABILITY_BAR


def test_end_to_end_registration_through_the_package():
    import shot_fpfh_b200.matching.ransac as ransac_module
    from shot_fpfh_b200.descriptors import ShotMultiprocessor
    from shot_fpfh_b200.keypoint_selection import select_keypoints_iss
    from shot_fpfh_b200.matching import match_descriptors, ransac_on_matches

    scan, normals, ref, ref_normals, _, rot, _, s = rigid_pair_30k()
    scan_kp = select_keypoints_iss(scan, 5 * s, 3.75 * s)
    ref_kp = select_keypoints_iss(ref, 5 * s, 3.75 * s)
    with ShotMultiprocessor(min_neighborhood_size=10, verbose=False) as shot:
        d_scan = shot.compute_descriptor_single_scale(scan, normals, scan[scan_kp], 5 * s)
        d_ref = shot.compute_descriptor_single_scale(ref, ref_normals, ref[ref_kp], 5 * s)
    a, b = match_descriptors(d_scan, d_ref, None, filter_nonreciprocal=True, verbose=False)
    ransac_module.rng = np.random.default_rng(seed=72)
    ratio, coarse = ransac_on_matches(a, b, scan[scan_kp], ref[ref_kp], n_draws=1000, distance_threshold=s)
    print(f"{a.shape[0]} matches, inlier ratio {ratio:.3f}, rotation error {np.abs(coarse.rotation - rot).max():.2e}")
    assert np.abs(coarse.rotation - rot).max() < 0.1


def _reference_available():
    import sys

    sys.path.insert(0, ROOT)
    from baseline import reference_loader

    return reference_loader.available()


@pytest.mark.skipif(not _reference_available(), reason="baseline/_ref was not shipped")
def test_reference_pipeline_with_iss_keypoints():
    import shot_fpfh_b200.dropin as dropin
    import shot_fpfh_b200.matching.ransac as ransac_module
    from baseline import reference_loader
    from shot_fpfh_b200.keypoint_selection import select_keypoints_iss

    reference_loader.load()
    dropin.install()
    try:
        pipeline = importlib.import_module("shot_fpfh.pipeline")
        n = 60_000
        scan, directions = synthetic.bumpy_sphere(n, seed=0)
        normals = synthetic.bumpy_sphere_true_normals(directions)
        ref, ref_normals, _, rot, _ = synthetic.rigid_pair(scan, normals)
        s = synthetic.mean_spacing(n)
        pipe = pipeline.RegistrationPipeline(scan=scan, scan_normals=normals, ref=ref, ref_normals=ref_normals)
        pipe.scan_keypoints = select_keypoints_iss(pipe.scan, 5 * s, 3.75 * s)
        pipe.ref_keypoints = select_keypoints_iss(pipe.ref, 5 * s, 3.75 * s)
        assert pipe.scan_keypoints.shape[0] > 200
        pipe.compute_descriptors(radius=5.0 * s, descriptor_choice="shot_single_scale", subsample_support=False,
                                 min_neighborhood_size=10, disable_progress_bars=True, verbose=False)
        assert pipe.scan_descriptors.shape == (pipe.scan_keypoints.shape[0], 352)
        pipe.find_descriptors_matches("simple", reject_threshold=0.8, threshold_multiplier=4.0)
        ransac_module.rng = np.random.default_rng(seed=72)
        coarse, ratio = pipe.run_ransac(n_draws=1000, max_inliers_distance=s, disable_progress_bar=True)
        assert np.abs(coarse.rotation - rot).max() < 0.1
    finally:
        dropin.uninstall()


def test_one_million_points_by_sampling():
    from sklearn.neighbors import KDTree

    n = 1_000_000
    pts, _ = synthetic.bumpy_sphere(n, seed=12)
    s = synthetic.mean_spacing(n)
    rs, rn, m = 5 * s, 3.75 * s, 5
    d = device_details(pts, rs, rn, m)
    kp = d["keypoints"]
    assert kp.shape[0] > 1000 and kp.min() >= 0 and kp.max() < n and np.all(np.diff(kp) > 0)
    assert (d["saliency"][kp] > 0).all() and (d["nms_counts"][kp] >= m).all()
    rng = np.random.default_rng(0)
    tree = KDTree(pts)
    sample_kp = rng.choice(kp, min(2000, kp.shape[0]), replace=False)
    for i, nb in zip(sample_kp, tree.query_radius(pts[sample_kp], rn)):
        assert d["saliency"][i] >= d["saliency"][nb].max()
    sample = rng.choice(n, 2000, replace=False)
    counts, eig, _ = iss_oracle.covariance_eigenvalues(pts, rs, sample)
    tol = 1e-12 * rs**2
    assert np.array_equal(d["counts"][sample], counts)
    assert np.abs(d["eigenvalues"][sample] - eig).max() <= tol
    sal = iss_oracle.saliency_of(counts, eig, m, G21, G32)
    margin = iss_oracle.margin_points(eig, G21, G32, rs)
    assert np.abs(d["saliency"][sample] - sal)[~margin].max(initial=0.0) <= tol
    print(f"1M points: {kp.shape[0]} keypoints, {int(margin.sum())} margin points in the sample")
