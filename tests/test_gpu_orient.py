"""
GPU: consistent normal orientation (csrc/orient.cu, descriptors.orient_normals) against the oracle
(oracle/orientation_oracle.py) given the device's own k-NN lists: the signs must be IDENTICAL, bit for bit, and the
number of trees equal. Clouds: the bumpy sphere with eigh-sign normals, random sign flips of true normals, two separate
spheres, a plane, a duplicate-laden cloud and a 1M-point sphere (the oracle runs on the full 1M-point graph). Also
agreement with the true outward normals, viewpoints, degenerate inputs and run-to-run reproducibility.
"""

import numpy as np
import pytest

from oracle import orientation_oracle as oo
from shot_fpfh_b200 import synthetic

pytestmark = pytest.mark.gpu

K = 10


def device_orient(points, normals, k=K, towards=None):
    """(device output, number of trees, the device's (n, k + 1) lists) through the ops layer."""
    from shot_fpfh_b200 import ops
    from shot_fpfh_b200.descriptors.pca_based_descriptors import knn_device
    from shot_fpfh_b200.device import upload

    pts, nrm = upload(points), upload(normals)
    nbr = knn_device(pts, pts, k + 1)
    out, trees = ops.orient_normals(pts, nrm, nbr, towards)
    return out.cpu().numpy(), trees, nbr.cpu().numpy()


def check_against_oracle(points, normals, k=K, towards=None, label=""):
    from shot_fpfh_b200.descriptors import orient_normals

    out, trees, nbr = device_orient(points, normals, k, towards)
    want, d = oo.orient(points, normals, nbr, towards, details=True)
    assert out.tobytes() == want.tobytes(), f"{label}: {int((out != want).any(axis=1).sum())} rows differ"
    assert trees == d["n_trees"]
    assert orient_normals(points, normals, k, towards).tobytes() == want.tobytes()
    print(f"{label}: {points.shape[0]} points, {d['n_edges']} edges, {trees} tree(s), identical to the oracle")
    return out, d


def outward_share(out, true):
    agree = np.einsum("ij,ij->i", out, true) > 0
    return float(max(agree.mean(), 1.0 - agree.mean()))


def test_bumpy_sphere_20k_eigh_normals():
    from shot_fpfh_b200.descriptors import compute_normals

    n = 20_000
    pts, dirs = synthetic.bumpy_sphere(n, seed=0)
    true = synthetic.bumpy_sphere_true_normals(dirs)
    nrm = compute_normals(pts, pts, k=K)
    before = float((np.einsum("ij,ij->i", nrm, true) > 0).mean())
    out, d = check_against_oracle(pts, nrm, label="sphere 20k eigh")
    print(f"eigh signs outward {before:.4f} -> oriented {outward_share(out, true):.4f} (up to one global sign)")
    assert 0.4 < before < 0.6 and d["n_trees"] == 1 and outward_share(out, true) == 1.0


def test_random_sign_flips_of_true_normals():
    n = 30_000
    pts, dirs = synthetic.bumpy_sphere(n, seed=6)
    true = synthetic.bumpy_sphere_true_normals(dirs)
    flipped = true * np.random.default_rng(6).choice([-1.0, 1.0], size=(n, 1))
    out, _ = check_against_oracle(pts, flipped, label="sphere 30k flipped")
    assert outward_share(out, true) == 1.0


def test_two_separate_spheres_are_two_trees():
    a, da = synthetic.bumpy_sphere(8000, seed=7)
    b, db = synthetic.bumpy_sphere(8000, seed=8)
    pts = np.concatenate([a, b + [6.0, 0.0, 0.0]])
    true = synthetic.bumpy_sphere_true_normals(np.concatenate([da, db]))
    flipped = true * np.random.default_rng(7).choice([-1.0, 1.0], size=(16000, 1))
    out, d = check_against_oracle(pts, flipped, label="two spheres")
    assert d["n_trees"] == 2
    assert outward_share(out[:8000], true[:8000]) == 1.0 and outward_share(out[8000:], true[8000:]) == 1.0
    # each tree's lowest member keeps its input sign
    assert np.array_equal(out[0], flipped[0]) and np.array_equal(out[8000], flipped[8000])


def test_plane():
    rng = np.random.default_rng(9)
    xy = rng.uniform(-1.0, 1.0, size=(20_000, 2))
    pts = np.concatenate([xy, 0.002 * rng.normal(size=(20_000, 1))], axis=1)
    nrm = np.tile([0.0, 0.0, 1.0], (20_000, 1)) + 0.05 * rng.normal(size=(20_000, 3))
    nrm *= rng.choice([-1.0, 1.0], size=(20_000, 1))
    out, _ = check_against_oracle(pts, nrm, label="plane")
    assert (out[:, 2] > 0).all() or (out[:, 2] < 0).all()
    up, _ = check_against_oracle(pts, nrm, towards=(0.2, 0.1, 3.0), label="plane, viewpoint above")
    assert (up[:, 2] > 0).all()


def test_duplicate_laden_cloud():
    base, dirs = synthetic.bumpy_sphere(10_000, seed=10)
    true = synthetic.bumpy_sphere_true_normals(dirs)
    pts = np.concatenate([base, base[:3000], base[:500]])
    rng = np.random.default_rng(10)
    t = np.concatenate([true, true[:3000], true[:500]])
    nrm = t * rng.choice([-1.0, 1.0], size=(13_500, 1))
    nrm[::97] = 0.0  # zero normals: weight 1, no flip
    out, _ = check_against_oracle(pts, nrm, label="duplicates")
    nonzero = np.abs(nrm).sum(axis=1) > 0
    assert outward_share(out[nonzero], t[nonzero]) > 0.99


def test_towards_inside_and_outside_the_sphere():
    n = 20_000
    pts, dirs = synthetic.bumpy_sphere(n, seed=11)
    true = synthetic.bumpy_sphere_true_normals(dirs)
    flipped = true * np.random.default_rng(11).choice([-1.0, 1.0], size=(n, 1))
    inside, _ = check_against_oracle(pts, flipped, towards=pts.mean(axis=0), label="towards the centre")
    assert (np.einsum("ij,ij->i", inside, true) < 0).all()  # every normal points inward
    check_against_oracle(pts, flipped, towards=(4.0, 1.0, -2.0), label="towards an outside viewpoint")


def test_one_million_points_against_the_full_oracle():
    n = 1_000_000
    pts, dirs = synthetic.bumpy_sphere(n, seed=12)
    true = synthetic.bumpy_sphere_true_normals(dirs)
    flipped = true * np.random.default_rng(12).choice([-1.0, 1.0], size=(n, 1))
    out, d = check_against_oracle(pts, flipped, label="sphere 1M")
    assert d["n_trees"] == 1 and outward_share(out, true) == 1.0


def test_degenerate_inputs():
    from shot_fpfh_b200 import ops
    from shot_fpfh_b200._lib import SfError
    from shot_fpfh_b200.descriptors import orient_normals
    from shot_fpfh_b200.device import upload

    out = orient_normals(np.empty((0, 3)), np.empty((0, 3)))
    assert out.shape == (0, 3) and out.dtype == np.float64
    pts, _ = synthetic.bumpy_sphere(50, seed=13)
    nrm = np.ones((50, 3))
    with pytest.raises(ValueError, match="n_neighbors = 51, n_samples_fit = 50"):
        orient_normals(pts, nrm, k=50)
    with pytest.raises(ValueError, match="Expected n_neighbors > 0"):
        orient_normals(pts, nrm, k=0)
    bad = nrm.copy()
    bad[3, 0] = np.nan
    with pytest.raises(ValueError, match="finite"):
        orient_normals(pts, bad)
    bad_pts = pts.copy()
    bad_pts[7, 2] = np.inf
    with pytest.raises(ValueError, match="finite"):
        orient_normals(bad_pts, nrm)
    with pytest.raises(ValueError, match="finite"):
        orient_normals(pts, nrm, towards=(0.0, np.nan, 0.0))
    # lists holding only the point itself: every point is a lone tree and keeps its sign
    import torch

    signed = nrm * np.random.default_rng(13).choice([-1.0, 1.0], size=(50, 1))
    alone = torch.arange(50, dtype=torch.int32, device="cuda").reshape(50, 1)
    out, trees = ops.orient_normals(upload(pts), upload(signed), alone)
    assert trees == 50 and out.cpu().numpy().tobytes() == signed.tobytes()
    # an index outside the cloud is refused by the C ABI
    nbr = torch.full((50, 2), 50, dtype=torch.int32, device="cuda")
    with pytest.raises(SfError, match="outside"):
        ops.orient_normals(upload(pts), upload(nrm), nbr)


def test_two_runs_are_bit_identical():
    from shot_fpfh_b200.descriptors import compute_normals, orient_normals

    pts, _ = synthetic.bumpy_sphere(200_000, seed=14)
    nrm = compute_normals(pts, pts, k=30)
    a = orient_normals(pts, nrm)
    b = orient_normals(pts, nrm)
    assert a.tobytes() == b.tobytes()
    c = orient_normals(pts, nrm, towards=(0.0, 0.0, 0.0))
    assert c.tobytes() == orient_normals(pts, nrm, towards=(0.0, 0.0, 0.0)).tobytes()
