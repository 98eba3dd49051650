"""
The reference's registration flow (scripts/register_point_clouds.py:80-127 -> pipeline.py: select_keypoints,
compute_descriptors, find_descriptors_matches, run_ransac, run_icp) through THIS package's reference-shaped API, host
NumPy arrays in and out at every stage, on a synthetic rigid pair (SURVEY.md 8d generator). BASELINE.json configs[4]
names a 10M-point pair; the size is an argument:

    python scripts/run_registration_flow.py [n_points] [fpfh] [voxel|iss] [pca|pca_raw] [adaptive]

The keypoint selector is `voxel` (select_keypoints_subsampling, 3.75 spacings: the default) or `iss`
(select_keypoints_iss, salient radius 5 spacings, non-max radius 3.75 spacings: far fewer keypoints, on salient points).
The normals are the synthetic surface's analytic ones (the default), or `pca`: compute_normals(k=30) of each cloud,
oriented by orient_normals (k = 10) towards the cloud's centroid and then negated, so that both clouds' normals point
away from it, as the analytic ones do. `pca_raw` keeps compute_normals' signs (LAPACK's, a coin flip per point): it
measures what sign noise does to matching.
The coarse alignment is the reference's `ransac_on_matches` (10 000 draws of 4 matches), or with `adaptive`
ransac_on_matches_adaptive (device-drawn 3-match hypotheses until 99.9 % confidence), same threshold.
Prints wall-clock per stage and the error of the recovered transform against the known one. (`/root/reference` is not
on the GPU box, so its `RegistrationPipeline` object cannot be run there; `dropin.install()` binds exactly these
callables into it.)
"""

import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from shot_fpfh_b200 import synthetic  # noqa: E402
from shot_fpfh_b200.core import RigidTransform  # noqa: E402
from shot_fpfh_b200.descriptors import (  # noqa: E402
    ShotMultiprocessor,
    compute_fpfh_descriptor,
    compute_normals,
    orient_normals,
)
from shot_fpfh_b200.icp import icp_point_to_plane  # noqa: E402
from shot_fpfh_b200.keypoint_selection import select_keypoints_iss, select_keypoints_subsampling  # noqa: E402
from shot_fpfh_b200.matching import match_descriptors, ransac_on_matches, ransac_on_matches_adaptive  # noqa: E402


def run(n: int, with_fpfh: bool = False, verbose: bool = True, keypoints: str = "voxel",
        normals_from: str = "analytic", adaptive: bool = False) -> dict:
    times = {}

    def stage(name, fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        times[name] = time.perf_counter() - t0
        if verbose:
            print(f"  {name:34s} {1e3 * times[name]:10.1f} ms")
        return out

    scan, directions = synthetic.bumpy_sphere(n, seed=0)
    normals = synthetic.bumpy_sphere_true_normals(directions)  # the surface's own normals: ICP needs them (see there)
    ref, ref_normals, perm, rot, trans = synthetic.rigid_pair(scan, normals)
    s = synthetic.mean_spacing(n)
    radius = 5.0 * s
    if verbose:
        print(f"pair of {n} points, radius {radius:.5f}, {normals_from} normals")
    if normals_from in ("pca", "pca_raw"):
        def pca(cloud):
            nrm = compute_normals(cloud, cloud, k=30)
            return nrm if normals_from == "pca_raw" else -orient_normals(cloud, nrm, k=10, towards=cloud.mean(axis=0))

        normals = stage(f"normals {normals_from} (scan)", lambda: pca(scan))
        ref_normals = stage(f"normals {normals_from} (ref)", lambda: pca(ref))
    elif normals_from != "analytic":
        raise ValueError(f"unknown normals {normals_from!r} (analytic, pca or pca_raw)")
    if keypoints == "iss":
        select = lambda cloud: select_keypoints_iss(cloud, 5.0 * s, 3.75 * s)  # noqa: E731
    elif keypoints == "voxel":
        select = lambda cloud: select_keypoints_subsampling(cloud, 3.75 * s)  # noqa: E731
    else:
        raise ValueError(f"unknown keypoint selector {keypoints!r} (voxel or iss)")
    scan_kp = stage(f"select_keypoints {keypoints} (scan)", lambda: select(scan))
    ref_kp = stage(f"select_keypoints {keypoints} (ref)", lambda: select(ref))
    with ShotMultiprocessor(min_neighborhood_size=10, verbose=False) as shot:
        scan_desc = stage("SHOT single scale (scan)", lambda: shot.compute_descriptor_single_scale(
            scan, normals, scan[scan_kp], radius))
        ref_desc = stage("SHOT single scale (ref)", lambda: shot.compute_descriptor_single_scale(
            ref, ref_normals, ref[ref_kp], radius))
    if with_fpfh:
        stage("FPFH 33-d on the keypoints (scan)", lambda: compute_fpfh_descriptor(
            scan_kp, scan, normals, radius, n_bins=11, decorrelated=True, verbose=False))
    # the two clouds' keypoints are different points of the surface (voxel selection of a rotated copy): reciprocity is
    # the filter that fits, as in pipeline.py:376-399 with `filter_nonreciprocal`
    matches = stage("match_descriptors (reciprocal)", lambda: match_descriptors(
        scan_desc, ref_desc, None, filter_nonreciprocal=True, verbose=False))
    del scan_desc, ref_desc
    import shot_fpfh_b200.matching.ransac as ransac_module

    ransac_module.rng = np.random.default_rng(seed=72)  # the reference's module-level generator (ransac.py:14)
    if adaptive:
        ratio, coarse = stage("ransac_on_matches_adaptive", lambda: ransac_on_matches_adaptive(
            matches[0], matches[1], scan[scan_kp], ref[ref_kp], distance_threshold=4 * s))
    else:
        ratio, coarse = stage("ransac_on_matches (10000 draws)", lambda: ransac_on_matches(
            matches[0], matches[1], scan[scan_kp], ref[ref_kp], n_draws=10_000, distance_threshold=4 * s))
    fine, rms, _ = stage("icp_point_to_plane (<= 20 iters)", lambda: icp_point_to_plane(
        scan, ref, ref_normals, RigidTransform(coarse.rotation, coarse.translation), d_max=2 * s, voxel_size=3.75 * s,
        max_iter=20, rms_threshold=1e-9))
    out = {
        "n_points": n, "keypoint_selector": keypoints, "normals": normals_from, "adaptive_ransac": adaptive, "keypoints": (int(scan_kp.shape[0]), int(ref_kp.shape[0])), "matches": int(matches[0].shape[0]),
        "ransac_inlier_ratio": float(ratio),
        "coarse_rotation_error": float(np.abs(coarse.rotation - rot).max()),
        "fine_rotation_error": float(np.abs(fine.rotation - rot).max()),
        "fine_translation_error": float(np.abs(fine.translation - trans).max()),
        "seconds": times, "total_seconds": float(sum(times.values())),
        "peak_device_GiB": torch.cuda.max_memory_allocated() / 2**30,
    }
    if verbose:
        print({k: v for k, v in out.items() if k != "seconds"})
    return out


if __name__ == "__main__":
    size = int(sys.argv[1]) if len(sys.argv) > 1 else 10_000_000
    words = sys.argv[2:]
    normals_from = "pca" if "pca" in words else ("pca_raw" if "pca_raw" in words else "analytic")
    run(size, with_fpfh="fpfh" in words, keypoints="iss" if "iss" in words else "voxel", normals_from=normals_from,
        adaptive="adaptive" in words)
