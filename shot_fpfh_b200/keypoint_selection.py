"""
Keypoint selection with the reference's signatures (shot_fpfh/keypoint_selection.py), for the two selectors that
are voxel-grid reductions of the cloud (SURVEY.md §8f row 1): they sit immediately upstream of the descriptors and
are Python loops over voxels in the reference (4.4 s at 1M points).

  select_keypoints_subsampling(points, voxel_size)                       keypoint_selection.py:34-46
  select_keypoints_with_density_threshold(points, voxel_size, value, radius=None)        :65-122

Both run on the device (csrc/subsample.cu; the density variant with a radius different from the voxel size also
uses the uniform grid's fixed-radius count, csrc/grid.cu). The iterative and the random selectors of the reference
are not data-parallel (a sequential greedy cover; NumPy's global RNG) and are left to the reference.

A voxel selector keeps one point per voxel whatever the geometry. This module also has the salient-keypoint detector
that SHOT and FPFH are usually paired with, which the reference does not have:

  select_keypoints_iss(points, salient_radius=0.0, non_max_radius=0.0, gamma_21=0.975, gamma_32=0.975,
                       min_neighbors=5)                                     ISS (Zhong 2009), csrc/iss.cu

It has no name in the reference for `dropin.install()` to rebind. With the reference's `RegistrationPipeline`, assign
its result before computing descriptors; the pipeline keeps keypoints that are already set:

    pipe.scan_keypoints = select_keypoints_iss(pipe.scan)
    pipe.ref_keypoints = select_keypoints_iss(pipe.ref)
    pipe.compute_descriptors(...)
"""

from __future__ import annotations

import numpy as np
import numpy.typing as npt


def select_keypoints_subsampling(points: npt.NDArray[np.float64], voxel_size: float) -> npt.NDArray[np.int64]:
    """Indices of the points closest to the barycentre of each occupied voxel (= `grid_subsampling`)."""
    from .subsampling import grid_subsampling_gpu

    return grid_subsampling_gpu(points, voxel_size)


def select_keypoints_with_density_threshold(
    points: npt.NDArray[np.float64],
    voxel_size: float,
    density_threshold_value: int,
    density_threshold_radius: float | None = None,
) -> npt.NDArray[np.int64]:
    """
    The voxel representatives of `select_keypoints_subsampling`, kept only where the density exceeds the threshold:
    more than `density_threshold_value` points in the voxel when the radius is the voxel size (or None), else more
    than that many points of the cloud within `density_threshold_radius` of the representative (itself included,
    as `KDTree.query_radius` counts it) — keypoint_selection.py:104-118. Lexicographic voxel order, like the
    reference's `np.unique(axis=0)`.
    """
    import torch

    from . import ops
    from .device import Grid, upload

    pts = upload(points)
    picked, members = ops.voxel_subsample(pts, float(voxel_size), want_members=True)
    if picked.shape[0] == 0:
        return np.array([])  # what `np.array([])` of the reference's empty list is
    if density_threshold_radius is None or density_threshold_radius == voxel_size:
        keep = members > int(density_threshold_value)
    else:
        grid = Grid().build(pts, None, float(density_threshold_radius))
        offsets, _, _, _ = ops.radius_csr(grid, pts[picked].contiguous(), float(density_threshold_radius), count_only=True)
        keep = (offsets[1:] - offsets[:-1]) > int(density_threshold_value)
        torch.cuda.synchronize()
        grid.close()
    out = picked[keep].cpu().numpy()
    return out if out.shape[0] else np.array([])


def _resolution(pts) -> float:
    """Mean distance from each point to its nearest OTHER point (a duplicate counts 0), on the device."""
    from .descriptors.pca_based_descriptors import knn_device

    nbr = knn_device(pts, pts, 2)  # nearest first; the second is another point or, for a duplicate, at distance 0
    return float((pts[nbr[:, 1].long()] - pts).norm(dim=1).mean())


def select_keypoints_iss(
    points: npt.NDArray[np.float64],
    salient_radius: float = 0.0,
    non_max_radius: float = 0.0,
    gamma_21: float = 0.975,
    gamma_32: float = 0.975,
    min_neighbors: int = 5,
) -> npt.NDArray[np.int64]:
    """
    ISS salient keypoints (Intrinsic Shape Signatures, Zhong 2009; Open3D's definition and defaults). For each point,
    e3 <= e2 <= e1 are the eigenvalues of the covariance of the points within `salient_radius`; its saliency is e3 when
    that neighbourhood holds at least `min_neighbors` points and e2 / e1 < gamma_21 and e3 / e2 < gamma_32, else 0.
    A point is a keypoint when its saliency is positive, at least `min_neighbors` points lie within `non_max_radius`,
    and none of them has a larger saliency (equal saliencies keep both points).
    A radius of 0.0 derives both from the cloud's resolution `res` (mean distance to the nearest other point):
    salient_radius = 6 res, non_max_radius = 4 res.
    Returns the keypoints' indices into `points`, int64, ascending (empty when there are none).
    oracle/iss_oracle.py states the same computation in NumPy.
    """
    import torch

    from . import ops
    from .device import Grid, require_cuda, upload

    require_cuda()
    for name, value in (("salient_radius", salient_radius), ("non_max_radius", non_max_radius)):
        if not (np.isfinite(value) and value >= 0.0):
            raise ValueError(f"{name} must be finite and >= 0, got {value}")
    if not (np.isfinite(gamma_21) and np.isfinite(gamma_32)):
        raise ValueError("gamma_21 and gamma_32 must be finite")
    if int(min_neighbors) < 1:
        raise ValueError(f"min_neighbors must be >= 1, got {min_neighbors}")
    pts = upload(np.asarray(points, dtype=np.float64).reshape(-1, 3))
    n = int(pts.shape[0])
    empty = np.empty(0, dtype=np.int64)
    if n == 0:
        return empty
    r_s, r_n = float(salient_radius), float(non_max_radius)
    if r_s == 0.0 or r_n == 0.0:
        # a lone point has no resolution; where every point has a duplicate the resolution is 0, every neighbourhood
        # is one position, every covariance 0 and every saliency 0: no keypoints either way
        res = _resolution(pts) if n >= 2 else 0.0
        if res == 0.0:
            return empty
        r_s, r_n = 6.0 * res, 4.0 * res
    grid = Grid().build(pts, None, max(r_s, r_n))
    try:
        saliency, _, _ = ops.iss_saliency(grid, r_s, int(min_neighbors), float(gamma_21), float(gamma_32))
        keypoints = ops.iss_select(grid, saliency, r_n, int(min_neighbors))
        out = keypoints.cpu().numpy().astype(np.int64)
        torch.cuda.current_stream().synchronize()
    finally:
        grid.close()
    return out
