"""
`compute_normals` with the reference's signature (shot_fpfh/descriptors/pca_based_descriptors.py:29-59) on the GPU:
k-nearest-neighbour (or fixed-radius) neighbourhoods on the uniform grid of csrc/grid.cu, then the eigenvector of the
smallest eigenvalue of each neighbourhood's covariance (csrc/normals.cu, LAPACK-path 3x3 eigensolver so that the sign
of a normal that is NOT re-oriented by `pre_computed_normals` is the one np.linalg.eigh gives).

This is a "next" row (SURVEY.md §8f #2): it runs upstream of the hot path, in `get_data` (helpers/io_ply.py:259-301).
`orient_normals` (no counterpart in the reference) gives those normals consistent signs (csrc/orient.cu).
The other functions of the reference module (sphericity, linearity ... features and their plots) are not on any path
the pipeline takes and are not provided.
"""

from __future__ import annotations

import numpy as np
import numpy.typing as npt
import torch

from .. import ops
from ..device import Grid, download, require_cuda, upload


def _calibrate_reach(grid_points: torch.Tensor, queries: torch.Tensor, k: int) -> float:
    """A reach with ~4k cloud points inside for the median query (two rounds on a 2 000-query sample)."""
    n = int(grid_points.shape[0])
    lo, hi = grid_points.min(dim=0).values, grid_points.max(dim=0).values
    extent = (hi - lo).clamp_min(1e-300)
    volume = float(torch.prod(extent))
    reach = (3.0 * 4 * k * volume / (4.0 * np.pi * n)) ** (1.0 / 3.0) if volume > 0 else float(extent.max())
    reach = max(reach, 1e-300)
    sample = queries[torch.randperm(queries.shape[0], device=queries.device)[:2000]].contiguous()
    for _ in range(3):
        grid = Grid().build(grid_points, None, reach)
        offsets, _, _, _ = ops.radius_csr(grid, sample, reach, want_sorted=False)
        grid.close()
        counts = (offsets[1:] - offsets[:-1]).double()
        median = float(counts.median())
        if 2.5 * k <= median <= 6 * k:
            break
        reach *= (4.0 * k / max(median, 0.5)) ** 0.4  # count ~ reach^2 (surfaces) .. reach^3 (volumes)
    return reach


def knn_device(points: torch.Tensor, queries: torch.Tensor, k: int):
    """k nearest cloud points of every query -> int32 (Q, k) ORIGINAL point indices, nearest first."""
    if k > points.shape[0]:
        raise ValueError(f"Expected n_neighbors <= n_samples_fit, but n_neighbors = {k}, n_samples_fit = {points.shape[0]}")
    nq = int(queries.shape[0])
    nbr = torch.empty((nq, k), dtype=torch.int32, device=points.device)
    status = torch.zeros(nq, dtype=torch.int32, device=points.device)
    reach = _calibrate_reach(points, queries, k) if nq else 1.0
    grid = Grid().build(points, None, reach)
    ops.knn_attempt(grid, queries, k, reach, nbr, status)
    # status: 1 = solved, 0 = fewer than k points within reach, 2 = more than the kernel can rank within reach
    small = reach
    for _ in range(40):  # denser-than-median places: shrink the reach on the same grid
        crowded = status == 2
        if not bool(crowded.any()):
            break
        small /= 1.5
        attempt = torch.where(crowded, 0, 1).to(torch.int32)  # only the crowded queries take part
        ops.knn_attempt(grid, queries, k, small, nbr, attempt)
        status = torch.where(crowded, attempt, status)
    for _ in range(60):  # sparser-than-median places: grow the reach, which needs a coarser grid
        if bool((status == 1).all()):
            break
        if bool((status == 2).any()):
            break
        reach *= 1.6
        grid.build(points, None, reach)
        ops.knn_attempt(grid, queries, k, reach, nbr, status)
    grid.close()
    if not bool((status == 1).all()):
        raise RuntimeError("k-nearest-neighbour search did not converge (more than 512 coincident points?)")
    return nbr


def compute_normals(
    query_points: npt.NDArray[np.float64],
    cloud_points: npt.NDArray[np.float64],
    *,
    k: int | None = None,
    radius: float | None = None,
    pre_computed_normals: npt.NDArray[np.float64] | None = None,
) -> npt.NDArray[np.float64]:
    """
    Computes PCA-based normals on a point cloud. Reorients normals based on pre-computed normals if provided.
    (Reference: pca_based_descriptors.py:29-59; `k` takes precedence over `radius`, as there.)
    """
    assert k is not None or radius is not None, "No parameter provided for the neighborhood search."
    pts, q = upload(cloud_points), upload(query_points)
    pre = upload(pre_computed_normals) if pre_computed_normals is not None else None
    if k is not None:
        nbr = knn_device(pts, q, int(k))
        normals = ops.pca_normals(pts, int(q.shape[0]), nbr.reshape(-1), fixed_k=int(k), pre_normals=pre)
    else:
        grid = Grid().build(pts, None, radius)
        offsets, _, nbr, _ = ops.radius_csr(grid, q, radius, want_sorted=False, want_index=True)
        grid.close()
        normals = ops.pca_normals(pts, int(q.shape[0]), nbr, offsets=offsets, pre_normals=pre)
    return download(normals)


def orient_normals(
    points: npt.NDArray[np.float64],
    normals: npt.NDArray[np.float64],
    k: int = 10,
    towards: npt.ArrayLike | None = None,
) -> npt.NDArray[np.float64]:
    """
    Consistently oriented normals (Hoppe et al. 1992; Open3D's `orient_normals_consistent_tangent_plane`): the signs
    of `normals` (e.g. `compute_normals` output, whose signs are LAPACK's) are propagated along the minimum spanning
    forest of the k-nearest-neighbour graph, with edge weight 1 - |n_i . n_j|. Returns a new (n, 3) float64 array: the
    input normals with some of them negated.
    Each tree of the forest (one per connected piece of the graph) gets one sign: by default its member with the
    lowest index keeps its input sign; with `towards` = (x, y, z), a viewpoint, the tree takes the sign under which
    more of its members have n . (towards - p) > 0 than < 0 (a tie keeps the default).
    No counterpart in the reference; oracle/orientation_oracle.py states the same computation in NumPy.
    """
    require_cuda()
    pts_h = np.asarray(points, dtype=np.float64).reshape(-1, 3)
    nrm_h = np.asarray(normals, dtype=np.float64).reshape(-1, 3)
    if pts_h.shape != nrm_h.shape:
        raise ValueError(f"points {pts_h.shape} and normals {nrm_h.shape} differ in shape")
    if not (np.isfinite(pts_h).all() and np.isfinite(nrm_h).all()):
        raise ValueError("orient_normals: points and normals must be finite")
    if towards is not None:
        towards = np.asarray(towards, dtype=np.float64).reshape(3)
        if not np.isfinite(towards).all():
            raise ValueError("orient_normals: towards must be finite")
    n, k = pts_h.shape[0], int(k)
    if n == 0:
        return np.empty((0, 3), dtype=np.float64)
    if k < 1:
        raise ValueError(f"Expected n_neighbors > 0. Got {k}")
    pts, nrm = upload(pts_h), upload(nrm_h)
    nbr = knn_device(pts, pts, k + 1)  # raises for k >= n; the point itself is among its k + 1 nearest
    out, _ = ops.orient_normals(pts, nrm, nbr, towards)
    return download(out)
