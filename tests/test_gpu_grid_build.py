"""
GPU: the grid's counting-sort build (cell-mates ranked by original index) writes the same bytes as the stable
radix-sort build it replaced (SF_GRID_RADIX=1), so a change to either cannot alter any result: cell-sorted coordinates and
normals in float64 and float32, cell_start, perm and inv_perm — on the 1M-point benchmark cloud, a crowded cell,
duplicated points, a cloud without normals, a speculative rebuild on the previous box and a build in a caller's box.
"""

import os

import numpy as np
import pytest

from shot_fpfh_b200 import synthetic

pytestmark = pytest.mark.gpu


def _host_arrays(grid, normals: bool) -> dict:
    """Every array of a built grid, copied to the host as raw bytes."""
    from shot_fpfh_b200 import ops

    out = ops.grid_arrays(grid, normals)
    out["perm"], out["inv_perm"] = ops.grid_permutation(grid)
    return {k: v.cpu().numpy().view(np.uint8) for k, v in out.items()}


def _build(radix: str, xyz, nrm, radius, box=None, speculative=False) -> dict:
    from shot_fpfh_b200.device import Grid

    os.environ["SF_GRID_RADIX"] = radix
    try:
        grid = Grid()
        if speculative:  # the first build reads the box back, the second assumes it (as in a repeated step)
            grid.set_speculative(builds=True)
            grid.build(xyz, nrm, radius)
        grid.build(xyz, nrm, radius, box=box)
        arrays = _host_arrays(grid, nrm is not None)
        assert grid.poll() == 0
        grid.close()
        return arrays
    finally:
        del os.environ["SF_GRID_RADIX"]


def _crowded(n: int, seed: int):
    """A bumpy sphere with 20 000 of its points moved into one small cube (one cell holds thousands of points)."""
    pts, nrm = synthetic.bumpy_sphere(n, seed=seed)
    rng = np.random.default_rng(seed)
    pts[::10][:20_000] = pts[0] + 1e-4 * rng.random((20_000, 3))
    return pts, nrm


def _duplicated(n: int, seed: int):
    pts, nrm = synthetic.bumpy_sphere(n, seed=seed)
    pts[1000:3000] = pts[17]                       # 2000 copies of one point
    pts[5000:9000] = pts[5000:9000].round(2)       # many exact duplicates on a lattice
    pts[20_000:40_000] = pts[40_000:60_000]        # 20 000 points twice, far apart in input order
    return pts, nrm


CASES = {
    "c2_cloud": lambda: (*synthetic.bumpy_sphere(1_000_000, seed=0), 5.0 * synthetic.mean_spacing(1_000_000)),
    "crowded_cell": lambda: (*_crowded(200_000, 5), 5.0 * synthetic.mean_spacing(200_000)),
    "duplicates": lambda: (*_duplicated(200_000, 6), 5.0 * synthetic.mean_spacing(200_000)),
    "few_large_cells": lambda: (np.random.default_rng(7).random((30_000, 3)), None, 0.4),
}


@pytest.mark.parametrize("case", sorted(CASES))
@pytest.mark.parametrize("with_normals", [True, False])
@pytest.mark.parametrize("mode", ["sync", "speculative", "in_box"])
def test_counting_sort_build_is_byte_identical_to_radix_build(case, with_normals, mode):
    from shot_fpfh_b200.device import upload

    pts, nrm, radius = CASES[case]()
    if with_normals and nrm is None:
        nrm = np.random.default_rng(8).standard_normal(pts.shape)
    xyz = upload(pts)
    nrm_dev = upload(nrm) if with_normals else None
    box = None
    if mode == "in_box":  # a box larger than the cloud, as a rank of the halo partition gets it
        lo, hi = pts.min(axis=0), pts.max(axis=0)
        box = (lo - 0.25 * (hi - lo), hi + 0.1 * (hi - lo))
    want = _build("1", xyz, nrm_dev, radius, box=box, speculative=mode == "speculative")
    got = _build("0", xyz, nrm_dev, radius, box=box, speculative=mode == "speculative")
    assert set(got) == set(want) == ({"pts", "xyzc", "cell_start", "perm", "inv_perm"}
                                     | ({"nrm", "nrm32"} if with_normals else set()))
    for name in want:
        assert got[name].shape == want[name].shape, name
        assert np.array_equal(got[name], want[name]), f"{name} differs ({case}, normals={with_normals}, {mode})"
    perm = want["perm"].view(np.int32)
    assert np.array_equal(np.sort(perm), np.arange(pts.shape[0], dtype=np.int32))
