"""
GPU: the per-call device scratch of the C ABI (sf::Scratch, csrc/sf_common.cuh) goes back to the device's default memory
pool on every return path, the rejected calls included. The library takes its per-call temporaries from that pool and
torch's caching allocator does not use it, so the pool's used-memory counter reads the same before and after each call.
"""

import ctypes
import os

import numpy as np
import pytest
from conftest import registration_case

from shot_fpfh_b200 import synthetic

pytestmark = pytest.mark.gpu

CU_MEMPOOL_ATTR_USED_MEM_CURRENT = 7  # cuda.h, CUmemPool_attribute


@pytest.fixture(scope="module")
def pool_used():
    """() -> bytes in use in the current device's default memory pool, read after the device has finished."""
    import torch

    if "cudaMallocAsync" in os.environ.get("PYTORCH_CUDA_ALLOC_CONF", ""):
        pytest.skip("torch allocates from the default memory pool itself")
    torch.cuda.init()
    cuda = ctypes.CDLL("libcuda.so.1")
    device = ctypes.c_int(0)
    assert cuda.cuDeviceGet(ctypes.byref(device), torch.cuda.current_device()) == 0
    pool = ctypes.c_void_p()
    assert cuda.cuDeviceGetDefaultMemPool(ctypes.byref(pool), device) == 0

    def used() -> int:
        torch.cuda.synchronize()
        value = ctypes.c_uint64(0)
        assert cuda.cuMemPoolGetAttribute(pool, CU_MEMPOOL_ATTR_USED_MEM_CURRENT, ctypes.byref(value)) == 0
        return int(value.value)

    return used


def returns_scratch(used, call):
    """Runs call() and asserts that the pool holds as much as before it; returns what call() returned."""
    before = used()
    result = call()
    assert used() == before
    return result


def cloud(n=20_000):
    from shot_fpfh_b200.device import Grid, upload

    pts, normals = synthetic.bumpy_sphere(n, seed=4)
    radius = 5.0 * synthetic.mean_spacing(n)
    p_dev = upload(pts)
    return p_dev, Grid().build(p_dev, upload(normals), radius), radius


def test_rejected_calls_release_their_scratch(pool_used):
    import torch

    from shot_fpfh_b200 import ops
    from shot_fpfh_b200._lib import SfError

    # more flagged queries than one launch's 65535 query tiles of 64
    gen = torch.Generator(device="cuda").manual_seed(0)
    a = torch.rand((8, 33), dtype=torch.float64, device="cuda", generator=gen)
    b = torch.rand((8, 33), dtype=torch.float64, device="cuda", generator=gen)
    rows = torch.arange(8, dtype=torch.int64, device="cuda")
    n_which = 65535 * 64 + 1
    which = torch.zeros(n_which, dtype=torch.int64, device="cuda")
    limit = torch.ones(n_which, dtype=torch.float64, device="cuda")
    before = pool_used()
    with pytest.raises(SfError, match="flagged queries"):
        ops.match_exhaustive(a, rows, which, limit, b, rows, 1.0, 10.0)
    assert pool_used() == before
    del which, limit

    # SHOT rows that are not 16-byte aligned, rejected after the work list has been allocated
    p_dev, grid, radius = cloud()
    queries = p_dev[:500].contiguous()
    offsets, nbr, _, _ = ops.radius_csr(grid, queries, radius)
    lrf = ops.shot_lrf(grid, queries, radius, offsets, nbr)
    nq = int(queries.shape[0])
    out = torch.empty(nq * 352 + 1, dtype=torch.float32, device="cuda")[1:].view(nq, 352)
    before = pool_used()
    with pytest.raises(SfError, match="16-byte aligned"):
        ops.shot_descriptor(grid, queries, radius, offsets, nbr, lrf, 10, True, out=out)
    assert pool_used() == before
    grid.close()


def test_successful_calls_release_their_scratch(pool_used):
    import torch

    from shot_fpfh_b200 import ops
    from shot_fpfh_b200.device import Grid, download_sparse_rows, upload

    used = pool_used
    p_dev, grid, radius = cloud()
    n = grid.n
    kp = torch.arange(0, n, 2, dtype=torch.int64, device="cuda")  # >= 4096: the rows stage sorts the keypoints
    fused, pairs = returns_scratch(used, lambda: ops.fpfh_cloud(grid, radius, 11, True, kp, out_dtype=torch.float32))
    assert pairs > 0
    block = returns_scratch(used, lambda: ops.FpfhBlock(grid, radius, 11, True, 0, n, p_dev.device))
    spfh_all = returns_scratch(used, lambda: block.spfh(want_pairs=True))
    assert block.pairs == pairs
    assert torch.equal(returns_scratch(used, lambda: block.rows(spfh_all, kp)), fused)
    offsets, nbr, _, dist = ops.radius_csr(grid, None, radius, want_dist=True)
    spfh = ops.spfh(grid, offsets, nbr, 11, True)
    returns_scratch(used, lambda: ops.fpfh(grid, offsets, nbr, dist, spfh, kp, out_dtype=torch.float32))

    queries = p_dev[:500].contiguous()
    q_offsets, q_nbr, _, _ = ops.radius_csr(grid, queries, radius)
    lrf = ops.shot_lrf(grid, queries, radius, q_offsets, q_nbr)
    desc = returns_scratch(used, lambda: ops.shot_descriptor(grid, queries, radius, q_offsets, q_nbr, lrf, 10, True))
    returns_scratch(used, lambda: download_sparse_rows(desc.float().contiguous(), 2))

    rows = returns_scratch(used, lambda: ops.nonempty_rows(desc))
    packed, sqnorm = ops.match_pack(desc, rows, 1.0)
    returns_scratch(used, lambda: ops.match_topk(packed, packed, sqnorm, 8, 0, tensor_cores=True))
    which = torch.arange(100, dtype=torch.int64, device="cuda")  # positions in `rows`
    limit = torch.full((100,), 0.5, dtype=torch.float64, device="cuda")
    returns_scratch(used, lambda: ops.match_exhaustive(desc, rows, which, limit, desc, rows, 1.0, 4.0))

    sal, _, _ = ops.iss_saliency(grid, radius, 5, 0.975, 0.975)
    returns_scratch(used, lambda: ops.iss_select(grid, sal, radius, 5))
    grid.close()

    scan, ref, ref_normals, _, _ = registration_case()
    s = np.sqrt(3.0 / scan.shape[0])
    scan_dev = upload(scan)
    sub = returns_scratch(used, lambda: ops.voxel_subsample(scan_dev, 3 * s))
    ref_grid = Grid().build(upload(ref), upload(ref_normals), 4 * s)
    row = np.concatenate([np.eye(3).ravel(), np.zeros(3)])
    returns_scratch(used, lambda: ops.icp_plane_step(ref_grid, scan_dev[sub].contiguous(), row, 4 * s))
    ref_grid.close()
