"""
Thin device-level wrappers: one Python function per C-ABI entry point (include/shotfpfh_b200.h), taking and
returning CUDA tensors. No arithmetic happens here.
"""

from __future__ import annotations

import ctypes

import numpy as np
import torch

from ._lib import check, lib
from .device import Grid, ptr, require_cuda, stream_ptr

SHOT_LEN = 352
FPFH_RANGES = ((-1.0, 1.0), (-1.0, 1.0), (-np.pi / 2, np.pi / 2))


def radius_csr(
    grid: Grid,
    queries: torch.Tensor | None,
    radius: float,
    want_sorted: bool = True,
    want_index: bool = False,
    want_dist: bool = False,
    self_range: tuple[int, int] | None = None,
    count_only: bool = False,
):
    """
    Fixed-radius search (sf_radius_count + sf_radius_fill; `count_only` stops after the count: offsets only). `queries=None` searches around the cloud's own
    points at cell-sorted positions `self_range = (first, count)` (default: all of them).
    Returns (offsets int64[q+1], nbr_sorted|None, nbr_index|None, dist|None).
    """
    dev = require_cuda()
    first, count = self_range if self_range is not None else (0, grid.n)
    nq = int(count) if queries is None else int(queries.shape[0])
    if nq == 0:  # an empty query set (a NULL pointer would mean "the cloud itself" to the C ABI)
        e32 = torch.empty(0, dtype=torch.int32, device=dev)
        return (
            torch.zeros(1, dtype=torch.int64, device=dev),
            e32 if want_sorted else None,
            e32.clone() if want_index else None,
            torch.empty(0, dtype=torch.float64, device=dev) if want_dist else None,
        )
    offsets = torch.empty(nq + 1, dtype=torch.int64, device=dev)
    total = ctypes.c_int64(0)
    check(
        lib.sf_radius_count(
            grid.handle, ptr(queries), int(first), nq, float(radius), ptr(offsets), ctypes.byref(total), stream_ptr()
        )
    )
    if count_only:
        return offsets, None, None, None
    p = int(total.value)
    nbr_sorted = torch.empty(p, dtype=torch.int32, device=dev) if want_sorted else None
    nbr_index = torch.empty(p, dtype=torch.int32, device=dev) if want_index else None
    dist = torch.empty(p, dtype=torch.float64, device=dev) if want_dist else None
    check(
        lib.sf_radius_fill(
            grid.handle, ptr(queries), int(first), nq, float(radius), ptr(offsets), ptr(nbr_sorted), ptr(nbr_index),
            ptr(dist), stream_ptr(),
        )
    )
    return offsets, nbr_sorted, nbr_index, dist


def grid_permutation(grid: Grid) -> tuple[torch.Tensor, torch.Tensor]:
    """(perm, inv_perm) as int32 CUDA tensors (copies; the grid keeps the originals)."""
    dev = require_cuda()
    perm = torch.empty(grid.n, dtype=torch.int32, device=dev)
    inv = torch.empty(grid.n, dtype=torch.int32, device=dev)
    check(lib.sf_grid_permutation(grid.handle, ptr(perm), ptr(inv), stream_ptr()))
    return perm, inv


def grid_arrays(grid: Grid, normals: bool) -> dict[str, torch.Tensor]:
    """Copies of the grid's cell-sorted arrays as CUDA tensors: pts (n, 4) float64, xyzc (n, 4) float32, cell_start
    (ncells + 1) int32 and, when `normals` (the grid must have been built with them), nrm and nrm32."""
    dev = require_cuda()
    info = grid.info()
    n, ncells = info["n"], info["ncells"]
    out = {
        "pts": torch.empty((n, 4), dtype=torch.float64, device=dev),
        "xyzc": torch.empty((n, 4), dtype=torch.float32, device=dev),
        "cell_start": torch.empty(ncells + 1, dtype=torch.int32, device=dev),
    }
    if normals:
        out["nrm"] = torch.empty((n, 4), dtype=torch.float64, device=dev)
        out["nrm32"] = torch.empty((n, 4), dtype=torch.float32, device=dev)
    check(lib.sf_grid_arrays(grid.handle, ptr(out["pts"]), ptr(out.get("nrm")), ptr(out["xyzc"]), ptr(out.get("nrm32")),
                             ptr(out["cell_start"]), stream_ptr()))
    return out


def voxel_subsample(xyz: torch.Tensor, voxel_size: float, want_members: bool = False):
    """
    Indices (int64, device) of one point per occupied voxel — `grid_subsampling` semantics, see csrc/subsample.cu.
    With `want_members` also the number of points of each of those voxels: (indices, members).
    """
    n = int(xyz.shape[0])
    if n == 0:
        empty = torch.empty(0, dtype=torch.int64, device=xyz.device)
        return (empty, empty.clone()) if want_members else empty
    picked = torch.empty(n, dtype=torch.int32, device=xyz.device)
    members = torch.empty(n, dtype=torch.int32, device=xyz.device) if want_members else None
    count = ctypes.c_int64(0)
    check(lib.sf_voxel_subsample(ptr(xyz), n, float(voxel_size), ptr(picked), ptr(members), ctypes.byref(count),
                                 stream_ptr()))
    picked = picked[: int(count.value)].long()
    return (picked, members[: int(count.value)].long()) if want_members else picked


def knn_attempt(grid: Grid, queries: torch.Tensor, k: int, reach: float, nbr_index: torch.Tensor, status: torch.Tensor):
    """One sf_knn attempt at `reach` (see include/shotfpfh_b200.h); updates nbr_index / status in place."""
    check(
        lib.sf_knn(grid.handle, ptr(queries), int(queries.shape[0]), int(k), float(reach), ptr(nbr_index), ptr(status),
                   stream_ptr())
    )


def pca_normals(xyz: torch.Tensor, nq: int, nbr_index: torch.Tensor, offsets: torch.Tensor | None = None,
                fixed_k: int = 0, pre_normals: torch.Tensor | None = None) -> torch.Tensor:
    """PCA normals of neighbourhoods given as ORIGINAL point indices into `xyz` (CSR or fixed_k per query)."""
    out = torch.empty((nq, 3), dtype=torch.float64, device=xyz.device)
    if nq:
        check(
            lib.sf_pca_normals(ptr(xyz), nq, ptr(offsets), int(fixed_k), ptr(nbr_index), ptr(pre_normals), ptr(out),
                               stream_ptr())
        )
    return out


def orient_normals(xyz: torch.Tensor, normals: torch.Tensor, nbr_index: torch.Tensor,
                   towards=None) -> tuple[torch.Tensor, int]:
    """Consistently oriented `normals` (sf_orient_normals) from the (n, K) neighbour lists `nbr_index` (ORIGINAL
    indices, int32) -> (oriented normals float64 (n, 3), number of trees of the spanning forest)."""
    n = int(xyz.shape[0])
    out = torch.empty((n, 3), dtype=torch.float64, device=xyz.device)
    trees = ctypes.c_int64(0)
    t = None if towards is None else np.ascontiguousarray(towards, dtype=np.float64).reshape(3)
    check(lib.sf_orient_normals(ptr(xyz), ptr(normals), n, ptr(nbr_index), int(nbr_index.shape[1]) if n else 1,
                                None if t is None else t.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), ptr(out),
                                ctypes.byref(trees), stream_ptr()))
    return out, int(trees.value)


def iss_saliency(grid: Grid, salient_radius: float, min_neighbors: int, gamma_21: float, gamma_32: float,
                 want_counts: bool = False, want_eigvals: bool = False):
    """
    ISS saliency of every cloud point (sf_iss_saliency), in CELL-SORTED order (`grid_permutation` maps it to original
    order). Returns (saliency float64 (n,), counts int32 (n,) | None, eigenvalues float64 (n, 3) ascending | None).
    """
    dev = require_cuda()
    n = grid.n
    sal = torch.empty(n, dtype=torch.float64, device=dev)
    counts = torch.empty(n, dtype=torch.int32, device=dev) if want_counts else None
    eig = torch.empty((n, 3), dtype=torch.float64, device=dev) if want_eigvals else None
    check(lib.sf_iss_saliency(grid.handle, float(salient_radius), int(min_neighbors), float(gamma_21), float(gamma_32),
                              ptr(sal), ptr(counts), ptr(eig), stream_ptr()))
    return sal, counts, eig


def iss_select(grid: Grid, saliency: torch.Tensor, non_max_radius: float, min_neighbors: int) -> torch.Tensor:
    """Non-maximum suppression of the cell-sorted `saliency` (sf_iss_select) -> int64 original indices, ascending."""
    dev = require_cuda()
    out = torch.empty(max(grid.n, 1), dtype=torch.int32, device=dev)
    count = ctypes.c_int64(0)
    check(lib.sf_iss_select(grid.handle, ptr(saliency), float(non_max_radius), int(min_neighbors), ptr(out),
                            ctypes.byref(count), stream_ptr()))
    return out[: int(count.value)].long()


def shot_lrf(grid: Grid, queries: torch.Tensor, radius: float, offsets: torch.Tensor, nbr_sorted: torch.Tensor):
    nq = int(queries.shape[0])
    lrf = torch.empty((nq, 3, 3), dtype=torch.float64, device=queries.device)
    check(lib.sf_shot_lrf(grid.handle, ptr(queries), nq, float(radius), ptr(offsets), ptr(nbr_sorted), ptr(lrf), stream_ptr()))
    return lrf


def shot_descriptor(
    grid: Grid,
    queries: torch.Tensor,
    radius: float,
    offsets: torch.Tensor,
    nbr_sorted: torch.Tensor,
    lrf: torch.Tensor,
    min_neighborhood_size: int,
    normalize: bool,
    out_dtype: torch.dtype = torch.float64,
    out: torch.Tensor | None = None,
):
    nq = int(queries.shape[0])
    if out is None:
        out = torch.empty((nq, SHOT_LEN), dtype=out_dtype, device=queries.device)
    assert out.shape == (nq, SHOT_LEN) and out.dtype in (torch.float32, torch.float64)
    check(
        lib.sf_shot_descriptor(
            grid.handle, ptr(queries), nq, float(radius), ptr(offsets), ptr(nbr_sorted), ptr(lrf),
            int(min_neighborhood_size), int(bool(normalize)), ptr(out), int(out.dtype == torch.float64), stream_ptr(),
        )
    )
    return out


def shot_single_scale(
    grid: Grid,
    queries: torch.Tensor,
    radius: float,
    min_neighborhood_size: int,
    normalize: bool,
    out_dtype: torch.dtype = torch.float64,
    out: torch.Tensor | None = None,
    want_lrf: bool = False,
    want_pairs: bool = False,
):
    """
    The fused single-scale driver (sf_shot_single_scale): search + frames + descriptors on the same neighbourhoods.
    Returns (descriptors, lrf | None, number of neighbour pairs | None).
    """
    nq = int(queries.shape[0])
    if out is None:
        out = torch.empty((nq, SHOT_LEN), dtype=out_dtype, device=queries.device)
    assert out.shape == (nq, SHOT_LEN) and out.dtype in (torch.float32, torch.float64)
    lrf = torch.empty((nq, 3, 3), dtype=torch.float64, device=queries.device) if want_lrf else None
    pairs = ctypes.c_int64(0)
    check(
        lib.sf_shot_single_scale(
            grid.handle, ptr(queries), nq, float(radius), int(min_neighborhood_size), int(bool(normalize)), ptr(out),
            int(out.dtype == torch.float64), ptr(lrf), ctypes.byref(pairs) if want_pairs else None, stream_ptr(),
        )
    )
    return out, lrf, (int(pairs.value) if want_pairs else None)


def shot_last_deferred() -> int:
    """Queries the float32 kernel handed to the float64 kernel in the last `shot_single_scale(want_pairs=True)`."""
    n = ctypes.c_int64(0)
    check(lib.sf_shot_last_deferred(ctypes.byref(n)))
    return int(n.value)


def profile_enable(enable: bool) -> None:
    check(lib.sf_profile_enable(int(bool(enable))))


def profile_read() -> tuple[float, float, float]:
    """(search + moments, eigen, votes + descriptor) milliseconds of the last fused single-scale call."""
    ms = (ctypes.c_float * 3)()
    check(lib.sf_profile_read(ms))
    return float(ms[0]), float(ms[1]), float(ms[2])


def fpfh_edges(n_bins: int) -> np.ndarray:
    """(3, n_bins + 1) float64 histogram edges, built on the host exactly as NumPy builds them."""
    return np.ascontiguousarray(np.stack([np.linspace(lo, hi, n_bins + 1) for lo, hi in FPFH_RANGES]))


def spfh(
    grid: Grid,
    offsets: torch.Tensor,
    nbr_sorted: torch.Tensor,
    n_bins: int,
    decorrelated: bool,
    self_range: tuple[int, int] | None = None,
):
    """SPFH rows of the cell-sorted points `self_range = (first, count)` (default all), CSR from the same range."""
    width = 3 * n_bins if decorrelated else n_bins**3
    first, count = self_range if self_range is not None else (0, grid.n)
    out = torch.empty((int(count), width), dtype=torch.float32, device=offsets.device)
    edges = fpfh_edges(n_bins)
    check(
        lib.sf_spfh(
            grid.handle, int(first), int(count), ptr(offsets), ptr(nbr_sorted), int(n_bins), int(bool(decorrelated)),
            edges.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), ptr(out), stream_ptr(),
        )
    )
    return out


def fpfh_cloud(grid: Grid, radius: float, n_bins: int, decorrelated: bool, keypoints: torch.Tensor,
               out_dtype: torch.dtype = torch.float64, out: torch.Tensor | None = None, want_pairs: bool = True):
    """
    The fused FPFH driver (sf_fpfh_cloud): search around every cloud point, SPFH, FPFH rows of `keypoints` (original
    point indices, int64). Returns (rows (Q, width), number of neighbour pairs | None).
    """
    width = 3 * n_bins if decorrelated else n_bins**3
    nq = int(keypoints.shape[0])
    if out is None:
        out = torch.empty((nq, width), dtype=out_dtype, device=keypoints.device)
    assert out.shape == (nq, width) and out.is_contiguous()
    edges = fpfh_edges(n_bins)
    pairs = ctypes.c_int64(0)
    check(
        lib.sf_fpfh_cloud(
            grid.handle, float(radius), int(n_bins), int(bool(decorrelated)),
            edges.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), ptr(keypoints), nq, ptr(out),
            int(out.dtype == torch.float64), ctypes.byref(pairs) if want_pairs else None, stream_ptr(),
        )
    )
    return out, (int(pairs.value) if want_pairs else None)



def fpfh_row_stride(width: int) -> int:
    """Floats between consecutive rows of the fused drivers' SPFH tables (rows padded to 16 bytes up to 128 bins)."""
    stride = ctypes.c_int32(0)
    check(lib.sf_fpfh_row_stride(int(width), ctypes.byref(stride)))
    return int(stride.value)


class FpfhBlock:
    """
    The fused FPFH driver on ONE block [first, first + count) of the cell-sorted cloud (one block per GPU):
    `spfh()` scans the candidates once (padded lists + weights kept here) and returns the block's SPFH rows;
    after the caller's all-gather, `rows(spfh_all, keypoints)` gives the FPFH rows of the keypoints (original
    indices) whose cell-sorted position lies in the block. first = 0, count = n reproduces `fpfh_cloud` bit for bit.
    """

    def __init__(self, grid: Grid, radius: float, n_bins: int, decorrelated: bool, first: int, count: int, device):
        self.grid, self.radius, self.n_bins, self.decorrelated = grid, float(radius), int(n_bins), bool(decorrelated)
        self.first, self.count = int(first), int(count)
        self.width = 3 * self.n_bins if self.decorrelated else self.n_bins**3
        self.stride = fpfh_row_stride(self.width)
        self.offsets = torch.empty(self.count + 1, dtype=torch.int64, device=device)
        total = ctypes.c_int64(0)
        check(lib.sf_fpfh_block_begin(grid.handle, self.radius, self.first, self.count, ptr(self.offsets),
                                      ctypes.byref(total), stream_ptr()))
        cap = max(int(total.value), 1)
        self.nbr = torch.empty(cap, dtype=torch.int32, device=device)
        self.weights = torch.empty(cap, dtype=torch.float32, device=device)
        self.counts = torch.empty(max(self.count, 1), dtype=torch.int32, device=device)
        self.pairs = 0

    def spfh(self, want_pairs: bool = False) -> torch.Tensor:
        rows = torch.empty((self.count, self.stride), dtype=torch.float32, device=self.offsets.device)
        edges = fpfh_edges(self.n_bins)
        pairs = ctypes.c_int64(0)
        check(lib.sf_fpfh_block_spfh(
            self.grid.handle, self.radius, self.n_bins, int(self.decorrelated),
            edges.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), self.first, self.count, ptr(self.offsets),
            ptr(self.nbr), ptr(self.weights), ptr(self.counts), ptr(rows),
            ctypes.byref(pairs) if want_pairs else None, stream_ptr(),
        ))
        self.pairs = int(pairs.value)
        return rows

    def rows(self, spfh_all: torch.Tensor, keypoints: torch.Tensor, out_dtype: torch.dtype = torch.float32) -> torch.Tensor:
        assert spfh_all.shape == (self.grid.n, self.stride) and spfh_all.dtype == torch.float32 and spfh_all.is_contiguous()
        nq = int(keypoints.shape[0])
        out = torch.empty((nq, self.width), dtype=out_dtype, device=spfh_all.device)
        check(lib.sf_fpfh_block_rows(
            self.grid.handle, self.first, self.count, ptr(self.offsets), ptr(self.counts), ptr(self.nbr),
            ptr(self.weights), ptr(spfh_all), self.width, ptr(keypoints), nq, ptr(out),
            int(out_dtype == torch.float64), stream_ptr(),
        ))
        return out


def fpfh(
    grid: Grid,
    offsets: torch.Tensor,
    nbr_sorted: torch.Tensor,
    dist: torch.Tensor,
    spfh_rows: torch.Tensor,
    keypoints: torch.Tensor,
    out_dtype: torch.dtype = torch.float64,
    csr_by_keypoint: bool = False,
):
    """
    FPFH rows of the keypoints (original indices). `spfh_rows` covers the WHOLE cloud in cell-sorted order. The CSR
    is the whole-cloud self-search (default) or, with `csr_by_keypoint`, a search around the keypoints' coordinates.
    """
    nq, width = int(keypoints.shape[0]), int(spfh_rows.shape[1])
    assert int(spfh_rows.shape[0]) == grid.n
    out = torch.empty((nq, width), dtype=out_dtype, device=offsets.device)
    if nq == 0:
        return out
    check(
        lib.sf_fpfh(
            grid.handle, ptr(offsets), ptr(nbr_sorted), ptr(dist), int(bool(csr_by_keypoint)), ptr(spfh_rows), width,
            ptr(keypoints), nq, ptr(out), int(out_dtype == torch.float64), stream_ptr(),
        )
    )
    return out


# ---- matching -------------------------------------------------------------------------------------------------
def nonempty_rows(desc: torch.Tensor, want_absmax: bool = False):
    """Ids of the rows with a non-zero entry; with `want_absmax` also the largest |x| of the array (same pass; NaN or
    inf when the array holds one): (rows, absmax)."""
    n, width = int(desc.shape[0]), int(desc.shape[1])
    rows = torch.empty(max(n, 1), dtype=torch.int64, device=desc.device)
    count = ctypes.c_int64(0)
    absmax = ctypes.c_double(0.0)
    check(lib.sf_nonempty_rows(ptr(desc), n, width, ptr(rows), ctypes.byref(count),
                               ctypes.byref(absmax) if want_absmax else None, stream_ptr()))
    rows = rows[: int(count.value)]
    return (rows, float(absmax.value)) if want_absmax else rows


def padded_width(width: int) -> int:
    return (width + 63) // 64 * 64


def match_pack(desc: torch.Tensor, rows: torch.Tensor, scale: float):
    """-> (float16 (count, padded_width) operand, float32 squared norms of the rounded rows)."""
    width, count = int(desc.shape[1]), int(rows.shape[0])
    wp = padded_width(width)
    packed = torch.empty((count, wp), dtype=torch.float16, device=desc.device)
    sqnorm = torch.empty(count, dtype=torch.float32, device=desc.device)
    check(lib.sf_match_pack(ptr(desc), width, ptr(rows), count, float(scale), ptr(packed), wp, ptr(sqnorm), stream_ptr()))
    return packed, sqnorm


def match_topk(a_packed, b_packed, b_sqnorm, k: int, index_offset: int = 0, tensor_cores: bool = True):
    qa, qb, wp = int(a_packed.shape[0]), int(b_packed.shape[0]), int(a_packed.shape[1])
    score = torch.empty((qa, k), dtype=torch.float32, device=a_packed.device)
    idx = torch.empty((qa, k), dtype=torch.int32, device=a_packed.device)
    check(
        lib.sf_match_topk(
            ptr(a_packed), qa, ptr(b_packed), ptr(b_sqnorm), qb, wp, int(k), int(index_offset), ptr(score), ptr(idx),
            int(bool(tensor_cores)), stream_ptr(),
        )
    )
    return score, idx


def topk_merge(score: torch.Tensor, idx: torch.Tensor):
    """(parts, qa, k) -> (qa, k)."""
    parts, qa, k = (int(s) for s in score.shape)
    so = torch.empty((qa, k), dtype=torch.float32, device=score.device)
    io = torch.empty((qa, k), dtype=torch.int32, device=score.device)
    check(lib.sf_topk_merge(ptr(score.contiguous()), ptr(idx.contiguous()), parts, qa, k, ptr(so), ptr(io), stream_ptr()))
    return so, io


def nearest_merge(packed: torch.Tensor):
    """(parts, q, 3) float64 (d1, global nearest index, d2) per target shard -> (nn int64, d1, d2) against the union."""
    parts, q = int(packed.shape[0]), int(packed.shape[1])
    nn = torch.empty(q, dtype=torch.int64, device=packed.device)
    d1 = torch.empty(q, dtype=torch.float64, device=packed.device)
    d2 = torch.empty(q, dtype=torch.float64, device=packed.device)
    check(lib.sf_nearest_merge(ptr(packed.contiguous()), parts, q, ptr(nn), ptr(d1), ptr(d2), stream_ptr()))
    return nn, d1, d2


def match_certify(score, a_sqnorm, d1, d2, scale: float, b_norm_max: float, width: int, qb: int, want_second: bool):
    """uint8 (qa,) flags: 1 where the shortlist does not provably contain the nearest (second-nearest) neighbour."""
    qa, k = int(score.shape[0]), int(score.shape[1])
    flags = torch.empty(qa, dtype=torch.uint8, device=score.device)
    check(lib.sf_match_certify(ptr(score.contiguous()), k, ptr(a_sqnorm), ptr(d1), ptr(d2), qa, float(scale),
                               float(b_norm_max), int(width), int(qb), int(bool(want_second)), ptr(flags), stream_ptr()))
    return flags


def match_exhaustive(a_desc, rows_a, which, limit, b_desc, rows_b, scale: float, norm_bound: float) -> torch.Tensor:
    """(n_which, 16) int32 lists of the flagged queries `which`: every target within `limit` (float64 per flagged query;
    found in float32 on the rows times `scale` with a proven slack: `norm_bound` >= |a| + |b| over the scaled rows);
    row[0] == -2 where more than 16
    targets qualified (see sf_match_exhaustive)."""
    n = int(which.shape[0])
    cand = torch.empty((n, 16), dtype=torch.int32, device=a_desc.device)
    check(lib.sf_match_exhaustive(ptr(a_desc), ptr(rows_a), ptr(which.contiguous()), n, ptr(limit.contiguous()), ptr(b_desc),
                                  ptr(rows_b), int(rows_b.shape[0]), int(a_desc.shape[1]), float(scale), float(norm_bound), ptr(cand),
                                  stream_ptr()))
    return cand


def match_exhaustive_topk(a_desc, rows_a, which, b_desc, rows_b, cand_idx) -> None:
    """Rewrites the rows `which` of the (qa, k) shortlist `cand_idx` with the exhaustive float64 k nearest targets."""
    k = int(cand_idx.shape[1])
    check(lib.sf_match_exhaustive_topk(ptr(a_desc), ptr(rows_a), ptr(which.contiguous()), int(which.shape[0]), ptr(b_desc),
                                       ptr(rows_b), int(rows_b.shape[0]), int(a_desc.shape[1]), k, ptr(cand_idx),
                                       stream_ptr()))


def match_rerank(a_desc, rows_a, b_desc, rows_b, cand_idx):
    qa, k, width = int(cand_idx.shape[0]), int(cand_idx.shape[1]), int(a_desc.shape[1])
    nn = torch.empty(qa, dtype=torch.int32, device=a_desc.device)
    d1 = torch.empty(qa, dtype=torch.float64, device=a_desc.device)
    d2 = torch.empty(qa, dtype=torch.float64, device=a_desc.device)
    check(
        lib.sf_match_rerank(
            ptr(a_desc), ptr(rows_a), qa, ptr(b_desc), ptr(rows_b), width, ptr(cand_idx.contiguous()), k, ptr(nn),
            ptr(d1), ptr(d2), stream_ptr(),
        )
    )
    return nn, d1, d2


def ransac_count_inliers(matched_scan: torch.Tensor, matched_ref: torch.Tensor, transforms: torch.Tensor,
                         threshold: float) -> torch.Tensor:
    """Inliers of each candidate transform ((D, 12) rows: rotation row-major, translation) -> int32 (D,)."""
    m, d = int(matched_scan.shape[0]), int(transforms.shape[0])
    assert transforms.dtype == torch.float64 and transforms.shape[1:] == (12,) and matched_ref.shape == matched_scan.shape
    counts = torch.zeros(d, dtype=torch.int32, device=matched_scan.device)
    check(lib.sf_ransac_count_inliers(ptr(matched_scan), ptr(matched_ref), m, ptr(transforms), d, float(threshold),
                                      ptr(counts), stream_ptr()))
    return counts


def ransac_adaptive(matched_scan: torch.Tensor, matched_ref: torch.Tensor, threshold: float, edge_similarity: float,
                    seed: int, max_draws: int, confidence: float) -> dict:
    """
    Adaptive RANSAC (sf_ransac_adaptive) on (m, 3) float64 device tensors: {"transform": float64 (12,) host array
    (rotation row-major, translation), "best_draw", "best_count", "draws_used", "valid": ints, "mask": uint8 (m,)
    device tensor of the winner's inliers}; best_draw is -1 and valid 0 when no draw passed the checks.
    """
    import numpy as np

    m = int(matched_scan.shape[0])
    assert matched_scan.dtype == torch.float64 and matched_ref.shape == matched_scan.shape
    transform = np.zeros(12, dtype=np.float64)
    counters = [ctypes.c_int64() for _ in range(4)]
    mask = torch.empty(m, dtype=torch.uint8, device=matched_scan.device)
    check(lib.sf_ransac_adaptive(ptr(matched_scan), ptr(matched_ref), m, float(threshold), float(edge_similarity),
                                 int(seed) & 0xFFFFFFFFFFFFFFFF, int(max_draws), float(confidence),
                                 transform.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
                                 *(ctypes.byref(c) for c in counters), ptr(mask), stream_ptr()))
    best_draw, best_count, draws_used, valid = (c.value for c in counters)
    return {"transform": transform, "best_draw": best_draw, "best_count": best_count, "draws_used": draws_used,
            "valid": valid, "mask": mask}


def ransac_adaptive_batch(matched_scan: torch.Tensor, matched_ref: torch.Tensor, threshold: float,
                          edge_similarity: float, seed: int, first_draw: int, n_draws: int) -> dict:
    """One batch of sf_ransac_adaptive (sf_ransac_adaptive_batch): {"survivors": uint32 as int64 device tensor of the
    draws that pass the edge check, "valid_draws", "transforms" (V, 12), "counts": the valid draws, their transforms
    and inlier counts}, each sorted by draw index."""
    m = int(matched_scan.shape[0])
    assert matched_scan.dtype == torch.float64 and matched_ref.shape == matched_scan.shape
    dev = matched_scan.device
    survivors = torch.empty(n_draws, dtype=torch.int32, device=dev)
    valid_draws = torch.empty(n_draws, dtype=torch.int32, device=dev)
    transforms = torch.empty((n_draws, 12), dtype=torch.float64, device=dev)
    counts = torch.empty(n_draws, dtype=torch.int32, device=dev)
    n = (ctypes.c_int64 * 2)()
    check(lib.sf_ransac_adaptive_batch(ptr(matched_scan), ptr(matched_ref), m, float(threshold),
                                       float(edge_similarity), int(seed) & 0xFFFFFFFFFFFFFFFF, int(first_draw),
                                       int(n_draws), ptr(survivors), ptr(valid_draws), ptr(transforms), ptr(counts),
                                       n, stream_ptr()))

    def as_draws(t: torch.Tensor) -> torch.Tensor:  # uint32 bits -> int64
        return t.to(torch.int64) & 0xFFFFFFFF

    order = torch.argsort(as_draws(valid_draws[: n[1]]))
    return {"survivors": torch.sort(as_draws(survivors[: n[0]])).values, "valid_draws": as_draws(valid_draws[: n[1]])[order],
            "transforms": transforms[: n[1]][order], "counts": counts[: n[1]][order]}


def icp_plane_step(ref_grid: Grid, scan: torch.Tensor, transform_row, d_max: float, want_nearest: bool = False):
    """
    One point-to-plane ICP iteration's sums (sf_icp_plane_step): float64 (29,) host array = 21 entries of g^T g
    (upper triangle, row order), 6 of g^T h, sum of |residual|, number of pairs. With `want_nearest` also the
    int32 device tensor of each scan point's nearest reference index (-1: none within d_max).
    """
    import numpy as np

    row = np.ascontiguousarray(transform_row, dtype=np.float64)
    assert row.shape == (12,)
    sums = np.zeros(29, dtype=np.float64)
    n = int(scan.shape[0])
    nearest = torch.empty(n, dtype=torch.int32, device=scan.device) if want_nearest else None
    dp = ctypes.POINTER(ctypes.c_double)
    check(lib.sf_icp_plane_step(ref_grid.handle, ptr(scan), n, row.ctypes.data_as(dp), float(d_max),
                                sums.ctypes.data_as(dp), ptr(nearest), stream_ptr()))
    return (sums, nearest) if want_nearest else sums
