"""
The float32 SHOT kernel (shot.cu::shot_fast_kernel) against the float64 kernel it hands queries to
(shot_descriptor_block_kernel, which runs every query under SF_SHOT_EXACT=1), and the float64 kernel against the
oracle, on realistic clouds and on clouds built to put neighbours on the decision boundaries.

Bars, the same in every case and without exemptions:
  - frames of the fused driver are identical (both paths flip the same raw eigenvectors, y = z x x in float64);
  - the all-zero rows are the same rows;
  - every row agrees to 1e-5 relative L2 (one misbinned neighbour moves a row by ~1e-2);
  - at least as many rows are bit-identical as queries were handed over (those run the float64 kernel both times).
"""

import numpy as np
import pytest
import torch
from conftest import rel_l2
from sklearn.neighbors import KDTree

from oracle import shot_oracle, shot_probes
from shot_fpfh_b200 import synthetic

pytestmark = pytest.mark.gpu

TOL = 1e-5
MIN_NB = 10


def _grid(pts, nrm, radius):
    from shot_fpfh_b200.device import Grid, upload

    return Grid().build(upload(pts), upload(nrm), radius)


def _fused(grid, queries, radius, dtype=torch.float32, normalize=True, min_nb=MIN_NB):
    from shot_fpfh_b200 import ops
    from shot_fpfh_b200.device import upload

    d, lrf, _ = ops.shot_single_scale(grid, upload(queries), radius, min_nb, normalize, out_dtype=dtype, want_lrf=True,
                                      want_pairs=True)
    torch.cuda.synchronize()
    return d.cpu(), lrf.cpu(), ops.shot_last_deferred()


def _caller(grid, queries, radius, frames, dtype=torch.float32, normalize=True, min_nb=MIN_NB, search_radius=None):
    from shot_fpfh_b200 import ops
    from shot_fpfh_b200.device import upload

    q = upload(queries)
    offsets, nbr, _, _ = ops.radius_csr(grid, q, radius)
    d = ops.shot_descriptor(grid, q, radius, offsets, nbr, upload(frames), min_nb, normalize, out_dtype=dtype)
    torch.cuda.synchronize()
    return d.cpu(), None, None


def _twice(monkeypatch, call):
    """The same call by default and with SF_SHOT_EXACT=1 (launch_descriptor reads it on every call)."""
    monkeypatch.delenv("SF_SHOT_EXACT", raising=False)
    fast = call()
    monkeypatch.setenv("SF_SHOT_EXACT", "1")
    exact = call()
    monkeypatch.delenv("SF_SHOT_EXACT", raising=False)
    return fast, exact


def _oracle_rows(pts, nrm, queries, radius, frames, normalize=True, min_nb=MIN_NB):
    nbh = KDTree(pts).query_radius(queries, radius)
    return np.array([shot_oracle.shot_descriptor(q, pts[nb], nrm[nb], radius, f, normalize, min_nb)
                     for q, nb, f in zip(queries, nbh, frames)]).reshape(len(queries), 352)


def _row_err(got, want):
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    zero = ~want.any(axis=1)
    assert np.array_equal(~got.any(axis=1), zero), "all-zero rows differ"
    return rel_l2(got[~zero], want[~zero]) if (~zero).any() else np.zeros(1)


def _check(tag, fast, exact, oracle=None, oracle_idx=None):
    """Fast vs exact bars; exact vs oracle (rows `oracle_idx`) when given. Returns (deferred, fast-exact max)."""
    rows_f, fr_f, deferred = fast
    rows_e, fr_e, _ = exact
    if fr_f is not None:
        assert torch.equal(fr_f, fr_e), f"{tag}: frames differ"
    err = _row_err(rows_f.double().numpy(), rows_e.double().numpy())
    identical = int((rows_f == rows_e).all(dim=1).sum())
    nq = rows_f.shape[0]
    line = f"{tag}: nq {nq}, deferred {deferred}, identical {identical}, fast-exact max {err.max():.1e}"
    if oracle is not None:
        idx = np.arange(nq) if oracle_idx is None else oracle_idx
        oerr = _row_err(rows_e.double().numpy()[idx], oracle)
        line += f", exact-oracle max {oerr.max():.1e}"
    print(line)
    assert err.max() <= TOL, f"{tag}: fast vs exact {err.max():.2e}"
    if deferred is not None:
        assert identical >= deferred, f"{tag}: {identical} identical rows < {deferred} deferred"
    if oracle is not None:
        assert oerr.max() <= TOL, f"{tag}: exact vs oracle {oerr.max():.2e}"
    return deferred, err.max()


def _noisy_sphere(n, seed, noise=0.1):
    pts, dirs = synthetic.bumpy_sphere(n, seed=seed)
    rng = np.random.default_rng(seed + 1)
    nrm = dirs + noise * rng.normal(size=dirs.shape)
    return pts, nrm / np.linalg.norm(nrm, axis=1, keepdims=True)


@pytest.fixture(scope="module")
def sphere200k():
    return _noisy_sphere(200_000, 41)


# ---- a. realistic clouds, fused driver ------------------------------------------------------------------------------
@pytest.mark.parametrize("spacings,stride", [(5.0, 4), (8.0, 20)])
def test_fused_realistic(monkeypatch, sphere200k, spacings, stride):
    pts, nrm = sphere200k
    radius = spacings * synthetic.mean_spacing(pts.shape[0])
    queries = np.ascontiguousarray(pts[::stride])
    grid = _grid(pts, nrm, radius)
    sub = np.random.default_rng(2).choice(queries.shape[0], 600, replace=False)
    for dtype in (torch.float32, torch.float64):
        for normalize in (True, False):
            fast, exact = _twice(monkeypatch, lambda: _fused(grid, queries, radius, dtype, normalize))
            want = None
            if dtype == torch.float32:  # the oracle on the device's frames, on a sample
                want = _oracle_rows(pts, nrm, queries[sub], radius, exact[1].numpy()[sub], normalize)
            deferred, _ = _check(f"sphere K~{'70' if spacings == 5 else '190'} {dtype} norm={normalize}", fast, exact,
                                 want, sub)
            if spacings == 5.0:  # the fast kernel decides nearly everything (DESIGN.md: 0.6 % handed over at C2)
                assert deferred < 0.02 * queries.shape[0]
            else:  # K ~ 190 > 128: handed over
                assert deferred > 0.9 * queries.shape[0]
    grid.close()


# ---- b. adversarial clouds, fused driver ----------------------------------------------------------------------------
@pytest.mark.parametrize("tilt", [(0.0, 0.0), (0.3, -0.2)])
def test_fused_planar(monkeypatch, tilt):
    """Z is 0 or rounding noise: every query is handed over; the float64 rows follow the oracle (kAcosHalfPiMax,
    frame_dot in sf_math.cuh)."""
    rng = np.random.default_rng(8)
    n = 40_000
    xy = rng.uniform(0, 1, (n, 2))
    pts = np.column_stack([xy, tilt[0] * xy[:, 0] + tilt[1] * xy[:, 1]])
    nrm = np.array([-tilt[0], -tilt[1], 1.0]) + 0.1 * rng.normal(size=(n, 3))
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    radius = 5.0 / np.sqrt(n)
    queries = np.ascontiguousarray(pts[::40])
    grid = _grid(pts, nrm, radius)
    fast, exact = _twice(monkeypatch, lambda: _fused(grid, queries, radius))
    want = _oracle_rows(pts, nrm, queries, radius, exact[1].numpy())
    deferred, _ = _check(f"plane {tilt}", fast, exact, want)
    assert deferred == queries.shape[0] and torch.equal(fast[0], exact[0])
    grid.close()


def test_fused_cubic_lattice_ties(monkeypatch):
    """Exact distance ties (the fast kernel must defer them through amb_margin); the rows are deterministic."""
    h = 2.0**-6
    g = np.arange(36) * h
    pts = np.stack(np.meshgrid(g, g, g, indexing="ij"), axis=-1).reshape(-1, 3) + 0.5
    rng = np.random.default_rng(9)
    nrm = rng.normal(size=pts.shape)
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    radius = 2.5 * h
    queries = np.ascontiguousarray(pts[::7])
    grid = _grid(pts, nrm, radius)
    fast, exact = _twice(monkeypatch, lambda: _fused(grid, queries, radius))
    _check("cubic lattice", fast, exact)
    fast2, exact2 = _twice(monkeypatch, lambda: _fused(grid, queries, radius))
    assert torch.equal(fast[0], fast2[0]) and torch.equal(exact[0], exact2[0]), "rows are not deterministic"
    grid.close()


def test_fused_duplicates_and_normal_lengths(monkeypatch):
    """Exact duplicates of the query points (counted in K and in the votes, not in `positive`), and normals with
    |n|^2 on both sides of the fast kernel's 1.001 (kFastN2)."""
    pts, nrm = _noisy_sphere(60_000, 43)
    rng = np.random.default_rng(10)
    qi = rng.choice(pts.shape[0], 3000, replace=False)
    dup = qi[: 1500]
    scale = rng.choice([1.0, 1.001 * (1 - 1e-6), 1.001, 1.001 * (1 + 1e-6), 1.002, 0.998], pts.shape[0])
    nrm = nrm * np.sqrt(scale)[:, None]
    # a copy keeps its point's normal: for the other queries the copies are an exact distance tie, which the reference
    # breaks by its unstable argsort (DESIGN.md §2), and identical copies make the winner irrelevant
    pts_d = np.concatenate([pts, pts[dup], pts[dup[:500]]])
    nrm_d = np.concatenate([nrm, nrm[dup], nrm[dup[:500]]])
    radius = 5.0 * synthetic.mean_spacing(pts.shape[0])
    queries = np.ascontiguousarray(pts[qi])
    grid = _grid(pts_d, nrm_d, radius)
    fast, exact = _twice(monkeypatch, lambda: _fused(grid, queries, radius))
    sub = np.arange(0, 3000, 3)
    want = _oracle_rows(pts_d, nrm_d, queries[sub], radius, exact[1].numpy()[sub])
    _check("duplicates + |n|^2 ~ 1.001", fast, exact, want, sub)
    grid.close()


# ---- c. caller-provided lists with frames chosen by the test ---------------------------------------------------------
def _with_outside_clusters(pts, nrm, r, seed=14):
    """Four queries 0.3 r outside the bounding box of the probe clouds (cell coordinate -1 or dims, shot_rel32's
    wrapped cell codes), each with 30 neighbours inside the box, between the rows and columns of probe clusters."""
    rng = np.random.default_rng(seed)
    lo, hi = pts.min(axis=0), pts.max(axis=0)
    mid = 1.0 + 2.0 * r
    queries = np.array([[lo[0] - 0.3 * r, mid, 0.0], [hi[0] + 0.3 * r, mid, 0.0], [mid, lo[1] - 0.3 * r, 0.0],
                        [mid, hi[1] + 0.3 * r, 0.0]])
    inward = np.array([[1.0, 0.0, 0.0], [-1.0, 0.0, 0.0], [0.0, 1.0, 0.0], [0.0, -1.0, 0.0]])
    new_p, new_n = [], []
    for q, d in zip(queries, inward):
        off = rng.normal(size=(30, 3)) * [1.0, 1.0, 0.3]
        off -= (off @ d)[:, None] * d
        off *= (rng.uniform(0.05, 0.6, 30) * r / np.linalg.norm(off, axis=1))[:, None]
        off += rng.uniform(0.35, 0.6, 30)[:, None] * r * d
        new_p.append(q + off)
        n = rng.normal(size=(30, 3))
        new_n.append(n / np.linalg.norm(n, axis=1, keepdims=True))
    return np.concatenate([pts, *new_p]), np.concatenate([nrm, *new_n]), queries


def test_caller_lists_on_decision_boundaries(monkeypatch):
    pts, nrm, queries, frames, kinds = shot_probes.probe_set()
    r = shot_probes.RADIUS
    lo, hi = pts.min(axis=0), pts.max(axis=0)
    pts, nrm, extra = _with_outside_clusters(pts, nrm, r)
    assert np.array_equal(pts.min(axis=0), lo) and np.array_equal(pts.max(axis=0), hi)
    perms = shot_probes.signed_permutations()
    queries = np.concatenate([queries, extra])
    frames = np.concatenate([frames, np.array([perms[5 * i] for i in range(extra.shape[0])])])
    counts = np.array([len(nb) for nb in KDTree(pts).query_radius(extra, r)])
    assert (counts >= 30).all(), counts  # outside the box, neighbourhoods not empty
    want = {nz: _oracle_rows(pts, nrm, queries, r, frames, nz) for nz in (True, False)}
    for grid_radius in (r, 4 * r):  # the margin e_abs scales with the cell edge
        grid = _grid(pts, nrm, grid_radius)
        for normalize in (True, False):
            for dtype in (torch.float32, torch.float64):
                fast, exact = _twice(monkeypatch, lambda: _caller(grid, queries, r, frames, dtype, normalize))
                _check(f"probes grid {grid_radius / r:g}r {dtype} norm={normalize}", fast, exact, want[normalize])
        grid.close()


# ---- d. neighbour-count edges, both paths -----------------------------------------------------------------------------
def _clusters(sizes, duplicate, r=2.0**-4, seed=12):
    rng = np.random.default_rng(seed)
    pts, nrm, queries = [], [], []
    for i, k in enumerate(sizes):
        centre = np.array([1.0 + 4 * r * i, 1.0, 0.5])
        m = k - 1 - int(duplicate and k >= 2)
        off = rng.normal(size=(max(m, 0), 3))
        off *= (rng.uniform(0.05, 0.95, max(m, 0)) * r / np.linalg.norm(off, axis=1))[:, None]
        off[:, 2] *= 0.3
        block = [centre[None], centre + off] + ([centre[None]] if duplicate and k >= 2 else [])
        pts += block
        n = rng.normal(size=(k, 3)) * 0.2 + [0.0, 0.0, 1.0]
        nrm.append(n / np.linalg.norm(n, axis=1, keepdims=True))
        queries.append(centre)
    return np.concatenate(pts), np.concatenate(nrm), np.array(queries), r


@pytest.mark.parametrize("duplicate", [False, True])
def test_neighbour_count_edges(monkeypatch, duplicate):
    sizes = [1, 2, MIN_NB - 1, MIN_NB, MIN_NB + 1, MIN_NB + 2, 31, 32, 33, 63, 64, 65, 127, 128, 129, 130, 256]
    pts, nrm, queries, r = _clusters(sizes, duplicate)
    counts = np.array([len(nb) for nb in KDTree(pts).query_radius(queries, r)])
    assert np.array_equal(counts, sizes)
    grid = _grid(pts, nrm, r)
    fast, exact = _twice(monkeypatch, lambda: _fused(grid, queries, r))
    frames = exact[1].numpy()
    _check(f"cluster sizes fused dup={duplicate}", fast, exact, _oracle_rows(pts, nrm, queries, r, frames))
    fast, exact = _twice(monkeypatch, lambda: _caller(grid, queries, r, frames))
    _check(f"cluster sizes caller dup={duplicate}", fast, exact, _oracle_rows(pts, nrm, queries, r, frames))
    grid.close()


# ---- e. schedule and instantiations ------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def mixed():
    """A sphere (ordinary queries), a tilted plane patch (handed over), dense blobs (> 128 neighbours) and points off
    the cloud (empty), with the queries ordered so that each warp's consecutive queries cycle through the four kinds
    (the default fast grid has 148 x 2 x 8 = 2368 warps)."""
    rng = np.random.default_rng(13)
    n = 150_000
    sph, sn = _noisy_sphere(n, 44)
    radius = 5.0 * synthetic.mean_spacing(n)
    xy = rng.uniform(0, 0.6, (6000, 2))
    plane = np.column_stack([xy[:, 0] + 2.0, xy[:, 1], 0.3 * xy[:, 0] - 0.2 * xy[:, 1]])
    pn = np.tile(np.array([-0.3, 0.2, 1.0]) / np.linalg.norm([-0.3, 0.2, 1.0]), (plane.shape[0], 1))
    blob_c = sph[rng.choice(n, 64, replace=False)] * 1.0
    blobs = (blob_c[:, None, :] + rng.normal(size=(64, 200, 3)) * 0.15 * radius).reshape(-1, 3)
    bn = rng.normal(size=blobs.shape)
    bn /= np.linalg.norm(bn, axis=1, keepdims=True)
    pts = np.concatenate([sph, plane, blobs])
    nrm = np.concatenate([sn, pn, bn])
    kinds = [sph[rng.choice(n, 20000, replace=False)], plane[rng.choice(plane.shape[0], 20000)],
             blob_c[rng.integers(0, 64, 20000)], sph[rng.choice(n, 20000)] * 1.5]
    warps = 148 * 2 * 8
    q = np.empty((60000, 3))
    idx = np.arange(60000)
    for k in range(4):
        sel = (idx // warps) % 4 == k
        q[sel] = kinds[k][: sel.sum()]
    return pts, nrm, np.ascontiguousarray(q), radius


@pytest.mark.parametrize("nq", [1, 7, 2367, 2368, 2369, 60000])
def test_schedule_mixed_queries(monkeypatch, mixed, nq):
    pts, nrm, queries, radius = mixed
    queries = np.ascontiguousarray(queries[:nq])
    grid = _grid(pts, nrm, radius)
    fast, exact = _twice(monkeypatch, lambda: _fused(grid, queries, radius))
    _check(f"mixed nq={nq}", fast, exact)
    grid.close()


def test_float64_output_is_the_float32_rows_widened(monkeypatch, mixed):
    pts, nrm, queries, radius = mixed
    queries = np.ascontiguousarray(queries[:12000])
    grid = _grid(pts, nrm, radius)
    for exact_flag in (None, "1"):
        if exact_flag:
            monkeypatch.setenv("SF_SHOT_EXACT", "1")
        f32 = _fused(grid, queries, radius, torch.float32)
        f64 = _fused(grid, queries, radius, torch.float64)
        assert torch.equal(f32[0].double(), f64[0]) and torch.equal(f32[1], f64[1]), f"fused, SF_SHOT_EXACT={exact_flag}"
        frames = f32[1].numpy()
        c32 = _caller(grid, queries, radius, frames, torch.float32)
        c64 = _caller(grid, queries, radius, frames, torch.float64)
        assert torch.equal(c32[0].double(), c64[0]), f"caller lists, SF_SHOT_EXACT={exact_flag}"
        monkeypatch.delenv("SF_SHOT_EXACT", raising=False)
    grid.close()


# ---- f. power-of-two scale and a large translation --------------------------------------------------------------------
def test_power_of_four_scale_changes_nothing(monkeypatch):
    """Every float64 and float32 operation of both kernels and of the grid commutes with scaling by 4^k while the
    values stay normal: rows and frames are bit for bit those at k = 0."""
    pts, nrm = _noisy_sphere(40_000, 45)
    radius = 5.0 * synthetic.mean_spacing(pts.shape[0])
    queries = np.ascontiguousarray(pts[::8])
    ppts, pnrm, pq, pframes, _ = shot_probes.probe_set()
    pr = shot_probes.RADIUS

    def run(s):
        grid = _grid(pts * s, nrm, radius * s)
        fused = _twice(monkeypatch, lambda: _fused(grid, queries * s, radius * s))
        grid.close()
        pgrid = _grid(ppts * s, pnrm, pr * s)
        caller = _twice(monkeypatch, lambda: _caller(pgrid, pq * s, pr * s, pframes))
        pgrid.close()
        return fused, caller

    base = run(1.0)
    for k in (-20, -10, 10, 20):
        got = run(4.0**k)
        for (b_fast, b_exact), (g_fast, g_exact), what in zip(base, got, ("fused", "caller")):
            for b, g, path in ((b_fast, g_fast, "fast"), (b_exact, g_exact, "exact")):
                assert torch.equal(b[0], g[0]), f"4^{k}: {what} {path} rows differ"
                if b[1] is not None:
                    assert torch.equal(b[1], g[1]), f"4^{k}: {what} {path} frames differ"
    shift = 2.0**30
    grid = _grid(pts + shift, nrm, radius)
    fast, exact = _twice(monkeypatch, lambda: _fused(grid, queries + shift, radius))
    _check("translated by 2^30", fast, exact)
    grid.close()
