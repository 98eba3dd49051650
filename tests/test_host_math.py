"""
CPU check of the arithmetic the sm_100a kernels inline (shot_fpfh_b200/csrc/sf_math.cuh), through its g++ host
instantiation tests/host_math/libhost_math.so, against the oracle (which is pinned bit-exactly to the reference).
This is what can be verified about the kernels without a GPU: bin decisions, interpolation weights, the
winner-table formulation of the reference's last-writer-wins binning, the Jacobi eigen-solver, the FPFH features
and the NumPy-compatible histogram binning. Tolerance for descriptors: 1e-4 relative L2 per row (north_star).
"""

import ctypes
import os

import numpy as np
import pytest
from conftest import ROOT, rel_l2

from oracle import fpfh_oracle, shot_oracle
from shot_fpfh_b200 import synthetic
from sklearn.neighbors import KDTree

DP = ctypes.POINTER(ctypes.c_double)


def _p(a):
    return a.ctypes.data_as(DP)


@pytest.fixture(scope="module")
def hm():
    lib = ctypes.CDLL(os.path.join(ROOT, "tests", "host_math", "libhost_math.so"))
    lib.hm_rdist3.restype = ctypes.c_double
    lib.hm_rdist3.argtypes = [ctypes.c_double] * 3
    lib.hm_azimuth_octant.argtypes = [ctypes.c_double] * 2
    lib.hm_histogram_bin.argtypes = [ctypes.c_double, DP, ctypes.c_int]
    lib.hm_histogram_bin_scaled.argtypes = [ctypes.c_double, DP, ctypes.c_int]
    lib.hm_theta_bin.argtypes = [ctypes.c_double, ctypes.c_double, DP, ctypes.c_int]
    lib.hm_theta_bin_float64.argtypes = [ctypes.c_double, ctypes.c_double, DP, ctypes.c_int]
    lib.hm_eigh3.argtypes = [DP, DP, DP]
    lib.hm_lrf.argtypes = [DP, DP, ctypes.c_int, ctypes.c_double, DP]
    lib.hm_shot_descriptor.argtypes = [DP, DP, DP, ctypes.c_int, ctypes.c_double, DP, ctypes.c_int, ctypes.c_int,
                                       ctypes.POINTER(ctypes.c_float)]
    lib.hm_spfh_counts.argtypes = [DP, DP, DP, DP, ctypes.c_int, ctypes.c_int, ctypes.c_int, DP,
                                   ctypes.POINTER(ctypes.c_int)]
    lib.hm_fpfh_fast_check.argtypes = [ctypes.c_long, DP, DP, DP, ctypes.c_int, DP, ctypes.POINTER(ctypes.c_long),
                                       ctypes.POINTER(ctypes.c_long)]
    return lib


@pytest.fixture(scope="module")
def cloud():
    n = 6000
    pts, normals = synthetic.bumpy_sphere(n, seed=5)
    rng = np.random.default_rng(0)
    normals = normals + 0.2 * rng.normal(size=normals.shape)
    normals /= np.linalg.norm(normals, axis=1, keepdims=True)
    radius = 5.0 * synthetic.mean_spacing(n)
    return pts, normals, radius, KDTree(pts)


def test_eigh3_matches_lapack(hm):
    rng = np.random.default_rng(1)
    for trial in range(500):
        a = rng.normal(size=(20, 3)) * rng.uniform(0.01, 1.0, size=3) * 10.0 ** rng.integers(-4, 2)
        m = a.T @ a / 20
        packed = np.array([m[0, 0], m[0, 1], m[0, 2], m[1, 1], m[1, 2], m[2, 2]])
        ev, vec = np.zeros(3), np.zeros(9)
        hm.hm_eigh3(_p(packed), _p(ev), _p(vec))
        w, v = np.linalg.eigh(m)
        assert np.allclose(ev, w, rtol=1e-12, atol=1e-14 * np.abs(w).max())
        vec = vec.reshape(3, 3)
        for c in range(3):
            gap = min(abs(w[c] - w[o]) for o in range(3) if o != c) / max(np.abs(w).max(), 1e-300)
            if gap > 1e-6:
                assert abs(abs(vec[c] @ v[:, c]) - 1.0) < 1e-10 / gap * 1e-4 + 1e-12


def test_static_dsteqr_is_the_transcribed_dsteqr_bit_for_bit(hm):
    """sf_eigh3.cuh: the kernels run dsteqr with every index resolved at compile time (blocks of 1, 2, 3; QL or QR);
    the loop-for-loop transcription of LAPACK's routine is kept beside it as its specification."""
    rng = np.random.default_rng(11)
    n = 200_000
    d = rng.normal(size=(n, 3)) * 10.0 ** rng.integers(-6, 3, size=(n, 1))
    e = rng.normal(size=(n, 2)) * 10.0 ** rng.integers(-6, 3, size=(n, 1))
    kind = rng.integers(0, 12, size=n)
    d[kind == 0] = np.abs(d[kind == 0])                      # positive diagonals (covariances)
    e[kind == 1, 0] = 0.0                                    # exact splits
    e[kind == 2, 1] = 0.0
    e[kind == 3] = 0.0
    e[kind == 4, 0] *= 1e-17                                 # negligible off-diagonal entries (the eps tests)
    e[kind == 5, 1] *= 1e-17
    e[kind == 6] *= 1e-9                                     # nearly diagonal: deflation inside the iterations
    d[kind == 7] = d[kind == 7][:, :1]                       # equal diagonal entries
    d[kind == 8, 2] = d[kind == 8, 0]                        # |d3| == |d1|: the QL / QR choice at its boundary
    d[kind == 9] = 0.0                                       # zero diagonal
    d[kind == 10] *= 1e-150                                  # tiny values (safmin matters)
    e[kind == 10] *= 1e-150
    hm.hm_dsteqr3_static_vs_generic.restype = ctypes.c_long
    hm.hm_dsteqr3_static_vs_generic.argtypes = [DP, DP, ctypes.c_long]
    d, e = np.ascontiguousarray(d), np.ascontiguousarray(e)
    assert hm.hm_dsteqr3_static_vs_generic(_p(d), _p(e), n) == 0


def test_azimuth_octant_table(hm):
    g = np.load(os.path.join(ROOT, "tests", "golden", "edge_cases.npz"))
    got = [hm.hm_azimuth_octant(float(x), float(y)) for x, y in zip(g["azimuth_x"], g["azimuth_y"])]
    assert np.array_equal(got, g["azimuth_idx"])
    rng = np.random.default_rng(2)
    xy = rng.normal(size=(20000, 2))
    got = np.array([hm.hm_azimuth_octant(float(x), float(y)) for x, y in xy])
    assert np.array_equal(got, shot_oracle.azimuth_octant(xy[:, 0], xy[:, 1]))
    assert np.array_equal(got, np.floor((np.arctan2(xy[:, 1], xy[:, 0]) + np.pi) / (np.pi / 4)).astype(int))


def test_rdist_is_sklearn_order(hm):
    rng = np.random.default_rng(3)
    for d in rng.normal(size=(2000, 3)):
        sq = d * d
        assert hm.hm_rdist3(*map(float, d)) == (sq[0] + sq[1]) + sq[2]


def test_lrf_matches_oracle(hm, cloud):
    pts, _, radius, tree = cloud
    worst = 0.0
    for i in range(0, pts.shape[0], 40):
        nb = tree.query_radius(pts[i : i + 1], radius)[0]
        want = shot_oracle.local_reference_frame(pts[i], pts[nb], radius)
        got = np.zeros(9)
        hm.hm_lrf(_p(pts[i].copy()), _p(np.ascontiguousarray(pts[nb])), nb.shape[0], radius, _p(got))
        worst = max(worst, np.abs(got.reshape(3, 3) - want).max())
    assert worst < 1e-9, worst
    got = np.zeros(9)
    hm.hm_lrf(_p(pts[0].copy()), _p(np.zeros((0, 3))), 0, radius, _p(got))
    assert np.array_equal(got.reshape(3, 3), np.eye(3))


@pytest.mark.parametrize("normalize", [True, False])
def test_shot_winner_tables_match_oracle(hm, cloud, normalize):
    """The winner-table formulation (7 tables, packed 64-bit max) against the bit-exact oracle."""
    pts, normals, radius, tree = cloud
    errs = []
    for i in range(0, pts.shape[0], 12):
        nb = tree.query_radius(pts[i : i + 1], radius)[0]
        lrf = shot_oracle.local_reference_frame(pts[i], pts[nb], radius)
        want = shot_oracle.shot_descriptor(pts[i], pts[nb], normals[nb], radius, lrf, normalize, 10)
        got = np.zeros(352, dtype=np.float32)
        hm.hm_shot_descriptor(
            _p(pts[i].copy()), _p(np.ascontiguousarray(pts[nb])), _p(np.ascontiguousarray(normals[nb])), nb.shape[0],
            radius, _p(np.ascontiguousarray(lrf)), int(normalize), 10, got.ctypes.data_as(ctypes.POINTER(ctypes.c_float)),
        )
        errs.append(float(rel_l2(got.astype(np.float64), want)))
    errs = np.array(errs)
    assert errs.shape[0] == 500
    assert (errs > 1e-4).sum() == 0, f"{(errs > 1e-4).sum()} rows above 1e-4, max {errs.max():.3e}"
    assert np.median(errs) < 1e-6


def test_shot_sparse_neighbourhood_is_zero(hm, cloud):
    pts, normals, radius, tree = cloud
    nb = tree.query_radius(pts[:1], radius)[0][:8]
    got = np.ones(352, dtype=np.float32)
    hm.hm_shot_descriptor(
        _p(pts[0].copy()), _p(np.ascontiguousarray(pts[nb])), _p(np.ascontiguousarray(normals[nb])), nb.shape[0],
        radius, _p(np.eye(3)), 1, 10, got.ctypes.data_as(ctypes.POINTER(ctypes.c_float)),
    )
    assert not got.any()


# ---- the float32-filtered fast path (shot.cu::shot_fast_kernel, sf_math.cuh::shot_decide_fast) ---------------------
FP = ctypes.POINTER(ctypes.c_float)
LP = ctypes.POINTER(ctypes.c_long)


def _fast_lib(hm):
    hm.hm_shot_descriptor_fast.argtypes = [DP, DP, DP, ctypes.c_int, ctypes.c_double, DP, ctypes.c_double, DP,
                                           ctypes.c_int, ctypes.c_int, ctypes.c_int, FP, DP, LP]
    hm.hm_shot_decide_fast_check.argtypes = [ctypes.c_long, DP, FP, ctypes.c_double, ctypes.c_double, ctypes.c_int, LP]
    hm.hm_shot_trig_check.argtypes = [ctypes.c_long, FP, FP, FP]
    hm.hm_shot_trig_check.restype = ctypes.c_double
    return hm


def test_shot_polynomial_weights_match_libm(hm):
    """atan / asin polynomials of the fast path against atan2f / acosf of the exact path, on float32 inputs."""
    _fast_lib(hm)
    rng = np.random.default_rng(11)
    n = 400_000
    fx = rng.normal(size=n).astype(np.float32)
    fy = rng.normal(size=n).astype(np.float32)
    ratio = np.clip(rng.normal(scale=0.4, size=n), -1, 1).astype(np.float32)
    ratio[:1000] = np.linspace(-1, 1, 1000, dtype=np.float32)
    fx[:8] = [1, 1, 0, -1, -1, -1, 0, 1]
    fy[:8] = [0, 1, 1, 1, 0, -1, -1, -1]
    worst = hm.hm_shot_trig_check(n, fx.ctypes.data_as(FP), fy.ctypes.data_as(FP), ratio.ctypes.data_as(FP))
    assert worst < 1e-6, worst  # two float32 evaluations, each within ~3e-7 of the exact angle


@pytest.mark.parametrize("relative", [1, 0])
def test_shot_float32_decisions_never_disagree_with_float64(hm, relative):
    """
    Whenever shot_decide_fast is sure, every bin, octant, half-space and interpolation sign equals shot_decide's on
    the float64 values, for float32 inputs perturbed by up to the documented error bounds — `relative`: the fused
    driver's (8 u rho on X, Y, Z, rho), else the gathered coordinates' (24 u edge); 7 u on the cosine — including
    inputs placed on and next to every boundary.
    """
    _fast_lib(hm)
    rng = np.random.default_rng(12)
    radius, edge = 0.0177, 0.0177 * 1.001
    n = 1_500_000
    u = 2.0**-24
    rho = radius * rng.uniform(0.0, 1.0, n)
    direction = rng.normal(size=(n, 3))
    direction /= np.linalg.norm(direction, axis=1, keepdims=True)
    direction[:, 2] *= rng.choice([1.0, 1e-3, 1e-6], n)  # surfaces: Z clusters around 0
    direction /= np.linalg.norm(direction, axis=1, keepdims=True)
    xyz = direction * rho[:, None]
    cosine = np.clip(rng.normal(0.8, 0.3, n), -1.2, 1.2)
    # boundary cases: X = 0, Y = 0, |X| = |Y|, Z = 0, rho = r/2, cosine on bin centres / bin edges / the clip
    m = 200_000
    k = rng.integers(0, 7, m)
    tiny = rng.choice([0.0, 1e-12, 1e-9, 1e-8, 1e-7], m) * rng.choice([-1, 1], m) * radius
    xyz[:m][k == 0, 0] = tiny[k == 0]
    xyz[:m][k == 1, 1] = tiny[k == 1]
    sel = k == 2
    xyz[:m][sel, 1] = xyz[:m][sel, 0] * rng.choice([-1, 1], sel.sum()) + tiny[sel]
    xyz[:m][k == 3, 2] = tiny[k == 3]
    rho = np.linalg.norm(xyz, axis=1)
    sel = np.zeros(n, bool)
    sel[:m] = k == 4
    scale = (radius / 2 + np.resize(tiny, n)) / np.maximum(rho, 1e-300)
    xyz[sel] *= scale[sel, None]
    rho = np.linalg.norm(xyz, axis=1)
    sel[:] = False
    sel[:m] = k == 5
    cosine[sel] = (rng.integers(0, 23, sel.sum()) * 0.5 + 0.5) * 2 / 11 - 1 + np.resize(tiny, n)[sel] / radius
    sel[:] = False
    sel[:m] = k == 6
    cosine[sel] = rng.choice([-1.0, 1.0], sel.sum()) * (1 + np.resize(tiny, n)[sel])
    keep = rho > 0
    exact = np.ascontiguousarray(np.column_stack([xyz, cosine, rho])[keep])
    n = exact.shape[0]
    bound = (7.7 * u * exact[:, 4:5]) if relative else np.full((n, 1), 23.0 * u * edge)
    noise = rng.uniform(-1, 1, size=(n, 5)) * np.concatenate([bound, bound, bound, np.full((n, 1), 7 * u), bound], axis=1)
    approx = np.ascontiguousarray((exact + noise).astype(np.float32))
    stats = (ctypes.c_long * 3)()
    hm.hm_shot_decide_fast_check(n, _p(exact), approx.ctypes.data_as(FP), radius, edge, relative, stats)
    print(f"float32 decisions: {stats[0]} of {n} sure, {stats[1]} disagreements, largest weight gap {stats[2] * 1e-9:.2e}")
    assert stats[1] == 0
    assert stats[0] > 0.3 * n  # (a third of the samples have Z squashed into the margin, a quarter a clipped cosine)
    assert stats[2] * 1e-9 < 4e-4  # worst case of the bounds where the weights are worst conditioned (sf_math.cuh)


@pytest.mark.parametrize("shift", [None, (4.0e5, -2.5e6, 1.0e4)])
def test_shot_fast_kernel_mirror_matches_oracle(hm, cloud, shift):
    """
    The fast kernel's control flow (cell-relative float32 coordinates, votes on the raw eigenvectors, float32-filtered
    decisions, unique keys, five value sub-phases) for 500 queries against the bit-exact oracle; queries the kernel
    would hand to the exact kernel are counted. Second case: the cloud moved far from the origin.
    """
    _fast_lib(hm)
    pts, normals, radius, tree = cloud
    if shift is not None:
        pts = pts + np.array(shift)
        tree = KDTree(pts)
    origin = pts.min(axis=0)
    edge = radius * 1.001
    errs, deferred, deferred2, frame_err = [], 0, 0, 0.0
    stats = (ctypes.c_long * 2)()
    for i in range(0, pts.shape[0], 12):
        nb = tree.query_radius(pts[i : i + 1], radius)[0]
        rel = pts[nb] - pts[i]
        w = radius - np.linalg.norm(rel, axis=1)
        _, vec = np.linalg.eigh(rel.T @ (rel * w[:, None]) / w.sum())
        raw = np.ascontiguousarray(np.concatenate([vec[:, 2], vec[:, 0]]))
        lrf = shot_oracle.local_reference_frame(pts[i], pts[nb], radius)
        want = shot_oracle.shot_descriptor(pts[i], pts[nb], normals[nb], radius, lrf, True, 10)
        got = np.zeros(352, dtype=np.float32)
        frame = np.zeros(9)
        rc = hm.hm_shot_descriptor_fast(
            _p(pts[i].copy()), _p(np.ascontiguousarray(pts[nb])), _p(np.ascontiguousarray(normals[nb])), nb.shape[0],
            radius, _p(origin.copy()), edge, _p(raw), 1, 1, 10, got.ctypes.data_as(FP), _p(frame), stats)  # fused mode
        if rc:
            deferred += 1
            continue
        frame_err = max(frame_err, np.abs(frame.reshape(3, 3) - lrf).max())
        errs.append(float(rel_l2(got.astype(np.float64), want)))
        # the same query from the grid's cell-relative coordinates with the final frame (sf_shot_descriptor's mode)
        got2 = np.zeros(352, dtype=np.float32)
        rc2 = hm.hm_shot_descriptor_fast(
            _p(pts[i].copy()), _p(np.ascontiguousarray(pts[nb])), _p(np.ascontiguousarray(normals[nb])), nb.shape[0],
            radius, _p(origin.copy()), edge, _p(np.ascontiguousarray(lrf)), 0, 1, 10, got2.ctypes.data_as(FP), None, None)
        deferred2 += rc2
        assert rc2 or float(rel_l2(got2.astype(np.float64), want)) < 1e-5
    errs = np.array(errs)
    print(f"fast mirror: {errs.shape[0]} rows kept, {deferred} handed over, median {np.median(errs):.2e}, max "
          f"{errs.max():.2e}; unsure neighbours {stats[1]} of {stats[0]}; frame error {frame_err:.1e}")
    print(f"caller-list mode: {deferred2} more handed over")
    assert errs.shape[0] + deferred == 500 and deferred < 40 and deferred2 < 40
    assert (errs > 1e-5).sum() == 0, f"{(errs > 1e-5).sum()} rows above 1e-5, max {errs.max():.3e}"
    assert frame_err < 1e-12


def test_histogram_bin_is_numpy(hm):
    rng = np.random.default_rng(4)
    for n_bins in (5, 11, 7):
        edges = fpfh_oracle.bin_edges(n_bins)
        for f in range(3):
            e = np.ascontiguousarray(edges[f])
            lo, hi = e[0], e[-1]
            vals = np.concatenate([
                rng.uniform(lo * 1.2, hi * 1.2, 4000), e, np.nextafter(e, np.inf), np.nextafter(e, -np.inf),
                [np.nan, np.inf, -np.inf],
            ])
            got = np.array([hm.hm_histogram_bin(float(v), _p(e), n_bins) for v in vals])
            finite = np.isfinite(vals)
            assert np.array_equal(got[finite], fpfh_oracle.bin_index(vals[finite], e))
            assert (got[~finite] == -1).all()
            counts = np.bincount(got[got >= 0], minlength=n_bins)
            assert np.array_equal(counts, np.histogram(vals[finite], bins=n_bins, range=(lo, hi))[0])


def test_filtered_theta_bin_equals_float64_bin(hm):
    """sf_math.cuh::fpfh_theta_bin (float32 angle unless it lands near an edge) == bin of the float64 atan2, also
    for angles ON the edges, one ulp / 1e-9 / 1e-6 / 2e-5 rad around them, the +-pi/2 ends and the axes."""
    rng = np.random.default_rng(9)
    for n_bins in (5, 11, 16):
        e = np.ascontiguousarray(np.linspace(-np.pi / 2, np.pi / 2, n_bins + 1))
        angles = [rng.uniform(-np.pi, np.pi, 20000)]
        for eps in (0.0, 1e-16, 1e-12, 1e-9, 1e-7, 1e-6, 9e-6, 1.1e-5, 2e-5):
            angles += [e + eps, e - eps]
        angles = np.concatenate(angles)
        radii = 10.0 ** rng.uniform(-6, 2, angles.shape[0])
        ny, nx = radii * np.sin(angles), radii * np.cos(angles)
        extra = np.array([[0.0, 1.0], [0.0, -1.0], [1.0, 0.0], [-1.0, 0.0], [0.0, 0.0], [-0.0, -1.0], [1e-40, 1e-40],
                          [1e-300, -1e-300]])
        ny, nx = np.concatenate([ny, extra[:, 0]]), np.concatenate([nx, extra[:, 1]])
        for y, x in zip(ny, nx):
            # against the same libm atan2 (np.arctan2 may differ from it by an ulp, which decides an angle that is
            # exactly ON an edge)
            want = hm.hm_theta_bin_float64(float(y), float(x), _p(e), n_bins)
            assert hm.hm_theta_bin(float(y), float(x), _p(e), n_bins) == want, (y, x)
            theta = float(np.arctan2(y, x))
            assert hm.hm_histogram_bin_scaled(theta, _p(e), n_bins) == hm.hm_histogram_bin(theta, _p(e), n_bins)


def _unit(v):
    return v / np.linalg.norm(v, axis=1, keepdims=True)


@pytest.mark.parametrize("n_bins", [5, 11, 4, 16])
def test_float32_filtered_bins_never_disagree_with_float64(hm, n_bins):
    """sf_math.cuh::fpfh_bins_fast: whenever the float32 filter accepts a pair, its three bins are the float64
    path's. Random pairs at several scales, non-unit normals, and pairs built to put phi / theta / alpha ON a bin
    edge or 1e-16 .. 1e-5 away from it (the filter must then either agree or decline)."""
    rng = np.random.default_rng(21)
    edges = np.ascontiguousarray(fpfh_oracle.bin_edges(n_bins))
    rels, us, njs = [], [], []
    m = 60_000
    for scale_c, scale_n, spread in ((0.02, 1.0, 0.3), (1.0, 1.0, 3.0), (5.0, 0.5, 0.05), (1e-4, 2.0, 1.0), (0.02, 1.0, 0.0)):
        u = _unit(rng.normal(size=(m, 3))) * scale_n
        nj = _unit(u / scale_n + spread * rng.normal(size=(m, 3))) * rng.choice([1.0, scale_n], size=(m, 1))
        rel = rng.normal(size=(m, 3)) * scale_c
        rels.append(rel); us.append(u); njs.append(nj)
    # phi = (rel . u) / |rel| on / next to every edge: rel = cos(phi) u^ + sin(phi) t, u unit
    for delta in (0.0, 1e-16, 1e-12, 1e-9, 1e-8, 1e-7, 1e-6, 3e-6, 1e-5, -1e-16, -1e-9, -1e-7, -1e-6, -1e-5):
        for e in edges[1]:
            k = 200
            u = _unit(rng.normal(size=(k, 3)))
            t = _unit(np.cross(u, rng.normal(size=(k, 3))))
            c = np.clip(e + delta, -1.0, 1.0)
            rel = (c * u + np.sqrt(max(0.0, 1.0 - c * c)) * t) * 10.0 ** rng.uniform(-3, 0, size=(k, 1))
            rels.append(rel); us.append(u); njs.append(_unit(u + 0.2 * rng.normal(size=(k, 3))))
    # theta = atan2(nj . w, nj . u) on / next to every edge: nj = cos(theta) u + sin(theta) w^, w = u x (rel x u)
    for delta in (0.0, 1e-16, 1e-9, 1e-7, 1e-6, 3e-6, 1e-5, -1e-9, -1e-7, -1e-6, -1e-5):
        for e in edges[2]:
            k = 200
            u = _unit(rng.normal(size=(k, 3)))
            rel = rng.normal(size=(k, 3))
            w = np.cross(u, np.cross(rel, u))
            theta = e + delta
            # ny = nj . w = sin(theta) |w| s, nx = cos(theta) s  with nj = s (cos(theta) u + sin(theta) w / |w|^2)
            nj = np.cos(theta) * u + np.sin(theta) * w / np.sum(w * w, axis=1, keepdims=True)
            rels.append(rel); us.append(u); njs.append(nj)
    # alpha = (rel x u) . nj == 0 up to rounding (an edge when n_bins is even): nj in the plane of rel and u
    k = 5000
    u = _unit(rng.normal(size=(k, 3)))
    rel = rng.normal(size=(k, 3)) * 0.02
    nj = _unit(u + rng.uniform(-1, 1, size=(k, 1)) * rel)
    rels.append(rel); us.append(u); njs.append(nj)
    # degenerate: zero and denormal offsets, zero normals, huge offsets
    rels.append(np.array([[0.0, 0.0, 0.0], [1e-200, 0.0, 0.0], [1e-20, 1e-20, 0.0], [1e20, 0.0, 0.0], [0.1, 0.0, 0.0]]))
    us.append(np.array([[0.0, 0.0, 1.0]] * 4 + [[0.0, 0.0, 0.0]]))
    njs.append(np.array([[0.0, 0.0, 1.0]] * 3 + [[0.0, 1.0, 0.0], [0.0, 0.0, 0.0]]))
    rel, u, nj = (np.ascontiguousarray(np.concatenate(a)) for a in (rels, us, njs))
    stats = (ctypes.c_long * 2)()
    first_bad = ctypes.c_long(-1)
    hm.hm_fpfh_fast_check(rel.shape[0], _p(rel), _p(u), _p(nj), n_bins, _p(edges), stats, ctypes.byref(first_bad))
    assert stats[1] == 0, (first_bad.value, rel[first_bad.value], u[first_bad.value], nj[first_bad.value])
    assert stats[0] > 0.7 * 5 * m  # and the filter decides the generic pairs (alpha == 0 is an edge when n_bins is even)


@pytest.mark.parametrize("n_bins,decorrelated", [(5, False), (11, True), (11, False)])
def test_spfh_counts_match_oracle(hm, cloud, n_bins, decorrelated):
    pts, normals, radius, tree = cloud
    edges = np.ascontiguousarray(fpfh_oracle.bin_edges(n_bins))
    width = 3 * n_bins if decorrelated else n_bins**3
    mismatched = 0
    for i in range(0, pts.shape[0], 15):
        nb = tree.query_radius(pts[i : i + 1], radius)[0]
        a, p, t = fpfh_oracle.pair_features(pts[i], normals[i], pts[nb], normals[nb])
        want = fpfh_oracle.spfh_row(a, p, t, nb.shape[0], n_bins, decorrelated, edges) * nb.shape[0]
        hist = np.zeros(width, dtype=np.int32)
        hm.hm_spfh_counts(
            _p(pts[i].copy()), _p(normals[i].copy()), _p(np.ascontiguousarray(pts[nb])),
            _p(np.ascontiguousarray(normals[nb])), nb.shape[0], n_bins, int(decorrelated), _p(edges),
            hist.ctypes.data_as(ctypes.POINTER(ctypes.c_int)),
        )
        mismatched += int(not np.array_equal(hist, np.rint(want).astype(np.int32)))
    assert mismatched == 0


# ---- planar neighbourhoods and hand-built boundary probes (oracle/shot_probes.py) -----------------------------------
def test_arccos_half_pi_window_is_numpys(hm):
    """sf_math.cuh::kAcosHalfPiMax is the largest Z / rho > 0 for which np.arccos returns exactly np.pi / 2 (the
    reference then writes `lower` = 0 although the neighbour is binned in the upper half)."""
    from oracle import shot_probes

    hm.hm_acos_half_pi_max.restype = ctypes.c_double
    lo, hi = 1e-18, 1e-15  # arccos(lo) == pi/2 > arccos(hi): bisect on the doubles between them
    assert np.arccos(lo) == np.pi / 2 and np.arccos(hi) < np.pi / 2
    lo_i, hi_i = np.float64(lo).view(np.int64), np.float64(hi).view(np.int64)
    while hi_i - lo_i > 1:
        mid = (lo_i + hi_i) // 2
        if np.arccos(np.int64(mid).view(np.float64)) == np.pi / 2:
            lo_i = mid
        else:
            hi_i = mid
    window = float(np.int64(lo_i).view(np.float64))
    assert window == hm.hm_acos_half_pi_max() == shot_probes.A_HALF_PI_MAX
    assert np.arccos(np.nextafter(window, 1.0)) < np.pi / 2
    assert np.arccos(-window) > np.pi / 2  # below zero the window is narrower, and Z <= 0 takes the other branch


def test_numpy_matmul_rounds_like_frame_dot(hm):
    """The oracle's `rel @ lrf` equals sf_math.cuh::frame_dot bit for bit (fused multiply-adds, k = 0, 1, 2): on a
    plane the sign of Z is rounding noise and picks the elevation bin."""
    hm.hm_frame_local.argtypes = [DP, ctypes.c_long, DP, DP]
    rng = np.random.default_rng(31)
    n = 20000
    xy = rng.uniform(0, 1, (n, 2))
    for rel in (rng.normal(size=(n, 3)), np.column_stack([xy, 0.3 * xy[:, 0] - 0.2 * xy[:, 1]]) - [0.5, 0.5, 0.05]):
        rel = np.ascontiguousarray(rel)
        frame = shot_oracle.local_reference_frame(np.zeros(3), rel[:200], 0.1)
        got = np.zeros_like(rel)
        hm.hm_frame_local(_p(rel), n, _p(np.ascontiguousarray(frame)), _p(got))
        assert np.array_equal(got, rel @ frame)


def _host_row(hm, point, nbrs, normals, radius, frame, normalize=True, min_nb=10):
    got = np.zeros(352, dtype=np.float32)
    hm.hm_shot_descriptor(
        _p(np.ascontiguousarray(point)), _p(np.ascontiguousarray(nbrs)), _p(np.ascontiguousarray(normals)),
        nbrs.shape[0], radius, _p(np.ascontiguousarray(frame)), int(normalize), min_nb, got.ctypes.data_as(FP))
    return got.astype(np.float64)


@pytest.mark.parametrize("tilt", [(0.0, 0.0), (0.3, -0.2)])
def test_shot_planar_neighbourhoods_match_oracle(hm, tilt):
    """On a plane every Z is 0 or rounding noise: the float64 path (what the fast kernel hands such queries to) must
    follow the oracle there too, including Z / rho inside the arccos window (sf_math.cuh::kAcosHalfPiMax)."""
    rng = np.random.default_rng(7)
    n = 20000
    xy = rng.uniform(0, 1, (n, 2))
    pts = np.column_stack([xy, tilt[0] * xy[:, 0] + tilt[1] * xy[:, 1]])
    normals = np.array([-tilt[0], -tilt[1], 1.0]) + 0.1 * rng.normal(size=(n, 3))
    normals /= np.linalg.norm(normals, axis=1, keepdims=True)
    radius = 5.0 / np.sqrt(n)
    tree = KDTree(pts)
    errs = []
    for i in range(0, n, 67):
        nb = tree.query_radius(pts[i : i + 1], radius)[0]
        lrf = shot_oracle.local_reference_frame(pts[i], pts[nb], radius)
        want = shot_oracle.shot_descriptor(pts[i], pts[nb], normals[nb], radius, lrf, True, 10)
        errs.append(float(rel_l2(_host_row(hm, pts[i], pts[nb], normals[nb], radius, lrf), want)))
    errs = np.array(errs)
    print(f"plane {tilt}: {errs.shape[0]} rows, median {np.median(errs):.1e}, max {errs.max():.1e}")
    assert errs.max() <= 1e-5


def test_shot_boundary_probes_match_oracle(hm):
    """oracle/shot_probes.py: a neighbour on (and 1 ulp .. 1e-5 r off) every decision boundary, frames that copy
    coordinates exactly: the float64 path equals the oracle to 1e-5 on every row."""
    from oracle import shot_probes

    pts, normals, queries, frames, kinds = shot_probes.probe_set()
    radius = shot_probes.RADIUS
    tree = KDTree(pts)
    worst = {}
    for q, frame, kind in zip(queries, frames, kinds):
        nb = tree.query_radius(q[None], radius)[0]
        for normalize in (True, False):
            want = shot_oracle.shot_descriptor(q, pts[nb], normals[nb], radius, frame, normalize, 10)
            assert want.any()
            err = float(rel_l2(_host_row(hm, q, pts[nb], normals[nb], radius, frame, normalize), want))
            worst[kind] = max(worst.get(kind, 0.0), err)
    print({k: f"{v:.1e}" for k, v in worst.items()})
    assert max(worst.values()) <= 1e-5, worst
