"""
CPU: the orientation oracle (oracle/orientation_oracle.py, the specification of descriptors.orient_normals) — held to
its stored outputs, checked on hand-built graphs with known answers, and its Borůvka form (the device algorithm) held
to Kruskal + propagation on random graphs. Also the public function's signature and its refusal to run without a
device.
"""

import inspect

import numpy as np
import pytest
import torch
from conftest import load_golden

from oracle import orientation_oracle as oo
from oracle.make_orient_pins import K, ORIENT_CASES, case_inputs
from shot_fpfh_b200 import synthetic


def signs_from_boruvka(n, lo, hi, w, flip):
    """Parity relative to each tree's lowest member, from the Borůvka form."""
    comp, par, _ = oo.boruvka(n, lo, hi, w, flip)
    low = np.full(n, n)
    np.minimum.at(low, comp, np.arange(n))
    return low[comp], par ^ par[low[comp]]


def test_oracle_reproduces_its_pins():
    g = load_golden("orient_pins")
    for name, kind, view in ORIENT_CASES:
        pts, nrm = case_inputs(kind)
        towards = pts.mean(axis=0) if view == "centre" else view
        _, d = oo.orient(pts, nrm, oo.sklearn_knn(pts, K), towards, details=True)
        assert np.array_equal(d["parity"], g[f"{name}_parity"]), name
        assert np.array_equal(d["low"], g[f"{name}_low"]), name
        assert d["n_trees"] == int(g[f"{name}_n_trees"]), name


def test_path_aligns_every_sign_with_the_first_point():
    n = 6
    pts = np.stack([np.arange(n, dtype=np.float64), np.zeros(n), np.zeros(n)], axis=1)
    signs = np.array([1, -1, -1, 1, -1, 1], dtype=np.float64)
    nrm = np.tile([0.0, 0.6, 0.8], (n, 1)) * signs[:, None]
    nbr = np.array([[i, min(i + 1, n - 1)] for i in range(n)])  # i -> i + 1: a path
    out, d = oo.orient(pts, nrm, nbr, details=True)
    assert np.array_equal(out, np.tile([0.0, 0.6, 0.8], (n, 1)))
    assert d["n_trees"] == 1 and d["n_edges"] == n - 1


def test_frustrated_cycle_of_equal_weights_breaks_ties_by_index():
    # pairwise dots all -3 (exact): every edge weighs 1 - 3 = -2 and flips, so the triangle has no consistent
    # orientation and the answer depends on which edge the forest drops: keys (w, 0, 1) < (w, 0, 2) < (w, 1, 2)
    nrm = np.array([[2.0, -1.0, -1.0], [-1.0, 2.0, -1.0], [-1.0, -1.0, 2.0]])
    pts = np.eye(3)
    nbr = np.array([[0, 1, 2], [1, 2, 0], [2, 0, 1]])
    lo, hi = oo.knn_graph(nbr)
    w, flip = oo.edge_keys(nrm, lo, hi)
    assert np.array_equal(w, [-2.0, -2.0, -2.0]) and flip.all()
    assert np.array_equal(oo.msf_kruskal(3, lo, hi, w), [True, True, False])
    out = oo.orient(pts, nrm, nbr)
    assert np.array_equal(out, nrm * [[1.0], [-1.0], [-1.0]])
    assert np.array_equal(signs_from_boruvka(3, lo, hi, w, flip)[1], [0, 1, 1])
    # a square of equal weights: (0, 1), (0, 3), (1, 2) are kept, (2, 3) is dropped
    sq = np.array([[0, 1, 3], [1, 2, 0], [2, 3, 1], [3, 0, 2]])
    lo, hi = oo.knn_graph(sq)
    assert np.array_equal(oo.msf_kruskal(4, lo, hi, np.zeros(4)), [True, True, True, False])


def test_two_disconnected_pieces_each_keep_their_lowest_member():
    tri = np.array([[0.0, 0.0, 1.0], [0.0, 0.1, -1.0], [0.1, 0.0, -1.0]])
    nrm = np.concatenate([tri, -tri])
    pts = np.concatenate([np.eye(3), np.eye(3) + 10.0])
    nbr = np.array([[0, 1, 2], [1, 0, 2], [2, 0, 1], [3, 4, 5], [4, 3, 5], [5, 3, 4]])
    out, d = oo.orient(pts, nrm, nbr, details=True)
    assert d["n_trees"] == 2 and np.array_equal(d["low"], [0, 0, 0, 3, 3, 3])
    assert np.array_equal(out[:3], [[0.0, 0.0, 1.0], [0.0, -0.1, 1.0], [-0.1, 0.0, 1.0]])
    assert np.array_equal(out[3:], -out[:3])


def test_zero_normals_weigh_one_and_never_flip():
    nrm = np.array([[0.0, 0.0, 1.0], [0.0, 0.0, 0.0], [0.0, 0.0, -1.0], [0.0, 0.0, -1.0]])
    pts = np.arange(12, dtype=np.float64).reshape(4, 3)
    nbr = np.array([[0, 1], [1, 2], [2, 3], [3, 2]])  # path 0 - 1 - 2 - 3
    lo, hi = oo.knn_graph(nbr)
    w, flip = oo.edge_keys(nrm, lo, hi)
    assert np.array_equal(w, [1.0, 1.0, 0.0]) and np.array_equal(flip, [False, False, False])
    out = oo.orient(pts, nrm, nbr)
    assert np.array_equal(out, nrm)  # the zero normal carries no sign across: 2 and 3 keep theirs


def test_duplicates_with_opposite_normals_are_aligned_and_edges_counted_once():
    rng = np.random.default_rng(4)
    base, d = synthetic.bumpy_sphere(400, seed=4)
    true = synthetic.bumpy_sphere_true_normals(d)
    pts = np.concatenate([base, base[:60]])
    nrm = np.concatenate([true, -true[:60]]) * rng.choice([-1.0, 1.0], size=(460, 1))
    nbr = oo.sklearn_knn(pts, 8)
    lo, hi = oo.knn_graph(nbr)
    assert np.unique(lo * 460 + hi).shape[0] == lo.shape[0] and (lo < hi).all()
    out, det = oo.orient(pts, nrm, nbr, details=True)
    agree = np.einsum("ij,ij->i", out, np.concatenate([true, true[:60]])) > 0
    assert det["n_trees"] == 1 and (agree.all() or not agree.any())
    w, flip = oo.edge_keys(nrm, lo, hi)
    assert np.array_equal(signs_from_boruvka(460, lo, hi, w, flip), oo.propagate(460, lo, hi, flip,
                                                                                 oo.msf_kruskal(460, lo, hi, w)))


@pytest.mark.parametrize("seed", range(6))
def test_boruvka_equals_kruskal_on_random_graphs(seed):
    rng = np.random.default_rng(100 + seed)
    n = int(rng.integers(50, 400))
    kk = int(rng.integers(1, 6))
    nbr = rng.integers(0, n, size=(n, kk))
    nbr[:, 0] = np.arange(n)  # self entries, as the k + 1 lists carry them
    # normals drawn from a small set (many equal weights: the index tie-break decides), a few zero
    palette = rng.normal(size=(5, 3))
    palette[0] = 0.0
    nrm = palette[rng.integers(0, 5, n)] * rng.choice([-1.0, 1.0], size=(n, 1))
    lo, hi = oo.knn_graph(nbr)
    w, flip = oo.edge_keys(nrm, lo, hi)
    low_k, par_k = oo.propagate(n, lo, hi, flip, oo.msf_kruskal(n, lo, hi, w))
    low_b, par_b = signs_from_boruvka(n, lo, hi, w, flip)
    assert np.array_equal(low_k, low_b) and np.array_equal(par_k, par_b)


def test_bumpy_sphere_20k_eigh_normals_all_agree_with_the_outward_normal():
    n = 20_000
    pts, d = synthetic.bumpy_sphere(n, seed=0)
    true = synthetic.bumpy_sphere_true_normals(d)
    from oracle.make_orient_pins import eigh_normals

    nbr = oo.sklearn_knn(pts, 10)
    nrm = eigh_normals(pts, nbr)
    before = float((np.einsum("ij,ij->i", nrm, true) > 0).mean())
    out, det = oo.orient(pts, nrm, nbr, details=True)
    agree = np.einsum("ij,ij->i", out, true) > 0
    print(f"eigh signs outward {before:.4f}; oriented: {agree.mean():.4f} outward, {det['n_trees']} tree(s)")
    assert 0.4 < before < 0.6 and det["n_trees"] == 1 and (agree.all() or not agree.any())
    lo, hi = oo.knn_graph(nbr)
    w, flip = oo.edge_keys(nrm, lo, hi)
    assert oo.boruvka(n, lo, hi, w, flip)[2] <= 12
    assert np.array_equal(signs_from_boruvka(n, lo, hi, w, flip)[1], det["parity"] ^ det["parity"][0])


def test_towards_takes_the_majority_and_ties_keep_the_default():
    rng = np.random.default_rng(8)
    xy = rng.uniform(-1, 1, size=(300, 2))
    pts = np.concatenate([xy, np.zeros((300, 1))], axis=1)
    nrm = np.tile([0.0, 0.0, 1.0], (300, 1)) * rng.choice([-1.0, 1.0], size=(300, 1))
    nbr = oo.sklearn_knn(pts, 6)
    assert (oo.orient(pts, nrm, nbr, towards=(0.0, 0.0, 3.0))[:, 2] == 1.0).all()
    assert (oo.orient(pts, nrm, nbr, towards=(0.0, 0.0, -3.0))[:, 2] == -1.0).all()
    # a viewpoint in the plane: every dot is 0, a 0 : 0 tie -> point 0 keeps its sign
    assert np.array_equal(oo.orient(pts, nrm, nbr, towards=(5.0, 5.0, 0.0)), oo.orient(pts, nrm, nbr))


def test_non_finite_input_raises():
    pts = np.zeros((4, 3))
    nbr = np.zeros((4, 2), dtype=np.int64)
    for bad in (np.nan, np.inf):
        nrm = np.ones((4, 3))
        nrm[2, 1] = bad
        with pytest.raises(ValueError, match="finite"):
            oo.orient(pts, nrm, nbr)


def test_signature_pinned():
    from shot_fpfh_b200.descriptors import orient_normals

    params = [(p.name, p.default) for p in inspect.signature(orient_normals).parameters.values()]
    assert params == [("points", inspect.Parameter.empty), ("normals", inspect.Parameter.empty), ("k", 10),
                      ("towards", None)]


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the behaviour without a CUDA device")
def test_no_cpu_fallback():
    from shot_fpfh_b200.descriptors import orient_normals

    with pytest.raises(RuntimeError, match="no CPU fallback"):
        orient_normals(np.zeros((10, 3)), np.ones((10, 3)))
