"""
TEST INFRASTRUCTURE — CPU restatement of consistent normal orientation (Hoppe et al. 1992: signs propagated along a
minimum spanning tree of the k-NN graph) as shot_fpfh_b200.descriptors.orient_normals computes it. Only tests/ and
oracle/ may import this module.

The reference has no orientation step, so this module IS the specification (DESIGN.md §2, "pinned to a documented
restatement"):

  1. Graph: every entry j != i of point i's neighbour list (`knn_device(points, points, k + 1)`, ORIGINAL indices) is
     an undirected edge {i, j}; an edge found from both ends is one edge.
  2. d = (n_i.x*n_j.x + n_i.y*n_j.y) + n_i.z*n_j.z in float64, every product and sum rounded (no FMA). Weight
     w = 1 - |d|; key (w, min(i, j), max(i, j)), compared lexicographically: keys are unique, so the minimum
     spanning forest (MSF) is unique. Flip bit: d < 0 (d == 0, e.g. a zero normal, does not flip).
  3. A point's parity relative to another point of its tree is the XOR of the flip bits on the tree path between
     them (Hoppe's s_j = s_i * sign(n_i . n_j)).
  4. Default: in each tree the member with the lowest index keeps its input sign. With `towards` = t: a member votes
     + when n . (t - p) > 0 and - when < 0 under the tree's signs (t - p per component, then the dot of step 2); the
     tree takes the sign with more + than - votes; a tie keeps the default.
  5. Output: the input normals, negated where the final parity is 1.

`orient` runs Kruskal (scipy's minimum_spanning_tree on the keys' ranks) and propagates the flip bits down each tree;
`boruvka` is the data-parallel algorithm of csrc/orient.cu in NumPy (parity labels, mutual choices broken by id),
which the tests hold to the same signs. Pinned by tests/golden/orient_pins.npz (oracle/make_orient_pins.py).
"""

from __future__ import annotations

import numpy as np
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import minimum_spanning_tree


def dot3(a: np.ndarray, b: np.ndarray) -> np.ndarray:
    """(a.x*b.x + a.y*b.y) + a.z*b.z row by row; NumPy rounds every product and sum (what __dmul_rn/__dadd_rn do)."""
    return (a[:, 0] * b[:, 0] + a[:, 1] * b[:, 1]) + a[:, 2] * b[:, 2]


def knn_graph(nbr: np.ndarray) -> tuple[np.ndarray, np.ndarray]:
    """(n, K) neighbour lists -> the undirected edges (lo, hi), lo < hi, each once, in ascending (lo, hi) order."""
    nbr = np.asarray(nbr, dtype=np.int64)
    n = nbr.shape[0]
    src = np.repeat(np.arange(n, dtype=np.int64), nbr.shape[1])
    dst = nbr.reshape(-1)
    keep = src != dst
    packed = np.unique(np.minimum(src, dst)[keep] * n + np.maximum(src, dst)[keep])
    return packed // max(n, 1), packed % max(n, 1)


def edge_keys(normals: np.ndarray, lo: np.ndarray, hi: np.ndarray) -> tuple[np.ndarray, np.ndarray]:
    """(w, flip) of each edge: w = 1 - |d|, flip = d < 0."""
    d = dot3(normals[lo], normals[hi])
    return 1.0 - np.abs(d), d < 0.0


def key_order(lo: np.ndarray, hi: np.ndarray, w: np.ndarray) -> np.ndarray:
    """Edge ids in ascending key order (w, lo, hi)."""
    return np.lexsort((hi, lo, w))


def msf_kruskal(n: int, lo: np.ndarray, hi: np.ndarray, w: np.ndarray) -> np.ndarray:
    """Boolean mask of the MSF's edges: Kruskal on the keys. The keys' ranks 1..m are distinct positive weights with
    the keys' order, so scipy's (Kruskal) forest on them is the unique MSF of the keys (a zero weight would be read as
    a missing edge, hence ranks rather than w)."""
    m = lo.shape[0]
    tree = np.zeros(m, dtype=bool)
    if m == 0:
        return tree
    order = key_order(lo, hi, w)
    rank = np.empty(m, dtype=np.float64)
    rank[order] = np.arange(1, m + 1, dtype=np.float64)
    mst = minimum_spanning_tree(coo_matrix((rank, (lo, hi)), shape=(n, n)).tocsr()).tocoo()
    tree[order[mst.data.astype(np.int64) - 1]] = True
    return tree


def _jump(pred: np.ndarray, acc: np.ndarray) -> np.ndarray:
    """acc XOR-accumulated along pred pointers up to the roots (pred[root] = root, acc[root] = 0), by pointer jumping."""
    pred, acc = pred.copy(), acc.copy()
    while True:
        nxt = pred[pred]
        if np.array_equal(nxt, pred):
            return acc
        acc = acc ^ acc[pred]
        pred = nxt


def propagate(n: int, lo: np.ndarray, hi: np.ndarray, flip: np.ndarray, tree: np.ndarray):
    """
    (low, parity): for every point the lowest index of its tree, and its parity relative to that member (the XOR of
    the flip bits on the tree path). The tree is rooted at its lowest member by a breadth-first walk.
    """
    from scipy.sparse.csgraph import breadth_first_order, connected_components

    tl, th, tf = lo[tree], hi[tree], flip[tree].astype(np.uint8)
    adj = coo_matrix((np.ones(tl.shape[0]), (tl, th)), shape=(n, n)).tocsr()
    _, label = connected_components(adj, directed=False)
    low_of_label = np.full(label.max() + 1 if n else 0, n, dtype=np.int64)
    np.minimum.at(low_of_label, label, np.arange(n))
    low = low_of_label[label]
    # a super root n joined to every tree's lowest member: one breadth-first walk roots every tree
    roots = low_of_label
    rows = np.concatenate([tl, th, np.full(roots.shape[0], n)])
    cols = np.concatenate([th, tl, roots])
    walk = coo_matrix((np.ones(rows.shape[0]), (rows, cols)), shape=(n + 1, n + 1)).tocsr()
    _, pred = breadth_first_order(walk, n, directed=True, return_predecessors=True)
    pred = pred[:n].astype(np.int64)
    # the flip bit of the edge from each point to its predecessor
    edge_flip = np.zeros(n, dtype=np.uint8)
    child = np.where(pred[th] == tl, th, tl)
    edge_flip[child] = tf
    pred[pred == n] = np.flatnonzero(pred == n)  # the trees' lowest members become roots
    return low, _jump(pred, edge_flip)


def boruvka(n: int, lo: np.ndarray, hi: np.ndarray, w: np.ndarray, flip: np.ndarray):
    """
    The device algorithm (csrc/orient.cu) in NumPy: Borůvka rounds with parity labels. Returns (comp, parity, rounds):
    comp[i] = the representative of i's tree, parity[i] = i's parity relative to it.
    """
    comp = np.arange(n, dtype=np.int64)
    par = np.zeros(n, dtype=np.uint8)
    flip = flip.astype(np.uint8)
    live = np.arange(lo.shape[0])
    rounds = 0
    while True:
        live = live[comp[lo[live]] != comp[hi[live]]]  # compact: drop the edges inside a component
        if live.shape[0] == 0:
            return comp, par, rounds
        rounds += 1
        # min-edge pass: every live edge is offered to the components of both its endpoints
        side = np.concatenate([comp[lo[live]], comp[hi[live]]])
        cand = np.concatenate([live, live])
        order = np.lexsort((hi[cand], lo[cand], w[cand], side))
        first = np.ones(order.shape[0], dtype=bool)
        first[1:] = side[order][1:] != side[order][:-1]
        C, e = side[order][first], cand[order][first]
        best = np.full(n, -1, dtype=np.int64)
        best[C] = e
        # hook: C -> D along its chosen edge (u in C, v in D); when D chose the same edge only the higher id hooks
        u = np.where(comp[lo[e]] == C, lo[e], hi[e])
        v = np.where(comp[lo[e]] == C, hi[e], lo[e])
        D = comp[v]
        hooks = ~((best[D] == e) & (C < D))
        hook = np.arange(n, dtype=np.int64)
        hpar = np.zeros(n, dtype=np.uint8)
        hook[C[hooks]] = D[hooks]
        hpar[C[hooks]] = (par[u] ^ flip[e] ^ par[v])[hooks]
        # pointer jumping over the representatives, then relabel every point
        while True:
            nxt = hook[hook]
            if np.array_equal(nxt, hook):
                break
            hpar = hpar ^ hpar[hook]
            hook = nxt
        par = par ^ hpar[comp]
        comp = hook[comp]


def tree_signs(points, normals, low, par, towards=None) -> np.ndarray:
    """Final parity of every point from its parity relative to its tree's lowest member (step 4)."""
    par = par.astype(np.uint8)
    if towards is None:
        return par
    t = np.asarray(towards, dtype=np.float64).reshape(3)
    s = dot3(normals, np.stack([t[0] - points[:, 0], t[1] - points[:, 1], t[2] - points[:, 2]], axis=1))
    plus = ((s > 0) & (par == 0)) | ((s < 0) & (par == 1))
    minus = ((s < 0) & (par == 0)) | ((s > 0) & (par == 1))
    n = points.shape[0]
    flip_tree = np.bincount(low, weights=minus, minlength=n) > np.bincount(low, weights=plus, minlength=n)
    return par ^ flip_tree[low].astype(np.uint8)


def check_inputs(points, normals) -> tuple[np.ndarray, np.ndarray]:
    pts = np.asarray(points, dtype=np.float64).reshape(-1, 3)
    nrm = np.asarray(normals, dtype=np.float64).reshape(-1, 3)
    if pts.shape != nrm.shape:
        raise ValueError(f"points {pts.shape} and normals {nrm.shape} differ in shape")
    if not (np.isfinite(pts).all() and np.isfinite(nrm).all()):
        raise ValueError("orient_normals: points and normals must be finite")
    return pts, nrm


def orient(points, normals, nbr, towards=None, details: bool = False):
    """Oriented normals from the neighbour lists `nbr` (n, K) (ORIGINAL indices). With `details` also a dict: the
    final parity, the lowest member of each point's tree and the number of trees."""
    pts, nrm = check_inputs(points, normals)
    n = pts.shape[0]
    lo, hi = knn_graph(nbr)
    w, flip = edge_keys(nrm, lo, hi)
    low, par = propagate(n, lo, hi, flip, msf_kruskal(n, lo, hi, w))
    final = tree_signs(pts, nrm, low, par, towards)
    out = np.where(final[:, None] == 1, -nrm, nrm)
    if not details:
        return out
    return out, {"parity": final, "low": low, "n_trees": int(np.unique(low).shape[0]), "n_edges": int(lo.shape[0])}


def sklearn_knn(points: np.ndarray, k: int) -> np.ndarray:
    """(n, k + 1) neighbour lists from sklearn's KDTree (the hand-built tests; the GPU tests use the device's own)."""
    from sklearn.neighbors import KDTree

    return KDTree(points).query(points, k + 1, return_distance=False)
