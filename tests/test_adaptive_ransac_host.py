"""
CPU checks of the adaptive RANSAC specification (oracle/adaptive_ransac_oracle.py): the stored pins, the draw
formula against a plain-Python restatement, the T rewrite of the inlier predicate, the stopping rule, hand-made fits,
and the argument checks of ransac_on_matches_adaptive that run before any device work.
"""

import math
import os

import numpy as np
import pytest

from oracle import adaptive_ransac_oracle as oracle
from oracle import make_adaptive_ransac_pins as pins

MASK = (1 << 64) - 1


def test_oracle_reproduces_pins():
    stored = np.load(os.path.join(os.path.dirname(__file__), "golden", "adaptive_ransac_pins.npz"))
    fresh = pins.compute()
    assert sorted(stored.files) == sorted(fresh)
    for key in stored.files:
        assert np.array_equal(stored[key], fresh[key]), key


def _splitmix64(z: int) -> int:
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & MASK
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & MASK
    return z ^ (z >> 31)


def _draw(seed: int, d: int, m: int) -> list[int]:
    u = [_splitmix64((seed * 0x9E3779B97F4A7C15 + 3 * d + s) & MASK) >> 32 for s in range(3)]
    j0 = (u[0] * m) >> 32
    j1 = (u[1] * (m - 1)) >> 32
    j1 += j1 >= j0
    j2 = (u[2] * (m - 2)) >> 32
    j2 += j2 >= min(j0, j1)
    j2 += j2 >= max(j0, j1)
    return [j0, j1, j2]


@pytest.mark.parametrize("m", [3, 4, 7, 1000, (1 << 31) + 11, (1 << 32) - 1])
@pytest.mark.parametrize("seed", [0, 1, 12345678901234567, -3])
def test_draw_formula(m, seed):
    draws = np.concatenate([np.arange(2000), np.array([(1 << 32) - 2, (1 << 31) + 7])])
    got = oracle.draw_indices(seed, draws, m)
    want = np.array([_draw(seed, int(d), m) for d in draws])
    assert np.array_equal(got, want)
    assert (got >= 0).all() and (got < m).all()
    assert ((got[:, 0] != got[:, 1]) & (got[:, 0] != got[:, 2]) & (got[:, 1] != got[:, 2])).all()


def test_draws_distinct_and_uniform_at_m3_and_m7():
    for m in (3, 7):
        j = oracle.draw_indices(0, np.arange(200_000), m)
        assert ((j[:, 0] != j[:, 1]) & (j[:, 0] != j[:, 2]) & (j[:, 1] != j[:, 2])).all()
        for s in range(3):  # every index in every slot, about equally often
            freq = np.bincount(j[:, s], minlength=m) / j.shape[0]
            assert np.abs(freq - 1.0 / m).max() < 0.01


@pytest.mark.parametrize("threshold", [1.0, 0.01, 0.1, 3.0, 1e-150, 1e150, 0.3 * 4 * 0.0056])
def test_threshold_sq_rewrite(threshold):
    t = oracle.threshold_sq(threshold)
    assert math.sqrt(t) <= threshold < math.sqrt(math.nextafter(t, math.inf))
    probes = [t]
    for direction in (0.0, math.inf):
        x = t
        for _ in range(64):
            x = math.nextafter(x, direction)
            probes.append(x)
    probes += [threshold * threshold, math.nextafter(threshold * threshold, 0.0)]
    for d2 in probes:
        assert (d2 <= t) == (math.sqrt(d2) <= threshold), d2


@pytest.mark.parametrize("count,m,confidence,batches", [
    (27, 100, 0.999, 1), (2, 100, 0.999, 1), (1, 100, 0.999, 7), (1, 100, 0.99, 5), (1, 200, 0.999, 53),
    (5, 1000, 0.5, 6),
])
def test_stopping_rule(count, m, confidence, batches):
    k = 1
    while not oracle.should_stop(k, count, m, confidence):
        k += 1
    assert k == batches
    r = count / m  # the closed form: the smallest k with k B >= log(1 - confidence) / log(1 - r^3)
    assert k == math.ceil(math.log(1 - confidence) / math.log1p(-r ** 3) / oracle.BATCH)
    assert not oracle.should_stop(1, 0, m, confidence)


def test_collinear_triples_rejected():
    a = np.array([[[0.0, 0.0, 0.0], [1.0, 2.0, 3.0], [2.5, 5.0, 7.5]]])
    b = a + np.array([0.3, -1.0, 2.0])
    assert oracle.edges_consistent(a, b, 0.9).all()
    _, ok = oracle.kabsch3(a, b)
    assert not ok.any()
    # a near-collinear triple is still a fit
    a2 = a.copy()
    a2[0, 2] += [0.0, 0.1, 0.0]
    _, ok = oracle.kabsch3(a2, a2 + 1.0)
    assert ok.all()


def test_edge_check():
    a = np.array([[[0.0, 0.0, 0.0], [1.0, 0.0, 0.0], [0.0, 1.0, 0.0]]])
    assert oracle.edges_consistent(a, a * 1.05, 0.9).all()
    assert not oracle.edges_consistent(a, a * 1.2, 0.9).any()
    assert oracle.edges_consistent(a, a * 1.2, 0.8).all()


def test_pure_rotation_recovered_from_three_pairs():
    from shot_fpfh_b200.synthetic import rotation_from_rotvec

    rng = np.random.default_rng(4)
    for _ in range(20):
        rot = rotation_from_rotvec(rng.normal(size=3))
        # a well-shaped triangle (singular values of H within a factor 4) in a random pose
        a = (np.array([[0.0, 0.0, 0.0], [1.0, 0.0, 0.0], [0.3, 1.5, 0.0]]) @ rotation_from_rotvec(rng.normal(size=3)).T)[None]
        b = a @ rot.T
        tr, ok = oracle.kabsch3(a, b)
        assert ok.all()
        assert np.abs(tr[0, :9].reshape(3, 3) - rot).max() <= 1e-14
        assert np.abs(tr[0, 9:]).max() <= 1e-14
        assert np.linalg.det(tr[0, :9].reshape(3, 3)) == pytest.approx(1.0, abs=1e-14)


def test_all_collinear_input_has_no_winner():
    line = np.zeros((40, 3))
    line[:, 0] = np.linspace(0.0, 1.0, 40)
    out = oracle.ransac_adaptive(line, line + 0.5, 0.01, max_draws=50_000)
    assert out["valid"] == 0 and out["best_count"] == 0 and out["best_draw"] == -1
    assert out["survivors"] > 0 and out["draws_used"] == 50_000


def test_public_function_checks_arguments():
    from shot_fpfh_b200 import synthetic
    from shot_fpfh_b200.matching import ransac_on_matches_adaptive

    scan, ref, si, ri, *_ = synthetic.corrupted_matches(100, 0.5, seed=3)
    for kwargs in ({"distance_threshold": 0.0}, {"distance_threshold": -1.0}, {"distance_threshold": math.inf},
                   {"confidence": 1.0}, {"confidence": 0.0}, {"edge_similarity": 0.0}, {"edge_similarity": 1.5},
                   {"max_draws": 0}, {"max_draws": 1 << 32}):
        with pytest.raises(ValueError):
            ransac_on_matches_adaptive(si, ri, scan, ref, **kwargs)
    with pytest.raises(ValueError):
        ransac_on_matches_adaptive(si[:2], ri[:2], scan, ref)
    huge = np.broadcast_to(np.zeros(1, dtype=np.int64), (1 << 32,))
    with pytest.raises(ValueError):
        ransac_on_matches_adaptive(huge, huge, scan, ref)
    bad = scan.copy()
    bad[si[0], 1] = np.inf
    with pytest.raises(ValueError):
        ransac_on_matches_adaptive(si, ri, bad, ref)


def test_corrupted_matches():
    from shot_fpfh_b200 import synthetic

    scan, ref, si, ri, rot, trans = synthetic.corrupted_matches(5000, 0.1, noise=0.0, seed=2)
    correct = np.linalg.norm(scan[si] @ rot.T + trans - ref[ri], axis=1) < 1e-12
    assert correct.sum() >= 500 and correct.sum() <= 510  # 500 chosen, and a random pick may hit its true partner
