"""
TEST INFRASTRUCTURE ONLY. Hand-built SHOT neighbourhoods whose neighbours sit ON the decision boundaries of the
descriptor (and next to them), for comparing the float32 kernel, the float64 kernels and the oracle.

Every query is the centre of an isolated cluster (clusters 4 radii apart) at z = 0; its generic neighbours lie
within r / 4, so that the probe is the farthest neighbour and its values are the ones the oracle keeps (last writer
wins). Its frame is a signed permutation matrix (det +1): X, Y, Z and the cosine are then exact copies of offset and
normal components, whatever the summation order, so the boundary a probe is placed on is the boundary every
implementation sees. Radius and coordinates are dyadic; the distances inside a cluster are distinct.
"""

from __future__ import annotations

import itertools

import numpy as np

RADIUS = 2.0**-4
N_GENERIC = 30
A_HALF_PI_MAX = 1.7225464241988333e-16  # largest Z / rho > 0 with np.arccos(Z / rho) == np.pi / 2 (sf_math.cuh)


def signed_permutations() -> list[np.ndarray]:
    """The 24 rotations that permute the axes with signs; columns are the frame's [x y z] axes."""
    out = []
    for perm in itertools.permutations(range(3)):
        for signs in itertools.product((1.0, -1.0), repeat=3):
            m = np.zeros((3, 3))
            for col, (axis, s) in enumerate(zip(perm, signs)):
                m[axis, col] = s
            if np.linalg.det(m) > 0:
                out.append(m)
    return out


def deltas(r: float) -> list[float]:
    """0 and +-{1 ulp of r, 1e-12, 1e-9, 1e-7, 1e-6, 1e-5} x r: the distances from a boundary a probe is put at."""
    out = [0.0]
    for m in (np.spacing(r) / r, 1e-12, 1e-9, 1e-7, 1e-6, 1e-5):
        out += [m * r, -m * r]
    return out


def cosine_boundaries(max_hits: int = 2) -> list[float]:
    """Cosines c for which the oracle's (c + 1) * 11 / 2 - 0.5 is exactly an integer or a half-integer (bin centres
    and bin edges of the cosine histogram), found by stepping np.nextafter around the real solution, and the
    neighbouring doubles on either side of each."""
    out = []
    for twice in range(-1, 22):
        target = twice / 2.0
        c = np.clip((target + 0.5) * 2.0 / 11.0 - 1.0, -1.0, 1.0)
        lo = c
        for _ in range(64):
            lo = np.nextafter(lo, -2.0)
        hits, cur, closest = [], lo, []
        for _ in range(128):
            if -1.0 <= cur <= 1.0:
                gap = abs((cur + 1.0) * 11 / 2.0 - 0.5 - target)
                if gap == 0.0:
                    hits.append(float(cur))
                closest.append((gap, float(cur)))
            cur = np.nextafter(cur, 2.0)
        if not hits:  # no double lands exactly on it: the nearest ones
            hits = [c for _, c in sorted(closest)[:max_hits]]
        for h in hits[:max_hits]:
            out += [h, float(np.nextafter(h, -2.0)), float(np.nextafter(h, 2.0))]
    return [c for c in out if -1.0 <= c <= 1.0]


def _window_ratios() -> list[float]:
    a = A_HALF_PI_MAX
    ratios = [a, float(np.nextafter(a, 1.0)), float(np.nextafter(a, 0.0)), a / 2, 1e-17, 2e-16, 1e-300]
    ratios += [-1e-17, -4.9e-17, -5.1e-17, -1e-16]
    for e in (1e-10,):  # the oracle's equator rule |phi - pi/2| < 1e-10
        ratios += [e, e * (1 - 1e-6), e * (1 + 1e-6), -e, -e * (1 - 1e-6), -e * (1 + 1e-6)]
    return ratios


def _z_for_ratio(t: float, rho: float) -> float:
    """A z with z / rho == t in float64 when one exists (else the nearest one)."""
    z = t * rho
    best = z
    for _ in range(8):
        if z / rho == t:
            return z
        z = np.nextafter(z, np.inf if z / rho < t else -np.inf)
        if abs(z / rho - t) < abs(best / rho - t):
            best = z
    return best


def probe_set(seed: int = 0, r: float = RADIUS):
    """
    Returns (points (n, 3), normals (n, 3), queries (q, 3), frames (q, 3, 3), kinds: list of q strings).
    Each query is a cloud point (a neighbour at distance 0), with N_GENERIC generic neighbours and one probe.
    """
    rng = np.random.default_rng(seed)
    perms = signed_permutations()
    z_perms = [m for m in perms if abs(m[2, 2]) == 1.0]  # local Z along world z: the query's z = 0 keeps tiny Z exact
    q = 2.0**-30  # grid of the generic coordinates
    x0, y0, z0, a = (np.round(v * r / q) * q for v in (0.3, 0.41, 0.22, 0.35))
    probes = []  # (kind, local offset[, cosine, |n|^2 of the probe's normal])
    for d in deltas(r):
        probes += [("X=0", (d, y0, z0)), ("Y=0", (x0, d, z0)), ("|X|=|Y|", (a, a + d, z0)),
                   ("|X|=|Y|", (a, -(a + d), -z0)), ("Z=0", (x0, y0, d))]
        for frac in (0.25, 0.5, 0.75, 1.0):
            rb = frac * r + d
            probes += [(f"rho={frac}r", (rb, 0.0, 0.0)), (f"rho={frac}r", tuple(rb * np.array([2.0, 3.0, 6.0]) / 7.0))]
    for m in (1e-12, 1e-9, 1e-6, 1e-3):
        probes.append(("tiny rho", tuple(m * r * np.array([0.36, 0.48, 0.8]))))
    xw, yw = (np.round(v * r / q) * q for v in (0.588, 0.784))
    rho_w = float(np.linalg.norm([xw, yw, 0.0]))  # (z^2 is far below half an ulp of rho^2)
    for t in _window_ratios():
        probes.append(("Z/rho", (xw, yw, _z_for_ratio(t, rho_w))))
    cos_list = cosine_boundaries()
    for c in cos_list:
        probes.append(("cos", (x0, y0, z0), c, 1.0))
    for c in cos_list[::6]:
        for d in (1e-12, 1e-9, 1e-7, 1e-6, 1e-5):
            probes += [("cos", (x0, -y0, z0), float(np.clip(c + d, -1, 1)), 1.0),
                       ("cos", (x0, -y0, z0), float(np.clip(c - d, -1, 1)), 1.0)]
    for s in (1.001 * (1 - 1e-6), 1.001 * (1 - 1e-7), 1.001, 1.001 * (1 + 1e-7), 1.001 * (1 + 1e-6), 1.01):
        probes.append(("|n|^2", (x0, y0, -z0), 0.3, s))

    pts, nrm, queries, frames, kinds = [], [], [], [], []
    side = int(np.ceil(np.sqrt(len(probes))))
    for i, pr in enumerate(probes):
        kind, loc = pr[0], np.array(pr[1], dtype=np.float64)
        centre = np.array([1.0 + 4.0 * r * (i % side), 1.0 + 4.0 * r * (i // side), 0.0])
        frame = (z_perms if kind == "Z/rho" else perms)[i % (8 if kind == "Z/rho" else 24)]
        # generic neighbours: distinct distances below r / 4 (so that the probe, farther out, wins every bin it
        # addresses), dyadic coordinates, random unit normals
        while True:
            g = rng.normal(size=(N_GENERIC, 3))
            g *= (rng.uniform(0.02, 0.24, N_GENERIC) * r / np.linalg.norm(g, axis=1))[:, None]
            g = np.round(g / q) * q
            rho = np.linalg.norm(g, axis=1)
            if np.unique(rho).shape[0] == N_GENERIC and rho.min() > 0:
                break
        gn = rng.normal(size=(N_GENERIC, 3))
        gn /= np.linalg.norm(gn, axis=1, keepdims=True)
        probe = centre + frame @ loc
        if len(pr) > 2:  # a normal with the cosine c and |n|^2 = scale (local frame: (s, 0, c))
            c, scale = pr[2], pr[3]
            n_loc = np.array([np.sqrt(max(0.0, 1.0 - c * c)), 0.0, c]) * np.sqrt(scale)
            n_loc[2] = c * np.sqrt(scale) if scale != 1.0 else c  # (the cosine itself exactly when |n| = 1)
            pn = frame @ n_loc
        else:
            pn = gn[0]
        pts += [centre[None], centre + g, probe[None]]
        nrm += [gn[1:2], gn, pn[None]]
        queries.append(centre)
        frames.append(frame)
        kinds.append(kind)
    return np.concatenate(pts), np.concatenate(nrm), np.array(queries), np.array(frames), kinds
