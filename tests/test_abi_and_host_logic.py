"""
CPU: the C-ABI library loads and exports every symbol include/shotfpfh_b200.h declares (no compute call), the
product fails loudly without a GPU, the host-side mirror keeps the reference's signatures, and the pure host
logic (voxel subsampling, filters, synthetic generator) behaves like the reference's.
"""

import ctypes
import inspect
import os
import re

import numpy as np
import pytest
from conftest import ROOT

from oracle.reference_harness import reference_available


def _declared_symbols():
    with open(os.path.join(ROOT, "include", "shotfpfh_b200.h")) as f:
        text = f.read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(sf_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from shot_fpfh_b200 import _lib

    names = _declared_symbols()
    assert len(names) >= 18
    raw = ctypes.CDLL(_lib.LIB_PATH)
    for name in names:
        assert hasattr(raw, name), f"{name} is declared in the header but not exported"
    assert set(names) == set(_lib.EXPORTS), set(names) ^ set(_lib.EXPORTS)
    with open(os.path.join(ROOT, "include", "shotfpfh_b200.h")) as f:
        declared_version = int(re.search(r"#define SF_ABI_VERSION (\d+)", f.read()).group(1))
    assert _lib.lib.sf_abi_version() == declared_version == _lib.ABI_VERSION
    assert _lib.lib.sf_last_error() is not None


def test_library_is_native_sm100a_code():
    """The .so carries sm_100a SASS with the Blackwell tensor-core / TMA instructions (no PTX-only fallback)."""
    import subprocess

    from shot_fpfh_b200 import _lib

    out = subprocess.run(["cuobjdump", "-lelf", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out
    obj = os.path.join(ROOT, "shot_fpfh_b200", "csrc", "match_tc.o")
    if os.path.exists(obj):
        sass = subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True).stdout
        for mnemonic in ("UTCHMMA", "LDTM", "UTMALDG"):
            assert mnemonic in sass, mnemonic


def test_no_cpu_fallback():
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from shot_fpfh_b200.descriptors import ShotMultiprocessor, compute_fpfh_descriptor
    from shot_fpfh_b200.matching import basic_matching

    pts = np.random.default_rng(0).random((50, 3))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        with ShotMultiprocessor() as shot:
            shot.compute_descriptor_single_scale(pts, pts, pts[:5], 0.1)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        compute_fpfh_descriptor(np.arange(5), pts, pts, 0.1, 5)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        basic_matching(pts, pts)


def test_product_never_imports_the_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "shot_fpfh_b200")):
        for name in files:
            if name.endswith((".py", ".cu", ".cuh", ".h")):
                with open(os.path.join(dirpath, name)) as f:
                    text = f.read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", text, flags=re.M), os.path.join(dirpath, name)
                assert "/root/reference" not in text, os.path.join(dirpath, name)


def test_per_call_scratch_has_one_owner():
    """Per-call device scratch is taken through sf::Scratch (csrc/sf_common.cuh), which frees it on every return path:
    no other source allocates from or frees to the stream-ordered pool itself."""
    csrc = os.path.join(ROOT, "shot_fpfh_b200", "csrc")
    for name in sorted(os.listdir(csrc)):
        if name.endswith((".cu", ".cuh", ".cpp", ".h")) and name != "sf_common.cuh":
            with open(os.path.join(csrc, name)) as f:
                text = f.read()
            for word in ("cudaMallocAsync", "cudaFreeAsync", "scratch_alloc"):
                assert word not in text, f"{name} names {word}"


def test_signatures_pinned():
    """The reference-shaped API keeps the parameter lists stored in tests/golden/api_signatures.json (what the live
    comparison below checks against the reference itself)."""
    import json

    from oracle.make_oracle_pins import api_signatures

    with open(os.path.join(ROOT, "tests", "golden", "api_signatures.json")) as f:
        want = json.load(f)
    got = api_signatures()
    assert sorted(got) == sorted(want)
    for name in want:
        assert got[name] == want[name], name


@pytest.mark.skipif(not reference_available(), reason="/root/reference only exists in the build container")
def test_signatures_mirror_the_reference():
    from oracle.reference_harness import import_reference

    import_reference()
    import shot_fpfh.descriptors as ref_d
    import shot_fpfh.descriptors.shot as ref_shot
    import shot_fpfh.matching as ref_m

    import shot_fpfh_b200.descriptors as d
    import shot_fpfh_b200.descriptors.shot as shot
    import shot_fpfh_b200.matching as m

    def params(fn):
        return [(p.name, p.kind, p.default) for p in inspect.signature(fn).parameters.values()]

    for name in ("compute_fpfh_descriptor", "compute_normals"):
        assert params(getattr(d, name)) == params(getattr(ref_d, name)), name
    for name in ("basic_matching", "match_descriptors", "double_matching_with_rejects", "threshold_filter",
                 "quantile_filter", "left_median_filter"):
        assert params(getattr(m, name)) == params(getattr(ref_m, name)), name
    for name in ("get_local_rf", "get_azimuth_idx", "interpolate_on_adjacent_husks", "interpolate_vertical_volumes",
                 "compute_single_shot_descriptor", "compute_shot_descriptor"):
        assert params(getattr(shot, name)) == params(getattr(ref_shot, name)), name
    import shot_fpfh.keypoint_selection as ref_k

    import shot_fpfh_b200.keypoint_selection as k

    for name in ("select_keypoints_subsampling", "select_keypoints_with_density_threshold"):
        assert params(getattr(k, name)) == params(getattr(ref_k, name)), name
    import shot_fpfh.core as ref_core
    import shot_fpfh.icp as ref_icp

    import shot_fpfh_b200.core as core
    import shot_fpfh_b200.icp as icp

    assert params(m.ransac_on_matches) == params(ref_m.ransac_on_matches)
    assert params(icp.icp_point_to_plane) == params(ref_icp.icp_point_to_plane)
    for name in ("solver_point_to_point", "solver_point_to_plane"):
        assert params(getattr(core, name)) == params(getattr(ref_core, name)), name
    for method in ("__init__", "__matmul__", "__invert__", "__getitem__", "transform", "inv", "normalize_rotation"):
        got, want = params(getattr(core.RigidTransform, method)), params(getattr(ref_core.RigidTransform, method))
        assert [p[:2] for p in got] == [p[:2] for p in want], method  # the defaults are arrays: compared by name/kind
    import dataclasses

    ref_fields = [(f.name, f.default) for f in dataclasses.fields(ref_d.ShotMultiprocessor)]
    assert [(f.name, f.default) for f in dataclasses.fields(d.ShotMultiprocessor)] == ref_fields
    for method in ("compute_local_rf", "compute_descriptor", "compute_descriptor_single_scale",
                   "compute_descriptor_bi_scale", "compute_descriptor_multiscale", "__enter__", "__exit__"):
        assert params(getattr(d.ShotMultiprocessor, method)) == params(getattr(ref_d.ShotMultiprocessor, method)), method


def _reference_grid_subsampling(points, voxel_size):
    """Restatement of core/subsampling.py:5-39 (loop over voxels) used to check the vectorised version."""
    keys, inverse, counts = np.unique(((points - points.min(axis=0)) // voxel_size).astype(int), axis=0,
                                      return_inverse=True, return_counts=True)
    order = np.argsort(inverse.ravel(), kind="stable")
    out, seen = [], 0
    for c in counts:
        ids = order[seen : seen + c]
        out.append(ids[np.linalg.norm(points[ids] - points[ids].mean(axis=0), axis=1).argmin()])
        seen += c
    return np.array(out)


def test_grid_subsampling_matches_reference_semantics():
    from shot_fpfh_b200 import synthetic
    from shot_fpfh_b200.subsampling import grid_subsampling

    pts, _ = synthetic.bumpy_sphere(20000, seed=3)
    for voxel in (0.05, 0.11, 0.5, 3.0):
        got = grid_subsampling(pts, voxel)
        assert np.array_equal(got, _reference_grid_subsampling(pts, voxel))
    if reference_available():
        from oracle.reference_harness import import_reference

        import_reference()
        from shot_fpfh.core import grid_subsampling as ref

        # The reference walks each voxel in the order of an UNSTABLE np.argsort (subsampling.py:19), so when two
        # points are equidistant from the barycentre (every 2-point voxel, up to rounding) its pick depends on
        # the sort implementation. Everything else must be identical.
        got, want = grid_subsampling(pts, 0.08), np.asarray(ref(pts, 0.08))
        assert got.shape == want.shape
        keys = ((pts - pts.min(axis=0)) // 0.08).astype(int)
        differ = np.nonzero(got != want)[0]
        assert differ.shape[0] < 0.02 * got.shape[0]
        for i in differ:
            assert np.array_equal(keys[got[i]], keys[want[i]])
            members = np.nonzero((keys == keys[got[i]]).all(axis=1))[0]
            centre = pts[members].mean(axis=0)
            assert abs(np.linalg.norm(pts[got[i]] - centre) - np.linalg.norm(pts[want[i]] - centre)) < 1e-12
    assert grid_subsampling(np.zeros((0, 3)), 0.1).shape == (0,)


def test_filters():
    from shot_fpfh_b200.matching import left_median_filter, quantile_filter, threshold_filter

    d = np.array([0.0, 0.2, 0.1, 0.5, 0.31, 0.0, 0.29])
    assert np.array_equal(threshold_filter(d, 3.0), d <= 0.1 * 3.0)
    assert np.array_equal(quantile_filter(d, (0.25, 0.75)), (d >= np.quantile(d, 0.25)) & (d <= np.quantile(d, 0.75)))
    med = np.median(d)
    assert np.array_equal(left_median_filter(d), (d <= med) & (d >= (med + 1) / 2))  # index 1 is the first non-zero


def test_synthetic_generator_is_seeded_and_matches_the_survey_shape():
    from shot_fpfh_b200 import synthetic

    a, d = synthetic.bumpy_sphere(5000, seed=0)
    b, _ = synthetic.bumpy_sphere(5000, seed=0)
    assert np.array_equal(a, b) and np.allclose(np.linalg.norm(d, axis=1), 1.0)
    rho = np.linalg.norm(a, axis=1)
    assert 0.79 < rho.min() and rho.max() < 1.21
    ref, ref_n, perm, rot, t = synthetic.rigid_pair(a, d)
    assert np.allclose(ref, (a @ rot.T + t)[perm]) and np.allclose(rot @ rot.T, np.eye(3))
    kp = synthetic.voxel_first_point_queries(a, 0.3)
    assert kp.shape[0] < 5000 and np.all(np.diff(kp) > 0)
    rows = synthetic.sparse_unit_rows(100)
    assert np.allclose(np.linalg.norm(rows, axis=1), 1.0, atol=1e-6) and (rows == 0).mean() > 0.8


def test_host_row_expansion_rebuilds_dense_float64_rows():
    """csrc/host_io.cpp (no GPU involved): compact rows -> dense float64, every thread count, odd shapes, bad input."""
    from shot_fpfh_b200._lib import SF_ERR_ARG, check, lib

    rng = np.random.default_rng(3)
    for n_rows, width in ((0, 352), (1, 352), (3, 352), (777, 352), (5000, 33), (300, 125), (64, 4096)):
        dense = (rng.random((n_rows, width)) * (rng.random((n_rows, width)) < 0.14)).astype(np.float32)
        if n_rows > 2:
            dense[1] = 0.0  # an empty row
            dense[2] = -1.5  # a full row, negative values
        r, c = np.nonzero(dense)
        offsets = np.zeros(n_rows + 1, np.int64)
        np.cumsum(np.bincount(r, minlength=n_rows), out=offsets[1:])
        cols, vals = c.astype(np.uint16), dense[r, c]
        for threads in (1, 3, 8):
            out = np.full((n_rows, width), 7.0)
            check(lib.sf_host_expand_rows_begin(offsets.ctypes.data, cols.ctypes.data, vals.ctypes.data, n_rows, width,
                                                out.ctypes.data, threads))
            check(lib.sf_host_wait())
            assert np.array_equal(out, dense.astype(np.float64)), (n_rows, width, threads)
    bad = cols.copy()
    bad[0] = 5000  # column outside the row
    out = np.zeros((n_rows, width))
    check(lib.sf_host_expand_rows_begin(offsets.ctypes.data, bad.ctypes.data, vals.ctypes.data, n_rows, width,
                                        out.ctypes.data, 2))
    assert lib.sf_host_wait() == SF_ERR_ARG
    assert lib.sf_host_expand_rows_begin(None, None, None, 4, 352, None, 2) == SF_ERR_ARG
    assert lib.sf_host_expand_rows_begin(offsets.ctypes.data, cols.ctypes.data, vals.ctypes.data, 1, 5000,
                                         out.ctypes.data, 2) == SF_ERR_ARG
    assert lib.sf_host_wait() == 0


def test_host_widening_equals_astype_float64():
    """csrc/host_io.cpp::sf_host_widen_begin (no GPU involved): dst = double(src) exactly, any length / alignment /
    thread count, jobs queued back to back."""
    from shot_fpfh_b200._lib import SF_ERR_ARG, check, lib

    rng = np.random.default_rng(5)
    for n in (0, 1, 7, 4095, 4096, 100_003, 1_000_000):
        src = rng.standard_normal(n + 3).astype(np.float32)
        for shift in (0, 1, 3):  # unaligned starts on both sides
            for threads in (1, 3, 8):
                dst = np.full(n + 5, 7.0)
                check(lib.sf_host_widen_begin(src[shift:].ctypes.data, n, dst[1:].ctypes.data, threads))
                check(lib.sf_host_wait())
                assert np.array_equal(dst[1 : 1 + n], src[shift : shift + n].astype(np.float64))
                assert dst[0] == 7.0 and (dst[1 + n :] == 7.0).all()
    # two jobs in flight: the second waits for the first
    a, b = rng.standard_normal(500_000).astype(np.float32), rng.standard_normal(300_001).astype(np.float32)
    out = np.zeros(800_001)
    check(lib.sf_host_widen_begin(a.ctypes.data, a.size, out.ctypes.data, 4))
    check(lib.sf_host_widen_begin(b.ctypes.data, b.size, out[a.size :].ctypes.data, 4))
    check(lib.sf_host_wait())
    assert np.array_equal(out, np.concatenate([a, b]).astype(np.float64))
    assert lib.sf_host_widen_begin(None, 5, None, 2) == SF_ERR_ARG


def test_result_buffers_are_recycled_only_when_the_caller_dropped_them(monkeypatch):
    """device.result_buffer: a buffer goes out again only when no reference to the previous result (views and slices
    included) is left; results the caller keeps are never touched."""
    from shot_fpfh_b200 import device

    monkeypatch.setattr(device, "_RESULT_POOL", [])
    kept = [device.result_buffer((50, 8))[1] for _ in range(4)]  # a pipeline that keeps its descriptors
    for i, k in enumerate(kept):
        k[...] = i
    assert len({k.ctypes.data for k in kept}) == 4
    view = kept[0][10:20]
    first = kept[1].ctypes.data
    del kept
    d = device.result_buffer((50, 8))[1]  # one of the three dropped buffers comes back ...
    d[...] = 9.0
    assert np.all(view == 0)  # ... never the one a slice still points into
    addresses = {d.ctypes.data}
    for _ in range(6):  # a loop `d = f()`: the previous result is alive during the call -> buffers alternate
        d = device.result_buffer((50, 8))[1]
        d[...] = 7.0
        addresses.add(d.ctypes.data)
    assert np.all(view == 0)
    assert len(addresses) <= 3 and first in addresses and d.dtype == np.float64 and d.shape == (50, 8)


def test_bench_reference_arm_prints_one_contract_line():
    """`bench.py --impl reference` (the CPU arm, no GPU needed): exactly one JSON line on stdout with the contract's keys."""
    import json
    import subprocess
    import sys

    proc = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                           "--warmup", "0", "--cpu-seconds", "1.0"], capture_output=True, text=True, timeout=600)
    assert proc.returncode == 0, proc.stderr[-2000:]
    lines = [ln for ln in proc.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and line["metric"] == "SHOT descriptors/sec" and line["unit"] == "descriptors/s"
    assert line["higher_is_better"] is True and line["n_gpus"] == 1 and line["steps"] == 1 and line["value"] > 0
    assert line["config"]["workload"].startswith("C2: SHOT single-scale, 1M-point")
    cpu = line["cpu_baseline"]
    # the unmodified reference from baseline/_ref when it is installed, else the oracle port
    assert cpu["kind"] in ("reference", "port") and cpu["cores"] >= 1 and cpu["value"] == line["value"]
    assert "queries" in cpu["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["gpu_launches"] == 0


def test_replayed_ransac_draws_are_numpys_draws():
    """matching/ransac.py::replay_choices == the loop of `rng.choice(n, k, replace=False, shuffle=False)` calls of the
    reference (ransac.py:48-53): same draws, same generator state afterwards (so later calls continue the same
    stream), with and without a buffered 32-bit half at entry, collisions (tiny populations), Lemire rejections
    (populations of millions), and the regimes that fall back to the calls themselves."""
    from shot_fpfh_b200.matching.ransac import replay_choices

    cases = [(20000, 4, 10000), (100, 4, 5000), (6, 4, 3000), (5, 4, 100), (3_000_000, 4, 4000), (30_000_000, 4, 1500),
             (2**31 + 7, 4, 2000), (3 * 2**30 + 1, 3, 1000), (20000, 1, 10), (40000, 7, 2000), (12000, 300, 5),
             (9000, 300, 5), (2**33, 4, 50), (4, 4, 20), (20000, 4, 0)]
    for seed in (72, 5):
        for pop, size, n in cases:
            for buffered in (False, True):
                a, b = np.random.default_rng(seed), np.random.default_rng(seed)
                if buffered:
                    a.integers(0, 100, dtype=np.uint32)
                    b.integers(0, 100, dtype=np.uint32)
                    assert b.bit_generator.state["has_uint32"] == 1
                want = [a.choice(pop, size, replace=False, shuffle=False) for _ in range(n)]
                got = replay_choices(b, pop, size, n)
                assert got.shape == (n, size) and (n == 0 or np.array_equal(np.stack(want), got)), (seed, pop, size, n)
                assert a.bit_generator.state == b.bit_generator.state, (seed, pop, size, n, buffered)
                assert np.array_equal(a.choice(pop, size, replace=False, shuffle=False),
                                      b.choice(pop, size, replace=False, shuffle=False))
    # another bit generator: the calls themselves
    a, b = np.random.Generator(np.random.MT19937(3)), np.random.Generator(np.random.MT19937(3))
    want = np.stack([a.choice(500, 4, replace=False, shuffle=False) for _ in range(50)])
    assert np.array_equal(replay_choices(b, 500, 4, 50), want)


@pytest.mark.skipif(not reference_available(), reason="the reference package is only present in the build container")
def test_dropin_rebinds_the_names_the_pipeline_imports_and_restores_them():
    """dropin.install(): every hot-path name `pipeline.py` imports (pipeline.py:15, :24-30) resolves to this package
    inside the UNMODIFIED reference, the pipeline object can be built on top of them, and uninstall() puts the
    reference's own functions back. (No compute: there is no GPU here.)"""
    import importlib

    from oracle.reference_harness import import_reference

    import_reference()
    import shot_fpfh_b200.dropin as dropin
    from shot_fpfh_b200 import descriptors as d
    from shot_fpfh_b200 import icp, matching as m

    pipeline = importlib.import_module("shot_fpfh.pipeline")
    originals = {name: getattr(pipeline, name) for name in (
        "ShotMultiprocessor", "compute_fpfh_descriptor", "basic_matching", "match_descriptors",
        "double_matching_with_rejects", "ransac_on_matches", "icp_point_to_plane")}
    done = dropin.install()
    try:
        assert len(done) >= 30
        assert pipeline.ShotMultiprocessor is d.ShotMultiprocessor
        assert pipeline.compute_fpfh_descriptor is d.compute_fpfh_descriptor
        assert pipeline.basic_matching is m.basic_matching and pipeline.match_descriptors is m.match_descriptors
        assert pipeline.double_matching_with_rejects is m.double_matching_with_rejects
        assert pipeline.ransac_on_matches is m.ransac_on_matches and pipeline.icp_point_to_plane is icp.icp_point_to_plane
        ref_pkg = importlib.import_module("shot_fpfh")
        assert ref_pkg.compute_normals is d.compute_normals
        assert importlib.import_module("shot_fpfh.descriptors").ShotMultiprocessor is d.ShotMultiprocessor
        # the reference's own orchestration object builds on top of the rebound names
        rng = np.random.default_rng(0)
        pts = rng.random((50, 3))
        pipe = pipeline.RegistrationPipeline(scan=pts, scan_normals=pts, ref=pts, ref_normals=pts)
        assert hasattr(pipe, "compute_descriptors") and hasattr(pipe, "find_descriptors_matches")
    finally:
        dropin.uninstall()
    for name, fn in originals.items():
        assert getattr(pipeline, name) is fn, name
