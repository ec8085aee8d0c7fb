"""Pins the CPU oracle to the golden vectors produced by the reference's own sources (tests/golden/make_golden.py)."""
import os

import numpy as np
import pytest

from oracle.kicp_oracle_py import ref_available

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_map(ko, z):
    m = ko.OracleMap(float(z["voxel_size"]), float(z["max_range"]), int(z["max_points_per_voxel"]))
    m.add_points(z["map_points"])  # voxel-grouped, insertion order kept
    assert m.num_points() == len(z["map_points"])
    return m


@pytest.mark.parametrize("name", ["reg_cfg1", "reg_cfg2_small"])
def test_oracle_matches_reference_golden(oracle, name):
    ko = oracle
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    m = load_map(ko, z)
    keys, counts, pts = m.export_voxels()
    assert np.array_equal(keys, z["map_keys"]) and np.array_equal(counts, z["map_counts"]) and np.array_equal(pts, z["map_points"])
    for case in z["cases"]:
        max_iter, conv, adaptive, fixed, tau = int(case[0]), case[1], bool(case[2]), case[3], case[4]
        pose, st = m.register(z["scan"], z["last_pose"], z["rel_odom"], tau, max_iter=max_iter, conv=conv, adaptive=adaptive,
                              fixed_reg=fixed)
        # same sources of rounding, same order: the restatement reproduces the reference bit for bit
        assert np.array_equal(pose, case[5:]), (name, case[:5], ko.pose_delta(pose, case[5:]))


def test_threshold_matches_reference_golden(oracle):
    ko = oracle
    z = np.load(os.path.join(GOLDEN, "threshold.npz"))
    th = ko.OracleThreshold(float(z["map_err"]), float(z["max_range"]), True, 1.0)
    for e, tau in zip(z["errs"], z["taus"]):
        th.update(e)
        assert th.compute() == tau


def test_oracle_matches_reference_build_live(oracle, workload):
    """The restatement against the poses the reference's own Registration.cpp (oracle/_ref) produced on workload cfg2 with 1 and 3
    threads (tests/golden/reference_build.npz)."""
    ko = oracle
    z = np.load(os.path.join(GOLDEN, "reference_build.npz"))
    w = workload(2)
    po, _ = w.map.register(w.scan, w.last_pose, w.rel_odom, w.tau)
    assert len(z["cfg2_threads"]) == 2
    for thr, pr in zip(z["cfg2_threads"], z["cfg2_poses"]):
        dt, ang = ko.pose_delta(pr, po)
        assert dt < 1e-12 and ang < 1e-12, (thr, dt, ang)


@pytest.mark.skipif(not ref_available(), reason="oracle/_ref not built (the reference's sources were absent at build time)")
def test_pipeline_golden_is_reproducible(oracle):
    """The committed pipeline fixture equals a fresh run of the reference's own pipeline sources (threads = 1)."""
    from oracle import sequences as S
    ko = oracle
    z = np.load(os.path.join(GOLDEN, "pipeline_seq.npz"))
    seq = S.unpack_sequence(z, True)
    pipe = ko.ref_pipeline(max_num_threads=1, deskew=True)
    poses, n_src, n_map = S.run_pipeline(pipe, seq)
    pipe.close()
    assert np.array_equal(poses, z["deskew_poses"]) and np.array_equal(n_map, z["deskew_n_map"])


def fuzz_cases(ko):
    """Small random scenes and random solver settings (0..25 iterations, adaptive / fixed regularisation, gates from 5 cm to 3 m,
    empty scans), fixed seed.  Yields (oracle map, last pose, odometry, scan, tau, solver keywords)."""
    from oracle.workloads import unicycle as _unicycle
    rng = np.random.default_rng(20260923)

    def unicycle(_, d, th):
        return _unicycle(d, th)

    for case in range(40):
        vs = float(rng.choice([0.5, 1.0, 2.0]))
        cap = int(rng.choice([1, 5, 20]))
        # a bumpy ground patch plus two walls, mapped from a few random poses
        n_map = int(rng.integers(500, 6000))
        ground = np.c_[rng.uniform(-25, 25, (n_map, 2)), 0.05 * rng.standard_normal(n_map)]
        wall = np.c_[rng.uniform(-25, 25, n_map // 2), np.full(n_map // 2, 12.0) + 0.02 * rng.standard_normal(n_map // 2),
                     rng.uniform(0, 4, n_map // 2)]
        om = ko.OracleMap(vs, 100.0, cap)
        pts = np.concatenate([ground, wall])
        om.add_points(pts)
        last = ko.planar_pose(*rng.uniform(-3, 3, 2), rng.uniform(-3.1, 3.1))
        true_rel = unicycle(ko, rng.uniform(0.0, 1.0), rng.uniform(-0.1, 0.1))
        odom = unicycle(ko, rng.uniform(0.0, 1.1), rng.uniform(-0.12, 0.12))
        n_scan = int(rng.integers(0, 3000))
        world = pts[rng.integers(0, len(pts), n_scan)] + 0.01 * rng.standard_normal((n_scan, 3))
        scan = ko.se3_transform(ko.se3_inverse(ko.se3_compose(last, true_rel)), world) if n_scan else np.zeros((0, 3))
        tau = float(rng.choice([0.05, 0.3, 1.0, 3.0]))
        kw = dict(max_iter=int(rng.choice([0, 1, 3, 10, 25])), conv=float(rng.choice([1e-3, 1e-6, 1e-1])),
                  adaptive=bool(rng.integers(0, 2)), fixed_reg=float(rng.choice([0.0, 0.1, 10.0])))
        yield om, last, odom, scan, tau, kw


def test_oracle_matches_reference_build_fuzz(oracle):
    """Randomised pin of the restatement (fuzz_cases), the oracle against the poses the reference's own Registration.cpp (oracle/_ref,
    one thread = the same summation order) produced on the same scenes (tests/golden/reference_build.npz).  Same map sizes, same NaN
    pattern, poses within 1e-14 (most are bit-identical; the rest differ by one rounding: the test wrapper rebuilds Sophus::SE3d from
    a pose7, whose constructor re-normalises the quaternion)."""
    ko = oracle
    z = np.load(os.path.join(GOLDEN, "reference_build.npz"))
    exact = 0
    cases = list(fuzz_cases(ko))
    assert len(cases) == len(z["fuzz_poses"]) == 40
    for case, ((om, last, odom, scan, tau, kw), pr, n_ref) in enumerate(zip(cases, z["fuzz_poses"], z["fuzz_map_points"])):
        assert om.num_points() == n_ref, case
        po, _ = om.register(scan, last, odom, tau, **kw)
        assert np.array_equal(np.isnan(po), np.isnan(pr)), (case, kw)
        if np.isnan(po).any():
            continue
        dt, ang = ko.pose_delta(po, pr)
        assert dt < 1e-14 and ang < 1e-14, (case, kw, dt, ang)
        exact += int(np.array_equal(po, pr))
    assert exact >= 20
