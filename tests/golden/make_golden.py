"""Generates tests/golden/*.npz from the REFERENCE'S OWN sources compiled here (oracle/_ref/libkicp_ref.so =
/root/reference/cpp/kinematic_icp/{registration/Registration.cpp, correspondence_threshold/CorrespondenceThreshold.cpp,
pipeline/KinematicICP.cpp} built against header shims, see oracle/Makefile).  Run in the authoring container only
(/root/reference does not exist on the GPU box):

    python tests/golden/make_golden.py

Each fixture carries the inputs (scan, voxel-grouped map, poses, tau, parameters) and the reference's outputs, so the
tests need neither /root/reference nor oracle/_ref.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import kicp_oracle_py as ko  # noqa: E402
from oracle import workloads as W  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))


def registration_fixture(name, cfg_id, **kw):
    w = W.Workload(cfg_id, cache=False, **kw)
    keys, counts, pts = w.map.export_voxels()
    rm = ko.RefMap(w.voxel_size, w.max_range, w.max_points_per_voxel)
    rm.add_points(pts)
    assert rm.num_points() == len(pts)
    cases = []  # (max_iter, conv, adaptive, fixed_reg, tau)
    for max_iter, conv, adaptive, fixed, tau in [(10, 1e-3, 1, 0.0, w.tau), (1, 1e-3, 1, 0.0, w.tau), (10, 1e-3, 0, 0.5, w.tau),
                                                  (25, 1e-5, 0, 0.0, w.tau), (10, 1e-3, 1, 0.0, 0.35)]:
        pose = rm.register(w.scan, w.last_pose, w.rel_odom, tau, max_iter=max_iter, conv=conv, adaptive=bool(adaptive),
                           fixed_reg=fixed, threads=1)
        cases.append(np.concatenate([[max_iter, conv, adaptive, fixed, tau], pose]))
    np.savez_compressed(os.path.join(HERE, name + ".npz"), scan=w.scan, map_keys=keys, map_counts=counts, map_points=pts,
                        last_pose=w.last_pose, rel_odom=w.rel_odom, true_pose=w.true_pose, voxel_size=w.voxel_size,
                        max_range=w.max_range, max_points_per_voxel=w.max_points_per_voxel, cases=np.array(cases))
    print(name, "N", len(w.scan), "M", len(pts), "cases", len(cases))


def threshold_fixture():
    rng = np.random.default_rng(7)
    errs = np.array([ko.se3_exp(rng.normal(size=6) * [0.05, 0.02, 0.0, 0.0, 0.0, 0.004]) for _ in range(12)])
    taus = np.empty(len(errs))
    ko.ref_lib().kref_threshold_sequence(0.2236, 100.0, 1, 1.0, errs.ctypes.data_as(ko.c_dp), len(errs),
                                         taus.ctypes.data_as(ko.c_dp))
    np.savez_compressed(os.path.join(HERE, "threshold.npz"), errs=errs, taus=taus, map_err=0.2236, max_range=100.0)
    print("threshold", taus[:3])


def pipeline_fixture():
    """kinematic_icp::pipeline::KinematicICP::RegisterFrame over a short drive — the reference's own KinematicICP.cpp +
    Registration.cpp + CorrespondenceThreshold.cpp (oracle/_ref), single-threaded."""
    from oracle import sequences as S
    out = {}
    for tag, deskew in (("plain", False), ("deskew", True)):
        seq = S.make_sequence(deskew=deskew)
        pipe = ko.ref_pipeline(max_num_threads=1, deskew=deskew)
        poses, n_src, n_map = S.run_pipeline(pipe, seq)
        pipe.close()
        out[tag + "_poses"], out[tag + "_n_src"], out[tag + "_n_map"] = poses, n_src, n_map
        print("pipeline", tag, n_src.tolist(), n_map.tolist())
    out.update(S.pack_sequence(S.make_sequence(deskew=False)))  # the frames / odometry both runs consumed
    np.savez_compressed(os.path.join(HERE, "pipeline_seq.npz"), **out)


def reference_build_fixture():
    """The reference's own Registration.cpp on workload cfg2 (1 and 3 threads) and on the scenes of test_golden_cpu.fuzz_cases
    (one thread), each map filled with the oracle map's voxel-grouped points."""
    sys.path.insert(0, os.path.dirname(HERE))
    from test_golden_cpu import fuzz_cases
    w = W.Workload(2, cache=False)
    _, _, pts = w.map.export_voxels()
    rm = ko.RefMap(w.voxel_size, w.max_range, w.max_points_per_voxel)
    rm.add_points(pts)
    threads = [1, 3]
    cfg2 = [rm.register(w.scan, w.last_pose, w.rel_odom, w.tau, threads=t) for t in threads]
    fuzz, n_map = [], []
    for om, last, odom, scan, tau, kw in fuzz_cases(ko):
        _, _, stored = om.export_voxels()
        rm = ko.RefMap(om.voxel_size, om.max_distance, om.max_points_per_voxel)
        rm.add_points(stored)
        n_map.append(rm.num_points())
        fuzz.append(rm.register(scan, last, odom, tau, threads=1, **kw))
    np.savez_compressed(os.path.join(HERE, "reference_build.npz"), cfg2_threads=np.array(threads), cfg2_poses=np.array(cfg2),
                        fuzz_poses=np.array(fuzz), fuzz_map_points=np.array(n_map))
    print("reference_build cfg2", len(w.scan), "fuzz cases", len(fuzz))


if __name__ == "__main__":
    assert ko.ref_available(), "build oracle/_ref first: make -C oracle ref"
    registration_fixture("reg_cfg1", 1)
    registration_fixture("reg_cfg2_small", 2, M=30_000, n_az=450)
    threshold_fixture()
    pipeline_fixture()
    reference_build_fixture()
