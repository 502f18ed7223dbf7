"""Generates tests/golden/kitti00_pair.npz from the reference's data/kitti_00.

usage  : python tests/golden/make_kitti00.py <reference checkout>/data/kitti_00
Inputs : 000000.bin, 000001.bin of that directory -- packed float32 xyz (util/read_points.hpp:30-45), the two
         consecutive KITTI-00 scans the reference ships (BASELINE.json configs[4], SURVEY.md 8d cfg5).
Steps  : every 3rd point is kept (fixture size; 41,556 + 41,535 points); the test estimates covariances the way
         src/gtsam_points/features/covariance_estimation.cpp:18-77 does (k = 10, EIG regularisation) with the oracle, builds a
         0.5 m GaussianVoxelMap from frame 0 and runs the frame-to-map LM of tests/mini_lm.py from identity.
Outputs: the points (float32, as in the files) and the ORACLE-driven LM pose track + final pose as golden values.
Tests read only the .npz.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import mini_lm  # noqa: E402
import oracle_lib as orc  # noqa: E402

RESOLUTION = 0.5


def oracle_track(p0, p1, threads=4):
    c0 = orc.estimate_covariances(p0, 10, num_threads=threads)
    c1 = orc.estimate_covariances(p1, 10, num_threads=threads)
    vm = orc.VoxelMap(RESOLUTION)
    vm.insert(orc.Cloud(p0, c0))
    f = orc.Factor(vm, orc.Cloud(p1, c1), num_threads=1)  # one thread: deterministic summation order
    track = []
    values, hist = mini_lm.optimize([mini_lm.OracleFactorAdapter(f, None, 0, fixed_target_pose=np.eye(4))], {0: np.eye(4)}, on_iteration=lambda h, v: track.append(v[0].copy()))
    return vm, values[0], np.stack(track), hist


def main(data):
    frames = [np.fromfile(os.path.join(data, f"{i:06d}.bin"), dtype=np.float32).reshape(-1, 3)[::3].copy() for i in (0, 1)]
    p0, p1 = (f.astype(np.float64) for f in frames)
    vm, T, track, hist = oracle_track(p0, p1)
    out = os.path.join(HERE, "kitti00_pair.npz")
    np.savez_compressed(out, frame0=frames[0], frame1=frames[1], resolution=RESOLUTION, num_voxels=vm.num_voxels, T_final=T, track=track,
                        errors=np.array([h["error"] for h in hist]))
    print(out, os.path.getsize(out), "bytes;", len(p0), len(p1), "points; voxels", vm.num_voxels, "; iterations", len(track))
    print("final pose\n", T)


if __name__ == "__main__":
    main(sys.argv[1])
