"""Generates tests/golden/kitti07_frames.npz from the reference's own test data.

usage  : python tests/golden/make_kitti07_frames.py <reference checkout>/data/kitti_07_dump
Inputs : {graph.txt, 00000{0..4}/points.bin} of that directory -- the five submaps and ground-truth poses
         that src/test/test_matching_cost_factors.cpp:35-78 loads (packed float32 xyz; poses `tx ty tz qx qy qz qw`).
Content: every 2nd point of each submap (fixture size), the ground-truth poses, and noisy initial poses = ground truth composed
         with Exp(U(-0.1, 0.1)^6) -- the reference test's perturbation (:41-59), drawn ONCE here because std::mt19937 +
         uniform_real_distribution is not reproducible across standard libraries (the test's own comment says so).
Tests read only the .npz.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from gtsam_points_b200 import synthetic as syn  # noqa: E402
from make_golden import quat_pose  # noqa: E402


def main(data):
    gt = []
    for line in open(os.path.join(data, "graph.txt")):
        tok = line.split()
        if tok and tok[0].startswith("v"):
            gt.append(quat_pose([float(x) for x in tok[1:8]]))
    assert len(gt) == 5
    rng = np.random.default_rng(8191)
    noisy = [T @ syn.se3_exp(rng.uniform(-0.1, 0.1, 6)) for T in gt]
    out = {"poses_gt": np.stack(gt), "poses": np.stack(noisy)}
    for i in range(5):
        p = np.fromfile(os.path.join(data, f"{i:06d}", "points.bin"), dtype=np.float32).reshape(-1, 3)[::2]
        out[f"points{i}"] = np.ascontiguousarray(p)
    np.savez_compressed(os.path.join(HERE, "kitti07_frames.npz"), **out)
    print({k: v.shape for k, v in out.items()})


if __name__ == "__main__":
    main(sys.argv[1])
