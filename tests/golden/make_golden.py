"""Generates tests/golden/kitti07_pair.npz from the reference's own test data.

usage  : python tests/golden/make_golden.py <reference checkout>/data/kitti_07_dump
Inputs : {graph.txt, 000000/points.bin, 000001/points.bin} of that directory -- the submaps the reference's
         src/test/test_matching_cost_factors.cpp:62-78 loads (packed float32 xyz; poses `tx ty tz qx qy qz qw`).
Steps  : every 2nd point is kept (fixture size); covariances follow src/gtsam_points/features/covariance_estimation.cpp:18-77
         (k = 10 nearest neighbours incl. the point itself, cov = (sum p p^T - mean sum p^T) / k, eigenvalues replaced by
         (1e-3, 1, 1) in ascending-eigenvalue order), computed by golden_util.estimate_covariances (the oracle) -- they are
         not stored, the tests recompute them from the points the same way;
         noisy relative pose = ground truth composed with a fixed tangent perturbation;
         outputs = the CPU oracle's VGICP (1.0 m voxels, as in the reference test :84-90) and GICP linearize() / error() /
         correspondences with num_threads = 1 (deterministic summation order).
Tests read only the .npz.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import golden_util  # noqa: E402
import oracle_lib as orc  # noqa: E402
from gtsam_points_b200 import synthetic as syn  # noqa: E402


def quat_pose(v):
    tx, ty, tz, qx, qy, qz, qw = v
    n = np.sqrt(qx * qx + qy * qy + qz * qz + qw * qw)
    qx, qy, qz, qw = qx / n, qy / n, qz / n, qw / n
    R = np.array(
        [
            [1 - 2 * (qy * qy + qz * qz), 2 * (qx * qy - qz * qw), 2 * (qx * qz + qy * qw)],
            [2 * (qx * qy + qz * qw), 1 - 2 * (qx * qx + qz * qz), 2 * (qy * qz - qx * qw)],
            [2 * (qx * qz - qy * qw), 2 * (qy * qz + qx * qw), 1 - 2 * (qx * qx + qy * qy)],
        ]
    )
    T = np.eye(4)
    T[:3, :3] = R
    T[:3, 3] = [tx, ty, tz]
    return T


def main(data):
    poses = {}
    for line in open(os.path.join(data, "graph.txt")):
        tok = line.split()
        poses[int(tok[0][1:])] = quat_pose([float(x) for x in tok[1:8]])
    clouds = []
    for i in (0, 1):
        p = np.fromfile(os.path.join(data, f"{i:06d}", "points.bin"), dtype=np.float32).reshape(-1, 3)[::2]
        clouds.append(np.ascontiguousarray(p))
    pts = [c.astype(np.float64) for c in clouds]
    covs = [golden_util.estimate_covariances(p) for p in pts]

    T_target, T_source_gt = poses[0], poses[1]
    xi = np.array([0.03, -0.02, 0.025, 0.08, -0.06, 0.04])  # fixed tangent noise (the reference test draws U(-0.1, 0.1))
    T_source = T_source_gt @ syn.se3_exp(xi)
    delta = orc.calc_delta(T_target, T_source)
    delta_eval = orc.calc_delta(T_target, T_source_gt @ syn.se3_exp(0.5 * xi))

    tgt = orc.Cloud(pts[0], covs[0])
    src = orc.Cloud(pts[1], covs[1])
    out = dict(
        target_points=clouds[0],
        source_points=clouds[1],
        T_target=T_target,
        T_source_gt=T_source_gt,
        T_source=T_source,
        delta=delta,
        delta_eval=delta_eval,
        resolution=np.array(1.0),
    )
    vm = orc.VoxelMap(1.0)
    vm.insert(tgt)
    ex = vm.export()
    out["voxel_coords"] = ex["coords"]
    out["voxel_num_points"] = ex["n"]
    f = orc.Factor(vm, src, num_threads=1)
    out["vgicp_linearized"] = f.linearize_raw(delta)
    out["vgicp_corr"] = f.correspondences().astype(np.int32)
    out["vgicp_error_eval"] = np.array(f.error(delta_eval))
    tree = orc.KdTree(tgt)
    g = orc.Factor(tgt, src, tree=tree, num_threads=1)
    out["gicp_linearized"] = g.linearize_raw(delta)
    out["gicp_corr"] = g.correspondences().astype(np.int32)
    out["gicp_error_eval"] = np.array(g.error(delta_eval))
    path = os.path.join(HERE, "kitti07_pair.npz")
    np.savez_compressed(path, **out)
    print(path, os.path.getsize(path) // 1024, "KiB;", "voxels", len(ex["coords"]), "vgicp inliers", int(out["vgicp_linearized"][121]), "gicp inliers", int(out["gicp_linearized"][121]))


if __name__ == "__main__":
    main(sys.argv[1])
