"""BASELINE.json configs[4] / SURVEY.md 8d cfg5: KITTI-00 frame-to-map VGICP on the two scans the reference ships
(tests/golden/kitti00_pair.npz, made by tests/golden/make_kitti00.py).  The CPU test pins the oracle against the committed
golden pose track; the GPU test drives the same LM with the CUDA factor and must follow the oracle pose for pose."""
import os

import numpy as np
import pytest

import mini_lm
import oracle_lib as orc

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "kitti00_pair.npz")


@pytest.fixture(scope="module")
def data():
    z = np.load(GOLD)
    d = {k: z[k] for k in z.files}
    d["p0"], d["p1"] = d["frame0"].astype(np.float64), d["frame1"].astype(np.float64)
    threads = max(1, min(8, orc.max_threads()))
    d["c0"] = orc.estimate_covariances(d["p0"], 10, num_threads=threads)
    d["c1"] = orc.estimate_covariances(d["p1"], 10, num_threads=threads)
    return d


def oracle_factor(d):
    vm = orc.VoxelMap(float(d["resolution"]))
    vm.insert(orc.Cloud(d["p0"], d["c0"]))
    f = orc.Factor(vm, orc.Cloud(d["p1"], d["c1"]), num_threads=1)
    return vm, f


def run_lm(factor):
    track = []
    values, hist = mini_lm.optimize([factor], {0: np.eye(4)}, on_iteration=lambda h, v: track.append(v[0].copy()))
    return values[0], np.stack(track), hist


def test_oracle_reproduces_the_golden_pose_track(data):
    vm, f = oracle_factor(data)
    assert vm.num_voxels == int(data["num_voxels"])
    T, track, hist = run_lm(mini_lm.OracleFactorAdapter(f, None, 0, fixed_target_pose=np.eye(4)))
    assert track.shape == data["track"].shape and np.abs(track - data["track"]).max() < 1e-9
    assert np.abs(T - data["T_final"]).max() < 1e-9
    # a plausible KITTI ego-motion: ~0.68 m forward, < 0.01 rad
    rot, trans = mini_lm.pose_error(T, np.eye(4))
    assert 0.5 < trans < 0.9 and rot < 0.01
    # hit rate at identity (SURVEY.md 8d: 77 % of the full scan at 0.5 m; the third-density fixture sees a sparser map)
    assert 0.4 < vm.overlap(orc.Cloud(data["p1"], data["c1"]), np.eye(4)) < 0.95


@pytest.mark.gpu
def test_cuda_frame_to_map_follows_the_oracle_track(data):
    import gtsam_points_b200 as g

    vm = g.GaussianVoxelMapGPU(float(data["resolution"]))
    vm.insert(g.PointCloud(data["p0"], data["c0"]))
    assert vm.num_voxels == int(data["num_voxels"])
    f = g.IntegratedVGICPFactor(np.eye(4), 0, vm, g.PointCloud(data["p1"], data["c1"]))
    T, track, hist = run_lm(f)
    assert track.shape == data["track"].shape
    assert np.abs(track - data["track"]).max() < 1e-7  # same pose at every LM iteration as the CPU-driven optimisation
    assert np.abs(T - data["T_final"]).max() < 1e-7
    # correspondences at the final pose are the oracle's, bit for bit
    ovm, of = oracle_factor(data)
    f.linearize({0: T})
    of.linearize(T)
    assert np.array_equal(f.correspondences(), of.correspondences())
