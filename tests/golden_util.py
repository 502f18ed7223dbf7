import os

import numpy as np

import oracle_lib as orc

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "kitti07_pair.npz")


def estimate_covariances(points):
    """The reference's estimate_covariances (k = 10, EIG regularisation) through the oracle: the covariances are a function of
    the stored points, so the fixture keeps only the points (in float64 the covariances were three quarters of its size).
    V diag(e) V^T leaves a few entries one ulp off their transpose; the fixture's covariances are exactly symmetric."""
    c = orc.estimate_covariances(points, 10, num_threads=max(1, min(8, orc.max_threads())))
    return 0.5 * (c + c.transpose(0, 2, 1))


def load():
    z = np.load(GOLDEN)
    d = {k: z[k] for k in z.files}
    d["target_points"] = d["target_points"].astype(np.float64)
    d["source_points"] = d["source_points"].astype(np.float64)
    d["target_covs"] = estimate_covariances(d["target_points"])
    d["source_covs"] = estimate_covariances(d["source_points"])
    d["resolution"] = float(d["resolution"])
    return d
