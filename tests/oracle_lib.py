"""ctypes binding of oracle/liboracle.so -- TEST INFRASTRUCTURE ONLY.

Importable from tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / reference legs.
The product package (gtsam_points_b200/) never imports this module.
"""
import ctypes as C
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
_LIB = None

LINEARIZED_DOUBLES = 122


def build(force=False):
    native_dir = os.environ.get("B2_ORACLE_NATIVE")
    if native_dir:
        # secondary CPU number of bench.py: the same code with -march=native, ALWAYS rebuilt on the host that runs it, into the
        # directory B2_ORACLE_NATIVE names (bench.py runs from a tree that may be read-only)
        so = os.path.join(os.path.abspath(native_dir), "liboracle_native.so")
        subprocess.check_call(["make", "-B", "-C", ORACLE_DIR, f"NATIVE_OUT={so}", so], stdout=subprocess.DEVNULL)
        return so
    so = os.path.join(ORACLE_DIR, "liboracle.so")
    src = [os.path.join(ORACLE_DIR, f) for f in ("oracle.cpp", "oracle.h", "Makefile")]
    if force or not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in src):
        subprocess.check_call(["make", "-C", ORACLE_DIR, "liboracle.so"], stdout=subprocess.DEVNULL)
    return so


def lib():
    global _LIB
    if _LIB is None:
        L = C.CDLL(build())
        vp, dp, ip, lp = C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int32), C.POINTER(C.c_int64)
        L.orc_cloud_create.restype = vp
        L.orc_cloud_create.argtypes = [dp, dp, C.c_size_t]
        L.orc_cloud_destroy.argtypes = [vp]
        L.orc_voxelmap_create.restype = vp
        L.orc_voxelmap_create.argtypes = [C.c_double]
        L.orc_voxelmap_destroy.argtypes = [vp]
        L.orc_voxelmap_set_lru.argtypes = [vp, C.c_int, C.c_int]
        L.orc_voxelmap_insert.argtypes = [vp, vp]
        L.orc_voxelmap_num_voxels.restype = C.c_size_t
        L.orc_voxelmap_num_voxels.argtypes = [vp]
        L.orc_voxelmap_export.argtypes = [vp, ip, dp, dp, ip]
        L.orc_voxelmap_lookup.argtypes = [vp, dp, C.c_size_t, ip]
        L.orc_kdtree_create.restype = vp
        L.orc_kdtree_create.argtypes = [vp, C.c_int]
        L.orc_kdtree_destroy.argtypes = [vp]
        L.orc_kdtree_num_nodes.restype = C.c_size_t
        L.orc_kdtree_num_nodes.argtypes = [vp]
        L.orc_kdtree_knn.argtypes = [vp, dp, C.c_size_t, C.c_int, C.c_double, C.POINTER(C.c_uint64), dp, ip, C.c_int]
        L.orc_estimate_covariances.argtypes = [vp, C.c_int, dp, C.c_int, dp]
        L.orc_vgicp_create.restype = vp
        L.orc_vgicp_create.argtypes = [vp, vp]
        L.orc_gicp_create.restype = vp
        L.orc_gicp_create.argtypes = [vp, vp, vp]
        L.orc_factor_destroy.argtypes = [vp]
        L.orc_factor_set_num_threads.argtypes = [vp, C.c_int]
        L.orc_factor_set_max_correspondence_distance.argtypes = [vp, C.c_double]
        L.orc_factor_linearize.argtypes = [vp, dp, dp]
        L.orc_factor_error.restype = C.c_double
        L.orc_factor_error.argtypes = [vp, dp]
        L.orc_factor_correspondences.argtypes = [vp, lp]
        L.orc_calc_delta.argtypes = [dp, dp, dp]
        L.orc_max_threads.restype = C.c_int
        L.orc_icp_create.restype = vp
        L.orc_icp_create.argtypes = [vp, vp, vp, C.c_int]
        L.orc_cloud_set_normals.argtypes = [vp, dp]
        L.orc_factor_set_fused_cov_cache_mode.argtypes = [vp, C.c_int]
        L.orc_factor_set_correspondence_update_tolerance.argtypes = [vp, C.c_double, C.c_double]
        L.orc_overlap.restype = C.c_double
        L.orc_overlap.argtypes = [vp, vp, dp]
        L.orc_overlap_multi.restype = C.c_double
        L.orc_overlap_multi.argtypes = [C.POINTER(vp), C.c_int, vp, dp]
        L.orc_voxelmap_save_compact.restype = C.c_int
        L.orc_voxelmap_save_compact.argtypes = [vp, C.c_char_p]
        L.orc_voxelmap_load.restype = vp
        L.orc_voxelmap_load.argtypes = [C.c_char_p]
        L.orc_merge_frames.restype = C.c_size_t
        L.orc_merge_frames.argtypes = [dp, C.POINTER(vp), C.c_int, C.c_double, dp, dp]
        _LIB = L
    return _LIB


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def unpack_linearized(buf):
    buf = np.asarray(buf, dtype=np.float64)
    return dict(
        H_target=buf[0:36].reshape(6, 6).copy(),
        H_source=buf[36:72].reshape(6, 6).copy(),
        H_target_source=buf[72:108].reshape(6, 6).copy(),
        b_target=buf[108:114].copy(),
        b_source=buf[114:120].copy(),
        error=float(buf[120]),
        num_inliers=int(buf[121]),
    )


class Cloud:
    def __init__(self, pts, covs=None):
        self.pts = np.ascontiguousarray(pts, dtype=np.float64)
        self.covs = None if covs is None else np.ascontiguousarray(covs, dtype=np.float64).reshape(len(pts), 9)
        self.n = len(self.pts)
        dummy = np.zeros(1)  # keep the pointers non-NULL for empty clouds
        self.h = lib().orc_cloud_create(_dp(self.pts) if self.n else _dp(dummy), None if self.covs is None else (_dp(self.covs) if self.n else _dp(dummy)), self.n)

    def set_normals(self, normals):
        self.normals = np.ascontiguousarray(normals, dtype=np.float64).reshape(self.n, 3)
        lib().orc_cloud_set_normals(self.h, _dp(self.normals))

    def __del__(self):
        if getattr(self, "h", None):
            lib().orc_cloud_destroy(self.h)
            self.h = None


class VoxelMap:
    def __init__(self, resolution, _handle=None):
        self.resolution = resolution
        self.h = _handle if _handle is not None else lib().orc_voxelmap_create(resolution)
        self._clouds = []

    def insert(self, cloud: Cloud):
        lib().orc_voxelmap_insert(self.h, cloud.h)

    def set_lru(self, horizon, clear_cycle):
        lib().orc_voxelmap_set_lru(self.h, int(horizon), int(clear_cycle))

    def overlap(self, source: Cloud, T_target_source) -> float:
        T = np.ascontiguousarray(T_target_source, dtype=np.float64).reshape(16)
        return lib().orc_overlap(self.h, source.h, _dp(T))

    def save_compact(self, path):
        if lib().orc_voxelmap_save_compact(self.h, str(path).encode()) != 0:
            raise IOError(path)

    @staticmethod
    def load(path):
        h = lib().orc_voxelmap_load(str(path).encode())
        if not h:
            raise IOError(path)
        vm = VoxelMap(1.0, _handle=h)
        return vm

    @property
    def num_voxels(self):
        return lib().orc_voxelmap_num_voxels(self.h)

    def export(self):
        V = self.num_voxels
        coords = np.zeros((V, 3), dtype=np.int32)
        means = np.zeros((V, 3))
        covs = np.zeros((V, 3, 3))
        n = np.zeros(V, dtype=np.int32)
        lib().orc_voxelmap_export(self.h, coords.ctypes.data_as(C.POINTER(C.c_int32)), _dp(means), _dp(covs), n.ctypes.data_as(C.POINTER(C.c_int32)))
        return dict(coords=coords, means=means, covs=covs, n=n, resolution=self.resolution)

    def lookup(self, xyz):
        xyz = np.ascontiguousarray(xyz, dtype=np.float64)
        out = np.zeros(len(xyz), dtype=np.int32)
        lib().orc_voxelmap_lookup(self.h, _dp(xyz), len(xyz), out.ctypes.data_as(C.POINTER(C.c_int32)))
        return out

    def __del__(self):
        if getattr(self, "h", None):
            lib().orc_voxelmap_destroy(self.h)
            self.h = None


def estimate_covariances(points, k_neighbors=10, eigen_values=(1e-3, 1.0, 1.0), num_threads=1):
    """estimate_covariances(points, k, eigen_values, num_threads) of the reference (EIG regularisation) -> n x 3 x 3."""
    cloud = Cloud(points)
    out = np.zeros((len(points), 3, 3))
    ev = np.ascontiguousarray(eigen_values, dtype=np.float64)
    lib().orc_estimate_covariances(cloud.h, int(k_neighbors), _dp(ev), int(num_threads), _dp(out))
    return out


def overlap_multi(targets, source: Cloud, Ts_target_source) -> float:
    Ts = np.ascontiguousarray(Ts_target_source, dtype=np.float64).reshape(len(targets), 16)
    arr = (C.c_void_p * len(targets))(*[t.h for t in targets])
    return lib().orc_overlap_multi(arr, len(targets), source.h, _dp(Ts))


def merge_frames(poses, frames, resolution):
    poses = np.ascontiguousarray(poses, dtype=np.float64).reshape(len(frames), 16)
    total = sum(f.n for f in frames)
    xyz, cov = np.zeros((total, 3)), np.zeros((total, 3, 3))
    arr = (C.c_void_p * len(frames))(*[f.h for f in frames])
    m = lib().orc_merge_frames(_dp(poses), arr, len(frames), float(resolution), _dp(xyz), _dp(cov))
    return xyz[:m].copy(), cov[:m].copy()


class KdTree:
    def __init__(self, cloud: Cloud, num_threads=1):
        self.cloud = cloud
        self.h = lib().orc_kdtree_create(cloud.h, num_threads)

    @property
    def num_nodes(self):
        return lib().orc_kdtree_num_nodes(self.h)

    def knn(self, queries, k, max_sq_dist=np.finfo(np.float64).max, num_threads=1):
        q = np.ascontiguousarray(queries, dtype=np.float64)
        idx = np.zeros((len(q), k), dtype=np.uint64)
        sqd = np.zeros((len(q), k))
        found = np.zeros(len(q), dtype=np.int32)
        lib().orc_kdtree_knn(
            self.h, _dp(q), len(q), k, max_sq_dist, idx.ctypes.data_as(C.POINTER(C.c_uint64)), _dp(sqd), found.ctypes.data_as(C.POINTER(C.c_int32)), num_threads
        )
        return idx.view(np.int64), sqd, found

    def __del__(self):
        if getattr(self, "h", None):
            lib().orc_kdtree_destroy(self.h)
            self.h = None


class Factor:
    """IntegratedVGICPFactor (target = VoxelMap) or IntegratedGICPFactor (target = Cloud + KdTree)."""

    FULL, COMPACT, NONE = 0, 1, 2

    def __init__(self, target, source: Cloud, tree: KdTree = None, num_threads=1, icp=None):
        """icp: None (GICP / VGICP), "point" (IntegratedICPFactor) or "plane" (IntegratedPointToPlaneICPFactor)."""
        self.target, self.source, self.tree = target, source, tree
        if isinstance(target, VoxelMap):
            self.h = lib().orc_vgicp_create(target.h, source.h)
        elif icp:
            self.h = lib().orc_icp_create(target.h, tree.h, source.h, 1 if icp == "plane" else 0)
        else:
            self.h = lib().orc_gicp_create(target.h, tree.h, source.h)
        lib().orc_factor_set_num_threads(self.h, num_threads)

    def set_fused_cov_cache_mode(self, mode):
        lib().orc_factor_set_fused_cov_cache_mode(self.h, int(mode))

    def set_correspondence_update_tolerance(self, angle, trans):
        lib().orc_factor_set_correspondence_update_tolerance(self.h, float(angle), float(trans))

    def set_num_threads(self, n):
        lib().orc_factor_set_num_threads(self.h, n)

    def set_max_correspondence_distance(self, d):
        lib().orc_factor_set_max_correspondence_distance(self.h, d)

    def linearize_raw(self, delta):
        d = np.ascontiguousarray(delta, dtype=np.float64).reshape(16)
        out = np.zeros(LINEARIZED_DOUBLES)
        lib().orc_factor_linearize(self.h, _dp(d), _dp(out))
        return out

    def linearize(self, delta):
        return unpack_linearized(self.linearize_raw(delta))

    def error(self, delta):
        d = np.ascontiguousarray(delta, dtype=np.float64).reshape(16)
        return lib().orc_factor_error(self.h, _dp(d))

    def correspondences(self):
        out = np.zeros(self.source.n, dtype=np.int64)
        lib().orc_factor_correspondences(self.h, out.ctypes.data_as(C.POINTER(C.c_int64)))
        return out

    def __del__(self):
        if getattr(self, "h", None):
            lib().orc_factor_destroy(self.h)
            self.h = None


def calc_delta(T_target, T_source):
    a = np.ascontiguousarray(T_target, dtype=np.float64).reshape(16)
    b = np.ascontiguousarray(T_source, dtype=np.float64).reshape(16)
    d = np.zeros(16)
    lib().orc_calc_delta(_dp(a), _dp(b), _dp(d))
    return d.reshape(4, 4)


def max_threads():
    return lib().orc_max_threads()
