"""ctypes binding of the CPU oracle (oracle/ppf_oracle.cpp).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs.  The product package never imports this module.
PARITY UNPINNED (see oracle/ppf_oracle.h).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "_build", "libppf_oracle.so")

FEATURE_PCL_PFH, FEATURE_DROST_COS, FEATURE_DROST_ANGLE = 0, 1, 2
ALPHA_MODE_A, ALPHA_MODE_B = 0, 1
NALPHA_CEIL, NALPHA_FLOOR_DROP, NALPHA_FLOOR_CLAMP = 0, 1, 2
BIN_NAN, BIN_DROPPED = 0xFFFFFFFF, 0xFFFFFFFE

HYP_DTYPE = np.dtype(
    [("pose", np.float32, (12,)), ("votes", np.uint32), ("model_index", np.uint32),
     ("alpha_bin", np.uint32), ("scene_index", np.uint32)]
)
assert HYP_DTYPE.itemsize == 64


def build(force: bool = False) -> str:
    """Compile the oracle with the committed Makefile (g++, no external dependencies)."""
    src = [os.path.join(_HERE, f) for f in ("ppf_oracle.cpp", "icp_oracle.cpp", "prep_oracle.cpp", "cvppf_oracle.cpp", "ppf_oracle.h", "Makefile")]
    stale = (not os.path.exists(_LIB_PATH)) or any(
        os.path.getmtime(s) > os.path.getmtime(_LIB_PATH) for s in src)
    if force or stale:
        subprocess.run(["make", "-C", _HERE] + (["-B"] if force else []), check=True,
                       stdout=subprocess.DEVNULL)
    return _LIB_PATH


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            build()
        _lib = C.CDLL(_LIB_PATH)
        _declare(_lib)
    return _lib


def _declare(L):
    fp, vp, sz = C.POINTER(C.c_float), C.c_void_p, C.c_size_t
    L.oracle_pair_feature.argtypes = [C.c_int, vp, vp, vp, vp, vp]
    L.oracle_pair_feature.restype = C.c_int
    L.oracle_alpha.argtypes = [vp, vp, vp]
    L.oracle_alpha.restype = C.c_float
    L.oracle_ref_frame.argtypes = [vp, vp, vp, vp]
    L.oracle_ppf_estimation.argtypes = [C.c_int, vp, sz, vp]
    L.oracle_ppf_estimation.restype = sz
    L.oracle_ppf_estimation_mt.argtypes = [C.c_int, vp, sz, vp, C.c_int]
    L.oracle_ppf_estimation_mt.restype = sz
    L.oracle_hashmap_create.argtypes = [C.c_float, C.c_float]
    L.oracle_hashmap_create.restype = vp
    L.oracle_hashmap_destroy.argtypes = [vp]
    L.oracle_hashmap_set_features.argtypes = [vp, vp, sz]
    L.oracle_hashmap_set_features_mt.argtypes = [vp, vp, sz, C.c_int]
    L.oracle_vote_accumulate_from_pairs_mt.argtypes = [vp, C.c_int, sz, sz, vp, vp, vp, C.c_int]
    L.oracle_vote_accumulate_from_pairs_mt.restype = C.c_uint64
    L.oracle_hashmap_model_diameter.argtypes = [vp]
    L.oracle_hashmap_model_diameter.restype = C.c_float
    L.oracle_hashmap_num_entries.argtypes = [vp]
    L.oracle_hashmap_num_entries.restype = sz
    L.oracle_hashmap_num_keys.argtypes = [vp]
    L.oracle_hashmap_num_keys.restype = sz
    L.oracle_hashmap_quantise.argtypes = [vp, vp, vp]
    L.oracle_hashmap_query.argtypes = [vp, C.c_float, C.c_float, C.c_float, C.c_float, vp, sz]
    L.oracle_hashmap_query.restype = sz
    L.oracle_hashmap_query_key.argtypes = [vp, vp, vp, sz]
    L.oracle_hashmap_query_key.restype = sz
    L.oracle_hashmap_dump_keys.argtypes = [vp, vp, vp]
    L.oracle_hashmap_set_nalpha_rule.argtypes = [vp, C.c_int]
    L.oracle_num_alpha_bins.argtypes = [C.c_float, C.c_int]
    L.oracle_num_alpha_bins.restype = C.c_uint32
    L.oracle_alpha_bin.argtypes = [C.c_int, C.c_int, C.c_float, C.c_float, C.c_float]
    L.oracle_alpha_bin.restype = C.c_uint32
    L.oracle_scene_pairs.argtypes = [vp, C.c_int, vp, sz, sz, vp, vp, vp]
    L.oracle_scene_pairs.restype = sz
    L.oracle_vote_accumulate.argtypes = [vp, C.c_int, C.c_int, sz, vp, sz, sz, vp]
    L.oracle_vote_accumulate.restype = C.c_uint64
    L.oracle_vote_accumulate_from_pairs.argtypes = [vp, C.c_int, sz, sz, vp, vp, vp]
    L.oracle_vote_accumulate_from_pairs.restype = C.c_uint64
    L.oracle_vote.argtypes = [vp, C.c_int, C.c_int, vp, sz, vp, sz, sz, sz, sz, C.c_int, vp, vp]
    L.oracle_vote.restype = C.c_int
    L.oracle_vote_refs.argtypes = [vp, C.c_int, C.c_int, vp, sz, vp, sz, vp, sz, C.c_int, vp, vp]
    L.oracle_vote_refs.restype = C.c_int
    L.oracle_peak_pose.argtypes = [C.c_int, C.c_float, vp, sz, C.c_uint32, vp, sz, vp]
    L.oracle_cluster.argtypes = [vp, sz, C.c_float, C.c_float, vp, vp, vp, vp]
    L.oracle_cluster.restype = sz
    L.oracle_poses_within.argtypes = [vp, vp, C.c_float, C.c_float]
    L.oracle_poses_within.restype = C.c_int
    L.oracle_transform.argtypes = [vp, sz, vp, vp]
    L.oracle_register.argtypes = [vp, C.c_int, C.c_int, vp, sz, vp, sz, sz, C.c_float, C.c_float,
                                  C.c_int, vp, vp, vp, vp]
    L.oracle_register.restype = sz
    L.oracle_max_threads.restype = C.c_int
    L.oracle_voxel_grid.argtypes = [vp, sz, sz, vp, vp, C.POINTER(C.c_int)]
    L.oracle_voxel_grid.restype = sz
    L.oracle_knn.argtypes = [vp, sz, sz, C.c_int, vp, vp, C.c_int]
    L.oracle_sor.argtypes = [vp, sz, sz, C.c_int, C.c_double, vp, vp, C.POINTER(C.c_double), C.c_int]
    L.oracle_sor.restype = sz
    L.oracle_normals.argtypes = [vp, sz, sz, C.c_int, vp, C.c_int, vp, C.c_int]
    L.oracle_renormalize_normals.argtypes = [vp, sz, sz]
    L.oracle_frustum_corners.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double,
                                         C.c_double, C.c_double, vp]
    L.oracle_crop_pyramid.argtypes = [vp, sz, sz, vp, vp]
    L.oracle_crop_pyramid.restype = sz
    L.oracle_cv_create.argtypes = [C.c_double, C.c_double, C.c_double]
    L.oracle_cv_create.restype = vp
    L.oracle_cv_destroy.argtypes = [vp]
    L.oracle_cv_set_search_params.argtypes = [vp, C.c_double, C.c_double]
    L.oracle_cv_sample.argtypes = [vp, sz, C.c_float, vp]
    L.oracle_cv_sample.restype = sz
    L.oracle_cv_murmur.argtypes = [C.c_char_p, C.c_int, C.c_uint32]
    L.oracle_cv_murmur.restype = C.c_uint32
    L.oracle_cv_pair.argtypes = [vp, vp, C.c_double, C.c_double, vp]
    L.oracle_cv_pair.restype = C.c_uint32
    L.oracle_cv_train.argtypes = [vp, vp, sz]
    L.oracle_cv_train.restype = sz
    L.oracle_cv_model_points.argtypes = [vp, vp]
    L.oracle_cv_model_points.restype = sz
    L.oracle_cv_match.argtypes = [vp, vp, sz, C.c_double, C.c_double, vp, vp, sz, vp, C.POINTER(sz), C.c_int]
    L.oracle_cv_match.restype = sz
    L.oracle_cv_match_s2b.argtypes = [vp, vp, sz, vp, sz, C.c_double, C.c_double, vp, vp, sz, vp, C.POINTER(sz), C.c_int]
    L.oracle_cv_match_s2b.restype = sz
    L.oracle_cv_table_size.argtypes = [vp]
    L.oracle_cv_table_size.restype = sz
    L.oracle_cv_table_export.argtypes = [vp, vp, vp]
    L.oracle_cv_num_angles.argtypes = [vp]
    L.oracle_cv_num_angles.restype = C.c_int
    L.oracle_cv_bucket.argtypes = [vp, sz, vp, sz]
    L.oracle_cv_bucket.restype = sz
    L.oracle_cv_accumulator.argtypes = [vp, vp, sz, vp, sz, C.c_double, sz, vp]
    L.oracle_cv_accumulator.restype = sz


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def pair_feature(p1, n1, p2, n2, mode=FEATURE_PCL_PFH):
    a = [_f32(x) for x in (p1, n1, p2, n2)]
    f = np.zeros(4, np.float32)
    ok = lib().oracle_pair_feature(mode, *[_p(x) for x in a], _p(f))
    return bool(ok), f


def alpha(p_r, n_r, p):
    a = [_f32(x) for x in (p_r, n_r, p)]
    return float(lib().oracle_alpha(*[_p(x) for x in a]))


def ref_frame(p_r, n_r):
    a = [_f32(x) for x in (p_r, n_r)]
    R = np.zeros(9, np.float32)
    t = np.zeros(3, np.float32)
    lib().oracle_ref_frame(_p(a[0]), _p(a[1]), _p(R), _p(t))
    return R.reshape(3, 3), t


def ppf_estimation(cloud, mode=FEATURE_PCL_PFH, n_threads=1):
    """PPFEstimation::compute -> (N*N, 5) float32, NaN rows for invalid pairs (rows in parallel when n_threads > 1)."""
    cloud = _f32(cloud)
    n = cloud.shape[0]
    out = np.empty((n * n, 5), np.float32)
    lib().oracle_ppf_estimation_mt(mode, _p(cloud), n, _p(out), int(n_threads))
    return out


def host_threads():
    """cores this process may run on (OMP_NUM_THREADS is ignored: torchrun sets it to 1)"""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def num_alpha_bins(angle_step, nalpha_rule=NALPHA_CEIL):
    return int(lib().oracle_num_alpha_bins(np.float32(angle_step), nalpha_rule))


def alpha_bin(alpha_m, alpha_s, angle_step, mode=ALPHA_MODE_A, nalpha_rule=NALPHA_CEIL):
    """bin of one vote; BIN_NAN for a NaN angle, BIN_DROPPED for a vote the FLOOR_DROP rule loses"""
    return int(lib().oracle_alpha_bin(mode, nalpha_rule, np.float32(angle_step), np.float32(alpha_m),
                                      np.float32(alpha_s)))


class HashMap:
    """pcl::PPFHashMapSearch restated (unordered_multimap + alpha_m matrix)."""

    def __init__(self, angle_step=np.float32(12.0 / 180.0 * np.pi), dist_step=np.float32(0.01), nalpha_rule=NALPHA_CEIL):
        self.angle_step = np.float32(angle_step)
        self.dist_step = np.float32(dist_step)
        self._h = lib().oracle_hashmap_create(self.angle_step, self.dist_step)
        self.n = 0
        self.set_nalpha_rule(nalpha_rule)

    def set_nalpha_rule(self, rule):
        """columns of the voting accumulator: NALPHA_CEIL (default) | NALPHA_FLOOR_DROP | NALPHA_FLOOR_CLAMP"""
        self.nalpha_rule = int(rule)
        lib().oracle_hashmap_set_nalpha_rule(self._h, self.nalpha_rule)
        return self

    def __del__(self):
        if getattr(self, "_h", None):
            lib().oracle_hashmap_destroy(self._h)
            self._h = None

    def set_input_feature_cloud(self, feats, n_threads=1):
        """n_threads > 1 builds the container sharded by key (same bucket contents, minutes -> seconds at 10^8 pairs)"""
        feats = _f32(feats).reshape(-1, 5)
        lib().oracle_hashmap_set_features_mt(self._h, _p(feats), feats.shape[0], int(n_threads))
        self.n = int(np.sqrt(np.float32(feats.shape[0])))
        return self

    @property
    def model_diameter(self):
        return float(lib().oracle_hashmap_model_diameter(self._h))

    @property
    def num_entries(self):
        return int(lib().oracle_hashmap_num_entries(self._h))

    @property
    def num_keys(self):
        return int(lib().oracle_hashmap_num_keys(self._h))

    def quantise(self, f):
        f = _f32(f)
        d = np.zeros(4, np.int32)
        lib().oracle_hashmap_quantise(self._h, _p(f), _p(d))
        return d

    def query(self, f1, f2, f3, f4):
        cap = 1024
        while True:
            out = np.zeros((cap, 2), np.uint64)
            n = lib().oracle_hashmap_query(self._h, f1, f2, f3, f4, _p(out), cap)
            if n <= cap:
                return out[:n]
            cap = n

    def query_key(self, d):
        d = np.ascontiguousarray(d, np.int32)
        cap = 1024
        while True:
            out = np.zeros((cap, 2), np.uint64)
            n = lib().oracle_hashmap_query_key(self._h, _p(d), _p(out), cap)
            if n <= cap:
                return out[:n]
            cap = n

    def dump_keys(self):
        k = self.num_keys
        keys = np.zeros((k, 4), np.int32)
        lengths = np.zeros(k, np.uint32)
        lib().oracle_hashmap_dump_keys(self._h, _p(keys), _p(lengths))
        return keys, lengths

    def scene_pairs(self, scene, s_r, mode=FEATURE_PCL_PFH):
        scene = _f32(scene)
        n = scene.shape[0]
        inr = np.zeros(n, np.uint8)
        d = np.zeros((n, 4), np.int32)
        a = np.zeros(n, np.float32)
        lib().oracle_scene_pairs(self._h, mode, _p(scene), n, s_r, _p(inr), _p(d), _p(a))
        return inr, d, a

    def vote_accumulate(self, n_m, scene, s_r, mode=FEATURE_PCL_PFH, alpha_mode=ALPHA_MODE_A):
        scene = _f32(scene)
        acc = np.zeros((n_m, num_alpha_bins(self.angle_step, self.nalpha_rule)), np.uint32)
        votes = lib().oracle_vote_accumulate(self._h, mode, alpha_mode, n_m, _p(scene),
                                             scene.shape[0], s_r, _p(acc))
        return acc, int(votes)

    def vote_accumulate_from_pairs(self, n_m, d, alpha_s, alpha_mode=ALPHA_MODE_A, n_threads=1):
        d = np.ascontiguousarray(d, np.int32).reshape(-1, 4)
        alpha_s = _f32(alpha_s)
        acc = np.zeros((n_m, num_alpha_bins(self.angle_step, self.nalpha_rule)), np.uint32)
        votes = lib().oracle_vote_accumulate_from_pairs_mt(self._h, alpha_mode, n_m, d.shape[0], _p(d),
                                                           _p(alpha_s), _p(acc), int(n_threads))
        return acc, int(votes)

    def vote(self, model, scene, ref_first=0, ref_step=1, ref_count=None, n_threads=1,
             mode=FEATURE_PCL_PFH, alpha_mode=ALPHA_MODE_A):
        model, scene = _f32(model), _f32(scene)
        if ref_count is None:
            ref_count = (scene.shape[0] - ref_first + ref_step - 1) // ref_step
        hyps = np.zeros(ref_count, HYP_DTYPE)
        stats = np.zeros(4, np.uint64)
        rc = lib().oracle_vote(self._h, mode, alpha_mode, _p(model), model.shape[0], _p(scene),
                               scene.shape[0], ref_first, ref_step, ref_count, n_threads,
                               _p(hyps), _p(stats))
        if rc != 0:
            raise RuntimeError("oracle_vote failed (model/table size mismatch?)")
        return hyps, dict(zip(("pairs_examined", "pairs_in_radius", "nonempty_lookups", "votes"),
                              (int(x) for x in stats)))

    def vote_refs(self, model, scene, refs, n_threads=1, mode=FEATURE_PCL_PFH, alpha_mode=ALPHA_MODE_A):
        """the voting loop over an explicit list of reference points -> (hypotheses, counters)"""
        model, scene = _f32(model), _f32(scene)
        refs = np.ascontiguousarray(refs, np.uint64)
        hyps = np.zeros(len(refs), HYP_DTYPE)
        stats = np.zeros(4, np.uint64)
        rc = lib().oracle_vote_refs(self._h, mode, alpha_mode, _p(model), model.shape[0], _p(scene), scene.shape[0],
                                    _p(refs), len(refs), n_threads, _p(hyps), _p(stats))
        if rc != 0:
            raise RuntimeError("oracle_vote_refs failed (model/table size mismatch?)")
        return hyps, dict(zip(("pairs_examined", "pairs_in_radius", "nonempty_lookups", "votes"),
                              (int(x) for x in stats)))

    def register(self, model, scene, ref_rate=5, pos_thr=0.01, rot_thr=20.0 / 180.0 * np.pi,
                 n_threads=1, mode=FEATURE_PCL_PFH, alpha_mode=ALPHA_MODE_A):
        model, scene = _f32(model), _f32(scene)
        final = np.zeros(16, np.float32)
        poses = np.zeros((3, 16), np.float32)
        votes = np.zeros(3, np.uint32)
        stats = np.zeros(4, np.uint64)
        n = lib().oracle_register(self._h, mode, alpha_mode, _p(model), model.shape[0], _p(scene),
                                  scene.shape[0], ref_rate, np.float32(pos_thr), np.float32(rot_thr),
                                  n_threads, _p(final), _p(poses), _p(votes), _p(stats))
        return final.reshape(4, 4), poses[:n].reshape(n, 4, 4), votes[:n], stats


def peak_pose(model, model_index, bin_, scene, s_r, angle_step, alpha_mode=ALPHA_MODE_A):
    model, scene = _f32(model), _f32(scene)
    pose = np.zeros(12, np.float32)
    lib().oracle_peak_pose(alpha_mode, np.float32(angle_step), _p(model), model_index, bin_,
                           _p(scene), s_r, _p(pose))
    return pose.reshape(3, 4)


def cluster(hyps, pos_thr=0.01, rot_thr=20.0 / 180.0 * np.pi):
    hyps = np.ascontiguousarray(hyps, HYP_DTYPE)
    n = hyps.shape[0]
    poses = np.zeros((3, 16), np.float32)
    votes = np.zeros(3, np.uint32)
    assign = np.zeros(n, np.uint32)
    ncl = C.c_size_t(0)
    k = lib().oracle_cluster(_p(hyps), n, np.float32(pos_thr), np.float32(rot_thr), _p(poses),
                             _p(votes), _p(assign), C.byref(ncl))
    return poses[:k].reshape(k, 4, 4), votes[:k], assign, int(ncl.value)


def poses_within(a, b, pos_thr, rot_thr):
    a, b = _f32(a).reshape(-1)[:12], _f32(b).reshape(-1)[:12]
    return bool(lib().oracle_poses_within(_p(a), _p(b), np.float32(pos_thr), np.float32(rot_thr)))


def transform(cloud, pose16):
    cloud = _f32(cloud)
    M = _f32(pose16).reshape(16)
    out = np.zeros((cloud.shape[0], 3), np.float32)
    lib().oracle_transform(_p(cloud), cloud.shape[0], _p(M), _p(out))
    return out


def max_threads():
    return int(lib().oracle_max_threads())


def icp_refine(model, scene, poses, max_iterations=100, tolerance=0.005, rejection_scale=2.5, num_levels=8):
    """ICP::registerModelToScene(model, scene, poses) of the reference (icp_oracle.cpp).
    poses: (P, 4, 4) model -> scene.  Returns (refined (P,4,4) float64, residuals (P,), iterations run)."""
    model, scene = _f32(model), _f32(scene)
    P = np.ascontiguousarray(np.asarray(poses, np.float64).reshape(-1, 4, 4)).copy()
    res = np.zeros(P.shape[0], np.float64)
    iters = C.c_uint64(0)
    L = lib()
    L.oracle_icp_refine.restype = C.c_int
    L.oracle_icp_refine.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_int, C.c_float, C.c_float, C.c_int,
                                    C.c_void_p, C.c_size_t, C.c_void_p, C.POINTER(C.c_uint64)]
    rc = L.oracle_icp_refine(_p(model), model.shape[0], _p(scene), scene.shape[0], max_iterations, tolerance,
                             rejection_scale, num_levels, _p(P), P.shape[0], _p(res), C.byref(iters))
    if rc != 0:
        raise RuntimeError("oracle_icp_refine failed")
    return P, res, int(iters.value)


def solve6(N, g):
    """the ICP's minimum-norm solve of the 6 x 6 Gram system (icp_oracle.cpp solve6)"""
    N = np.ascontiguousarray(np.asarray(N, np.float64).reshape(6, 6)).copy()
    g = np.ascontiguousarray(np.asarray(g, np.float64).reshape(6)).copy()
    x = np.zeros(6, np.float64)
    L = lib()
    L.oracle_icp_solve6.restype = C.c_int
    L.oracle_icp_solve6.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    if L.oracle_icp_solve6(_p(N), _p(g), _p(x)) != 0:
        raise RuntimeError("oracle_icp_solve6 failed")
    return x


# ---- scene pre-processing (prep_oracle.cpp): VoxelGrid, StatisticalOutlierRemoval, NormalEstimationOMP -----------
COV_SHIFTED, COV_RAW = 0, 1  # computeMeanAndCovarianceMatrix of PCL >= 1.12 / PCL 1.8-1.11


def voxel_grid(xyz, leaf):
    """pcl::VoxelGrid<PointXYZ>: (N, >=3) -> (M, 3) centroids in ascending voxel order; (cloud, overflowed)."""
    xyz = _f32(xyz)
    leaf3 = _f32(np.broadcast_to(np.asarray(leaf, np.float32), (3,)))
    out = np.zeros((xyz.shape[0], 3), np.float32)
    status = C.c_int(0)
    m = lib().oracle_voxel_grid(_p(xyz), xyz.shape[0], xyz.shape[1], _p(leaf3), _p(out), C.byref(status))
    return out[:m].copy(), bool(status.value)


def knn(xyz, k, n_threads=None):
    """exact k nearest neighbours (self included), rows sorted by (d2, index): (idx (N,k) uint32, d2 (N,k) float32)"""
    xyz = _f32(xyz)
    k = min(int(k), xyz.shape[0])
    idx = np.zeros((xyz.shape[0], k), np.uint32)
    d2 = np.zeros((xyz.shape[0], k), np.float32)
    lib().oracle_knn(_p(xyz), xyz.shape[0], xyz.shape[1], k, _p(idx), _p(d2), n_threads or max_threads())
    return idx, d2


def statistical_outlier_removal(xyz, mean_k=50, std_mul=1.0, n_threads=None):
    """pcl::StatisticalOutlierRemoval<PointXYZ>: -> (keep mask (N,) bool, mean distances (N,), threshold)"""
    xyz = _f32(xyz)
    n = xyz.shape[0]
    dist = np.zeros(n, np.float32)
    keep = np.zeros(n, np.uint8)
    thr = C.c_double(0.0)
    lib().oracle_sor(_p(xyz), n, xyz.shape[1], mean_k, float(std_mul), _p(dist), _p(keep), C.byref(thr),
                     n_threads or max_threads())
    return keep.astype(bool), dist, thr.value


def normals(xyz, k=30, viewpoint=(0.0, 0.0, 0.0), cov_mode=COV_SHIFTED, n_threads=None):
    """pcl::NormalEstimationOMP<PointXYZ, Normal>::compute with setKSearch(k): -> (N, 4) [nx ny nz curvature]"""
    xyz = _f32(xyz)
    vp3 = _f32(viewpoint)
    out = np.zeros((xyz.shape[0], 4), np.float32)
    lib().oracle_normals(_p(xyz), xyz.shape[0], xyz.shape[1], k, _p(vp3), cov_mode, _p(out), n_threads or max_threads())
    return out


def renormalize_normals(nrm):
    """CloudProcessor::PointCloudXYZNormalToMat's normal re-normalisation; returns a new (N, 3) array"""
    out = _f32(nrm).copy()
    lib().oracle_renormalize_normals(_p(out), out.shape[0], out.shape[1])
    return out


def frustum_corners(depth, box, intrinsics):
    """SceneCropping's four far corners (left_top, left_bot, right_top, right_bot) for box = (x, y, w, h) and
    intrinsics = (fx, fy, ppx, ppy): -> (4, 3) float32"""
    depth = np.ascontiguousarray(depth, np.float32)
    out = np.zeros((4, 3), np.float32)
    fx, fy, ppx, ppy = (float(v) for v in intrinsics)
    lib().oracle_frustum_corners(_p(depth), depth.shape[0], depth.shape[1], int(box[0]), int(box[1]), int(box[2]), int(box[3]),
                                 fx, fy, ppx, ppy, _p(out))
    return out


def crop_pyramid(xyz, corners):
    """ConvexHull{corners, origin} + CropHull: boolean mask of the points inside"""
    xyz = _f32(xyz)
    corners = _f32(corners).reshape(12)
    keep = np.zeros(xyz.shape[0], np.uint8)
    lib().oracle_crop_pyramid(_p(xyz), xyz.shape[0], xyz.shape[1], _p(corners), _p(keep))
    return keep.astype(bool)


# ---- the engine the reference actually calls: cv::ppf_match_3d::PPF3DDetector (cvppf_oracle.cpp) --------------------
def cv_sample(pc, sample_step):
    """samplePCByQuantization over the cloud's own bounding box: (N, 6) -> (M, 6)"""
    pc = _f32(pc)
    out = np.zeros_like(pc)
    m = lib().oracle_cv_sample(_p(pc), pc.shape[0], np.float32(sample_step), _p(out))
    return out[:m].copy()


def cv_murmur(data: bytes, seed: int) -> int:
    """MurmurHash3_x86_32"""
    return int(lib().oracle_cv_murmur(data, len(data), seed))


def cv_pair(p1n1, p2n2, angle_step, distance_step):
    """(computePPFFeatures (4,), hashPPF) of one pair"""
    a, b = _f32(p1n1), _f32(p2n2)
    f = np.zeros(4, np.float64)
    h = lib().oracle_cv_pair(_p(a), _p(b), float(angle_step), float(distance_step), _p(f))
    return f, int(h)


class CvDetector:
    """PPF3DDetector(relativeSamplingStep, relativeDistanceStep = 0.05, numAngles = 30)"""

    def __init__(self, relative_sampling_step, relative_distance_step=0.05, num_angles=30):
        self._h = lib().oracle_cv_create(float(relative_sampling_step), float(relative_distance_step), float(num_angles))

    def __del__(self):
        if getattr(self, "_h", None):
            lib().oracle_cv_destroy(self._h)
            self._h = None

    def set_search_params(self, position_threshold=-1.0, rotation_threshold=-1.0):
        lib().oracle_cv_set_search_params(self._h, float(position_threshold), float(rotation_threshold))

    def train_model(self, model):
        model = _f32(model)
        self.n_model = int(lib().oracle_cv_train(self._h, _p(model), model.shape[0]))
        return self

    def model_points(self):
        out = np.zeros((self.n_model, 6), np.float32)
        lib().oracle_cv_model_points(self._h, _p(out))
        return out

    def match(self, scene, relative_scene_sample_step=1.0 / 5.0, relative_scene_distance=0.03, max_poses=16, n_threads=None):
        """-> (poses (P, 4, 4) float64, cluster votes (P,), raw per-reference (votes, model index, alpha index), #clusters)"""
        scene = _f32(scene)
        poses = np.zeros((max_poses, 16), np.float64)
        votes = np.zeros(max_poses, np.uint32)
        raw = np.zeros((scene.shape[0], 3), np.uint32)
        n_refs = C.c_size_t(0)
        ncl = lib().oracle_cv_match(self._h, _p(scene), scene.shape[0], float(relative_scene_sample_step),
                                    float(relative_scene_distance), _p(poses), _p(votes), max_poses, _p(raw), C.byref(n_refs),
                                    n_threads or max_threads())
        k = min(int(ncl), max_poses)
        return poses[:k].reshape(-1, 4, 4), votes[:k], raw[:n_refs.value].copy(), int(ncl)

    def match_s2b(self, scene, edge, relative_scene_sample_step=1.0 / 5.0, relative_scene_distance=0.03, max_poses=16, n_threads=None):
        """the fork's match_S2B as inferred: reference points from the scene, paired with the edge cloud; returns as match()"""
        scene, edge = _f32(scene), _f32(edge)
        poses = np.zeros((max_poses, 16), np.float64)
        votes = np.zeros(max_poses, np.uint32)
        raw = np.zeros((scene.shape[0], 3), np.uint32)
        n_refs = C.c_size_t(0)
        ncl = lib().oracle_cv_match_s2b(self._h, _p(scene), scene.shape[0], _p(edge), edge.shape[0], float(relative_scene_sample_step),
                                        float(relative_scene_distance), _p(poses), _p(votes), max_poses, _p(raw), C.byref(n_refs),
                                        n_threads or max_threads())
        k = min(int(ncl), max_poses)
        return poses[:k].reshape(-1, 4, 4), votes[:k], raw[:n_refs.value].copy(), int(ncl)

    @property
    def table_size(self):
        return int(lib().oracle_cv_table_size(self._h))

    def bucket(self, b):
        """ppfInd = i * M + j of the nodes chained in bucket b, ascending"""
        n = int(lib().oracle_cv_bucket(self._h, int(b), None, 0))
        out = np.zeros(n, np.uint32)
        if n:
            lib().oracle_cv_bucket(self._h, int(b), _p(out), n)
        return out

    @property
    def num_angles(self):
        """accumulator columns of the trained detector: floor(2 pi / angle_step)"""
        return int(lib().oracle_cv_num_angles(self._h))

    def table_export(self):
        """(offsets (table_size + 1,), nodes (M * (M - 1),)): the buckets as a CSR, nodes ascending inside a bucket"""
        off = np.zeros(self.table_size + 1, np.uint32)
        nodes = np.zeros(max(1, self.n_model * (self.n_model - 1)), np.uint32)
        lib().oracle_cv_table_export(self._h, _p(off), _p(nodes))
        return off, nodes[:self.n_model * (self.n_model - 1)]

    def accumulator(self, scene, sampled_index, relative_scene_distance, edge=None):
        """accumulator (M, num_angles) of the sampled scene point sampled_index"""
        scene = _f32(scene)
        edge = None if edge is None else _f32(edge)
        acc = np.zeros((self.n_model, self.num_angles), np.uint32)
        lib().oracle_cv_accumulator(self._h, _p(scene), scene.shape[0], _p(edge) if edge is not None else None,
                                    0 if edge is None else edge.shape[0], float(relative_scene_distance), int(sampled_index), _p(acc))
        return acc
