"""GPU tests: every host path returns the device memory it takes from the stream-ordered pool.

The library allocates clouds, tables and call-scoped scratch from the device's default memory pool, whose release
threshold b200ppf_create sets to "keep everything": memory a path forgets to free is never given back while the process
lives.  Each case runs three times and reads the pool's used-memory counter (cudaMemPoolAttrUsedMemCurrent, a read-only
query) after a device synchronisation: after a successful round whose handles are freed, and after each error that
inputs can reach once the table build has allocated, it must be back at its starting value.
"""
import ctypes
import os

import numpy as np
import pytest

from conftest import ANGLE_STEP, DIST_STEP, GOLDEN, load_cloud

pytestmark = pytest.mark.gpu

POOL_ATTR_USED_MEM_CURRENT = 0x7


def _cudart():
    for name in ("libcudart.so.12", os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "lib64", "libcudart.so.12")):
        try:
            return ctypes.CDLL(name)
        except OSError:
            continue
    pytest.fail("libcudart.so.12 not found")


@pytest.fixture(scope="module")
def pool_used():
    rt = _cudart()
    pool = ctypes.c_void_p()
    assert rt.cudaDeviceGetDefaultMemPool(ctypes.byref(pool), 0) == 0

    def used():
        assert rt.cudaDeviceSynchronize() == 0
        v = ctypes.c_uint64(0)
        assert rt.cudaMemPoolGetAttribute(pool, POOL_ATTR_USED_MEM_CURRENT, ctypes.byref(v)) == 0
        return v.value

    return used


@pytest.fixture(scope="module")
def setup(ctx, bottle, scene_crop):
    dm, ds = ctx.upload_cloud(bottle), ctx.upload_cloud(scene_crop)
    return dm, ds, ctx.table_build_from_cloud(dm, ANGLE_STEP, DIST_STEP)


def _rounds(pool_used, run):
    start = pool_used()
    for k in range(3):
        run()
        assert pool_used() == start, f"round {k}: {pool_used() - start} bytes still taken from the pool"


def _free(*handles):
    for h in handles:
        if h is not None:
            h.free()


def test_cloud_paths_return_their_memory(ctx, pool_used, bottle, setup):
    dm, ds, _ = setup
    raw = np.load(os.path.join(GOLDEN, "scene_crop_raw.npz"))["cloud"][::4].copy()

    def upload():
        _free(ctx.upload_cloud(bottle), ctx.upload_xyz(raw))

    def prep():
        xyz = ctx.upload_xyz(raw)
        vox = ctx.voxel_grid(xyz, 0.01)
        kept, _, _, _ = ctx.statistical_outlier_removal(vox, 20, 1.0)
        ctx.normal_estimation(kept, 30)
        edges = ctx.curvature_edges(kept, 0.03)
        ctx.normalize_normals(kept)
        ctx.knn(kept, 8)
        kept.download(curvature=True)
        _free(xyz, vox, kept, edges)

    def transform():
        ctx.transform(ds, np.eye(4, dtype=np.float32))

    def icp():
        ctx.icp_refine(dm, ds, [np.eye(4)], max_iterations=5, num_levels=2)

    for run in (upload, prep, transform, icp):
        _rounds(pool_used, run)


def test_table_paths_return_their_memory(ctx, pool_used, tmp_path, setup):
    from yolo_ppf_pose_estimation_b200 import capi
    dm, ds, table = setup
    path = str(tmp_path / "t.bin")

    def build():
        f = ctx.features_compute(dm)
        t1 = ctx.table_build(f, ANGLE_STEP, DIST_STEP)
        t2 = ctx.table_build_from_cloud(dm, ANGLE_STEP, DIST_STEP)
        _free(f, t1, t2)

    def save_load_clone():
        table.save(path)
        loaded = ctx.table_load(path)
        h = ctypes.c_void_p()
        ctx.check(capi.lib().b200ppf_table_clone(ctx._h, loaded._h, ctypes.byref(h)))
        _free(loaded, capi.Table(ctx, h))

    def alpha_m():
        table.alpha_m()

    for run in (build, save_load_clone, alpha_m):
        _rounds(pool_used, run)


def test_match_paths_return_their_memory(ctx, pool_used, setup):
    from yolo_ppf_pose_estimation_b200 import capi
    dm, ds, table = setup

    def vote_cluster():
        hyps = ctx.vote(dm, table, ds, 0, 5)
        ctx.cluster(hyps)
        ctx.register(dm, table, ds, ref_rate=5)

    def debug_hooks():
        ctx.vote_debug_pairs(table, ds, 0)
        ctx.vote_debug_accumulator(table, ds, 0)
        capi.debug_alpha_bins(np.zeros(8, np.float32), np.linspace(-3, 3, 8).astype(np.float32), ANGLE_STEP, ctx=ctx)
        keys = np.arange(3000, 0, -1, dtype=np.uint32) // 7
        ctx.debug_radix_sort(keys, 3000, v0=keys, v1=keys, v0_iota=True)
        ctx.debug_lower_bounds(np.sort(keys), 100, 2, dev_len=1000)
        ctx.debug_flag_scan(keys % 2)
        ctx.debug_flag_scan(keys % 2, host_total=True)
        ctx.debug_scan_rows(keys, 3, 1000)
        ctx.debug_run_heads(np.sort(keys))

    for run in (vote_cluster, debug_hooks):
        _rounds(pool_used, run)


def test_object_paths_return_their_memory(ctx, pool_used, bottle, scene_full):
    from yolo_ppf_pose_estimation_b200 import capi
    b = np.load(os.path.join(GOLDEN, "crop_box.npz"))
    depth = np.zeros(tuple(b["image"]), np.float32)
    for (r, c), d in zip(b["pixels"], b["depths"]):
        depth[r, c] = d
    cor = capi.frustum_corners(depth, b["box"], b["intrinsics"])
    scene, model = ctx.upload_xyz(scene_full[:, :3]), ctx.upload_cloud(bottle)
    table = ctx.table_build_from_cloud(model, ANGLE_STEP, DIST_STEP)
    det = capi.CvDetector(ctx, 0.025, 0.05).train_model(bottle)

    def match_object():
        _, obj, edges = ctx.match_object(scene, cor, model, table)
        _free(obj, edges)

    def cv_match_object():
        _, obj, edges = ctx.cv_match_object(det, scene, cor, model)
        _free(obj, edges)

    def cv_train():
        capi.CvDetector(ctx, 0.025, 0.05).train_model(bottle).close()

    for run in (match_object, cv_match_object, cv_train):
        _rounds(pool_used, run)
    _free(scene, model, table)
    det.close()


def test_table_build_errors_return_their_memory(ctx, pool_used, bottle, setup):
    from yolo_ppf_pose_estimation_b200.capi import B200PPFError
    dm = setup[0]
    long_normals = bottle.copy()
    long_normals[:, 3:] *= 2.0
    dl = ctx.upload_cloud(long_normals)
    model = load_cloud("bottle_1cm")[::4].copy()
    dsmall = ctx.upload_cloud(model)
    f = ctx.features_compute(dsmall).download()
    n = dsmall.size
    ij = next(k for k in range(n * n) if k // n != k % n and np.isfinite(f[k]).all())
    f[ij, 4] = 4.0  # an alpha_m outside [-pi, pi]

    def too_fine():  # a distance step this fine multiplies the key space past 2^31
        with pytest.raises(B200PPFError, match="discretisation too fine"):
            ctx.table_build_from_cloud(dm, ANGLE_STEP, 1e-7)

    def off_range():
        with pytest.raises(B200PPFError, match="left the analytic key range"):
            ctx.table_build_from_cloud(dl, ANGLE_STEP, DIST_STEP)

    def bad_alpha():
        feats = ctx.features_upload(f)
        with pytest.raises(B200PPFError, match="alpha_m lies outside"):
            ctx.table_build(feats, ANGLE_STEP, DIST_STEP)
        _free(feats)

    for run in (too_fine, off_range, bad_alpha):
        _rounds(pool_used, run)
    _free(dl, dsmall)
