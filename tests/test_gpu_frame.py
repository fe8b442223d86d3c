"""GPU tests of the frame calls: every box of a frame in one call (b200ppf_crop_pyramids, b200ppf_icp_refine_batch,
b200cv_match_frame, b200ppf_match_frame), and of the per-object calls as frames of one box.

Bars: the multi-box crop equals one crop per box bit for bit (rows, order, bounding box); the batched ICP equals one
icp_refine per job bit for bit (poses, residuals, summed iterations) with one launch per distinct cluster size; a frame call
equals the per-object calls box by box in every result field but the times; a failed box leaves the others as they would
be alone; errors of the call itself leave the default pool's used-memory counter where it was; a per-object call keeps its
own edge rule (edges for edges_out, or for Matching_S2B) and rejects handles of another context.
"""
import ctypes
import gc
import os
import subprocess

import numpy as np
import pytest

from conftest import ANGLE_STEP, DIST_STEP, ROOT

pytestmark = pytest.mark.gpu

INVALID, STATE, UNSUPPORTED = -1, -4, -5
POOL_ATTR_USED_MEM_CURRENT = 0x7
FIELDS = ("residual", "votes", "n_poses", "n_cropped", "n_sampled", "n_filtered", "n_edges")
N_LIBRARY = 8


@pytest.fixture(scope="module")
def pool_used():
    """the default pool's used-memory counter after a device synchronisation (the method of test_gpu_device_memory.py)"""
    rt = None
    for name in ("libcudart.so.12", os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "lib64", "libcudart.so.12")):
        try:
            rt = ctypes.CDLL(name)
            break
        except OSError:
            continue
    assert rt is not None, "libcudart.so.12 not found"
    pool = ctypes.c_void_p()
    assert rt.cudaDeviceGetDefaultMemPool(ctypes.byref(pool), 0) == 0

    def used():
        gc.collect()  # handles of earlier tests that wait in a reference cycle go back to the pool before the count
        assert rt.cudaDeviceSynchronize() == 0
        v = ctypes.c_uint64(0)
        assert rt.cudaMemPoolGetAttribute(pool, POOL_ATTR_USED_MEM_CURRENT, ctypes.byref(v)) == 0
        return v.value

    return used


def _library_box(model, k):
    """the far corners of library instance k's box: its projection grown by 0.03 on the image plane, 0.15 m behind it
    (tools/prep_bench.py:frame_case for k = 0)"""
    from yolo_ppf_pose_estimation_b200 import synth
    T = synth.library_pose(k)
    p = model[:, :3].astype(np.float64) @ T[:3, :3].T + T[:3, 3]
    zf = np.float32(p[:, 2].max() + 0.15)
    tx, ty = p[:, 0] / p[:, 2], p[:, 1] / p[:, 2]
    xl, xr, yt, yb = (np.float32(v * zf) for v in (tx.min() - 0.03, tx.max() + 0.03, ty.min() - 0.03, ty.max() + 0.03))
    return np.array([[xl, yt, zf], [xl, yb, zf], [xr, yt, zf], [xr, yb, zf]], np.float32)


@pytest.fixture(scope="module")
def library(ctx):
    """the synthetic 1 Mi-point frame with its 8 library instances: scene cloud, box corners, models (host and device),
    one PPF3DDetector(0.025, 0.05) per model"""
    from yolo_ppf_pose_estimation_b200 import capi, synth
    xyz = np.ascontiguousarray(synth.synth_library_scene(1 << 20)[:, :3], np.float32)
    models = [synth.synth_model(2000, 10 + k, k).astype(np.float32) for k in range(N_LIBRARY)]
    cors = np.stack([_library_box(m, k) for k, m in enumerate(models)])
    dets = [capi.CvDetector(ctx, 0.025, 0.05).train_model(m) for m in models]
    return dict(xyz=xyz, scene=ctx.upload_xyz(xyz), cors=cors, models=models, dmodels=[ctx.upload_cloud(m) for m in models],
                dets=dets)


@pytest.fixture(scope="module")
def reference(ctx, scene_full, bottle):
    """the reference frame (regenerated 1 cm scene, surrogate YOLO box), the bottle model, PPF3DDetector(0.025, 0.05)"""
    from yolo_ppf_pose_estimation_b200 import capi
    b = np.load(os.path.join(ROOT, "tests", "golden", "crop_box.npz"))
    depth = np.zeros(tuple(b["image"]), np.float32)
    for (r, c), d in zip(b["pixels"], b["depths"]):
        depth[r, c] = d
    cor = capi.frustum_corners(depth, b["box"], b["intrinsics"])
    det = capi.CvDetector(ctx, 0.025, 0.05).train_model(bottle)
    return dict(scene=ctx.upload_xyz(scene_full[:, :3]), cor=cor, model=ctx.upload_cloud(bottle), det=det, depth=depth,
                box=b["box"], K=b["intrinsics"])


def _code(fn):
    from yolo_ppf_pose_estimation_b200 import capi
    with pytest.raises(capi.B200PPFError) as e:
        fn()
    return e.value.code


def _same_result(got, want, what):
    assert got["pose"].tobytes() == want["pose"].tobytes(), what
    for f in FIELDS:
        assert np.asarray(got[f]).tobytes() == np.asarray(want[f]).tobytes(), (what, f, got[f], want[f])


def _free(clouds):
    for c in clouds:
        c.free()


# ---- 1. crop -----------------------------------------------------------------------------------------------------------
def _check_crops(ctx, scene, xyz, cors, leaf=0.005):
    many = ctx.crop_pyramids(scene, cors)
    kept_sets = []
    for k, cor in enumerate(cors):
        one, kept = ctx.crop_pyramid(scene, cor)
        rows = one.download(curvature=True)
        assert many[k].size == one.size, k
        assert many[k].download(curvature=True).tobytes() == rows.tobytes(), k
        assert np.array_equal(rows[:, :3], xyz[kept]), k  # the kept points, in input order
        if one.size:  # the voxel grid is laid out from the cloud's bounding box: equal grids, equal boxes
            assert ctx.voxel_grid(many[k], leaf).download().tobytes() == ctx.voxel_grid(one, leaf).download().tobytes(), k
        kept_sets.append(set(kept.tolist()))
        one.free()
    _free(many)
    return kept_sets


def test_crop_pyramids_library_boxes_equal_one_crop_each(ctx, library):
    sets = _check_crops(ctx, library["scene"], library["xyz"], library["cors"])
    assert all(len(s) > 1000 for s in sets)


def test_crop_pyramids_overlap_empty_and_sizes(ctx, library):
    scene, xyz, cors = library["scene"], library["xyz"], library["cors"]
    wide = cors[0].copy()
    wide[:, 0] += np.float32(0.05) * np.sign(wide[:, 0] - wide[:, 0].mean())  # box 0 grown sideways: overlaps box 0
    behind = cors[1] * np.array([1, 1, -1], np.float32)  # a pyramid behind the camera keeps nothing
    sets = _check_crops(ctx, scene, xyz, np.stack([cors[0], wide, behind, cors[4]]))
    assert sets[0] & sets[1] and sets[0] <= sets[1] and len(sets[2]) == 0
    for K in (1, 64):
        n0 = ctx.launch_count
        many = ctx.crop_pyramids(scene, np.repeat(cors[2:3], K, axis=0))
        launches = ctx.launch_count - n0
        one, _ = ctx.crop_pyramid(scene, cors[2])
        ref = one.download(curvature=True).tobytes()
        assert len(many) == K and all(c.download(curvature=True).tobytes() == ref for c in many)
        assert launches == 3, (K, launches)  # mask pass, tile scans, scatter: whatever K is
        _free(many + [one])


def test_crop_pyramids_bad_box_fails_the_call(ctx, library, pool_used):
    cors = library["cors"][:5].copy()
    cors[3, 3, 2] += np.float32(0.1)  # box 3's base is not planar
    start = pool_used()
    with pytest.raises(Exception) as e:
        ctx.crop_pyramids(library["scene"], cors)
    assert e.value.code == UNSUPPORTED and "box 3" in str(e.value)
    assert pool_used() == start
    bad = library["cors"][:2].copy()
    bad[1, 0, 0] = np.float32(np.nan)
    assert _code(lambda: ctx.crop_pyramids(library["scene"], bad)) == INVALID
    assert _code(lambda: ctx.crop_pyramids(library["scene"], np.zeros((65, 12), np.float32))) == INVALID
    assert pool_used() == start


# ---- 2. batched ICP -----------------------------------------------------------------------------------------------------
def _rigid(axis, angle, t):
    axis = np.asarray(axis, np.float64) / np.linalg.norm(axis)
    K = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
    T = np.eye(4)
    T[:3, :3] = np.eye(3) + np.sin(angle) * K + (1 - np.cos(angle)) * K @ K
    T[:3, 3] = t
    return T


@pytest.fixture(scope="module")
def icp_problems(ctx, bottle):
    """(model, scene, start poses) with models of 543 (1 CTA), 2 000 (2 CTAs) and 5 000 points (8 CTAs): the scene is
    the model under a known motion with 0.5 mm noise, the starts are that motion disturbed by a few degrees and cm"""
    from yolo_ppf_pose_estimation_b200 import synth
    rng = np.random.default_rng(11)
    out = []
    for m in (bottle, synth.synth_model(2000, 21, 1), synth.synth_model(5000, 22, 2)):
        m = np.ascontiguousarray(m, np.float32)
        G = _rigid(rng.normal(size=3), 0.6, rng.normal(scale=0.1, size=3) + (0, 0, 0.8))
        sc = np.concatenate([m[:, :3] @ G[:3, :3].T + G[:3, 3] + rng.normal(scale=5e-4, size=(len(m), 3)), m[:, 3:] @ G[:3, :3].T], 1)
        starts = np.stack([_rigid(rng.normal(size=3), 0.05, rng.normal(scale=0.01, size=3)) @ G for _ in range(3)])
        out.append((ctx.upload_cloud(m), ctx.upload_cloud(sc.astype(np.float32)), starts))
    return out


def _batch_equals_single(ctx, jobs):
    got, it = ctx.icp_refine_batch(jobs)
    total = 0
    for (m, s, P), (R, res) in zip(jobs, got):
        if len(P) == 0:
            assert R.shape == (0, 4, 4)
            continue
        R1, res1, it1 = ctx.icp_refine(m, s, P)
        assert R.tobytes() == R1.tobytes() and res.tobytes() == res1.tobytes()
        total += it1
    assert it == total
    return got


def test_icp_batch_equals_one_call_per_job(ctx, icp_problems):
    (b, bs, bp), (l, ls, lp), (g, gs, gp) = icp_problems
    jobs = [(l, ls, lp), (b, bs, bp), (g, gs, gp), (b, bs, bp[::-1]), (l, ls, lp[:0])]  # three sizes, a model twice, 0 poses
    n0 = ctx.launch_count
    ctx.icp_refine_batch(jobs)
    assert ctx.launch_count - n0 == 3  # one launch per distinct cluster size
    _batch_equals_single(ctx, jobs)
    n0 = ctx.launch_count
    got = _batch_equals_single(ctx, [(b, bs, bp), (b, bs, bp[1:]), (b, bs, bp[:1])])
    assert ctx.launch_count - n0 == 1 + 3  # the batch in one launch, then the three single calls
    assert got[0][0][1:].tobytes() == got[1][0].tobytes()  # a pose gives the same bits wherever it sits in a launch


def test_icp_batch_errors(ctx, icp_problems, bottle):
    from yolo_ppf_pose_estimation_b200 import capi
    (b, bs, bp), _, _ = icp_problems
    assert ctx.icp_refine_batch([]) == ([], 0)
    empty = ctx.upload_cloud(bottle[:0])
    assert _code(lambda: ctx.icp_refine_batch([(b, bs, bp), (b, empty, bp)])) == INVALID
    other = capi.Context(0)
    foreign = other.upload_cloud(bottle)
    assert _code(lambda: ctx.icp_refine_batch([(b, bs, bp), (foreign, bs, bp)])) == INVALID
    other.close()


# ---- 3. / 4. frame calls ----------------------------------------------------------------------------------------------
def _axis_angle_deg(R, Rt):
    a, b = R[:3, 2], Rt[:3, 2]  # the models are surfaces of revolution about z: the axis is what a pose fixes
    return float(np.degrees(np.arccos(np.clip(a @ b, -1.0, 1.0))))


@pytest.mark.parametrize("use_edges,icp_poses", [(1, 5), (1, 0), (0, 5), (0, 0)])
def test_cv_match_frame_equals_per_object_calls(ctx, library, use_edges, icp_poses):
    from yolo_ppf_pose_estimation_b200 import synth
    over = dict(leaf=0.005, use_edges=use_edges, icp_poses=icp_poses, relative_scene_sample_step=0.05 if use_edges else 1.0 / 14.0)
    res, status = ctx.cv_match_frame(library["scene"], library["cors"], library["dets"], library["dmodels"], **over)
    assert status.tolist() == [0] * N_LIBRARY
    for k in range(N_LIBRARY):
        one = ctx.cv_match_object(library["dets"][k], library["scene"], library["cors"][k], library["dmodels"][k], **over)[0]
        _same_result(res[k], one, k)
        assert res[k]["crop_ms"] == res[0]["crop_ms"] and res[k]["total_wall_ms"] == res[0]["total_wall_ms"]
        assert (res[k]["icp_ms"] > 0) == (icp_poses > 0)
    if icp_poses:  # a sanity bar, not the parity bar: the instances the chain finds are where synth put them
        found = [k for k in range(N_LIBRARY) if np.linalg.norm(res[k]["pose"][:3, 3] - synth.library_pose(k)[:3, 3]) < 0.01 and
                 _axis_angle_deg(res[k]["pose"], synth.library_pose(k)) < 5.0]
        # resultsSub[0] is the most-voted cluster after ICP, as in the reference; on this frame that cluster is a wrong
        # hypothesis for several instances (per-object call and frame call alike), so the bar names the ones it finds
        assert set(found) >= ({1, 7} if use_edges else {0, 2, 3, 5, 7}), found


def test_cv_match_frame_reference_box_twice(ctx, reference):
    r = reference
    res, status = ctx.cv_match_frame(r["scene"], [r["cor"], r["cor"]], [r["det"], r["det"]], [r["model"], r["model"]], leaf=0.01)
    one = ctx.cv_match_object(r["det"], r["scene"], r["cor"], r["model"], leaf=0.01)[0]
    assert status.tolist() == [0, 0]
    _same_result(res[0], one, 0)
    _same_result(res[1], one, 1)


@pytest.fixture(scope="module")
def library_tables(ctx, library):
    return [ctx.table_build_from_cloud(m, ANGLE_STEP, DIST_STEP) for m in library["dmodels"]]


@pytest.mark.parametrize("icp_poses", [5, 0])
def test_match_frame_equals_per_object_calls(ctx, library, library_tables, icp_poses):
    over = dict(leaf=0.005, ref_rate=20, icp_poses=icp_poses)
    res, status = ctx.match_frame(library["scene"], library["cors"], library["dmodels"], library_tables, **over)
    assert status.tolist() == [0] * N_LIBRARY
    for k in range(N_LIBRARY):
        one = ctx.match_object(library["scene"], library["cors"][k], library["dmodels"][k], library_tables[k], **over)[0]
        _same_result(res[k], one, k)


def test_match_frame_reference_box_twice(ctx, reference, bottle):
    r = reference
    table = ctx.table_build_from_cloud(r["model"], ANGLE_STEP, DIST_STEP)
    res, status = ctx.match_frame(r["scene"], [r["cor"], r["cor"]], [r["model"], r["model"]], [table, table], leaf=0.01, ref_rate=5)
    one = ctx.match_object(r["scene"], r["cor"], r["model"], table, leaf=0.01, ref_rate=5)[0]
    assert status.tolist() == [0, 0]
    _same_result(res[0], one, 0)
    _same_result(res[1], one, 1)


# ---- 5. per-box failure -------------------------------------------------------------------------------------------------
def test_a_failed_box_leaves_the_others(ctx, library, library_tables):
    L = library
    behind = L["cors"][1] * np.array([1, 1, -1], np.float32)
    cors = np.stack([L["cors"][0], behind, L["cors"][2]])
    idx = [0, 1, 2]
    res, status = ctx.cv_match_frame(L["scene"], cors, [L["dets"][k] for k in idx], [L["dmodels"][k] for k in idx], leaf=0.005)
    assert status.tolist() == [0, STATE, 0] and res[1]["n_cropped"] == 0
    for k in (0, 2):
        one = ctx.cv_match_object(L["dets"][k], L["scene"], cors[k], L["dmodels"][k], leaf=0.005)[0]
        _same_result(res[k], one, k)
    assert _code(lambda: ctx.cv_match_object(L["dets"][1], L["scene"], behind, L["dmodels"][1], leaf=0.005)) == STATE
    res, status = ctx.match_frame(L["scene"], cors, [L["dmodels"][k] for k in idx], [library_tables[k] for k in idx], leaf=0.005,
                                  ref_rate=20)
    assert status.tolist() == [0, STATE, 0]
    for k in (0, 2):
        one = ctx.match_object(L["scene"], cors[k], L["dmodels"][k], library_tables[k], leaf=0.005, ref_rate=20)[0]
        _same_result(res[k], one, k)
    # no curvature exceeds 1/3: no edge point for Matching_S2B in any box
    res, status = ctx.cv_match_frame(L["scene"], L["cors"][:2], L["dets"][:2], L["dmodels"][:2], leaf=0.005, edge_curvature=1.0)
    assert status.tolist() == [STATE, STATE] and res[0]["n_edges"] == 0 and res[0]["n_filtered"] > 0
    assert _code(lambda: ctx.cv_match_object(L["dets"][0], L["scene"], L["cors"][0], L["dmodels"][0], leaf=0.005,
                                             edge_curvature=1.0)) == STATE


# ---- 6. / 7. call errors and memory -------------------------------------------------------------------------------------
def test_frame_call_errors_and_memory(ctx, library, library_tables, bottle, pool_used):
    from yolo_ppf_pose_estimation_b200 import capi
    L = library
    dets, mods, cors = L["dets"][:3], L["dmodels"][:3], L["cors"][:3]
    lib = capi.lib()
    # warm: the context's grow-only buffers (not pool memory) reach their size before the counter is read
    ctx.cv_match_frame(L["scene"], cors, dets, mods, leaf=0.005)
    ctx.match_frame(L["scene"], cors, mods, library_tables[:3], leaf=0.005, ref_rate=20)
    start = pool_used()
    for _ in range(3):
        ctx.cv_match_frame(L["scene"], cors, dets, mods, leaf=0.005)
        ctx.match_frame(L["scene"], cors, mods, library_tables[:3], leaf=0.005, ref_rate=20)
        assert pool_used() == start

    c12 = np.ascontiguousarray(cors, np.float32).reshape(-1, 12)
    res = (capi.ObjectResult * 65)()
    status = np.zeros(65, np.int32)
    h_dets = (ctypes.c_void_p * 65)(*([dets[0]._h] * 65))
    h_mods = (ctypes.c_void_p * 65)(*([mods[0]._h] * 65))
    h_tabs = (ctypes.c_void_p * 65)(*([library_tables[0]._h] * 65))
    prm = capi.CvObjectParams()
    lib.b200cv_object_params_default(ctypes.byref(prm))
    cv = lambda n, d=h_dets, m=h_mods, st=status.ctypes.data, c=c12.ctypes.data, r=res: lib.b200cv_match_frame(  # noqa: E731
        ctx._h, L["scene"]._h, n, c, d, m, ctypes.byref(prm), r, st)
    pcl = lambda n, t=h_tabs, st=status.ctypes.data: lib.b200ppf_match_frame(  # noqa: E731
        ctx._h, L["scene"]._h, n, c12.ctypes.data, h_mods, t, None, res, st)
    assert cv(3, d=None) == INVALID and cv(3, m=None) == INVALID and cv(3, st=None) == INVALID and cv(3, c=None) == INVALID
    assert cv(3, r=None) == INVALID and pcl(3, t=None) == INVALID and pcl(3, st=None) == INVALID
    assert cv(0) == INVALID and cv(65) == INVALID and pcl(0) == INVALID and pcl(65) == INVALID
    assert _code(lambda: ctx.cv_match_frame(L["scene"], cors, dets, mods, leaf=0.005, edge_curvature=0.0)) == INVALID
    bad = cors.copy()
    bad[1, 3, 2] += np.float32(0.1)
    assert _code(lambda: ctx.cv_match_frame(L["scene"], bad, dets, mods, leaf=0.005)) == UNSUPPORTED
    untrained = capi.CvDetector(ctx, 0.025, 0.05)
    assert _code(lambda: ctx.cv_match_frame(L["scene"], cors, [dets[0], untrained, dets[2]], mods, leaf=0.005)) == STATE
    other = capi.Context(0)
    f_det = capi.CvDetector(other, 0.025, 0.05).train_model(L["models"][0])
    f_mod = other.upload_cloud(L["models"][0])
    f_scene = other.upload_xyz(L["xyz"][:1000])
    f_tab = other.table_build_from_cloud(f_mod, ANGLE_STEP, DIST_STEP)
    assert _code(lambda: ctx.cv_match_frame(L["scene"], cors, [dets[0], f_det, dets[2]], mods)) == INVALID
    assert _code(lambda: ctx.cv_match_frame(L["scene"], cors, dets, [mods[0], mods[1], f_mod])) == INVALID
    assert _code(lambda: ctx.cv_match_frame(f_scene, cors, dets, mods)) == INVALID
    assert _code(lambda: ctx.match_frame(L["scene"], cors, mods, [library_tables[0], f_tab, library_tables[2]])) == INVALID
    assert _code(lambda: ctx.match_frame(L["scene"], cors, [f_mod, mods[1], mods[2]], library_tables[:3])) == INVALID
    other.close()
    untrained.close()
    assert pool_used() == start


# ---- 8. C99 example -----------------------------------------------------------------------------------------------------
def test_c_abi_multi_box_example(tmp_path, ctx, scene_full, bottle, reference):
    """tests/cpp/c_abi_multi_box_example.c — the frame uploaded once, one b200cv_match_frame for all boxes, strict C99 —
    prints the poses of the Python frame call"""
    from yolo_ppf_pose_estimation_b200 import build
    r = reference
    lib = build.build()
    np.ascontiguousarray(scene_full[:, :3], np.float32).tofile(tmp_path / "scene.f32")
    r["depth"].tofile(tmp_path / "depth.f32")
    bottle.astype(np.float32).tofile(tmp_path / "model.f32")
    exe = tmp_path / "c_abi_multi_box_example"
    p = subprocess.run(["/usr/bin/gcc", "-std=c99", "-pedantic", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"),
                        os.path.join(ROOT, "tests", "cpp", "c_abi_multi_box_example.c"), "-o", str(exe), "-L", os.path.dirname(lib),
                        "-lb200ppf", f"-Wl,-rpath,{os.path.dirname(lib)}"], capture_output=True, text=True)
    assert p.returncode == 0, p.stderr
    box = [int(v) for v in r["box"]]  # the surrogate YOLO box twice: the golden depth image holds its four corner pixels only
    args = [str(tmp_path), "0.01", "0.025", str(r["depth"].shape[0]), str(r["depth"].shape[1])] + [repr(float(v)) for v in r["K"]] + \
           [str(v) for v in box * 2]
    p = subprocess.run([str(exe)] + args, capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stdout + p.stderr
    lines = p.stdout.strip().splitlines()
    assert len(lines) == 2
    res, status = ctx.cv_match_frame(r["scene"], [r["cor"]] * 2, [r["det"]] * 2, [r["model"]] * 2, leaf=0.01)
    for i, line in enumerate(lines):
        v = line.split()
        assert v[:3] == ["box", str(i), "0"] and status[i] == 0
        assert int(v[3]) == res[i]["votes"] and int(v[4]) == res[i]["n_poses"] and float(v[5]) == res[i]["residual"]
        assert np.array_equal(np.array([float(x) for x in v[6:]]), res[i]["pose"].reshape(16))


# ---- 9. the per-object calls: a frame of one box, plus its clouds ------------------------------------------------------
def _object_call(ctx, call, params_cls, default_fn, edges_out, **over):
    """a per-object call through ctypes with edges_out passed or NULL (Context's wrappers always pass both)
    -> (result dict, whether an edge cloud was handed out)"""
    from yolo_ppf_pose_estimation_b200 import capi
    prm = ctx._params(params_cls, default_fn, over)
    res = capi.ObjectResult()
    obj, edg = ctypes.c_void_p(), ctypes.c_void_p()
    ctx.check(call(ctypes.byref(prm), ctypes.byref(res), ctypes.byref(obj), ctypes.byref(edg) if edges_out else None))
    got_edges = bool(edg.value)
    _free([capi.Cloud(ctx, h) for h in (obj, edg) if h.value])
    return ctx._result(res), got_edges


def _edges_only_when_asked(ctx, call, params_cls, default_fn, **over):
    """edge_curvature > 0 and no engine need for the edges: they are extracted for edges_out only, and the rest of the
    result does not depend on them"""
    asked, got = _object_call(ctx, call, params_cls, default_fn, True, **over)
    plain, none = _object_call(ctx, call, params_cls, default_fn, False, **over)
    assert got and asked["n_edges"] > 0
    assert not none and plain["n_edges"] == 0 and plain["edges_ms"] == 0.0
    assert plain["pose"].tobytes() == asked["pose"].tobytes()
    for f in ("residual", "votes", "n_poses", "n_cropped", "n_sampled", "n_filtered"):
        assert plain[f] == asked[f], f


def test_match_object_extracts_edges_for_edges_out_only(ctx, reference):
    from yolo_ppf_pose_estimation_b200 import capi
    r, lib = reference, capi.lib()
    table = ctx.table_build_from_cloud(r["model"], ANGLE_STEP, DIST_STEP)
    c12 = np.ascontiguousarray(r["cor"], np.float32).reshape(12)
    _edges_only_when_asked(ctx, lambda *a: lib.b200ppf_match_object(ctx._h, r["scene"]._h, c12.ctypes.data, r["model"]._h, table._h, *a),
                           capi.ObjectParams, lib.b200ppf_object_params_default, leaf=0.01, ref_rate=5)


def test_cv_match_object_without_s2b_extracts_edges_for_edges_out_only(ctx, reference):
    from yolo_ppf_pose_estimation_b200 import capi
    r, lib = reference, capi.lib()
    c12 = np.ascontiguousarray(r["cor"], np.float32).reshape(12)
    _edges_only_when_asked(ctx, lambda *a: lib.b200cv_match_object(r["det"]._h, r["scene"]._h, c12.ctypes.data, r["model"]._h, *a),
                           capi.CvObjectParams, lib.b200cv_object_params_default, leaf=0.01, use_edges=0,
                           relative_scene_sample_step=1.0 / 14.0)


def test_match_object_rejects_handles_of_another_context(ctx, reference, scene_full, bottle):
    from yolo_ppf_pose_estimation_b200 import capi
    r = reference
    table = ctx.table_build_from_cloud(r["model"], ANGLE_STEP, DIST_STEP)
    other = capi.Context(0)
    f_scene, f_model = other.upload_xyz(scene_full[:, :3]), other.upload_cloud(bottle)
    f_table = other.table_build_from_cloud(f_model, ANGLE_STEP, DIST_STEP)
    assert _code(lambda: ctx.match_object(f_scene, r["cor"], r["model"], table, leaf=0.01)) == INVALID
    assert _code(lambda: ctx.match_object(r["scene"], r["cor"], f_model, table, leaf=0.01)) == INVALID
    assert _code(lambda: ctx.match_object(r["scene"], r["cor"], r["model"], f_table, leaf=0.01)) == INVALID
    other.close()
