"""GPU tests of verification against the depth image: b200ppf_depth_upload / b200ppf_cloud_from_depth,
b200ppf_score_poses_depth and the depth-verified frame calls (b200cv_match_frame_verified_depth,
b200ppf_match_frame_verified_depth).

Bars: the back-projection equals the numpy formula bit for bit (the reference crop is its own depth image back-projected);
the depth scores equal the float64 restatement (tests/verify_depth_reference.py) up to its borderline points, rms within 1e-5
relative; a record has the same bits alone, in a batch and on a second run with the batch's launch count; crafted cases
(no measurement, the model's own rendering, two plates) come out as the rule says; on the depth frame an occluded instance's
true pose keeps its fit while a pose 3 cm toward the camera is caught by its violations; the depth-verified frame calls equal
the unverified ones as the verified calls do; bad arguments are refused without leaking."""
import ctypes
import os

import numpy as np
import pytest

from conftest import ANGLE_STEP, DIST_STEP, ROOT
from test_gpu_frame import N_LIBRARY, _library_box, _rigid
from test_gpu_verify import SAME_FIELDS, _cv_expected, _object, _pcl_expected, _perturbed, pool_used, ref_frame  # noqa: F401
from verify_depth_reference import score_depth

pytestmark = pytest.mark.gpu

INVALID, STATE = -1, -4
UNUSED = 0xFFFFFFFF
COUNTS = ("inliers", "judged", "visible", "self_occluded", "occluded", "violations", "unknown")
PARAMS = [{}, dict(inlier_dist=0.005, normal_angle=np.radians(45.0)), dict(inlier_dist=0.02, normal_angle=np.pi)]


def _fit_bytes(f):
    return np.array([f[n] for n in COUNTS], np.uint32).tobytes() + np.array([f["fit"], f["rms"]], np.float32).tobytes()


def _backproject(depth, K):
    v, u = np.nonzero((depth > 0) & np.isfinite(depth))
    z = depth[v, u].astype(np.float64)
    return np.stack([(u - K[2]) * z / K[0], (v - K[3]) * z / K[1], z], 1).astype(np.float32)


def _ref_depth():
    """the reference crop as the 720 x 1280 depth image it was back-projected from (0 elsewhere)"""
    b = np.load(os.path.join(ROOT, "tests", "golden", "crop_box.npz"))
    K = b["intrinsics"].astype(np.float64)
    c = np.load(os.path.join(ROOT, "tests", "golden", "scene_crop_raw.npz"))["cloud"]
    cd = c.astype(np.float64)
    u = np.rint(K[0] * cd[:, 0] / cd[:, 2] + K[2]).astype(np.int64)
    v = np.rint(K[1] * cd[:, 1] / cd[:, 2] + K[3]).astype(np.int64)
    D = np.zeros(tuple(b["image"]), np.float32)
    D[v, u] = c[:, 2]
    return D, K, c


@pytest.fixture(scope="module")
def depth_frame(ctx):
    """the library depth frame: image, device image, scene cloud from it, boxes, models, detectors, tables"""
    from yolo_ppf_pose_estimation_b200 import capi, synth
    f = synth.synth_library_depth()
    dimg = ctx.upload_depth(f["depth"], f["K"])
    models = [synth.synth_model(2000, 10 + k, k).astype(np.float32) for k in range(N_LIBRARY)]
    dmodels = [ctx.upload_cloud(m) for m in models]
    return dict(f, dimg=dimg, scene=ctx.cloud_from_depth(dimg), cors=np.stack([_library_box(m, k) for k, m in enumerate(models)]),
                models=models, dmodels=dmodels, dets=[capi.CvDetector(ctx, 0.025, 0.05).train_model(m) for m in models],
                tables=[ctx.table_build_from_cloud(m, ANGLE_STEP, DIST_STEP) for m in dmodels])


@pytest.fixture(scope="module")
def ref_depth(ctx):
    D, K, c = _ref_depth()
    return dict(depth=D, K=K, cloud=c, dimg=ctx.upload_depth(D, K))


# ---- 1. back-projection ---------------------------------------------------------------------------------------------------
def test_back_projection_of_the_reference_crop(ctx, ref_depth):
    got = ctx.cloud_from_depth(ref_depth["dimg"]).download()
    assert got[:, :3].tobytes() == ref_depth["cloud"].tobytes()  # bit for bit and in order
    assert not got[:, 3:].any()


def test_back_projection_skips_pixels_without_a_measurement(ctx):
    rng = np.random.default_rng(11)
    D = rng.uniform(0.3, 3.0, (37, 53)).astype(np.float32)
    D[rng.random(D.shape) < 0.1] = 0.0
    D[rng.random(D.shape) < 0.05] = -1.0
    D[rng.random(D.shape) < 0.05] = np.nan
    D[rng.random(D.shape) < 0.05] = np.inf
    D[rng.random(D.shape) < 0.05] = -np.inf
    K = np.array([61.7, 59.3, 26.1, 17.9])
    want = _backproject(D, K)
    img = ctx.upload_depth(D, K)
    cloud = ctx.cloud_from_depth(img)
    got = cloud.download()
    assert got[:, :3].tobytes() == want.tobytes()
    # the bounding box drives the scoring grid: a pose on the cloud itself scores every visible point as an inlier
    model = np.concatenate([want, np.zeros_like(want)], 1)
    f = ctx.score_poses([(ctx.upload_cloud(model), cloud, np.eye(4)[None])], normal_angle=np.pi)[0][0]
    assert f["inliers"] == f["visible"] == len(want)
    empty = ctx.cloud_from_depth(ctx.upload_depth(np.zeros((4, 5), np.float32), K))
    assert empty.size == 0


# ---- 2. the restatement ------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def depth_cases(ctx, depth_frame, ref_frame, ref_depth, bottle):
    """[(model Cloud, model rows, scene Cloud, scene rows, poses, depth image, depth, K)]: the bottle on the reference object
    with the reference depth, library object 2 (a sphere hides half of it) on the depth frame with its model and the
    20 000-point model, the bottle on an empty scene"""
    from yolo_ppf_pose_estimation_b200 import synth
    rng = np.random.default_rng(7)
    r, L = ref_frame, depth_frame
    far = np.eye(4)
    far[:3, 3] = (100.0, -50.0, 80.0)
    robj, _ = _object(ctx, r["det"], r["scene"], r["cor"], r["model"], leaf=0.01)
    _, _, cands = ctx.cv_match_frame_verified(r["scene"], [r["cor"]], [r["det"]], [r["model"]], leaf=0.01)
    bposes = [c["pose"] for c in cands[0]][:2]
    bposes += _perturbed(rng, bposes[0], 3) + [far]
    k = synth.DEPTH_OCCLUDED[0]
    lobj, _ = _object(ctx, L["dets"][k], L["scene"], L["cors"][k], L["dmodels"][k], leaf=0.005)
    T = synth.library_pose(k)
    lposes = [T] + _perturbed(rng, T, 3) + [far]
    big = synth.synth_model(20000, 10 + k, k).astype(np.float32)
    empty = ctx.upload_cloud(np.zeros((0, 6), np.float32))
    rd, ld = (ref_depth["dimg"], ref_depth["depth"], ref_depth["K"]), (L["dimg"], L["depth"], L["K"])
    return [(r["model"], bottle, robj, robj.download(), bposes) + rd,
            (L["dmodels"][k], L["models"][k], lobj, lobj.download(), lposes) + ld,
            (ctx.upload_cloud(big), big, lobj, lobj.download(), lposes[:3]) + ld,
            (r["model"], bottle, empty, np.zeros((0, 6), np.float32), bposes[:3]) + rd]


def _check_against_restatement(got, model, scene, poses, depth, K, **prm):
    for f, T in zip(got, poses):
        r = score_depth(model, scene, T, depth, K, **prm)
        slack = int(r["borderline"].sum())
        for n in COUNTS:
            assert abs(f[n] - r[n]) <= slack, (n, f, {c: r[c] for c in COUNTS}, slack)
        if slack == 0:
            assert all(f[n] == r[n] for n in COUNTS), (f, {c: r[c] for c in COUNTS})
            assert abs(f["rms"] - r["rms"]) <= 1e-5 * max(r["rms"], 1e-12), (f["rms"], r["rms"])


@pytest.mark.parametrize("prm", PARAMS)
def test_score_poses_depth_equals_the_restatement(ctx, depth_cases, prm):
    full = {"inlier_dist": 0.01, "normal_angle": np.radians(30.0)} | prm
    for case in depth_cases:
        m, mrows, s, srows, P, dimg, D, K = case
        got = ctx.score_poses_depth([(m, s, np.stack(P))], dimg, **prm)[0]
        _check_against_restatement(got, mrows, srows, P, D, K, **full)
        if case is depth_cases[1]:
            assert got[0]["occluded"] > 0.2 * got[0]["visible"], got[0]  # the true pose of the occluded instance
    far = ctx.score_poses_depth([(depth_cases[0][0], depth_cases[0][2], depth_cases[0][4][-1][None])], depth_cases[0][5], **prm)[0][0]
    assert far["visible"] == 0 and far["judged"] == 0 and far["fit"] == 0.0
    empty = ctx.score_poses_depth([(depth_cases[3][0], depth_cases[3][2], np.stack(depth_cases[3][4]))], depth_cases[3][5], **prm)[0]
    assert all(f["inliers"] == 0 and f["rms"] == 0.0 for f in empty)


# ---- 3. batch independence ---------------------------------------------------------------------------------------------------
def test_a_pose_scores_the_same_bits_alone_and_in_any_batch(ctx, depth_cases):
    cases = [(m, s, np.stack(P[:3])) for m, _, s, _, P, *_ in depth_cases[1:3]] + [(depth_cases[0][0], depth_cases[1][2],
                                                                                     np.stack(depth_cases[1][4][:3]))]
    dimg = depth_cases[1][5]
    jobs = [cases[k % 3] for k in range(8)]
    n0 = ctx.launch_count
    batch = ctx.score_poses_depth(jobs, dimg)
    n_batch = ctx.launch_count - n0
    again = ctx.score_poses_depth(jobs, dimg)
    assert [[_fit_bytes(f) for f in j] for j in batch] == [[_fit_bytes(f) for f in j] for j in again]
    for k, (m, s, P) in enumerate(jobs[:3]):
        for i in range(3):
            n0 = ctx.launch_count
            alone = ctx.score_poses_depth([(m, s, P[i:i + 1])], dimg)[0][0]
            assert ctx.launch_count - n0 == n_batch
            assert _fit_bytes(alone) == _fit_bytes(batch[k][i]) == _fit_bytes(batch[k + 3][i]), (k, i)


# ---- 4. crafted cases ----------------------------------------------------------------------------------------------------------
K_CRAFT = np.array([300.0, 300.0, 63.5, 63.5])


def _plate(z, half=0.1, spacing=0.004):
    g = np.arange(-half, half + 1e-9, spacing)
    x, y = np.meshgrid(g, g)
    pts = np.stack([x.ravel(), y.ravel(), np.full(x.size, z)], 1)
    return np.concatenate([pts, np.tile([0.0, 0.0, -1.0], (len(pts), 1))], 1).astype(np.float32)


def _render(rows, T, K, shape):
    """a dense splat of the rows under T into a depth image: per pixel the nearest, 0 where nothing lands"""
    p = rows[:, :3].astype(np.float64) @ T[:3, :3].T + T[:3, 3]
    u = np.floor(K[0] * p[:, 0] / p[:, 2] + K[2] + 0.5).astype(np.int64)
    v = np.floor(K[1] * p[:, 1] / p[:, 2] + K[3] + 0.5).astype(np.int64)
    ok = (p[:, 2] > 0) & (u >= 0) & (u < shape[1]) & (v >= 0) & (v < shape[0])
    D = np.full(shape[0] * shape[1], np.inf)
    np.minimum.at(D, v[ok] * shape[1] + u[ok], p[ok, 2])
    return np.where(np.isfinite(D), D, 0.0).reshape(shape).astype(np.float32)


def test_crafted_cases(ctx):
    from yolo_ppf_pose_estimation_b200 import synth
    model = synth.synth_model(2000, 10, 0)
    T = synth.library_pose(0)
    T[:3, 3] = (0.0, 0.0, 0.8)
    dm = ctx.upload_cloud(model)
    moved = model.astype(np.float64).copy()
    moved[:, :3] = model[:, :3] @ T[:3, :3].T + T[:3, 3]
    moved[:, 3:] = model[:, 3:] @ T[:3, :3].T
    scene = ctx.upload_cloud(moved.astype(np.float32))
    shape = (128, 128)
    # no measurement anywhere: every visible point is unknown
    zero = ctx.upload_depth(np.zeros(shape, np.float32), K_CRAFT)
    f = ctx.score_poses_depth([(dm, scene, T[None])], zero)[0][0]
    assert f["visible"] > 0 and f["unknown"] == f["visible"] and f["judged"] == 0 and f["fit"] == 0.0 and f["inliers"] == 0
    # the model's own rendering at T: consistent everywhere
    dense = synth.synth_model(200000, 10 + 7919, 0)
    D = _render(dense, T, K_CRAFT, shape)
    f = ctx.score_poses_depth([(dm, scene, T[None])], ctx.upload_depth(D, K_CRAFT))[0][0]
    print("own rendering:", f)
    assert f["fit"] >= 0.99 and f["violations"] == 0, f
    _check_against_restatement([f], model, moved.astype(np.float32), [T], D, K_CRAFT)
    # two plates facing the camera, the back one 5 cm behind the front one and larger
    front, back = _plate(0.0, 0.05), _plate(0.05, 0.1)
    plates = np.concatenate([front, back])
    Tp = np.eye(4)
    Tp[2, 3] = 0.6
    scene_rows = plates.copy()
    scene_rows[:, 2] += 0.6
    Dp = _render(np.concatenate([_plate(0.0, 0.05, 0.001), _plate(0.05, 0.1, 0.001)]), Tp, K_CRAFT, shape)  # dense: no holes
    dimg = ctx.upload_depth(Dp, K_CRAFT)
    sc = ctx.upload_cloud(scene_rows)
    f2 = ctx.score_poses_depth([(ctx.upload_cloud(plates), sc, Tp[None])], dimg)[0][0]
    f1 = ctx.score_poses_depth([(ctx.upload_cloud(front), sc, Tp[None])], dimg)[0][0]
    r = score_depth(plates, scene_rows, Tp, Dp, K_CRAFT)
    hidden = int(r["self_occluded_mask"][len(front):].sum())
    under = np.all(np.abs(back[:, :2]) <= 0.05 - 0.004, axis=1).sum()  # back-plate points well inside the front plate's shadow
    print("two plates:", f2, "front alone:", f1, "hidden back points", hidden, "under the front plate", under)
    assert f2["self_occluded"] == hidden and hidden >= under
    assert f2["fit"] >= f1["fit"] - 1e-6 and f2["violations"] == 0


# ---- 5. occlusion and free space on the depth frame ---------------------------------------------------------------------------
def test_occlusion_keeps_the_fit_and_free_space_catches_a_near_pose(ctx, depth_frame):
    from yolo_ppf_pose_estimation_b200 import synth
    L = depth_frame
    occluded = [k for k in range(N_LIBRARY) if L["occluded_share"][k] > 0]
    assert len(occluded) >= 2 and all(0.3 <= L["occluded_share"][k] <= 0.6 for k in occluded)
    for k in occluded:
        obj, _ = _object(ctx, L["dets"][k], L["scene"], L["cors"][k], L["dmodels"][k], leaf=0.005)
        T = synth.library_pose(k)
        c = L["models"][k][:, :3].astype(np.float64).mean(0)
        about_centre = lambda R: T @ np.block([[R, (c - R @ c)[:, None]], [np.zeros((1, 3)), np.ones((1, 1))]])  # noqa: E731
        near = T.copy()
        near[:3, 3] -= 0.03 * T[:3, 3] / np.linalg.norm(T[:3, 3])
        shifted = T.copy()
        shifted[:3, 3] += 0.03 * T[:3, 2]
        poses = np.stack([T, near, T @ _rigid((0, 0, 1), np.radians(37.0), (0, 0, 0)), shifted,
                          about_centre(_rigid((1, 0, 0), np.pi, (0, 0, 0))[:3, :3]), about_centre(_rigid((1, 0, 0), np.pi / 2, (0, 0, 0))[:3, :3])])
        dfits = ctx.score_poses_depth([(L["dmodels"][k], obj, poses)], L["dimg"])[0]
        plain = ctx.score_poses([(L["dmodels"][k], obj, poses[:1])])[0][0]
        print(f"instance {k} (occluded {L['occluded_share'][k]:.2f}): depth fit {dfits[0]['fit']:.3f} plain {plain['fit']:.3f}; "
              f"near: violations {dfits[1]['violations']}/{dfits[1]['judged']} fit {dfits[1]['fit']:.3f}; turned "
              f"{dfits[2]['fit']:.3f} shifted {dfits[3]['fit']:.3f} upside-down {dfits[4]['fit']:.3f} tilted {dfits[5]['fit']:.3f}")
        assert dfits[0]["fit"] >= 0.85 and dfits[0]["fit"] >= plain["fit"] + 0.2, (k, dfits[0], plain)
        assert dfits[1]["violations"] >= 0.5 * dfits[1]["judged"] and dfits[1]["fit"] <= 0.5, (k, dfits[1])
        # the turn is about the model's axis of revolution: the same surface, so the same fit
        assert abs(dfits[2]["fit"] - dfits[0]["fit"]) <= 0.05 and max(f["fit"] for f in dfits[3:]) <= 0.7, (k, dfits)


# ---- 6. the depth-verified frame calls ----------------------------------------------------------------------------------------
def _check_verified_depth(ctx, res, status, vres, vstatus, vcands, expected, dimg):
    assert vstatus.tolist() == status.tolist()
    for b in range(len(res)):
        for f in SAME_FIELDS:
            assert vres[b][f] == res[b][f], (b, f)
        if status[b]:
            assert vcands[b] == []
            continue
        best = vcands[b][0]
        assert vres[b]["pose"].tobytes() == best["pose"].tobytes() and vres[b]["residual"] == best["residual"] and \
            vres[b]["votes"] == best["votes"]
        if best["rank"] == 0:
            assert vres[b]["pose"].tobytes() == res[b]["pose"].tobytes() and vres[b]["residual"] == res[b]["residual"]
        fits = [c["fit"]["fit"] for c in vcands[b]]
        assert fits == sorted(fits, reverse=True)
        poses, votes, residuals, obj, model = expected(b)
        by_rank = sorted(vcands[b], key=lambda c: c["rank"])
        assert [c["rank"] for c in by_rank] == list(range(len(poses)))
        for c, P, v, r in zip(by_rank, poses, votes, residuals):
            assert c["pose"].tobytes() == np.asarray(P, np.float64).tobytes() and c["votes"] == v and c["residual"] == r
        scored = ctx.score_poses_depth([(model, obj, np.stack([c["pose"] for c in by_rank]))], dimg)[0]
        assert [_fit_bytes(c["fit"]) for c in by_rank] == [_fit_bytes(f) for f in scored]


def _frames(depth_frame, ref_frame, ref_depth):
    L, r = depth_frame, ref_frame
    return ((L["scene"], L["dimg"], L["cors"], L["dets"], L["dmodels"], L["tables"], 0.005),
            (r["scene"], ref_depth["dimg"], np.stack([r["cor"]] * 2), [r["det"]] * 2, [r["model"]] * 2, [r["table"]] * 2, 0.01))


@pytest.mark.parametrize("use_edges,icp_poses", [(1, 5), (1, 0), (0, 5), (0, 0)])
def test_cv_depth_verified_equals_unverified(ctx, depth_frame, ref_frame, ref_depth, use_edges, icp_poses):
    for scene, dimg, cors, dets, mods, _, leaf in _frames(depth_frame, ref_frame, ref_depth):
        over = dict(leaf=leaf, use_edges=use_edges, icp_poses=icp_poses, relative_scene_sample_step=0.05 if use_edges else 1.0 / 14.0)
        res, status = ctx.cv_match_frame(scene, cors, dets, mods, **over)
        vres, vstatus, vcands = ctx.cv_match_frame_verified_depth(scene, dimg, cors, dets, mods, **over)
        _check_verified_depth(ctx, res, status, vres, vstatus, vcands, lambda b: _cv_expected(ctx, dets[b], scene, cors[b], mods[b], over),
                              dimg)


@pytest.mark.parametrize("icp_poses", [5, 0])
def test_pcl_depth_verified_equals_unverified(ctx, depth_frame, ref_frame, ref_depth, icp_poses):
    for scene, dimg, cors, dets, mods, tabs, leaf in _frames(depth_frame, ref_frame, ref_depth):
        over = dict(leaf=leaf, ref_rate=20, icp_poses=icp_poses)
        res, status = ctx.match_frame(scene, cors, mods, tabs, **over)
        vres, vstatus, vcands = ctx.match_frame_verified_depth(scene, dimg, cors, mods, tabs, **over)
        _check_verified_depth(ctx, res, status, vres, vstatus, vcands,
                              lambda b: _pcl_expected(ctx, tabs[b], scene, cors[b], mods[b], over, dets[b]), dimg)


def test_a_failed_box_has_empty_slots_and_leaves_the_others(ctx, depth_frame):
    from yolo_ppf_pose_estimation_b200 import capi
    L = depth_frame
    behind = L["cors"][1] * np.array([1, 1, -1], np.float32)
    cors = np.stack([L["cors"][0], behind, L["cors"][2]])
    dets, mods = [L["dets"][k] for k in (0, 1, 2)], [L["dmodels"][k] for k in (0, 1, 2)]
    prm = ctx._params(capi.CvObjectParams, capi.lib().b200cv_object_params_default, dict(leaf=0.005))
    res = (capi.ObjectResult * 3)()
    status = np.zeros(3, np.int32)
    cand = (capi.DepthCandidate * 15)()
    c12 = np.ascontiguousarray(cors, np.float32).reshape(-1, 12)
    ctx.check(capi.lib().b200cv_match_frame_verified_depth(ctx._h, L["scene"]._h, L["dimg"]._h, 3, c12.ctypes.data, ctx._handles(dets, 3),
                                                          ctx._handles(mods, 3), ctypes.byref(prm), None, res, status.ctypes.data, cand))
    assert status.tolist() == [0, STATE, 0]
    assert all(bytes(cand[5 + i].pose) == bytes(16 * 8) and cand[5 + i].rank == UNUSED and cand[5 + i].votes == 0 and
               bytes(cand[5 + i].fit) == bytes(ctypes.sizeof(capi.DepthFit)) for i in range(5))
    good, gstatus, gcands = ctx.cv_match_frame_verified_depth(L["scene"], L["dimg"], cors[[0, 2]], [dets[0], dets[2]], [mods[0], mods[2]],
                                                              leaf=0.005)
    assert gstatus.tolist() == [0, 0]
    for b, g in ((0, 0), (2, 1)):
        assert bytes(res[b].pose) == good[g]["pose"].tobytes()
        got = [cand[5 * b + i] for i in range(5) if cand[5 * b + i].rank != UNUSED]
        assert [(bytes(c.pose), c.rank, c.votes, c.residual, bytes(c.fit)) for c in got] == \
            [(x["pose"].tobytes(), x["rank"], x["votes"], x["residual"], _fit_bytes(x["fit"])) for x in gcands[g]]


# ---- 7. errors -------------------------------------------------------------------------------------------------------------------
def test_bad_images_and_arguments(ctx, depth_frame, depth_cases, pool_used):  # noqa: F811
    from yolo_ppf_pose_estimation_b200 import capi
    L = depth_frame
    cors, dets, mods, tabs = L["cors"][:2], L["dets"][:2], L["dmodels"][:2], L["tables"][:2]
    m, _, s, _, P, dimg, *_ = depth_cases[1]
    ctx.cv_match_frame_verified_depth(L["scene"], L["dimg"], cors, dets, mods, leaf=0.005)  # warm
    ctx.score_poses_depth([(m, s, np.stack(P))], dimg)
    ctx.cloud_from_depth(L["dimg"])
    start = pool_used()
    ctx.cv_match_frame_verified_depth(L["scene"], L["dimg"], cors, dets, mods, leaf=0.005)
    ctx.match_frame_verified_depth(L["scene"], L["dimg"], cors, mods, tabs, leaf=0.005, ref_rate=20)
    ctx.score_poses_depth([(m, s, np.stack(P))], dimg)
    ctx.cloud_from_depth(L["dimg"])
    assert pool_used() == start

    def code(fn):
        with pytest.raises(capi.B200PPFError) as e:
            fn()
        return e.value.code
    lib = capi.lib()
    good = np.ones((4, 5), np.float32)
    K = np.array([100.0, 100.0, 2.0, 1.5])
    for bad in (np.array([0.0, 100.0, 2.0, 1.5]), np.array([100.0, -1.0, 2.0, 1.5]), np.array([100.0, 100.0, np.nan, 1.5]),
                np.array([100.0, 100.0, 2.0, np.inf])):
        assert code(lambda: ctx.upload_depth(good, bad)) == INVALID, bad
    h = ctypes.c_void_p()
    Kc = np.ascontiguousarray(K)
    assert lib.b200ppf_depth_upload(ctx._h, good.ctypes.data, 0, 5, Kc.ctypes.data, ctypes.byref(h)) == INVALID
    assert lib.b200ppf_depth_upload(ctx._h, good.ctypes.data, 4, -1, Kc.ctypes.data, ctypes.byref(h)) == INVALID
    assert lib.b200ppf_depth_upload(ctx._h, good.ctypes.data, 1 << 16, 1 << 15, Kc.ctypes.data, ctypes.byref(h)) == INVALID
    assert lib.b200ppf_depth_upload(ctx._h, None, 4, 5, Kc.ctypes.data, ctypes.byref(h)) == INVALID
    assert lib.b200ppf_depth_upload(ctx._h, good.ctypes.data, 4, 5, None, ctypes.byref(h)) == INVALID
    assert lib.b200ppf_depth_upload(None, good.ctypes.data, 4, 5, Kc.ctypes.data, ctypes.byref(h)) == INVALID
    assert lib.b200ppf_cloud_from_depth(ctx._h, None, ctypes.byref(h)) == INVALID
    for bad in (dict(inlier_dist=0.0), dict(inlier_dist=np.nan), dict(normal_angle=-0.1), dict(normal_angle=np.nan)):
        assert code(lambda: ctx.cv_match_frame_verified_depth(L["scene"], L["dimg"], cors, dets, mods, leaf=0.005, **bad)) == INVALID
        assert code(lambda: ctx.match_frame_verified_depth(L["scene"], L["dimg"], cors, mods, tabs, leaf=0.005, **bad)) == INVALID
        assert code(lambda: ctx.score_poses_depth([(m, s, np.stack(P))], dimg, **bad)) == INVALID
    nan_pose = np.stack(P).copy()
    nan_pose[1, 0, 3] = np.nan
    assert code(lambda: ctx.score_poses_depth([(m, s, nan_pose)], dimg)) == INVALID
    other = capi.Context(0)
    foreign = other.upload_depth(good, K)
    assert code(lambda: ctx.score_poses_depth([(m, s, np.stack(P))], foreign)) == INVALID
    assert code(lambda: ctx.cloud_from_depth(foreign)) == INVALID
    assert code(lambda: ctx.cv_match_frame_verified_depth(L["scene"], foreign, cors, dets, mods, leaf=0.005)) == INVALID
    assert code(lambda: ctx.match_frame_verified_depth(L["scene"], foreign, cors, mods, tabs, leaf=0.005)) == INVALID
    foreign.free()
    other.close()
    fits = (capi.DepthFit * 4)()
    Pa = np.ascontiguousarray(np.stack(P[:2]))
    job = capi.IcpJob(m._h, s._h, Pa.ctypes.data, 2, None)
    assert lib.b200ppf_score_poses_depth(ctx._h, ctypes.byref(job), 1, None, None, fits) == INVALID  # depth NULL
    assert lib.b200ppf_score_poses_depth(ctx._h, ctypes.byref(job), 1, dimg._h, None, None) == INVALID  # fits NULL
    assert lib.b200ppf_score_poses_depth(ctx._h, None, 1, dimg._h, None, fits) == INVALID
    res = (capi.ObjectResult * 2)()
    st = np.zeros(2, np.int32)
    c12 = np.ascontiguousarray(cors, np.float32).reshape(-1, 12)
    assert lib.b200cv_match_frame_verified_depth(ctx._h, L["scene"]._h, None, 2, c12.ctypes.data, ctx._handles(dets, 2),
                                                 ctx._handles(mods, 2), None, None, res, st.ctypes.data, None) == INVALID
    assert lib.b200ppf_match_frame_verified_depth(ctx._h, L["scene"]._h, None, 2, c12.ctypes.data, ctx._handles(mods, 2),
                                                  ctx._handles(tabs, 2), None, None, res, st.ctypes.data, None) == INVALID
    assert lib.b200ppf_score_poses_depth(ctx._h, ctypes.byref(job), 1, dimg._h, None, fits) == 0
    assert pool_used() == start
