"""GPU tests of pose verification: b200ppf_score_poses and the verified frame calls (b200cv_match_frame_verified,
b200ppf_match_frame_verified).

Bars: the scores equal the float64 restatement (tests/verify_reference.py) up to its borderline points, rms within 1e-5
relative; a pose's record has the same bits alone, in a batch and on a second run, with a launch count that does not depend
on the batch; on the library frame the true pose outscores its decoys; a verified call equals the unverified one in every
result field but the best candidate's pose / residual / votes and the times, its candidates are the engine's matching and
ICP on the same object cloud and their fits are score_poses'; the library instances found with verification include those
found today; a failed box has empty candidate slots and leaves the others; bad verify values are refused without leaking.
"""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from conftest import ANGLE_STEP, DIST_STEP, ROOT
from test_gpu_frame import N_LIBRARY, _axis_angle_deg, _library_box, _rigid
from verify_reference import score

pytestmark = pytest.mark.gpu

INVALID, STATE = -1, -4
UNUSED = 0xFFFFFFFF
SAME_FIELDS = ("n_poses", "n_cropped", "n_sampled", "n_filtered", "n_edges")
ROT_THR = np.float32(20.0) / np.float32(180.0) * np.float32(3.14159265358979)  # b200ppf_object_params_default's, in float


@pytest.fixture(scope="module")
def lib_frame(ctx):
    """the 1 Mi-point library frame: scene, boxes, models (host, device), detectors, tables, leaf 0.005"""
    from yolo_ppf_pose_estimation_b200 import capi, synth
    xyz = np.ascontiguousarray(synth.synth_library_scene(1 << 20)[:, :3], np.float32)
    models = [synth.synth_model(2000, 10 + k, k).astype(np.float32) for k in range(N_LIBRARY)]
    dmodels = [ctx.upload_cloud(m) for m in models]
    return dict(scene=ctx.upload_xyz(xyz), cors=np.stack([_library_box(m, k) for k, m in enumerate(models)]), models=models,
                dmodels=dmodels, dets=[capi.CvDetector(ctx, 0.025, 0.05).train_model(m) for m in models],
                tables=[ctx.table_build_from_cloud(m, ANGLE_STEP, DIST_STEP) for m in dmodels])


@pytest.fixture(scope="module")
def ref_frame(ctx, scene_full, bottle):
    from yolo_ppf_pose_estimation_b200 import capi
    b = np.load(os.path.join(ROOT, "tests", "golden", "crop_box.npz"))
    depth = np.zeros(tuple(b["image"]), np.float32)
    for (r, c), d in zip(b["pixels"], b["depths"]):
        depth[r, c] = d
    model = ctx.upload_cloud(bottle)
    return dict(scene=ctx.upload_xyz(scene_full[:, :3]), cor=capi.frustum_corners(depth, b["box"], b["intrinsics"]), model=model,
                det=capi.CvDetector(ctx, 0.025, 0.05).train_model(bottle), table=ctx.table_build_from_cloud(model, ANGLE_STEP, DIST_STEP),
                depth=depth, box=b["box"], K=b["intrinsics"])


def _object(ctx, det, scene, cor, model, **over):
    """the pre-processed object cloud of one box (what the ICP and the scoring register to)"""
    _, obj, edges = ctx.cv_match_object(det, scene, cor, model, **over)
    return obj, edges


def _fit_bytes(f):
    return np.array([f["inliers"], f["visible"]], np.uint32).tobytes() + np.array([f["fit"], f["rms"]], np.float32).tobytes()


def _check_against_restatement(got, model, scene, poses, **prm):
    for f, T in zip(got, poses):
        r = score(model, scene, T, **prm)
        slack = int(r["borderline"].sum())
        assert abs(f["visible"] - r["visible"]) <= slack and abs(f["inliers"] - r["inliers"]) <= slack, (f, r["inliers"], r["visible"], slack)
        if slack == 0:
            assert f["inliers"] == r["inliers"] and f["visible"] == r["visible"]
            assert abs(f["rms"] - r["rms"]) <= 1e-5 * max(r["rms"], 1e-12), (f["rms"], r["rms"])


def _perturbed(rng, T, k):
    return [_rigid(rng.normal(size=3), rng.uniform(0.0, 0.1), rng.normal(scale=0.01, size=3)) @ T for _ in range(k)]


@pytest.fixture(scope="module")
def score_cases(ctx, lib_frame, ref_frame, bottle):
    """[(model Cloud, model rows, scene Cloud, scene rows, poses)]: the bottle on the reference object cloud, a 2 000-point
    library model and a 20 000-point model on library object 0, the bottle on an empty scene"""
    from yolo_ppf_pose_estimation_b200 import synth
    rng = np.random.default_rng(5)
    r, L = ref_frame, lib_frame
    far = np.eye(4)
    far[:3, 3] = (100.0, -50.0, 80.0)
    robj, _ = _object(ctx, r["det"], r["scene"], r["cor"], r["model"], leaf=0.01)
    _, _, cands = ctx.cv_match_frame_verified(r["scene"], [r["cor"]], [r["det"]], [r["model"]], leaf=0.01)
    bposes = [c["pose"] for c in cands[0]]
    bposes += _perturbed(rng, bposes[0], 6) + [far]
    lobj, _ = _object(ctx, L["dets"][0], L["scene"], L["cors"][0], L["dmodels"][0], leaf=0.005)
    T0 = synth.library_pose(0)
    lposes = [T0] + _perturbed(rng, T0, 6) + [far]
    big = synth.synth_model(20000, 10, 0).astype(np.float32)
    empty = ctx.upload_cloud(np.zeros((0, 6), np.float32))
    return [(r["model"], bottle, robj, robj.download(), bposes), (L["dmodels"][0], L["models"][0], lobj, lobj.download(), lposes),
            (ctx.upload_cloud(big), big, lobj, lobj.download(), lposes), (r["model"], bottle, empty, np.zeros((0, 6), np.float32), bposes[:3])]


# ---- 1. score_poses against the restatement ----------------------------------------------------------------------------
@pytest.mark.parametrize("prm", [{}, dict(inlier_dist=0.005, normal_angle=np.radians(45.0)), dict(inlier_dist=0.02, normal_angle=np.pi)])
def test_score_poses_equals_the_restatement(ctx, score_cases, prm):
    got = ctx.score_poses([(m, s, P) for m, _, s, _, P in score_cases], **prm)
    for (m, mrows, s, srows, P), fits in zip(score_cases, got):
        _check_against_restatement(fits, mrows, srows, P, **({"inlier_dist": 0.01, "normal_angle": np.radians(30.0)} | prm))
    assert got[0][-1]["visible"] > 0 and got[0][-1]["inliers"] == 0  # the far pose
    assert all(f["inliers"] == 0 and f["rms"] == 0.0 for f in got[3])  # the empty scene
    assert got[1][0]["fit"] > 0.5 and got[2][0]["fit"] > 0.5


# ---- 2. batch independence -----------------------------------------------------------------------------------------------
def test_a_pose_scores_the_same_bits_alone_and_in_any_batch(ctx, score_cases):
    cases = [(m, s, np.stack(P[:5])) for m, _, s, _, P in score_cases[:3]]
    jobs = [cases[k % 3] for k in range(8)]  # 8 jobs x 5 poses over three models and two scenes
    n0 = ctx.launch_count
    batch = ctx.score_poses(jobs)
    n_batch = ctx.launch_count - n0
    again = ctx.score_poses(jobs)
    assert [[_fit_bytes(f) for f in j] for j in batch] == [[_fit_bytes(f) for f in j] for j in again]
    for k, (m, s, P) in enumerate(jobs[:3]):
        for i in range(5):
            n0 = ctx.launch_count
            alone = ctx.score_poses([(m, s, P[i:i + 1])])[0][0]
            assert ctx.launch_count - n0 == n_batch  # the launch count does not depend on jobs or poses
            assert _fit_bytes(alone) == _fit_bytes(batch[k][i]), (k, i)
            assert _fit_bytes(alone) == _fit_bytes(batch[k + 3][i]), (k, i)


# ---- 3. decoys on the library frame ------------------------------------------------------------------------------------
def test_true_pose_outscores_its_decoys(ctx, lib_frame):
    from yolo_ppf_pose_estimation_b200 import synth
    L = lib_frame
    for k in range(N_LIBRARY):
        obj, _ = _object(ctx, L["dets"][k], L["scene"], L["cors"][k], L["dmodels"][k], leaf=0.005)
        T = synth.library_pose(k)
        c = L["models"][k][:, :3].astype(np.float64).mean(0)
        about_centre = lambda R: T @ np.block([[R, (c - R @ c)[:, None]], [np.zeros((1, 3)), np.ones((1, 1))]])  # noqa: E731
        shifted = T.copy()
        shifted[:3, 3] += 0.03 * T[:3, 2]
        poses = [T, T @ _rigid((0, 0, 1), np.radians(37.0), (0, 0, 0)), shifted, about_centre(_rigid((1, 0, 0), np.pi, (0, 0, 0))[:3, :3]),
                 about_centre(_rigid((1, 0, 0), np.pi / 2, (0, 0, 0))[:3, :3])]
        fits = [f["fit"] for f in ctx.score_poses([(L["dmodels"][k], obj, np.stack(poses))])[0]]
        print(f"instance {k}: true {fits[0]:.3f} turned {fits[1]:.3f} shifted {fits[2]:.3f} upside-down {fits[3]:.3f} "
              f"tilted {fits[4]:.3f}")
        assert sorted(range(5), key=lambda i: -fits[i])[:2] in ([0, 1], [1, 0]), (k, fits)
        assert fits[0] >= 0.85 and abs(fits[0] - fits[1]) <= 0.05 and max(fits[2:]) <= 0.7, (k, fits)


# ---- 4. verified equals unverified -------------------------------------------------------------------------------------
def _check_verified(ctx, res, status, vres, vstatus, vcands, expected):
    """expected(b) -> (poses, votes, residuals, object Cloud, model Cloud) of box b's candidates in rank order"""
    assert vstatus.tolist() == status.tolist()
    for b in range(len(res)):
        for f in SAME_FIELDS:
            assert vres[b][f] == res[b][f], (b, f)
        best = vcands[b][0]
        assert vres[b]["pose"].tobytes() == best["pose"].tobytes() and vres[b]["residual"] == best["residual"] and \
            vres[b]["votes"] == best["votes"]
        if best["rank"] == 0:
            assert vres[b]["pose"].tobytes() == res[b]["pose"].tobytes() and vres[b]["residual"] == res[b]["residual"] and \
                vres[b]["votes"] == res[b]["votes"]
        fits = [c["fit"]["fit"] for c in vcands[b]]
        assert fits == sorted(fits, reverse=True)
        poses, votes, residuals, obj, model = expected(b)
        by_rank = sorted(vcands[b], key=lambda c: c["rank"])
        assert [c["rank"] for c in by_rank] == list(range(len(poses)))
        for c, P, v, r in zip(by_rank, poses, votes, residuals):
            assert c["pose"].tobytes() == np.asarray(P, np.float64).tobytes() and c["votes"] == v and c["residual"] == r
        scored = ctx.score_poses([(model, obj, np.stack([c["pose"] for c in by_rank]))])[0]
        assert [_fit_bytes(c["fit"]) for c in by_rank] == [_fit_bytes(f) for f in scored]


def _cv_expected(ctx, det, scene, cor, model, over):
    obj, edges = _object(ctx, det, scene, cor, model, **over)
    use_edges, icp_poses = over["use_edges"], over["icp_poses"]
    top, n = det.match_cloud(obj, edges if use_edges else None, over["relative_scene_sample_step"], 0.05, max_poses=max(icp_poses, 1))
    n_c = max(min(icp_poses, len(top)), 1)
    P = np.stack([t["pose"].reshape(4, 4) for t in top[:n_c]])
    res = np.zeros(n_c)
    if icp_poses:
        [(P, res)], _ = ctx.icp_refine_batch([(model, obj, P)])
    return P, [int(t["num_votes"]) for t in top[:n_c]], res.tolist(), obj, model


def _pcl_expected(ctx, table, scene, cor, model, over, det_for_object):
    obj, _ = _object(ctx, det_for_object, scene, cor, model, leaf=over["leaf"])
    _, poses, votes = ctx.register(model, table, obj, ref_rate=over["ref_rate"], pos_thr=np.float32(0.01), rot_thr=ROT_THR)
    icp_poses = over["icp_poses"]
    n_c = max(min(icp_poses, len(poses)), 1)
    P = poses[:n_c].astype(np.float64)
    res = np.zeros(n_c)
    if icp_poses:
        [(P, res)], _ = ctx.icp_refine_batch([(model, obj, P)])
    return P, [int(v) for v in votes[:n_c]], res.tolist(), obj, model


@pytest.mark.parametrize("use_edges,icp_poses", [(1, 5), (1, 0), (0, 5), (0, 0)])
def test_cv_verified_equals_unverified(ctx, lib_frame, ref_frame, use_edges, icp_poses):
    for scene, cors, dets, mods, leaf in (
            (lib_frame["scene"], lib_frame["cors"], lib_frame["dets"], lib_frame["dmodels"], 0.005),
            (ref_frame["scene"], np.stack([ref_frame["cor"]] * 2), [ref_frame["det"]] * 2, [ref_frame["model"]] * 2, 0.01)):
        over = dict(leaf=leaf, use_edges=use_edges, icp_poses=icp_poses, relative_scene_sample_step=0.05 if use_edges else 1.0 / 14.0)
        res, status = ctx.cv_match_frame(scene, cors, dets, mods, **over)
        vres, vstatus, vcands = ctx.cv_match_frame_verified(scene, cors, dets, mods, **over)
        _check_verified(ctx, res, status, vres, vstatus, vcands, lambda b: _cv_expected(ctx, dets[b], scene, cors[b], mods[b], over))


@pytest.mark.parametrize("icp_poses", [5, 0])
def test_pcl_verified_equals_unverified(ctx, lib_frame, ref_frame, icp_poses):
    for scene, cors, dets, mods, tabs, leaf in (
            (lib_frame["scene"], lib_frame["cors"], lib_frame["dets"], lib_frame["dmodels"], lib_frame["tables"], 0.005),
            (ref_frame["scene"], np.stack([ref_frame["cor"]] * 2), [ref_frame["det"]] * 2, [ref_frame["model"]] * 2,
             [ref_frame["table"]] * 2, 0.01)):
        over = dict(leaf=leaf, ref_rate=20, icp_poses=icp_poses)
        res, status = ctx.match_frame(scene, cors, mods, tabs, **over)
        vres, vstatus, vcands = ctx.match_frame_verified(scene, cors, mods, tabs, **over)
        _check_verified(ctx, res, status, vres, vstatus, vcands,
                        lambda b: _pcl_expected(ctx, tabs[b], scene, cors[b], mods[b], over, dets[b]))


# ---- 5. instances found on the library frame ---------------------------------------------------------------------------
def _found(res):
    from yolo_ppf_pose_estimation_b200 import synth
    return {k for k in range(N_LIBRARY) if np.linalg.norm(res[k]["pose"][:3, 3] - synth.library_pose(k)[:3, 3]) < 0.01 and
            _axis_angle_deg(res[k]["pose"], synth.library_pose(k)) < 5.0}


@pytest.mark.parametrize("use_edges", [1, 0])
def test_verification_finds_the_library_instances(ctx, lib_frame, use_edges):
    L = lib_frame
    over = dict(leaf=0.005, use_edges=use_edges, icp_poses=5, relative_scene_sample_step=0.05 if use_edges else 1.0 / 14.0)
    res, _ = ctx.cv_match_frame(L["scene"], L["cors"], L["dets"], L["dmodels"], **over)
    vres, vstatus, vcands = ctx.cv_match_frame_verified(L["scene"], L["cors"], L["dets"], L["dmodels"], **over)
    plain, verified = _found(res), _found(vres)
    print(f"{'match_S2B' if use_edges else 'Matching'}: found without verification {sorted(plain)}, with verification "
          f"{sorted(verified)}; best ranks {[c[0]['rank'] for c in vcands]}; best fits {[round(c[0]['fit']['fit'], 3) for c in vcands]}")
    assert vstatus.tolist() == [0] * N_LIBRARY
    assert verified >= ({1, 7} if use_edges else {0, 2, 3, 5, 7}), verified


# ---- 6. failures and errors --------------------------------------------------------------------------------------------
def test_a_failed_box_has_empty_slots_and_leaves_the_others(ctx, lib_frame):
    L = lib_frame
    behind = L["cors"][1] * np.array([1, 1, -1], np.float32)
    cors, idx = np.stack([L["cors"][0], behind, L["cors"][2]]), [0, 1, 2]
    dets, mods = [L["dets"][k] for k in idx], [L["dmodels"][k] for k in idx]
    from yolo_ppf_pose_estimation_b200 import capi
    prm = ctx._params(capi.CvObjectParams, capi.lib().b200cv_object_params_default, dict(leaf=0.005))
    res = (capi.ObjectResult * 3)()
    status = np.zeros(3, np.int32)
    cand = (capi.Candidate * 15)()
    c12 = np.ascontiguousarray(cors, np.float32).reshape(-1, 12)
    ctx.check(capi.lib().b200cv_match_frame_verified(ctx._h, L["scene"]._h, 3, c12.ctypes.data, ctx._handles(dets, 3), ctx._handles(mods, 3),
                                                    ctypes.byref(prm), None, res, status.ctypes.data, cand))
    assert status.tolist() == [0, STATE, 0]
    assert all(bytes(cand[5 + i].pose) == bytes(16 * 8) and cand[5 + i].rank == UNUSED and cand[5 + i].votes == 0 and
               cand[5 + i].fit.inliers == 0 and cand[5 + i].fit.visible == 0 for i in range(5))
    good, gstatus, gcands = ctx.cv_match_frame_verified(L["scene"], cors[[0, 2]], [dets[0], dets[2]], [mods[0], mods[2]], leaf=0.005)
    assert gstatus.tolist() == [0, 0]
    for b, g in ((0, 0), (2, 1)):
        assert bytes(res[b].pose) == good[g]["pose"].tobytes()
        got = [cand[5 * b + i] for i in range(5) if cand[5 * b + i].rank != UNUSED]
        assert [(bytes(c.pose), c.rank, c.votes, c.residual, bytes(c.fit)) for c in got] == \
            [(x["pose"].tobytes(), x["rank"], x["votes"], x["residual"], _fit_bytes(x["fit"])) for x in gcands[g]]


def test_bad_verify_values_and_arguments(ctx, lib_frame, score_cases, pool_used):
    from yolo_ppf_pose_estimation_b200 import capi
    L = lib_frame
    cors, dets, mods, tabs = L["cors"][:2], L["dets"][:2], L["dmodels"][:2], L["tables"][:2]
    ctx.cv_match_frame_verified(L["scene"], cors, dets, mods, leaf=0.005)  # warm
    m, _, s, _, P = score_cases[0]
    ctx.score_poses([(m, s, np.stack(P))])
    start = pool_used()
    ctx.cv_match_frame_verified(L["scene"], cors, dets, mods, leaf=0.005)
    ctx.match_frame_verified(L["scene"], cors, mods, tabs, leaf=0.005, ref_rate=20)
    ctx.score_poses([(m, s, np.stack(P))])
    assert pool_used() == start

    def code(fn):
        with pytest.raises(capi.B200PPFError) as e:
            fn()
        return e.value.code
    for bad in (dict(inlier_dist=0.0), dict(inlier_dist=-0.01), dict(inlier_dist=np.nan), dict(inlier_dist=np.inf),
                dict(normal_angle=-0.1), dict(normal_angle=np.nan)):
        assert code(lambda: ctx.cv_match_frame_verified(L["scene"], cors, dets, mods, leaf=0.005, **bad)) == INVALID, bad
        assert code(lambda: ctx.match_frame_verified(L["scene"], cors, mods, tabs, leaf=0.005, **bad)) == INVALID, bad
        assert code(lambda: ctx.score_poses([(m, s, np.stack(P))], **bad)) == INVALID, bad
    nan_pose = np.stack(P).copy()
    nan_pose[1, 0, 3] = np.nan
    assert code(lambda: ctx.score_poses([(m, s, nan_pose)])) == INVALID
    other = capi.Context(0)
    foreign = other.upload_cloud(L["models"][0])
    assert code(lambda: ctx.score_poses([(m, s, np.stack(P)), (foreign, s, np.stack(P))])) == INVALID
    other.close()
    lib = capi.lib()
    fits = (capi.PoseFit * 4)()
    job = capi.IcpJob(m._h, s._h, None, 2, None)
    assert lib.b200ppf_score_poses(ctx._h, None, 1, None, fits) == INVALID
    assert lib.b200ppf_score_poses(ctx._h, ctypes.byref(job), 1, None, fits) == INVALID  # poses16 NULL
    Pa = np.ascontiguousarray(np.stack(P[:2]))
    job = capi.IcpJob(m._h, s._h, Pa.ctypes.data, 2, None)
    assert lib.b200ppf_score_poses(ctx._h, ctypes.byref(job), 1, None, None) == INVALID  # fits NULL
    assert lib.b200ppf_score_poses(ctx._h, ctypes.byref(job), 1, None, fits) == 0
    assert pool_used() == start


@pytest.fixture(scope="module")
def pool_used():
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
        import gc
        gc.collect()
        assert rt.cudaDeviceSynchronize() == 0
        v = ctypes.c_uint64(0)
        assert rt.cudaMemPoolGetAttribute(pool, 0x7, ctypes.byref(v)) == 0
        return v.value

    return used


# ---- 7. the C99 example ------------------------------------------------------------------------------------------------
def test_c_abi_verified_frame_example(tmp_path, ctx, scene_full, bottle, ref_frame):
    from yolo_ppf_pose_estimation_b200 import build
    r = ref_frame
    lib = build.build()
    np.ascontiguousarray(scene_full[:, :3], np.float32).tofile(tmp_path / "scene.f32")
    r["depth"].tofile(tmp_path / "depth.f32")
    bottle.astype(np.float32).tofile(tmp_path / "model.f32")
    exe = tmp_path / "c_abi_verified_frame_example"
    p = subprocess.run(["/usr/bin/gcc", "-std=c99", "-pedantic", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"),
                        os.path.join(ROOT, "tests", "cpp", "c_abi_verified_frame_example.c"), "-o", str(exe), "-L", os.path.dirname(lib),
                        "-lb200ppf", f"-Wl,-rpath,{os.path.dirname(lib)}"], capture_output=True, text=True)
    assert p.returncode == 0, p.stderr
    box = [int(v) for v in r["box"]]
    args = [str(tmp_path), "0.01", "0.025", str(r["depth"].shape[0]), str(r["depth"].shape[1])] + [repr(float(v)) for v in r["K"]] + \
           [str(v) for v in box * 2]
    p = subprocess.run([str(exe)] + args, capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stdout + p.stderr
    lines = p.stdout.strip().splitlines()
    assert len(lines) == 2
    print("\n".join(lines))
    res, status, cands = ctx.cv_match_frame_verified(r["scene"], [r["cor"]] * 2, [r["det"]] * 2, [r["model"]] * 2, leaf=0.01)
    for i, line in enumerate(lines):
        v = line.split()
        assert v[:3] == ["box", str(i), "0"] and status[i] == 0
        assert int(v[3]) == res[i]["votes"] and int(v[4]) == res[i]["n_poses"] and float(v[5]) == res[i]["residual"]
        best = cands[i][0]
        assert np.float32(float(v[6])) == np.float32(best["fit"]["fit"]) and int(v[7]) == best["fit"]["inliers"]
        assert int(v[8]) == best["fit"]["visible"] and int(v[9]) == best["rank"]
        assert np.array_equal(np.array([float(x) for x in v[10:]]), res[i]["pose"].reshape(16))
