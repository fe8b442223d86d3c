"""GPU tests of screening the pose clusters before ICP: b200cv_match_frame_screened and b200cv_match_frame_screened_depth.

Bars: screen_poses = max(icp_poses, 1) gives the verified call's results and candidates bit for bit; every other screen
equals its restatement through public calls (the object cloud of cv_match_object, every cluster of CvDetector.match_cloud,
score_poses / score_poses_depth of the first S, the selection by (fit desc, rank asc) in numpy, icp_refine_batch and a
second score) in pose, residual, votes, rank and fit, and every non-pose result field is cv_match_frame's; the launch count
is the same for S = 1 and S = 0 and grows with the boxes as the unverified call's does; with S = 0 the library instances
found include those the verified call finds; a failed box has empty slots and leaves the others; bad verify values and bad
depth images are refused without leaking.
"""
import ctypes

import numpy as np
import pytest

from test_gpu_frame import N_LIBRARY
from test_gpu_verify import SAME_FIELDS, _found, _object, lib_frame, pool_used, ref_frame  # noqa: F401
from test_gpu_verify_depth import depth_frame, ref_depth  # noqa: F401

pytestmark = pytest.mark.gpu

INVALID, STATE = -1, -4
UNUSED = 0xFFFFFFFF


def _over(leaf, use_edges=1, icp_poses=5):
    return dict(leaf=leaf, use_edges=use_edges, icp_poses=icp_poses, relative_scene_sample_step=0.05 if use_edges else 1.0 / 14.0)


def _cand_key(c):
    return c["pose"].tobytes(), c["residual"], c["votes"], c["rank"], c["fit"]


# ---- 1. screen_poses = max(icp_poses, 1) is the verified call --------------------------------------------------------------
def _lib_and_ref(lib_frame, ref_frame):
    L, r = lib_frame, ref_frame
    return ((L["scene"], L["cors"], L["dets"], L["dmodels"], 0.005),
            (r["scene"], np.stack([r["cor"]] * 2), [r["det"]] * 2, [r["model"]] * 2, 0.01))


@pytest.mark.parametrize("use_edges,icp_poses", [(1, 5), (1, 0), (0, 5), (0, 0)])
def test_screen_of_the_verified_clusters_is_the_verified_call(ctx, lib_frame, ref_frame, use_edges, icp_poses):
    for scene, cors, dets, mods, leaf in _lib_and_ref(lib_frame, ref_frame):
        over = _over(leaf, use_edges, icp_poses)
        vres, vstatus, vcands = ctx.cv_match_frame_verified(scene, cors, dets, mods, **over)
        sres, sstatus, scands = ctx.cv_match_frame_screened(scene, cors, dets, mods, screen_poses=max(icp_poses, 1), **over)
        assert sstatus.tolist() == vstatus.tolist()
        for a, b in zip(vres, sres):
            assert all(a[f] == b[f] for f in SAME_FIELDS + ("votes", "residual")) and a["pose"].tobytes() == b["pose"].tobytes()
        assert [[_cand_key(c) for c in box] for box in scands] == [[_cand_key(c) for c in box] for box in vcands]


@pytest.mark.parametrize("use_edges,icp_poses", [(1, 5), (0, 0)])
def test_depth_screen_of_the_verified_clusters_is_the_verified_call(ctx, depth_frame, ref_frame, ref_depth, use_edges, icp_poses):
    L, r = depth_frame, ref_frame
    for scene, dimg, cors, dets, mods, leaf in ((L["scene"], L["dimg"], L["cors"], L["dets"], L["dmodels"], 0.005),
                                                 (r["scene"], ref_depth["dimg"], np.stack([r["cor"]] * 2), [r["det"]] * 2,
                                                  [r["model"]] * 2, 0.01)):
        over = _over(leaf, use_edges, icp_poses)
        vres, vstatus, vcands = ctx.cv_match_frame_verified_depth(scene, dimg, cors, dets, mods, **over)
        sres, sstatus, scands = ctx.cv_match_frame_screened_depth(scene, dimg, cors, dets, mods, screen_poses=max(icp_poses, 1),
                                                                  **over)
        assert sstatus.tolist() == vstatus.tolist()
        for a, b in zip(vres, sres):
            assert all(a[f] == b[f] for f in SAME_FIELDS + ("votes", "residual")) and a["pose"].tobytes() == b["pose"].tobytes()
        assert [[_cand_key(c) for c in box] for box in scands] == [[_cand_key(c) for c in box] for box in vcands]


# ---- 2. the restatement through public calls ---------------------------------------------------------------------------------
def _screen_expected(ctx, det, scene, cor, model, over, S, score):
    """box's candidates as the screened call documents them, from public calls; score(model, obj, P) -> fit dicts"""
    obj, edges = _object(ctx, det, scene, cor, model, **over)
    top, n = det.match_cloud(obj, edges if over["use_edges"] else None, over["relative_scene_sample_step"], 0.05, max_poses=obj.size)
    assert len(top) == n >= 1
    s = n if S == 0 else min(S, n)
    P = np.stack([t["pose"].reshape(4, 4) for t in top[:s]]).astype(np.float64)
    fits = score(model, obj, P)
    icp_poses = over["icp_poses"]
    keep = sorted(sorted(range(s), key=lambda k: (-fits[k]["fit"], k))[:min(icp_poses, s) if icp_poses else 1])
    if icp_poses:
        [(R, res)], _ = ctx.icp_refine_batch([(model, obj, P[keep])])
        final = score(model, obj, R)
    else:
        R, res, final = P[keep], np.zeros(len(keep)), [fits[k] for k in keep]
    cands = [{"pose": R[i], "residual": float(res[i]), "votes": int(top[k]["num_votes"]), "rank": k, "fit": final[i]}
             for i, k in enumerate(keep)]
    order = sorted(range(len(cands)), key=lambda i: (-cands[i]["fit"]["fit"], i))
    return [cands[i] for i in order], n


def _check_restatement(ctx, screened, plain, scene, cors, dets, mods, over, S, score):
    res, status = plain
    sres, sstatus, scands = screened
    assert sstatus.tolist() == status.tolist() == [0] * len(dets)
    for b in range(len(dets)):
        for f in SAME_FIELDS:
            assert sres[b][f] == res[b][f], (b, f)
        want, n = _screen_expected(ctx, dets[b], scene, cors[b], mods[b], over, S, score)
        assert sres[b]["n_poses"] == n
        assert [_cand_key(c) for c in scands[b]] == [_cand_key(c) for c in want], b
        best = scands[b][0]
        assert sres[b]["pose"].tobytes() == best["pose"].tobytes() and sres[b]["residual"] == best["residual"] and \
            sres[b]["votes"] == best["votes"]


SCREENS = [(S, icp) for S in (0, 1, 7) for icp in (5, 1, 0)]


@pytest.mark.parametrize("S,icp_poses", SCREENS)
def test_screened_equals_its_restatement(ctx, lib_frame, ref_frame, S, icp_poses):
    L, r = lib_frame, ref_frame
    idx = [2, 3, 4]
    for scene, cors, dets, mods, leaf in ((L["scene"], L["cors"][idx], [L["dets"][k] for k in idx], [L["dmodels"][k] for k in idx], 0.005),
                                          (r["scene"], np.stack([r["cor"]]), [r["det"]], [r["model"]], 0.01)):
        over = _over(leaf, 1, icp_poses)
        screened = ctx.cv_match_frame_screened(scene, cors, dets, mods, screen_poses=S, **over)
        plain = ctx.cv_match_frame(scene, cors, dets, mods, **over)
        _check_restatement(ctx, screened, plain, scene, cors, dets, mods, over, S,
                           lambda m, o, P: ctx.score_poses([(m, o, P)])[0])


@pytest.mark.parametrize("S,icp_poses", SCREENS)
def test_depth_screened_equals_its_restatement(ctx, depth_frame, S, icp_poses):
    L = depth_frame
    idx = [2, 3]
    scene, dimg, cors, dets, mods = L["scene"], L["dimg"], L["cors"][idx], [L["dets"][k] for k in idx], [L["dmodels"][k] for k in idx]
    over = _over(0.005, 1, icp_poses)
    screened = ctx.cv_match_frame_screened_depth(scene, dimg, cors, dets, mods, screen_poses=S, **over)
    plain = ctx.cv_match_frame(scene, cors, dets, mods, **over)
    _check_restatement(ctx, screened, plain, scene, cors, dets, mods, over, S,
                       lambda m, o, P: ctx.score_poses_depth([(m, o, P)], dimg)[0])


# ---- 3. launch count -----------------------------------------------------------------------------------------------------------
def test_launch_count_does_not_grow_with_the_screen_or_the_boxes(ctx, lib_frame, depth_frame):
    L, D = lib_frame, depth_frame

    def launches(fn):
        n0 = ctx.launch_count
        fn()
        return ctx.launch_count - n0
    for name, F, call in (("object cloud", L, lambda s, c, d, m, **o: ctx.cv_match_frame_screened(s, c, d, m, **o)),
                          ("depth", D, lambda s, c, d, m, **o: ctx.cv_match_frame_screened_depth(s, D["dimg"], c, d, m, **o))):
        n = {}
        for K in (1, 3):
            cors, dets, mods = np.stack([F["cors"][2]] * K), [F["dets"][2]] * K, [F["dmodels"][2]] * K
            n["plain", K] = launches(lambda: ctx.cv_match_frame(F["scene"], cors, dets, mods, leaf=0.005))
            for S in (1, 0):
                n[S, K] = launches(lambda: call(F["scene"], cors, dets, mods, screen_poses=S, leaf=0.005))
        print(f"{name}: launches {n}")
        assert n[1, 1] == n[0, 1] and n[1, 3] == n[0, 3]
        assert n[0, 3] - n[0, 1] == n["plain", 3] - n["plain", 1]


# ---- 4. library instances ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("use_edges", [1, 0])
def test_screening_finds_the_verified_instances(ctx, lib_frame, use_edges):
    L = lib_frame
    over = _over(0.005, use_edges, 5)
    vres, vstatus, vcands = ctx.cv_match_frame_verified(L["scene"], L["cors"], L["dets"], L["dmodels"], **over)
    sres, sstatus, scands = ctx.cv_match_frame_screened(L["scene"], L["cors"], L["dets"], L["dmodels"], screen_poses=0, **over)
    verified, screened = _found(vres), _found(sres)
    print(f"{'match_S2B' if use_edges else 'Matching'}: found verified {sorted(verified)}, screened {sorted(screened)}; "
          f"clusters {[int(x['n_poses']) for x in sres]}; kept ranks {[sorted(c['rank'] for c in x) for x in scands]}; "
          f"best fits verified {[round(x[0]['fit']['fit'], 3) for x in vcands]} screened {[round(x[0]['fit']['fit'], 3) for x in scands]}")
    assert vstatus.tolist() == sstatus.tolist() == [0] * N_LIBRARY
    assert screened >= verified, (verified, screened)


# ---- 5. failures and errors ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("with_depth", [False, True])
def test_a_failed_box_has_empty_slots_and_leaves_the_others(ctx, lib_frame, depth_frame, with_depth):
    from yolo_ppf_pose_estimation_b200 import capi
    F = depth_frame if with_depth else lib_frame
    behind = F["cors"][1] * np.array([1, 1, -1], np.float32)
    cors = np.stack([F["cors"][0], behind, F["cors"][2]])
    dets, mods = [F["dets"][k] for k in (0, 1, 2)], [F["dmodels"][k] for k in (0, 1, 2)]
    prm = ctx._params(capi.CvObjectParams, capi.lib().b200cv_object_params_default, dict(leaf=0.005))
    res = (capi.ObjectResult * 3)()
    status = np.zeros(3, np.int32)
    c12 = np.ascontiguousarray(cors, np.float32).reshape(-1, 12)
    if with_depth:
        cand = (capi.DepthCandidate * 15)()
        ctx.check(capi.lib().b200cv_match_frame_screened_depth(ctx._h, F["scene"]._h, F["dimg"]._h, 3, c12.ctypes.data,
                                                               ctx._handles(dets, 3), ctx._handles(mods, 3), ctypes.byref(prm), None,
                                                               0, res, status.ctypes.data, cand))
        good, gstatus, gcands = ctx.cv_match_frame_screened_depth(F["scene"], F["dimg"], cors[[0, 2]], [dets[0], dets[2]],
                                                                  [mods[0], mods[2]], leaf=0.005)
    else:
        cand = (capi.Candidate * 15)()
        ctx.check(capi.lib().b200cv_match_frame_screened(ctx._h, F["scene"]._h, 3, c12.ctypes.data, ctx._handles(dets, 3),
                                                         ctx._handles(mods, 3), ctypes.byref(prm), None, 0, res, status.ctypes.data,
                                                         cand))
        good, gstatus, gcands = ctx.cv_match_frame_screened(F["scene"], cors[[0, 2]], [dets[0], dets[2]], [mods[0], mods[2]],
                                                            leaf=0.005)
    assert status.tolist() == [0, STATE, 0] and gstatus.tolist() == [0, 0]
    assert all(bytes(cand[5 + i].pose) == bytes(16 * 8) and cand[5 + i].rank == UNUSED and cand[5 + i].votes == 0 and
               bytes(cand[5 + i].fit) == bytes(ctypes.sizeof(type(cand[5 + i].fit))) for i in range(5))
    for b, g in ((0, 0), (2, 1)):
        assert bytes(res[b].pose) == good[g]["pose"].tobytes()
        got = [ctx._fit(cand[5 * b + i].fit) for i in range(5) if cand[5 * b + i].rank != UNUSED]
        assert [(bytes(cand[5 * b + i].pose), cand[5 * b + i].rank, cand[5 * b + i].votes, cand[5 * b + i].residual)
                for i in range(len(got))] == [(x["pose"].tobytes(), x["rank"], x["votes"], x["residual"]) for x in gcands[g]]
        assert got == [x["fit"] for x in gcands[g]]


def test_bad_verify_values_and_depth_images(ctx, lib_frame, depth_frame, pool_used):  # noqa: F811
    from yolo_ppf_pose_estimation_b200 import capi
    L, D = lib_frame, depth_frame
    cors, dets, mods = L["cors"][:2], L["dets"][:2], L["dmodels"][:2]
    dcors, ddets, dmods = D["cors"][:2], D["dets"][:2], D["dmodels"][:2]
    screened = lambda **o: ctx.cv_match_frame_screened(L["scene"], cors, dets, mods, leaf=0.005, **o)  # noqa: E731
    screened_depth = lambda img, **o: ctx.cv_match_frame_screened_depth(D["scene"], img, dcors, ddets, dmods, leaf=0.005, **o)  # noqa: E731
    screened(), screened_depth(D["dimg"])  # warm
    start = pool_used()
    screened()
    screened_depth(D["dimg"])
    assert pool_used() == start

    def code(fn):
        with pytest.raises(capi.B200PPFError) as e:
            fn()
        return e.value.code
    for bad in (dict(inlier_dist=0.0), dict(inlier_dist=-0.01), dict(inlier_dist=np.nan), dict(inlier_dist=np.inf),
                dict(normal_angle=-0.1), dict(normal_angle=np.nan)):
        assert code(lambda: screened(**bad)) == INVALID, bad
        assert code(lambda: screened_depth(D["dimg"], **bad)) == INVALID, bad
    other = capi.Context(0)
    foreign = other.upload_depth(np.ones((4, 5), np.float32), np.array([100.0, 100.0, 2.0, 1.5]))
    assert code(lambda: screened_depth(foreign)) == INVALID
    foreign.free()
    other.close()
    res = (capi.ObjectResult * 2)()
    st = np.zeros(2, np.int32)
    c12 = np.ascontiguousarray(dcors, np.float32).reshape(-1, 12)
    assert capi.lib().b200cv_match_frame_screened_depth(ctx._h, D["scene"]._h, None, 2, c12.ctypes.data, ctx._handles(ddets, 2),
                                                        ctx._handles(dmods, 2), None, None, 0, res, st.ctypes.data, None) == INVALID
    assert pool_used() == start
