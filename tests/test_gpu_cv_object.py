"""GPU tests of the OpenCV engine on device clouds (b200cv_detector_match_cloud) and of its per-object call
(b200cv_match_object: SceneCropping -> ... -> Matching_S2B -> ICP of the top poses, src/YOLO_cropping_ppf_test.cpp:91-122).

Bars: a device cloud and its downloaded rows sample, vote and cluster bit for bit alike (same kernels, same bounding box);
the one-call chain equals the stages called one by one bit for bit; against the CPU checker the cluster votes are equal and
the poses agree to rounding (1e-9, the bar of test_gpu_cvppf.py), the refined pose to 1e-5 m.
"""
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, load_cloud

pytestmark = pytest.mark.gpu


def _rigid(axis, angle, t):
    axis = np.asarray(axis, np.float64) / np.linalg.norm(axis)
    K = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
    T = np.eye(4)
    T[:3, :3] = np.eye(3) + np.sin(angle) * K + (1 - np.cos(angle)) * K @ K
    T[:3, 3] = t
    return T


@pytest.fixture(scope="module")
def case(bottle_5mm):
    """the bottle under a known rigid motion inside clutter, and a curvature-edge-like subset of the instance
    (the case of test_gpu_cvppf.py)"""
    G = _rigid((0.3, 1.0, 0.2), 0.7, (0.1, -0.05, 0.3))
    rng = np.random.default_rng(7)
    inst = np.concatenate([bottle_5mm[:, :3] @ G[:3, :3].T + G[:3, 3], bottle_5mm[:, 3:] @ G[:3, :3].T], axis=1)
    centre = inst[:, :3].mean(0)
    clutter = np.concatenate([centre + rng.normal(scale=0.15, size=(600, 3)), rng.normal(size=(600, 3))], axis=1)
    clutter[:, 3:] /= np.linalg.norm(clutter[:, 3:], axis=1, keepdims=True)
    scene = np.concatenate([inst, clutter]).astype(np.float32)
    z = bottle_5mm[:, :3] @ np.linalg.eigh(np.cov(bottle_5mm[:, :3].T))[1][:, -1]
    q = np.quantile(z, [0.03, 0.62, 0.72, 0.97])
    edge = inst[(z < q[0]) | ((z > q[1]) & (z < q[2])) | (z > q[3])].astype(np.float32)
    return bottle_5mm, scene, edge


def _crop_box():
    b = np.load(os.path.join(ROOT, "tests", "golden", "crop_box.npz"))
    depth = np.zeros(tuple(b["image"]), np.float32)
    for (r, c), d in zip(b["pixels"], b["depths"]):
        depth[r, c] = d
    return depth, b["box"], b["intrinsics"]


def _same_match(det, host_call, cloud_call):
    """host_call / cloud_call run one match each; every result of the detector's last match must be the same bits"""
    res_h, ncl_h = host_call()
    scene_h, raw_h, info_h = det.scene_points(), det.raw_poses(), det.info
    res_c, ncl_c = cloud_call()
    scene_c, raw_c, info_c = det.scene_points(), det.raw_poses(), det.info
    assert (info_c.n_scene_sampled, info_c.n_second_sampled) == (info_h.n_scene_sampled, info_h.n_second_sampled)
    assert np.array_equal(scene_c.view(np.uint32), scene_h.view(np.uint32))
    for f in ("num_votes", "model_index", "alpha_index"):
        assert np.array_equal(raw_c[f], raw_h[f]), f
    assert raw_c.tobytes() == raw_h.tobytes()
    assert ncl_c == ncl_h and np.array_equal(res_c["num_votes"], res_h["num_votes"])
    assert res_c.tobytes() == res_h.tobytes()
    return res_c, ncl_c


def test_match_cloud_equals_host_match_bit_for_bit(ctx, case):
    from yolo_ppf_pose_estimation_b200 import capi
    model, scene, edge = case
    det = capi.CvDetector(ctx, 0.04, 0.05).train_model(model)
    ds, de = ctx.upload_cloud(scene), ctx.upload_cloud(edge)
    assert np.array_equal(ds.download(), scene) and np.array_equal(de.download(), edge)
    _same_match(det, lambda: det.match(scene, 1.0 / 5.0, 0.04), lambda: det.match_cloud(ds, None, 1.0 / 5.0, 0.04))
    _, ncl = _same_match(det, lambda: det.match_s2b(scene, edge, 1.0 / 5.0, 0.04), lambda: det.match_cloud(ds, de, 1.0 / 5.0, 0.04))
    assert det.info.n_second_sampled > 0 and ncl > 0


def test_match_cloud_of_a_prep_cloud_never_reads_the_curvature(ctx, bottle):
    """the reference's crop through the device pre-processing: nrm.w carries the curvature, the sampling reads xyz + normal only"""
    from yolo_ppf_pose_estimation_b200 import capi
    d = ctx.voxel_grid(ctx.upload_xyz(load_cloud("scene_crop_raw")), 0.005)
    d, _, _, _ = ctx.statistical_outlier_removal(d, 50, 1.0)
    ctx.normal_estimation(d, 30)
    e = ctx.curvature_edges(d, 0.03)
    ctx.normalize_normals(d)
    ctx.normalize_normals(e)
    assert (d.download(curvature=True)[:, 6] > 0).mean() > 0.5 and e.size > 0
    obj, edg = d.download(), e.download()
    det = capi.CvDetector(ctx, 0.025, 0.05).train_model(bottle)
    _same_match(det, lambda: det.match(obj, 1.0 / 14.0, 0.05), lambda: det.match_cloud(d, None, 1.0 / 14.0, 0.05))
    _same_match(det, lambda: det.match_s2b(obj, edg, 0.05, 0.05), lambda: det.match_cloud(d, e, 0.05, 0.05))


@pytest.fixture(scope="module")
def frame(ctx, scene_full, bottle):
    """the reference frame (regenerated 1 cm scene, surrogate YOLO box), the bottle model, PPF3DDetector(0.025, 0.05)"""
    from yolo_ppf_pose_estimation_b200 import capi
    depth, box, K = _crop_box()
    cor = capi.frustum_corners(depth, box, K)
    det = capi.CvDetector(ctx, 0.025, 0.05).train_model(bottle)
    return ctx.upload_xyz(scene_full[:, :3]), cor, ctx.upload_cloud(bottle), det


def _stepwise(ctx, scene, cor):
    d, _ = ctx.crop_pyramid(scene, cor)
    n_crop = d.size
    d = ctx.voxel_grid(d, 0.01)
    n_vox = d.size
    d, _, _, _ = ctx.statistical_outlier_removal(d, 50, 1.0)
    ctx.normal_estimation(d, 30)
    e = ctx.curvature_edges(d, 0.03)
    ctx.normalize_normals(d)
    ctx.normalize_normals(e)
    return d, e, (n_crop, n_vox, d.size, e.size)


@pytest.mark.parametrize("use_edges", [1, 0])
def test_cv_match_object_equals_the_stepwise_chain(ctx, oracle, bottle, frame, use_edges):
    """Matching_S2B (use_edges=1, steps 0.05 / 0.05) and Matching (use_edges=0, step 1/14): one call = the stages one by
    one with the host-array match and the top 5 through icp_refine; the CPU checker on the device's own clouds agrees"""
    scene, cor, model, det = frame
    step = 0.05 if use_edges else 1.0 / 14.0
    res, obj, edges = ctx.cv_match_object(det, scene, cor, model, leaf=0.01, use_edges=use_edges, relative_scene_sample_step=step)
    d, e, sizes = _stepwise(ctx, scene, cor)
    assert (res["n_cropped"], res["n_sampled"], res["n_filtered"], res["n_edges"]) == sizes
    assert np.array_equal(obj.download(curvature=True), d.download(curvature=True))
    assert np.array_equal(edges.download(curvature=True), e.download(curvature=True))
    o, eh = d.download(), e.download()
    clusters, ncl = det.match_s2b(o, eh, step, 0.05) if use_edges else det.match(o, step, 0.05)
    top = clusters["pose"][:5].reshape(-1, 4, 4)
    P, resid, _ = ctx.icp_refine(model, d, top)
    assert res["n_poses"] == ncl and res["votes"] == clusters["num_votes"][0]
    assert np.array_equal(res["pose"], P[0]) and res["residual"] == resid[0]
    assert res["total_wall_ms"] > 0 and res["match_ms"] > 0 and res["icp_ms"] > 0
    # the CPU chain on the device's object and edge clouds
    ref = oracle.CvDetector(0.025, 0.05).train_model(bottle)
    rposes, rvotes, _, rncl = ref.match_s2b(o, eh, step, 0.05) if use_edges else ref.match(o, step, 0.05)
    k = min(len(clusters), len(rposes))
    assert rncl == ncl and np.array_equal(clusters["num_votes"][:k], rvotes[:k])
    assert np.abs(clusters["pose"][:k].reshape(k, 4, 4) - rposes[:k]).max() < 1e-9
    R, rres, _ = oracle.icp_refine(bottle, o, rposes[:5])
    msg = (f"use_edges={use_edges}: {sizes} points, {ncl} clusters, votes {res['votes']}, residual {res['residual']:.6g} "
           f"vs CPU {rres[0]:.6g}")
    if res["residual"] < 1e9 and rres[0] < 1e9:
        dt = float(np.linalg.norm(res["pose"][:3, 3] - R[0][:3, 3]))
        print(f"{msg}, |dt| vs CPU chain {dt:.3e} m, wall {res['total_wall_ms']:.2f} ms")
        assert dt < 1e-5
    else:
        print(f"{msg}: an ICP lost its correspondences, no translation comparison")


def test_cv_match_object_errors(ctx, case, scene_full, bottle, frame):
    from yolo_ppf_pose_estimation_b200 import capi
    scene, cor, model, det = frame
    INVALID, STATE = -1, -4

    def code(fn):
        with pytest.raises(capi.B200PPFError) as e:
            fn()
        return e.value.code

    untrained = capi.CvDetector(ctx, 0.025, 0.05)
    assert code(lambda: ctx.cv_match_object(untrained, scene, cor, model)) == STATE
    other = capi.Context(0)
    foreign = [other.upload_xyz(scene_full[:, :3]), other.upload_cloud(bottle), other.upload_cloud(case[1])]
    assert code(lambda: ctx.cv_match_object(det, foreign[0], cor, model)) == INVALID
    assert code(lambda: ctx.cv_match_object(det, scene, cor, foreign[1])) == INVALID
    assert code(lambda: det.match_cloud(foreign[2])) == INVALID
    other.close()  # frees the clouds still alive on it (the tracebacks above keep them) before the context itself
    assert all(c._h is None for c in foreign)
    assert code(lambda: ctx.cv_match_object(det, scene, cor, model, edge_curvature=0.0)) == INVALID
    assert code(lambda: ctx.cv_match_object(det, ctx.upload_xyz(scene_full[:, :3] + np.float32(10)), cor, model)) == STATE  # empty crop
    assert code(lambda: ctx.cv_match_object(det, scene, cor, model, edge_curvature=1.0)) == STATE  # no point has curvature > 1/3
    assert code(lambda: det.match_cloud(ctx.upload_cloud(case[1]), ctx.upload_cloud(case[2][:0]))) == INVALID
    # Matching needs no edges: edge_curvature <= 0 is fine there, and then no edge cloud is made
    res, _, edges = ctx.cv_match_object(det, scene, cor, model, use_edges=0, edge_curvature=0.0, relative_scene_sample_step=1.0 / 14.0)
    assert edges is None and res["n_edges"] == 0 and res["n_poses"] > 0
    # no ICP: the best cluster as matched
    res, obj, _ = ctx.cv_match_object(det, scene, cor, model, icp_poses=0)
    best, _ = det.match_s2b(obj.download(), _stepwise(ctx, scene, cor)[1].download(), 0.05, 0.05)
    assert res["residual"] == 0.0 and res["icp_ms"] == 0.0 and np.array_equal(res["pose"].reshape(16), best["pose"][0])


def test_c_abi_cv_frame_example(tmp_path, ctx, scene_full, bottle, frame):
    """tests/cpp/c_abi_cv_frame_example.c — the frame uploaded once, one b200cv_match_object per box, strict C99 — prints
    the pose of the Python call"""
    from yolo_ppf_pose_estimation_b200 import build
    scene, cor, model, det = frame
    lib = build.build()
    depth, box, K = _crop_box()
    np.ascontiguousarray(scene_full[:, :3], np.float32).tofile(tmp_path / "scene.f32")
    depth.tofile(tmp_path / "depth.f32")
    bottle.astype(np.float32).tofile(tmp_path / "model.f32")
    exe = tmp_path / "c_abi_cv_frame_example"
    r = subprocess.run(["/usr/bin/gcc", "-std=c99", "-pedantic", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"),
                        os.path.join(ROOT, "tests", "cpp", "c_abi_cv_frame_example.c"), "-o", str(exe), "-L", os.path.dirname(lib),
                        "-lb200ppf", f"-Wl,-rpath,{os.path.dirname(lib)}"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    args = [str(tmp_path), "0.01", "0.025", str(depth.shape[0]), str(depth.shape[1])] + [repr(float(v)) for v in K] + \
           [str(int(v)) for v in box] * 2
    r = subprocess.run([str(exe)] + args, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    lines = r.stdout.strip().splitlines()
    assert len(lines) == 2
    res, _, _ = ctx.cv_match_object(det, scene, cor, model, leaf=0.01)
    for i, line in enumerate(lines):
        v = line.split()
        assert v[:3] == ["box", str(i), "0"]
        assert int(v[3]) == res["votes"] and int(v[4]) == res["n_poses"] and float(v[5]) == res["residual"]
        assert np.array_equal(np.array([float(x) for x in v[6:]]), res["pose"].reshape(16))
