"""GPU tests of the engine the reference actually calls — cv::ppf_match_3d::PPF3DDetector on the device
(csrc/k7_cvppf.cu, b200cv_*): its errors and the OpenCV-shaped shim.  Its parity with the float64 restatement and the
CPU oracle, case by case, is tests/test_gpu_cvppf_steps.py.
"""
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT

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
    """the bottle under a known rigid motion inside clutter, and a curvature-edge-like subset of the instance"""
    G = _rigid((0.3, 1.0, 0.2), 0.7, (0.1, -0.05, 0.3))
    rng = np.random.default_rng(7)
    inst = np.concatenate([bottle_5mm[:, :3] @ G[:3, :3].T + G[:3, 3], bottle_5mm[:, 3:] @ G[:3, :3].T], axis=1)
    centre = inst[:, :3].mean(0)
    clutter = np.concatenate([centre + rng.normal(scale=0.15, size=(600, 3)), rng.normal(size=(600, 3))], axis=1)
    clutter[:, 3:] /= np.linalg.norm(clutter[:, 3:], axis=1, keepdims=True)
    scene = np.concatenate([inst, clutter]).astype(np.float32)
    # "edges": the instance points where the profile bends most (the shoulder and the rims of the bottle) — what
    # EdgeExtraction's curvature threshold keeps
    z = bottle_5mm[:, :3] @ np.linalg.eigh(np.cov(bottle_5mm[:, :3].T))[1][:, -1]
    q = np.quantile(z, [0.03, 0.62, 0.72, 0.97])
    edge = inst[(z < q[0]) | ((z > q[1]) & (z < q[2])) | (z > q[3])].astype(np.float32)
    return bottle_5mm, scene, edge, G


@pytest.fixture(scope="module")
def detectors(ctx, oracle, case):
    from yolo_ppf_pose_estimation_b200 import capi
    model = case[0]
    ref = oracle.CvDetector(0.04, 0.05).train_model(model)
    dev = capi.CvDetector(ctx, 0.04, 0.05).train_model(model)
    return dev, ref


def test_cv_errors_and_edges(ctx, case):
    from yolo_ppf_pose_estimation_b200 import capi
    model, scene, edge, G = case
    d = capi.CvDetector(ctx, 0.05, 0.05)
    with pytest.raises(capi.B200PPFError):
        d.match(scene)                                   # not trained
    with pytest.raises(capi.B200PPFError):
        d.train_model(model[:, :3])                      # no normals
    flat = model.copy()
    flat[:, 2] = 0.5
    with pytest.raises(capi.B200PPFError):
        d.train_model(flat)                              # zero extent: upstream divides by it
    d.train_model(model)
    with pytest.raises(capi.B200PPFError):
        d.match_s2b(scene, edge[:0])
    with pytest.raises(capi.B200PPFError):
        capi.CvDetector(ctx, 0.0, 0.05)
    # search parameters reach the clustering: a huge position threshold and rotation threshold merge everything
    d.set_search_params(1e3, 10.0)
    res, ncl = d.match(scene, 1.0 / 5.0, 0.05)
    assert ncl == 1 and res["num_votes"][0] == d.raw_poses()["num_votes"].sum()


def test_cpp_opencv_ppf_shim(tmp_path, ctx, oracle, case, detectors):
    """tests/cpp/cv_ppf_shim_example.cpp — PPF3DDetector(0.04, 0.05).trainModel / match / match_S2B and the ICP of the best
    poses, the reference's own call sequence, through include/opencv_compat — gives the C-ABI results."""
    from yolo_ppf_pose_estimation_b200 import build
    dev, ref = detectors
    model, scene, edge, G = case
    lib = build.build()
    model.astype(np.float32).tofile(tmp_path / "model.f32")
    scene.tofile(tmp_path / "scene.f32")
    edge.tofile(tmp_path / "edge.f32")
    exe = tmp_path / "cv_ppf_shim_example"
    cmd = ["/usr/bin/g++", "-std=c++14", "-O1", "-I", os.path.join(ROOT, "include", "opencv_compat"), "-I", os.path.join(ROOT, "include"),
           os.path.join(ROOT, "tests", "cpp", "cv_ppf_shim_example.cpp"), "-o", str(exe), "-L", os.path.dirname(lib), "-lb200ppf",
           f"-Wl,-rpath,{os.path.dirname(lib)}"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe), str(tmp_path)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    lines = {ln.split()[0]: ln for ln in r.stdout.strip().splitlines()}
    for tag, (res, ncl) in (("match", dev.match(scene, 1.0 / 5.0, 0.04)), ("match_S2B", dev.match_s2b(scene, edge, 1.0 / 5.0, 0.04))):
        parts = lines[tag].split(" | ")
        assert int(parts[0].split()[1]) == ncl
        for k, part in enumerate(parts[1:]):
            v = part.split()
            assert int(v[0]) == res["num_votes"][k] and int(v[1]) == res["model_index"][k]
            assert np.array_equal(np.array([float(x) for x in v[2:]]), res["pose"][k])
    icp = [float(x) for x in lines["icp"].split()[1:]]
    P = np.array(icp[1:]).reshape(4, 4)
    pts = model[:, :3].astype(np.float64)
    err = np.linalg.norm((pts @ P[:3, :3].T + P[:3, 3]) - (pts @ G[:3, :3].T + G[:3, 3]), axis=1).mean()
    assert err < 0.01, err      # the refined pose is at least as good as the matched one
