"""CPU tests of verification against the depth image: the float64 restatement (tests/verify_depth_reference.py) against a
brute-force per-point loop of the rule in include/b200ppf.h, the depth frame generator is deterministic, the new structs are
laid out in ctypes as the C compiler lays them out, the header compiles as C99 and C++14, and the library exports the new
symbols.  No device compute happens here."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from verify_depth_reference import score_depth

NEW_SYMBOLS = ("b200ppf_depth_upload", "b200ppf_depth_free", "b200ppf_cloud_from_depth", "b200ppf_score_poses_depth",
               "b200cv_match_frame_verified_depth", "b200ppf_match_frame_verified_depth")


def test_library_exports_the_depth_calls():
    from yolo_ppf_pose_estimation_b200 import capi
    L = C.CDLL(capi._build.LIB_PATH)
    for name in NEW_SYMBOLS:
        assert hasattr(L, name), name
        assert name in capi.SYMBOLS, name
    assert capi.lib().b200ppf_score_poses_depth(None, None, 0, None, None, None) == -1
    assert capi.lib().b200ppf_depth_upload(None, None, 1, 1, None, None) == -1


@pytest.mark.parametrize("struct,cls", [("b200ppf_depth_fit", "DepthFit"), ("b200ppf_depth_candidate", "DepthCandidate")])
def test_struct_layouts_match_the_header(tmp_path, struct, cls):
    from yolo_ppf_pose_estimation_b200 import capi
    ct = getattr(capi, cls)
    fields = [n for n, _ in ct._fields_]
    body = f'printf("size %zu\\n", sizeof({struct}));' + "".join(f'printf("{n} %zu\\n", offsetof({struct}, {n}));' for n in fields)
    src = tmp_path / "layout.c"
    src.write_text(f'#include <stdio.h>\n#include <stddef.h>\n#include "b200ppf.h"\nint main(void){{{body}return 0;}}\n')
    subprocess.run(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(tmp_path / "layout")], check=True)
    out = subprocess.run([str(tmp_path / "layout")], capture_output=True, text=True, check=True).stdout
    got = dict(line.split() for line in out.strip().splitlines())
    assert int(got.pop("size")) == C.sizeof(ct)
    assert {n: int(v) for n, v in got.items()} == {n: getattr(ct, n).offset for n in fields}


@pytest.mark.parametrize("lang,std,compiler", [("c", "c99", "gcc"), ("c++", "c++14", "g++")])
def test_header_compiles_strictly(tmp_path, lang, std, compiler):
    src = tmp_path / ("h.c" if lang == "c" else "h.cpp")
    src.write_text('#include "b200ppf.h"\nint main(void) { b200ppf_depth_fit f; b200ppf_depth_candidate c; (void)f; (void)c; '
                   'return B200PPF_DEPTH_SPLAT_MAX == 16 ? 0 : 1; }\n')
    r = subprocess.run([compiler, f"-std={std}", "-pedantic", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), "-c",
                        str(src), "-o", str(tmp_path / "h.o")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


# ---- the restatement against a per-point loop --------------------------------------------------------------------------------
def _brute(model, scene, T, D, K, tau, angle):
    """the rule of include/b200ppf.h, one point at a time"""
    tau = float(np.float32(tau))
    use_normals = not (np.float32(angle) >= np.float32(np.pi))
    cos_min = math.cos(float(np.float32(angle)))
    fx, fy, ppx, ppy = (float(k) for k in K)
    rows, cols = D.shape
    moved = []
    for m in model.astype(np.float64):
        p = [T[r, 0] * m[0] + T[r, 1] * m[1] + T[r, 2] * m[2] + T[r, 3] for r in range(3)]
        n = [T[r, 0] * m[3] + T[r, 1] * m[4] + T[r, 2] * m[5] for r in range(3)]
        facing = (m[3] == 0 and m[4] == 0 and m[5] == 0) or -(n[0] * p[0] + n[1] * p[1] + n[2] * p[2]) > 0
        pix = None
        if p[2] > 0:
            fu, fv = fx * p[0] / p[2] + ppx + 0.5, fy * p[1] / p[2] + ppy + 0.5
            if 0 <= fu < cols and 0 <= fv < rows:
                pix = (int(math.floor(fv)), int(math.floor(fu)))
        moved.append((p, n, facing, pix))
    zb = {}
    for p, _, _, pix in moved:
        if pix is None:
            continue
        h = int(min(math.floor(fx * tau / (2.0 * p[2])), 16))
        for v in range(max(pix[0] - h, 0), min(pix[0] + h, rows - 1) + 1):
            for u in range(max(pix[1] - h, 0), min(pix[1] + h, cols - 1) + 1):
                zb[v, u] = min(zb.get((v, u), math.inf), p[2])
    c = dict.fromkeys(("inliers", "judged", "visible", "self_occluded", "occluded", "violations", "unknown"), 0)
    d2s = []
    s = scene.astype(np.float64)
    for p, n, facing, pix in moved:
        if not facing or pix is None:
            continue
        if p[2] > zb[pix] + tau:
            c["self_occluded"] += 1
            continue
        c["visible"] += 1
        d = float(D[pix])
        if not (d > 0 and math.isfinite(d)):
            c["unknown"] += 1
            continue
        if p[2] > d + tau:
            c["occluded"] += 1
            continue
        c["judged"] += 1
        if p[2] < d - tau:
            c["violations"] += 1
            continue
        if len(s) == 0:
            continue
        e2 = ((s[:, :3] - np.array(p)) ** 2).sum(1)
        j = int(np.argmin(e2))
        if e2[j] <= tau * tau and (not use_normals or s[j, 3:6] @ np.array(n) >= cos_min):
            c["inliers"] += 1
            d2s.append(e2[j])
    c["fit"] = c["inliers"] / c["judged"] if c["judged"] else 0.0
    c["rms"] = math.sqrt(sum(d2s) / len(d2s)) if d2s else 0.0
    return c


def _case(seed):
    """a small random case: a model patch seen by a 24 x 32 camera, with an occluder, holes, NaN pixels, points behind the
    camera and outside the image"""
    rng = np.random.default_rng(seed)
    K = np.array([40.0, 41.0, 15.5, 11.5])
    n = 80
    xyz = np.stack([rng.uniform(-0.3, 0.3, n), rng.uniform(-0.2, 0.2, n), rng.uniform(-0.05, 0.05, n)], 1)
    nrm = rng.normal(size=(n, 3))
    nrm[:, 2] = -np.abs(nrm[:, 2]) - 0.5
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    nrm[:5] = 0.0  # zero normals count as facing
    model = np.concatenate([xyz, nrm], 1).astype(np.float32)
    T = np.eye(4)
    T[:3, 3] = (0.0, 0.0, 0.8)
    if seed % 2:
        T[:3, 3] = (0.25, 0.0, 0.6)  # a part outside the image
    p = model[:, :3].astype(np.float64) + T[:3, 3]
    # the depth: the model's surface with noise and offsets, an occluder, holes and NaN pixels
    D = rng.uniform(0.7, 1.2, (24, 32)).astype(np.float32)
    u = np.floor(K[0] * p[:, 0] / p[:, 2] + K[2] + 0.5).astype(int)
    v = np.floor(K[1] * p[:, 1] / p[:, 2] + K[3] + 0.5).astype(int)
    ok = (u >= 0) & (u < 32) & (v >= 0) & (v < 24)
    D[v[ok], u[ok]] = (p[ok, 2] + rng.choice([0.0, 0.004, -0.004, 0.05, -0.05], ok.sum())).astype(np.float32)
    D[2:9, 3:10] = 0.4  # occluder
    D[rng.random(D.shape) < 0.08] = 0.0
    D[rng.random(D.shape) < 0.04] = np.nan
    D[rng.random(D.shape) < 0.02] = -1.0
    scene = model.copy()
    scene[:, :3] = p + rng.normal(scale=0.003, size=p.shape)
    behind = T.copy()
    behind[2, 3] = -0.01  # part of the model behind the camera
    return model, scene, [T, behind], D, K


@pytest.mark.parametrize("seed", range(6))
@pytest.mark.parametrize("tau,angle", [(0.01, np.radians(30.0)), (0.02, np.pi), (0.005, np.radians(45.0))])
def test_restatement_equals_the_per_point_rule(seed, tau, angle):
    model, scene, poses, D, K = _case(seed)
    for T in poses:
        r = score_depth(model, scene, T, D, K, tau, angle)
        b = _brute(model, scene, T, D, K, tau, angle)
        slack = int(r["borderline"].sum())
        for k in ("inliers", "judged", "visible", "self_occluded", "occluded", "violations", "unknown"):
            assert abs(r[k] - b[k]) <= slack, (k, r[k], b[k], slack)
            if slack == 0:
                assert r[k] == b[k], (k, r[k], b[k])
        assert r["visible"] == r["judged"] + r["occluded"] + r["unknown"]
        if slack == 0:
            assert abs(r["rms"] - b["rms"]) <= 1e-12 + 1e-9 * b["rms"]


def test_restatement_cases_cover_every_outcome():
    seen = dict.fromkeys(("inliers", "self_occluded", "occluded", "violations", "unknown"), 0)
    for seed in range(6):
        model, scene, poses, D, K = _case(seed)
        for T in poses:
            r = score_depth(model, scene, T, D, K)
            for k in seen:
                seen[k] += r[k]
    assert all(v > 0 for v in seen.values()), seen


def test_depth_frame_is_deterministic():
    from yolo_ppf_pose_estimation_b200 import synth
    a, b = synth.synth_library_depth(), synth.synth_library_depth()
    assert a["depth"].dtype == np.float32 and a["depth"].shape == synth.DEPTH_SHAPE
    assert a["depth"].tobytes() == b["depth"].tobytes() and np.array_equal(a["K"], b["K"])
    assert np.array_equal(a["occluded_share"], b["occluded_share"])
    occluded = np.flatnonzero(a["occluded_share"])
    assert len(occluded) >= 2 and all(0.3 <= a["occluded_share"][k] <= 0.6 for k in occluded)
    # every instance is in view: its true pose projects inside the image
    for k in range(8):
        t = synth.library_pose(k)[:3, 3]
        u, v = a["K"][0] * t[0] / t[2] + a["K"][2], a["K"][1] * t[1] / t[2] + a["K"][3]
        assert 0 <= u < synth.DEPTH_SHAPE[1] and 0 <= v < synth.DEPTH_SHAPE[0]
