"""CPU tests of pose verification (b200ppf_score_poses and the verified frame calls): the library exports the new symbols,
the three new structs are laid out in ctypes as the C compiler lays them out, a NULL context is refused, the verified C99
example compiles under strict flags, and the float64 restatement (tests/verify_reference.py) that the GPU tests compare
against gives the right answers on hand-made clouds.  No device compute happens here."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from verify_reference import score

NEW_SYMBOLS = ("b200ppf_verify_params_default", "b200ppf_score_poses", "b200cv_match_frame_verified", "b200ppf_match_frame_verified")
TAU = 0.01


def test_library_exports_the_verification_calls():
    from yolo_ppf_pose_estimation_b200 import capi
    L = C.CDLL(capi._build.LIB_PATH)
    for name in NEW_SYMBOLS:
        assert hasattr(L, name), name
        assert name in capi.SYMBOLS, name
    prm = capi.VerifyParams()
    capi.lib().b200ppf_verify_params_default(C.byref(prm))
    assert prm.inlier_dist == np.float32(0.01) and abs(prm.normal_angle - np.radians(30.0)) < 1e-6


@pytest.mark.parametrize("struct,cls", [("b200ppf_verify_params", "VerifyParams"), ("b200ppf_pose_fit", "PoseFit"),
                                        ("b200ppf_candidate", "Candidate")])
def test_struct_layout_matches_the_header(tmp_path, struct, cls):
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


def test_verified_calls_refuse_a_null_context():
    from yolo_ppf_pose_estimation_b200 import capi
    L, INVALID = capi.lib(), -1
    c12 = (C.c_float * 12)()
    assert L.b200ppf_score_poses(None, None, 0, None, None) == INVALID
    assert L.b200cv_match_frame_verified(None, None, 1, c12, None, None, None, None, None, None, None) == INVALID
    assert L.b200ppf_match_frame_verified(None, None, 1, c12, None, None, None, None, None, None, None) == INVALID
    assert b"null context" in L.b200ppf_last_error(None)


def test_verified_frame_example_is_strict_c99(tmp_path):
    r = subprocess.run(["/usr/bin/gcc", "-std=c99", "-pedantic", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), "-c",
                        os.path.join(ROOT, "tests", "cpp", "c_abi_verified_frame_example.c"), "-o", str(tmp_path / "a.o")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


# ---- the restatement on hand-made clouds -------------------------------------------------------------------------------
def _plane(z, normal=(0.0, 0.0, -1.0), spacing=0.02, n=10):
    """an n x n grid of points at depth z with one normal for all: (n*n, 6) float32"""
    g = (np.arange(n) - n / 2) * spacing
    x, y = np.meshgrid(g, g)
    pts = np.stack([x.ravel(), y.ravel(), np.full(x.size, z)], 1)
    return np.concatenate([pts, np.broadcast_to(np.asarray(normal, np.float64), pts.shape)], 1).astype(np.float32)


def _at(z):
    T = np.eye(4)
    T[2, 3] = z
    return T


def test_plane_on_plane_every_visible_point_is_an_inlier():
    r = score(_plane(0.0), _plane(1.0), _at(1.0), TAU)
    assert r["visible"] == 100 and r["inliers"] == 100 and r["fit"] == 1.0 and r["rms"] == 0.0
    # seen from behind: nothing is visible
    r = score(_plane(0.0, (0.0, 0.0, 1.0)), _plane(1.0), _at(1.0), TAU)
    assert r["visible"] == 0 and r["inliers"] == 0 and r["fit"] == 0.0


def test_plane_shifted_by_the_inlier_distance():
    eps = 1e-3 * TAU
    inside = score(_plane(0.0), _plane(np.float32(1.0 + TAU - eps)), _at(1.0), TAU)
    outside = score(_plane(0.0), _plane(np.float32(1.0 + TAU + eps)), _at(1.0), TAU)
    assert inside["inliers"] == 100 and not inside["borderline"].any()
    assert abs(inside["rms"] - (np.float32(1.0 + TAU - eps) - 1.0)) < 1e-9
    assert outside["inliers"] == 0 and outside["visible"] == 100 and not outside["borderline"].any()


def test_flipped_scene_normals_give_no_inlier():
    r = score(_plane(0.0), _plane(1.0, (0.0, 0.0, 1.0)), _at(1.0), TAU)
    assert r["visible"] == 100 and r["inliers"] == 0
    # without the normal test the distance alone decides
    assert score(_plane(0.0), _plane(1.0, (0.0, 0.0, 1.0)), _at(1.0), TAU, normal_angle=np.pi)["inliers"] == 100


def test_zero_model_normals_are_visible():
    model = _plane(0.0, (0.0, 0.0, 0.0))
    r = score(model, _plane(1.0), _at(1.0), TAU)
    assert r["visible"] == 100 and r["inliers"] == 0  # 0 >= cos(30 degrees) fails
    assert score(model, _plane(1.0), _at(1.0), TAU, normal_angle=np.pi)["inliers"] == 100


def test_borderline_points():
    # every point exactly at the inlier distance
    r = score(_plane(0.0), _plane(np.float32(1.0 + TAU)), _at(1.0), TAU)
    assert r["borderline"].all()
    # scene normals turned by exactly the normal angle (the bound of the normal test)
    a = np.radians(30.0)
    r = score(_plane(0.0), _plane(1.0, (0.0, np.sin(a), -np.cos(a))), _at(1.0), TAU, normal_angle=np.float32(a))
    assert r["borderline"].all()
    # two scene points equally near every model point: a tie, and the lower index is taken
    scene = np.concatenate([_plane(1.0), _plane(1.0, (0.0, 0.0, 1.0))])
    r = score(_plane(0.0), scene, _at(1.0), TAU)
    assert r["borderline"].all() and r["inliers"] == 100
    r = score(_plane(0.0), scene[::-1].copy(), _at(1.0), TAU)
    assert r["inliers"] == 0  # the flipped-normal copy now has the lower indices
    # nothing borderline on the plain case
    assert not score(_plane(0.0), _plane(1.0), _at(1.0), TAU)["borderline"].any()
