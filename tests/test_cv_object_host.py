"""CPU tests of the per-object call of the OpenCV engine (b200cv_match_object): its parameter block is laid out in ctypes
as the C compiler lays it out, its defaults are the reference's, and the C99 frame example compiles under strict flags.
No device compute happens here."""
import ctypes as C
import os
import subprocess

import numpy as np

from conftest import ROOT


def test_cv_object_params_layout_matches_the_header(tmp_path):
    from yolo_ppf_pose_estimation_b200 import capi
    fields = [n for n, _ in capi.CvObjectParams._fields_]
    body = 'printf("size %zu\\n", sizeof(b200cv_object_params));' + "".join(
        f'printf("{n} %zu\\n", offsetof(b200cv_object_params, {n}));' for n in fields)
    src = tmp_path / "layout.c"
    src.write_text(f'#include <stdio.h>\n#include <stddef.h>\n#include "b200ppf.h"\nint main(void){{{body}return 0;}}\n')
    subprocess.run(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(tmp_path / "layout")], check=True)
    out = subprocess.run([str(tmp_path / "layout")], capture_output=True, text=True, check=True).stdout
    got = dict(line.split() for line in out.strip().splitlines())
    assert int(got.pop("size")) == C.sizeof(capi.CvObjectParams)
    assert {n: int(v) for n, v in got.items()} == {n: getattr(capi.CvObjectParams, n).offset for n in fields}


def test_cv_object_params_default_is_the_reference_chain():
    """src/YOLO_cropping_ppf_test.cpp:98-120 and include/CloudProcessing.h:481-530: OutlierProcessing(50), NormalEstimation(30),
    EdgeExtraction(0.03), match_S2B(object, edges, results, 0.05, 0.05), the top 5 poses through ICP(100, 0.005, 2.5, 8)"""
    from yolo_ppf_pose_estimation_b200 import capi
    p = capi.CvObjectParams()
    capi.lib().b200cv_object_params_default(C.byref(p))
    assert (p.sor_mean_k, p.sor_stddev_mul, p.normal_k, p.use_edges, p.icp_poses) == (50, 1.0, 30, 1, 5)
    assert p.leaf == np.float32(0.01) and p.edge_curvature == np.float32(0.03)
    assert (p.relative_scene_sample_step, p.relative_scene_distance) == (0.05, 0.05)
    assert (p.icp.max_iterations, p.icp.tolerance, p.icp.rejection_scale, p.icp.num_levels) == (100, np.float32(0.005), 2.5, 8)
    capi.lib().b200cv_object_params_default(None)  # a NULL block is ignored


def test_cv_frame_example_is_strict_c99(tmp_path):
    r = subprocess.run(["/usr/bin/gcc", "-std=c99", "-pedantic", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), "-c",
                        os.path.join(ROOT, "tests", "cpp", "c_abi_cv_frame_example.c"), "-o", str(tmp_path / "a.o")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
