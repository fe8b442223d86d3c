"""CPU tests of the frame calls (b200ppf_crop_pyramids, b200ppf_icp_refine_batch, b200cv_match_frame, b200ppf_match_frame):
the ICP job block is laid out in ctypes as the C compiler lays it out, the library exports the new symbols, the multi-box C99
example compiles under strict flags, and a NULL context is refused.  No device compute happens here."""
import ctypes as C
import os
import subprocess

from conftest import ROOT

NEW_SYMBOLS = ("b200ppf_crop_pyramids", "b200ppf_icp_refine_batch", "b200cv_match_frame", "b200ppf_match_frame")


def test_icp_job_layout_matches_the_header(tmp_path):
    from yolo_ppf_pose_estimation_b200 import capi
    fields = [n for n, _ in capi.IcpJob._fields_]
    body = 'printf("size %zu\\n", sizeof(b200ppf_icp_job));' + "".join(
        f'printf("{n} %zu\\n", offsetof(b200ppf_icp_job, {n}));' for n in fields)
    src = tmp_path / "layout.c"
    src.write_text(f'#include <stdio.h>\n#include <stddef.h>\n#include "b200ppf.h"\nint main(void){{{body}return 0;}}\n')
    subprocess.run(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(tmp_path / "layout")], check=True)
    out = subprocess.run([str(tmp_path / "layout")], capture_output=True, text=True, check=True).stdout
    got = dict(line.split() for line in out.strip().splitlines())
    assert int(got.pop("size")) == C.sizeof(capi.IcpJob)
    assert {n: int(v) for n, v in got.items()} == {n: getattr(capi.IcpJob, n).offset for n in fields}


def test_library_exports_the_frame_calls():
    from yolo_ppf_pose_estimation_b200 import capi
    L = C.CDLL(capi._build.LIB_PATH)
    for name in NEW_SYMBOLS:
        assert hasattr(L, name), name
        assert name in capi.SYMBOLS, name


def test_multi_box_example_is_strict_c99(tmp_path):
    r = subprocess.run(["/usr/bin/gcc", "-std=c99", "-pedantic", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), "-c",
                        os.path.join(ROOT, "tests", "cpp", "c_abi_multi_box_example.c"), "-o", str(tmp_path / "a.o")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def test_frame_calls_refuse_a_null_context():
    from yolo_ppf_pose_estimation_b200 import capi
    L, INVALID = capi.lib(), -1
    c12 = (C.c_float * 12)()
    out = (C.c_void_p * 1)()
    assert L.b200ppf_crop_pyramids(None, None, c12, 1, out) == INVALID
    assert L.b200ppf_icp_refine_batch(None, None, 0, None, None) == INVALID
    assert L.b200cv_match_frame(None, None, 1, c12, None, None, None, None, None) == INVALID
    assert L.b200ppf_match_frame(None, None, 1, c12, None, None, None, None, None) == INVALID
    assert b"null context" in L.b200ppf_last_error(None)
