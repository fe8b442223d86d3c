"""CPU tests of the host side: the C-ABI library loads and exports every declared symbol, fails
loudly without a GPU, the host build of the alpha-bin hot loop equals the literal form and the
oracle, the workload generators are deterministic, the multi-GPU sharding/all-gather plumbing is
exact under a 2-rank gloo run, the PCL-shaped C++ shim compiles and links, and bench.py's
reference arm prints the contract line.  No device compute happens here.
"""
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from conftest import ANGLE_STEP, ROOT


def _header_functions():
    text = open(os.path.join(ROOT, "include", "b200ppf.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(b200(?:ppf|cv)_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from yolo_ppf_pose_estimation_b200 import capi
    declared = _header_functions()
    assert len(declared) >= 35
    assert sorted(capi.SYMBOLS) == declared, set(declared) ^ set(capi.SYMBOLS)
    lib = capi.lib()  # resolves every symbol or raises
    for name in declared:
        assert hasattr(lib, name)
    assert lib.b200ppf_version() == 100


def test_struct_layouts_match_the_header():
    import ctypes as C
    from yolo_ppf_pose_estimation_b200 import capi
    assert capi.HYP_DTYPE.itemsize == 64 and capi.SIG_DTYPE.itemsize == 20
    assert capi.HYP_DTYPE.fields["votes"][1] == 48 and capi.HYP_DTYPE.fields["scene_index"][1] == 60
    # sizes and the offset of every struct's last member as the C compiler lays them out
    import subprocess
    import tempfile
    structs = {"b200ppf_table_info": (capi.TableInfo, "n_merged"), "b200ppf_timings": (capi.Timings, "prep_ms"),
               "b200ppf_icp_params": (capi.IcpParams, "num_levels"), "b200ppf_object_params": (capi.ObjectParams, "icp"),
               "b200ppf_object_result": (capi.ObjectResult, "total_wall_ms")}
    body = "".join(f'printf("{n} %zu %zu\\n", sizeof({n}), offsetof({n}, {last}));' for n, (_, last) in structs.items())
    with tempfile.TemporaryDirectory() as d:
        src = os.path.join(d, "layout.c")
        open(src, "w").write(f'#include <stdio.h>\n#include <stddef.h>\n#include "b200ppf.h"\nint main(void){{{body}return 0;}}\n')
        subprocess.run(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), src, "-o", os.path.join(d, "layout")], check=True)
        out = subprocess.run([os.path.join(d, "layout")], capture_output=True, text=True, check=True).stdout
    for line in out.strip().splitlines():
        name, size, off = line.split()
        cls, last = structs[name]
        assert C.sizeof(cls) == int(size) and getattr(cls, last).offset == int(off), line


def test_no_cpu_fallback_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from yolo_ppf_pose_estimation_b200 import capi
    with pytest.raises(capi.B200PPFError) as e:
        capi.Context(0)
    assert "no CPU fallback" in str(e.value)
    # the product never imports, links or loads anything under oracle/
    import yolo_ppf_pose_estimation_b200 as pkg
    bad = re.compile(r"(from\s+oracle|import\s+oracle|ppf_oracle|oracle/|oracle_)")
    for root, _, files in os.walk(os.path.dirname(pkg.__file__)):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(root, f)).read()
                assert not bad.search(src), f"{f} reaches into the oracle"


def test_hot_loop_alpha_bin_equals_literal_form_and_oracle(oracle):
    """alpha_bin_fast (guarded fp32 estimate) == alpha_bin_exact (PCL's double formula) == oracle,
    on random inputs and on inputs placed within a few ulps of every bin edge / wrap point."""
    from yolo_ppf_pose_estimation_b200 import capi
    rng = np.random.default_rng(1)
    L = oracle.lib()
    for step in (ANGLE_STEP, np.float32(0.25), np.float32(np.pi / 180), np.float32(0.5), np.float32(6 / 180 * np.pi)):
        nal = oracle.num_alpha_bins(step)
        n = 200_000
        am = rng.uniform(-np.pi, np.pi, n).astype(np.float32)
        as_ = rng.uniform(-np.pi, np.pi, n).astype(np.float32)
        k = rng.integers(-2 * nal - 2, 2 * nal + 2, n // 2)
        edge = np.concatenate([k * np.float64(step) - np.pi, rng.choice([-np.pi, np.pi, -2 * np.pi, 2 * np.pi, 0.0], n // 2)])
        as2 = rng.uniform(-np.pi, np.pi, n).astype(np.float32)
        am2 = (edge + as2.astype(np.float64)).astype(np.float32)
        am2 = (am2.view(np.int32) + rng.integers(-4, 5, n).astype(np.int32)).view(np.float32)
        AM, AS = np.concatenate([am, am2, [np.nan, 0.0]]).astype(np.float32), np.concatenate([as_, as2, [0.0, np.nan]]).astype(np.float32)
        for mode, rule in ((0, 0), (0, 1), (0, 2), (1, 0), (1, 2)):
            nal = oracle.num_alpha_bins(step, rule)
            fast, exact = capi.debug_alpha_bins(AM, AS, step, mode, nalpha_rule=rule)
            assert np.array_equal(fast, exact)
            sel = rng.choice(len(AM), 3000, replace=False)
            ref = np.array([L.oracle_alpha_bin(mode, rule, step, AM[i], AS[i]) for i in sel], np.uint32)
            ref[ref == oracle.BIN_DROPPED] = nal  # the device files a dropped vote in the row's spare cell
            assert np.array_equal(exact[sel], ref)
            assert exact[-1] == exact[-2] == 0xFFFFFFFF
            assert exact[:-2].max() <= (nal if rule == 1 else nal - 1)


def test_constant_shift_binning_over_many_angle_steps():
    """The kernel's vote arithmetic (phase cells, hot words, wrap through the unsigned max — alpha_bin_phase, the
    host build of the device functions) equals PCL's literal double-precision form for steps whose 2*pi/step is an
    integer (8 ... 720 positions: the constant-shift path) and for arbitrary steps (per-entry path), on random
    angles and on differences placed within a few ulps of every bin edge."""
    from yolo_ppf_pose_estimation_b200 import capi
    rng = np.random.default_rng(7)
    steps = [np.float32(2 * np.pi / k) for k in (8, 12, 30, 36, 60, 90, 180, 360, 720)]
    steps += [np.float32(x) for x in rng.uniform(0.02, 0.9, 6)]
    for step in steps:
        n = 60_000
        am = rng.uniform(-np.pi, np.pi, n).astype(np.float32)
        as_ = rng.uniform(-np.pi, np.pi, n).astype(np.float32)
        T = 2 * np.pi / float(step)
        k = rng.integers(0, int(T) + 1, n)
        as2 = rng.uniform(-np.pi, np.pi, n).astype(np.float32)
        am2 = ((k * np.float64(step) - np.pi + as2.astype(np.float64) + np.pi) % (2 * np.pi) - np.pi).astype(np.float32)
        am2 = (am2.view(np.int32) + rng.integers(-3, 4, n).astype(np.int32)).view(np.float32)
        ok = np.abs(am2) <= np.float32(3.14159274)
        for rule in (0, 1, 2):
            fast, exact = capi.debug_alpha_bins(np.concatenate([am, am2[ok]]), np.concatenate([as_, as2[ok]]), step, 0, nalpha_rule=rule)
            assert np.array_equal(fast, exact), (float(step), rule)


def test_constant_shift_binning_at_phase_cell_edges():
    """Entries whose alpha_m sits within a few ulps of a phase-cell edge are filed by an fp32 estimate that may name the
    neighbouring cell; their sub-phase byte then saturates at that cell's first / last value.  Scene phases just outside
    the guard band of the same edge, deeper inside the two cells, and in the entry's own sub-phase must all bin like PCL's
    literal form (the first version of the sub-phase byte moved one vote in a million by one bin here; and the guard band
    has to be circular: an entry at the very start of a bin and a scene phase at the very end of one are neighbours)."""
    from yolo_ppf_pose_estimation_b200 import capi
    rng = np.random.default_rng(23)
    for k in (12, 30, 36, 90, 360):
        step = np.float32(2 * np.pi / k)
        st = float(step)
        n = 120_000
        B = rng.integers(0, k, n)
        c = rng.integers(0, 17, n)  # 16 cells per bin: edges 0 ... 16
        am = (-np.pi + st * (B + c / 16.0)).astype(np.float32)
        am = (am.view(np.int32) + rng.integers(-6, 7, n).astype(np.int32)).view(np.float32)
        q = rng.integers(0, k, n)
        side = rng.choice([-1.0, 1.0], n)
        eps = np.concatenate([np.full(n // 4, 4.3e-6), np.full(n // 4, 1.2e-5), rng.uniform(0, 5e-6, n // 4),
                              rng.uniform(0, st / 16, n - 3 * (n // 4))])
        rng.shuffle(eps)
        a_s = st * (q + c / 16.0) + side * eps
        a_s = ((a_s + np.pi) % (2 * np.pi) - np.pi).astype(np.float32)
        ok = (np.abs(am) <= np.float32(3.14159274)) & (np.abs(a_s) <= np.float32(3.14159274))
        # and scene phases in the entry's own sub-phase: a few 2^-12 bins around the entry's position
        a_s2 = (st * (q + (B - B) + ((am.astype(np.float64) + np.pi) / st) % 1.0) + rng.uniform(-1, 1, n) * st * 2.0 ** -12)
        a_s2 = ((a_s2 + np.pi) % (2 * np.pi) - np.pi).astype(np.float32)
        AM = np.concatenate([am[ok], am[ok]])
        AS = np.concatenate([a_s[ok], a_s2[ok]])
        for rule in (0, 1, 2):
            fast, exact = capi.debug_alpha_bins(AM, AS, step, 0, nalpha_rule=rule)
            assert np.array_equal(fast, exact), (k, rule, int((fast != exact).sum()))


def test_synthetic_clouds():
    from yolo_ppf_pose_estimation_b200 import synth
    m = synth.synth_model(5000, 1)
    assert m.shape == (5000, 6) and m.dtype == np.float32
    assert np.array_equal(m, synth.synth_model(5000, 1)) and not np.array_equal(m, synth.synth_model(5000, 2))
    assert np.abs(np.linalg.norm(m[:, 3:], axis=1) - 1).max() < 1e-5
    assert m[:, 2].min() >= 0 and m[:, 2].max() <= 0.18 + 1e-6
    r = np.hypot(m[:, 0], m[:, 1])
    assert r.max() <= 0.05 + 1e-6
    # outward normals on the cylinder wall
    wall = (m[:, 2] > 0.01) & (m[:, 2] < 0.10)
    assert (np.einsum("ij,ij->i", m[wall, :2], m[wall, 3:5]) > 0).all()
    d = np.linalg.norm(m[:200, None, :3] - m[None, :200, :3], axis=-1).max()
    assert 0.15 < d < 0.2
    s = synth.synth_scene(20000, 2, model_seed=1)
    assert s.shape == (20000, 6) and np.array_equal(s, synth.synth_scene(20000, 2, model_seed=1))
    assert np.abs(np.linalg.norm(s[:, 3:], axis=1) - 1).max() < 1e-5
    assert (np.einsum("ij,ij->i", s[:, 3:], -s[:, :3]) >= 0).all()  # normals face the camera
    T = synth.gt_pose(2)
    assert np.allclose(T[:3, :3] @ T[:3, :3].T, np.eye(3), atol=1e-12) and np.allclose(T[:3, 3], [0.1, -0.05, 0.9])
    # the model instance is really there: ~10 % of the points lie on the posed surface
    p = (s[:, :3].astype(np.float64) - T[:3, 3]) @ T[:3, :3]
    on = (np.abs(np.hypot(p[:, 0], p[:, 1]) - 0.05) < 0.003) & (p[:, 2] > 0.0) & (p[:, 2] < 0.11)
    assert on.sum() > 0.02 * len(s)
    assert np.allclose(synth.uniform(7, 3, 4), synth.uniform(7, 3, 4)) and (synth.uniform(7, 3, 1000) < 1).all()


def test_workloads_and_shards():
    from yolo_ppf_pose_estimation_b200 import sharding, workloads
    c1, c2 = workloads.load("c1"), workloads.load("c2")
    assert c1.model.shape == (543, 6) and c1.scene.shape == (934, 6) and c1.n_ref == 187
    assert c2.scene.shape == (44893, 6) and c2.n_ref == 44893
    assert np.float32(c2.angle_step) == ANGLE_STEP
    for n_ref in (0, 1, 7, 187, 44893):
        for world in (1, 2, 3, 4, 8):
            seen = []
            for r in range(world):
                first, step, count = sharding.shard(n_ref, r, world)
                assert count <= sharding.chunk_size(n_ref, world)
                seen += [first + k * step for k in range(count)]
            assert sorted(seen) == list(range(n_ref))


_GLOO_WORKER = r"""
import os, sys, numpy as np, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from yolo_ppf_pose_estimation_b200 import sharding, workloads
from oracle import binding as ob
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo")
wl = workloads.load("c1")
feats = ob.ppf_estimation(wl.model)
hm = ob.HashMap(wl.angle_step, wl.dist_step).set_input_feature_cloud(feats)
n_ref = wl.n_ref
first, step, count = sharding.shard(n_ref, rank, world)
chunk = sharding.chunk_size(n_ref, world)
mine, _ = hm.vote(wl.model, wl.scene, first * wl.ref_rate, step * wl.ref_rate, count)   # this rank's shard
local = torch.zeros((chunk, 16), dtype=torch.float32)
local[:count] = torch.from_numpy(mine.view(np.float32).reshape(count, 16))
full = sharding.all_gather_hypotheses(local, n_ref, world, dist)[:n_ref].numpy().view(ob.HYP_DTYPE).reshape(-1)
ref, _ = hm.vote(wl.model, wl.scene, 0, wl.ref_rate, n_ref)                               # single-rank answer
assert full.tobytes() == ref.tobytes(), "gathered hypotheses differ from the single-rank run"
poses, votes, assign, ncl = ob.cluster(full, wl.pos_thr, wl.rot_thr)
rposes, rvotes, rassign, rncl = ob.cluster(ref, wl.pos_thr, wl.rot_thr)
assert np.array_equal(poses, rposes) and np.array_equal(votes, rvotes) and ncl == rncl
# every rank holds the same clustering result
t = torch.from_numpy(poses.reshape(-1).copy())
g = [torch.zeros_like(t) for _ in range(world)]
dist.all_gather(g, t)
assert all(torch.equal(g[0], x) for x in g)
dist.destroy_process_group()
print("GLOO_OK", rank)
"""


def test_two_rank_gloo_sharding(tmp_path):
    """N > 1 host path on CPU: interleaved shards + all-gather + reorder == single-rank hypotheses
    (the oracle stands in for the device vote; the plumbing is the code bench.py runs over NCCL)."""
    script = tmp_path / "worker.py"
    script.write_text(_GLOO_WORKER)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29617", OMP_NUM_THREADS="2")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29617", str(script), ROOT],
                       env=env, capture_output=True, text=True, timeout=600)
    assert r.stdout.count("GLOO_OK") == 2, r.stdout[-2000:] + r.stderr[-4000:]


def test_cpp_shim_compiles_and_links(tmp_path):
    """The PCL-shaped header shim (PPF operators, pre-processing operators) and the OpenCV-shaped ICP shim are valid
    C++14 and link against libb200ppf.so."""
    from yolo_ppf_pose_estimation_b200 import build
    lib = build.build()
    import torch
    for name, arg in (("pcl_shim_example", os.path.join(ROOT, "tests", "golden")), ("pcl_prep_example", "/nonexistent.f32"),
                      ("cv_icp_shim_example", "/nonexistent")):
        exe = tmp_path / name
        cmd = ["/usr/bin/g++", "-std=c++14", "-O1", "-Wall", "-Wextra", "-Werror",
               "-I", os.path.join(ROOT, "include", "pcl_compat"), "-I", os.path.join(ROOT, "include", "opencv_compat"),
               "-I", os.path.join(ROOT, "include"),
               os.path.join(ROOT, "tests", "cpp", name + ".cpp"), "-o", str(exe),
               "-L", os.path.dirname(lib), "-lb200ppf", f"-Wl,-rpath,{os.path.dirname(lib)}"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        # without a GPU the shim reports PCL-style errors and produces nothing (no crash, no fallback)
        if not torch.cuda.is_available():
            r = subprocess.run([str(exe), arg], capture_output=True, text=True, timeout=120)
            assert r.returncode == 3, (r.returncode, r.stdout, r.stderr)
            assert "no CPU fallback" in r.stderr


def test_opencv_icp_shim_marshalling_against_the_cpu_checker(tmp_path, oracle):
    """include/opencv_compat's ICP / Pose3D: the reference's call (include/CloudProcessing.h:518-523) built against a
    test double of the five C-ABI entry points it uses, backed by the CPU restatement of opencv_contrib's ICP — what the
    example writes equals oracle.icp_refine on the same clouds and poses (the GPU run of the same example is
    tests/test_gpu_zz_opencv_icp_shim.py)"""
    from yolo_ppf_pose_estimation_b200 import synth
    odir = os.path.join(ROOT, "oracle", "_build")
    model = synth.synth_model(3000, 1).astype(np.float32)
    G = synth.gt_pose(2)
    scene = np.concatenate([model[:, :3] @ G[:3, :3].T + G[:3, 3], model[:, 3:] @ G[:3, :3].T], axis=1).astype(np.float32)[::2]
    starts = []
    for k in range(3):
        D = np.eye(4)
        D[:3, 3] = (0.004 * (k + 1), -0.003, 0.002 * k)
        starts.append(D @ G)
    starts = np.ascontiguousarray(starts, np.float64)
    model.tofile(tmp_path / "model.f32")
    scene.tofile(tmp_path / "scene.f32")
    starts.tofile(tmp_path / "poses.f64")
    exe = tmp_path / "cv_icp_shim_mock"
    cmd = ["/usr/bin/g++", "-std=c++14", "-O1", "-I", os.path.join(ROOT, "include", "opencv_compat"), "-I",
           os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "cpp", "cv_icp_shim_example.cpp"),
           os.path.join(ROOT, "tests", "cpp", "mock_b200ppf_icp.cpp"), "-o", str(exe), "-L", odir, "-lppf_oracle",
           f"-Wl,-rpath,{odir}"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe), str(tmp_path)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    out = np.fromfile(tmp_path / "refined.f64", np.float64).reshape(-1, 17)
    P, res, _ = oracle.icp_refine(model, scene, starts)
    assert out.shape[0] == 3
    assert np.array_equal(out[:, :16].reshape(-1, 4, 4), P) and np.array_equal(out[:, 16], res)
    assert np.linalg.norm(P[0][:3, 3] - G[:3, 3]) < 1e-3 and "Pose to Model Index" in r.stdout


def test_header_is_plain_c(tmp_path):
    """include/b200ppf.h is the drop-in boundary: plain C types only — the INTEGRATION.md frame example compiles as
    strict C99 and the header as C++11"""
    inc = os.path.join(ROOT, "include")
    r = subprocess.run(["/usr/bin/gcc", "-std=c99", "-pedantic", "-Wall", "-Wextra", "-Werror", "-I", inc, "-c",
                        os.path.join(ROOT, "tests", "cpp", "c_abi_frame_example.c"), "-o", str(tmp_path / "a.o")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    src = tmp_path / "hdr.cpp"
    src.write_text('#include "b200ppf.h"\nint (*probe)(void) = &b200ppf_version;\n')
    r = subprocess.run(["/usr/bin/g++", "-std=c++11", "-Wall", "-Wextra", "-Werror", "-I", inc, "-c", str(src), "-o",
                        str(tmp_path / "b.o")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def test_bench_reference_arm_prints_the_contract_line(tmp_path, oracle):
    """The reference arm prints the JSON line, and --dump-outputs writes the clustering of its last step: the oracle's
    on that step's reference points."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "c1",
                        "--steps", "1", "--warmup", "0", "--cpu-sample", "8", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "pairs/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and "workload" in line["config"]
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    from yolo_ppf_pose_estimation_b200 import workloads
    wl = workloads.load("c1")
    refs = bench.sample_list(wl)[:8]  # the one step's reference points, in the order it votes on them
    assert sorted(refs) == line["sample_refs"]
    hm = oracle.HashMap(wl.angle_step, wl.dist_step).set_input_feature_cloud(oracle.ppf_estimation(wl.model))
    hyps, _ = hm.vote_refs(wl.model, wl.scene, refs, n_threads=oracle.host_threads())
    poses, votes, _, _ = oracle.cluster(hyps, wl.pos_thr, wl.rot_thr)
    dumped_poses, dumped_votes = np.load(tmp_path / "poses.npy"), np.load(tmp_path / "votes.npy")
    assert dumped_poses.dtype == np.float32 and dumped_votes.dtype == np.float64 and len(votes) > 0
    assert np.array_equal(dumped_poses, poses) and np.array_equal(dumped_votes, votes)


def test_bench_arms_print_the_same_config_and_a_fixed_cpu_sample():
    """The reference arm and the B200 arm describe the workload identically (the driver compares `config`), the CPU sample is
    a fixed list — same reference points on every box, every --gpus — and the thread count ignores OMP_NUM_THREADS."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    from yolo_ppf_pose_estimation_b200 import workloads
    wl = workloads.load("c3s")
    a, b = bench.workload_config(wl, 1), bench.workload_config(wl, 1)
    assert a == b and set(a) >= {"workload", "n_model", "n_scene", "n_ref", "l2"}
    s1, s2 = bench.sample_list(wl), bench.sample_list(wl)
    assert s1 == s2 and len(s1) == len(set(s1)) == 64 and max(s1) < wl.scene.shape[0]
    assert sorted(s1[:8]) == sorted(s1[:8]) and max(np.diff(sorted(s1[:8]))) < wl.scene.shape[0] // 4   # a prefix is spread out
    os.environ["OMP_NUM_THREADS"] = "1"
    try:
        assert bench.host_threads() == len(os.sched_getaffinity(0))
    finally:
        del os.environ["OMP_NUM_THREADS"]
    assert 1 <= bench.refs_per_cpu_step(workloads.load("c1"), 8, 0) <= 64 and bench.refs_per_cpu_step(wl, 8, 5) == 5
