#!/usr/bin/env python
"""One detected object start to finish with the engine the reference calls (b200cv_match_object): SceneCropping ->
Subsampling -> OutlierProcessing(50, 1.0) -> NormalEstimation(30) -> EdgeExtraction(0.03) -> re-normalise ->
PPF3DDetector::match_S2B(object, edges, 0.05, 0.05) -> ICP(100, 0.005, 2.5, 8) of the top 5 poses
(src/YOLO_cropping_ppf_test.cpp:91-122), the scene resident in HBM as it is for every box of a frame; vs the same chain
on the CPU (the oracle's restatements of the PCL operators and of PPF3DDetector / ICP) on all host threads.

Two inputs, those of tools/prep_bench.py's per-object lines: the reference frame (regenerated 1 cm scene, surrogate YOLO
box, bottle 1 cm) and the synthetic 1 Mi-point frame (library model 0); detector PPF3DDetector(0.025, 0.05) for both.
B200 arm: median of --repeat calls after one warm-up call, per-stage device times (CUDA events).  The card's name, power
limit and maximum SM clock are read (nvidia-smi, read-only) in the same run and written into every line.
Prints one JSON line per input (and appends it to --out when given).

usage: python tools/cv_object_bench.py [--repeat 20] [--no-cpu] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

SAMPLING_STEP, DISTANCE_STEP = 0.025, 0.05   # PPF3DDetector(relativeSamplingStep, relativeDistanceStep)
SCENE_STEP, SCENE_DISTANCE = 0.05, 0.05      # match_S2B(object, edges, results, 0.05, 0.05)
ICP_POSES = 5


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True)
    name, power, clock = (v.strip() for v in r.stdout.strip().splitlines()[0].split(","))
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def cpu_chain(scene, cor, model, leaf):
    """the same chain on the host: -> (stage times ms, pre-ICP clusters (poses, votes), refined best pose, residual)"""
    from oracle import binding as ob
    nt = ob.max_threads()
    ref = ob.CvDetector(SAMPLING_STEP, DISTANCE_STEP).train_model(model)  # training is offline, as on the device
    t = {}
    t0 = time.perf_counter()
    v = scene[ob.crop_pyramid(scene, cor)]
    t["crop"] = 1e3 * (time.perf_counter() - t0)
    t0 = time.perf_counter()
    v = ob.voxel_grid(v, leaf)[0]
    t["voxel"] = 1e3 * (time.perf_counter() - t0)
    t0 = time.perf_counter()
    v = v[ob.statistical_outlier_removal(v, 50, 1.0, n_threads=nt)[0]]
    t["outlier"] = 1e3 * (time.perf_counter() - t0)
    t0 = time.perf_counter()
    n = ob.normals(v, 30, n_threads=nt)
    t["normals"] = 1e3 * (time.perf_counter() - t0)
    t0 = time.perf_counter()
    obj = np.concatenate([v, ob.renormalize_normals(n[:, :3])], axis=1)
    edges = obj[n[:, 3] > np.float32(0.03)]
    t["edges"] = 1e3 * (time.perf_counter() - t0)
    t0 = time.perf_counter()
    poses, votes, _, _ = ref.match_s2b(obj, edges, SCENE_STEP, SCENE_DISTANCE, n_threads=nt)
    t["match"] = 1e3 * (time.perf_counter() - t0)
    t0 = time.perf_counter()
    R, res, _ = ob.icp_refine(model, obj, poses[:ICP_POSES])
    t["icp"] = 1e3 * (time.perf_counter() - t0)
    t["total"] = float(sum(t.values()))
    return t, nt, poses, votes, R[0], float(res[0]), {"n_filtered": int(obj.shape[0]), "n_edges": int(edges.shape[0])}


def frame_bench(c, name, repeat, with_cpu, gpu):
    from yolo_ppf_pose_estimation_b200 import capi
    from prep_bench import frame_case
    scene, cor, model, over = frame_case(name)
    leaf = over["leaf"]
    det = capi.CvDetector(c, SAMPLING_STEP, DISTANCE_STEP).train_model(model)
    dm = c.upload_cloud(model)
    t0 = time.perf_counter()
    ds = c.upload_xyz(scene)
    upload_ms = 1e3 * (time.perf_counter() - t0)
    runs = []
    for _ in range(repeat + 1):
        r, obj, edges = c.cv_match_object(det, ds, cor, dm, leaf=leaf)
        runs.append(r)
    runs = runs[1:]
    med = {k: float(np.median([x[k] for x in runs])) for k in runs[0] if k.endswith("_ms")}
    r = runs[-1]
    assert all(np.array_equal(x["pose"], r["pose"]) for x in runs), "the chain is deterministic"
    clusters, _ = det.match_cloud(obj, edges, SCENE_STEP, SCENE_DISTANCE)  # the poses before ICP
    rec = {"frame": name, "engine": "cv::ppf_match_3d::PPF3DDetector::match_S2B (b200cv_match_object)",
           "scene_points": int(scene.shape[0]), "model_points": int(model.shape[0]),
           "params": {"leaf": leaf, "detector": [SAMPLING_STEP, DISTANCE_STEP], "scene_steps": [SCENE_STEP, SCENE_DISTANCE],
                      "icp_poses": ICP_POSES, "icp": [100, 0.005, 2.5, 8]},
           "sizes": {k: int(r[k]) for k in ("n_cropped", "n_sampled", "n_filtered", "n_edges", "n_poses")},
           "detector": {"model_sampled": int(det.info.n_sampled), "scene_sampled": int(det.info.n_scene_sampled),
                        "edges_sampled": int(det.info.n_second_sampled)},
           "votes": int(r["votes"]), "residual": float(r["residual"]), "calls": repeat, "scene_upload_ms": upload_ms,
           "b200_ms_median": med, "gpu": gpu}
    if with_cpu:
        t, nt, poses, votes, R, cres, csizes = cpu_chain(scene, cor, model, leaf)
        rec["cpu_ms"] = t
        rec["cpu_threads"] = nt
        rec["cpu_note"] = ("CPU restatement of the PCL / OpenCV operators, all host threads (ICP: one thread per pose, "
                           "sequential); neighbour search by brute force; one call")
        rec["cpu_sizes"] = csizes
        k = min(len(poses), len(clusters))
        rec["cluster_votes_equal_cpu"] = bool(np.array_equal(clusters["num_votes"][:k], votes[:k]))
        rec["pose_max_abs_diff_vs_cpu_chain_before_icp"] = float(np.abs(clusters["pose"][:k].reshape(k, 4, 4) - poses[:k]).max())
        # the reference's ICP reports 1e10 when it loses its correspondences: a comparison of two diverged poses says nothing
        rec["icp_residual"] = {"b200": float(r["residual"]), "cpu": cres}
        if r["residual"] < 1e9 and cres < 1e9:
            rec["translation_diff_vs_cpu_m"] = float(np.linalg.norm(r["pose"][:3, 3] - R[:3, 3]))
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeat", type=int, default=20, help="timed calls per input (after one warm-up call)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--out", default=None, help="append the JSON lines to this file too")
    args = ap.parse_args()
    if args.repeat < 1:
        ap.error("--repeat must be at least 1")
    from yolo_ppf_pose_estimation_b200 import capi
    c = capi.Context(0)
    gpu = card()
    for name in ("reference frame", "synthetic 1Mi frame"):
        line = json.dumps(frame_bench(c, name, args.repeat, not args.no_cpu, gpu))
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(line + "\n")


if __name__ == "__main__":
    main()
