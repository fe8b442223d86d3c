#!/usr/bin/env python
"""Every box of a frame in one call (b200cv_match_frame: one crop pass, the per-object pre-processing and matching, one ICP
launch for the top 5 poses of every object) against one b200cv_match_object call per box, the frame resident in HBM.

Inputs:
  synthetic 1Mi frame  synth.synth_library_scene (1 Mi points, 8 instances), K = 1, 2, 4, 8 boxes: box k is the
                       projection of instance k built as tools/prep_bench.py:frame_case builds it for k = 0, with library
                       model k (2 000 points) and its own PPF3DDetector(0.025, 0.05); leaf 0.005
  reference frame      the regenerated 1 cm scene and surrogate YOLO box (tests/golden), the box repeated K times, one
                       bottle detector for all; leaf 0.01
Both arms run match_S2B(object, edges, 0.05, 0.05) and ICP(100, 0.005, 2.5, 8) of the top 5 poses.  Per K: --repeat frame
calls and --repeat serial rounds of K calls, alternated, after one warm-up of each; medians of the wall time and of the
per-stage device times (summed over the boxes for the serial arm and for the frame call's per-box stages; the frame call's
crop and ICP are one each).  Kernel launches per call and the ICP launches among them (launches with icp_poses = 5 minus
launches with icp_poses = 0) are counted with b200ppf_launch_count.  Every frame result must equal its serial call's bits.
The card's name, power limit and maximum SM clock (nvidia-smi, read-only) go into every line.

--verify: what pose verification adds.  For K = 1 and 8 boxes on both frames, --repeat b200cv_match_frame and
b200cv_match_frame_verified calls (default parameters: 1 cm, 30 degrees), alternated after one warm-up of each, medians of
the wall time; and b200ppf_score_poses alone on the verified call's candidates of the same boxes (each box's object cloud
from b200cv_match_object), --repeat calls timed with CUDA events on the context's stream.  The verified results must hold
the plain call's fields and the fits of score_poses.

usage: python tools/cv_frame_bench.py [--repeat 20] [--verify] [--out profiles/r4_cv_frame.jsonl | profiles/r5_verify.jsonl]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SAMPLING_STEP, DISTANCE_STEP = 0.025, 0.05
STAGES = ("voxel_ms", "outlier_ms", "normals_ms", "edges_ms", "match_ms")


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True)
    name, power, clock = (v.strip() for v in r.stdout.strip().splitlines()[0].split(","))
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def library_box(model, k):
    """tools/prep_bench.py:frame_case's box for instance k"""
    from yolo_ppf_pose_estimation_b200 import synth
    T = synth.library_pose(k)
    p = model[:, :3].astype(np.float64) @ T[:3, :3].T + T[:3, 3]
    zf = np.float32(p[:, 2].max() + 0.15)
    tx, ty = p[:, 0] / p[:, 2], p[:, 1] / p[:, 2]
    xl, xr, yt, yb = (np.float32(v * zf) for v in (tx.min() - 0.03, tx.max() + 0.03, ty.min() - 0.03, ty.max() + 0.03))
    return np.array([[xl, yt, zf], [xl, yb, zf], [xr, yt, zf], [xr, yb, zf]], np.float32)


def frames(c):
    """-> [(name, scene Cloud, [(corners, detector, model Cloud) per available box], leaf, K values)]"""
    from yolo_ppf_pose_estimation_b200 import capi, synth
    gold = os.path.join(ROOT, "tests", "golden")
    xyz = np.ascontiguousarray(synth.synth_library_scene(1 << 20)[:, :3], np.float32)
    boxes = []
    for k in range(8):
        m = synth.synth_model(2000, 10 + k, k).astype(np.float32)
        boxes.append((library_box(m, k), capi.CvDetector(c, SAMPLING_STEP, DISTANCE_STEP).train_model(m), c.upload_cloud(m)))
    out = [("synthetic 1Mi frame", c.upload_xyz(xyz), boxes, 0.005)]
    b = np.load(os.path.join(gold, "crop_box.npz"))
    depth = np.zeros(tuple(b["image"]), np.float32)
    for (r, col), d in zip(b["pixels"], b["depths"]):
        depth[r, col] = d
    bottle = np.load(os.path.join(gold, "bottle_1cm.npz"))["cloud"].astype(np.float32)
    one = (capi.frustum_corners(depth, b["box"], b["intrinsics"]), capi.CvDetector(c, SAMPLING_STEP, DISTANCE_STEP).train_model(bottle),
           c.upload_cloud(bottle))
    scene = np.load(os.path.join(gold, "scene_full_1cm.npz"))["cloud"][:, :3]
    out.append(("reference frame", c.upload_xyz(np.ascontiguousarray(scene, np.float32)), [one] * 8, 0.01))
    return out


def bench(c, name, scene, boxes, leaf, K, repeat, gpu):
    cors = np.stack([b[0] for b in boxes[:K]])
    dets, mods = [b[1] for b in boxes[:K]], [b[2] for b in boxes[:K]]

    def frame(**over):
        t0 = time.perf_counter()
        res, status = c.cv_match_frame(scene, cors, dets, mods, leaf=leaf, **over)
        wall = 1e3 * (time.perf_counter() - t0)
        assert status.tolist() == [0] * K, status
        return res, wall

    def serial(**over):
        t0 = time.perf_counter()
        res = [c.cv_match_object(dets[k], scene, cors[k], mods[k], leaf=leaf, **over)[0] for k in range(K)]
        return res, 1e3 * (time.perf_counter() - t0)

    def launches(fn, **over):
        n0 = c.launch_count
        fn(**over)
        return c.launch_count - n0

    fr, se = [], []
    frame(), serial()  # warm-up
    for _ in range(repeat):
        fr.append(frame())
        se.append(serial())
    identical = all(a["pose"].tobytes() == b["pose"].tobytes() and a["residual"] == b["residual"] and a["votes"] == b["votes"]
                    for (rf, _), (rs, _) in zip(fr, se) for a, b in zip(rf, rs))
    n_frame, n_serial = launches(frame), launches(serial)
    icp_frame, icp_serial = n_frame - launches(frame, icp_poses=0), n_serial - launches(serial, icp_poses=0)
    med = lambda v: float(np.median(v))  # noqa: E731
    f_stages = {"crop_ms": med([r[0]["crop_ms"] for r, _ in fr]), "icp_ms": med([r[0]["icp_ms"] for r, _ in fr])}
    f_stages.update({s: med([sum(x[s] for x in r) for r, _ in fr]) for s in STAGES})
    s_stages = {s: med([sum(x[s] for x in r) for r, _ in se]) for s in ("crop_ms", "icp_ms") + STAGES}
    f_wall, s_wall = med([w for _, w in fr]), med([w for _, w in se])
    r0 = fr[-1][0]
    return {"frame": name, "boxes": K, "calls": repeat, "leaf": leaf, "detector": [SAMPLING_STEP, DISTANCE_STEP],
            "n_cropped": [int(x["n_cropped"]) for x in r0], "n_filtered": [int(x["n_filtered"]) for x in r0],
            "n_edges": [int(x["n_edges"]) for x in r0],
            "frame_call": {"wall_ms_median": f_wall, "device_ms_median": f_stages, "launches": n_frame, "icp_launches": icp_frame},
            "serial_calls": {"wall_ms_median": s_wall, "device_ms_median_summed": s_stages, "launches": n_serial,
                             "icp_launches": icp_serial},
            "speedup_wall": s_wall / f_wall, "frame_wall_ms_per_object": f_wall / K, "identical_to_serial": identical, "gpu": gpu}


def bench_verify(c, name, scene, boxes, leaf, K, repeat, gpu):
    import torch
    cors = np.stack([b[0] for b in boxes[:K]])
    dets, mods = [b[1] for b in boxes[:K]], [b[2] for b in boxes[:K]]

    def timed(fn):
        t0 = time.perf_counter()
        out = fn(scene, cors, dets, mods, leaf=leaf)
        return out, 1e3 * (time.perf_counter() - t0)

    timed(c.cv_match_frame), timed(c.cv_match_frame_verified)  # warm-up
    plain, verified = [], []
    for _ in range(repeat):
        plain.append(timed(c.cv_match_frame))
        verified.append(timed(c.cv_match_frame_verified))
    (res, status), _ = plain[-1]
    (vres, vstatus, cands), _ = verified[-1]
    assert status.tolist() == vstatus.tolist() == [0] * K, (status, vstatus)
    same = all(a[f] == b[f] for a, b in zip(res, vres) for f in ("n_poses", "n_cropped", "n_sampled", "n_filtered", "n_edges"))
    # score_poses alone on the same candidates, against the same object clouds
    objects = [c.cv_match_object(dets[k], scene, cors[k], mods[k], leaf=leaf)[1] for k in range(K)]
    jobs = [(mods[k], objects[k], np.stack([x["pose"] for x in cands[k]])) for k in range(K)]
    fits = c.score_poses(jobs)
    fits_match = all(f["fit"] == x["fit"]["fit"] and f["inliers"] == x["fit"]["inliers"] for k in range(K)
                     for f, x in zip(fits[k], cands[k]))
    stream = torch.cuda.ExternalStream(c.stream)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(repeat)]
    n0 = c.launch_count
    c.score_poses(jobs)
    launches = c.launch_count - n0
    for e0, e1 in ev:
        e0.record(stream)
        c.score_poses(jobs)
        e1.record(stream)
    torch.cuda.synchronize()
    score_ms = [e0.elapsed_time(e1) for e0, e1 in ev]
    med = lambda v: float(np.median(v))  # noqa: E731
    p_wall, v_wall = med([w for _, w in plain]), med([w for _, w in verified])
    return {"frame": name, "boxes": K, "calls": repeat, "leaf": leaf, "verify": {"inlier_dist": 0.01, "normal_angle_deg": 30.0},
            "candidates": int(sum(len(x) for x in cands)), "model_points": [int(m.size) for m in mods],
            "object_points": [int(o.size) for o in objects],
            "plain_wall_ms_median": p_wall, "verified_wall_ms_median": v_wall, "added_wall_ms": v_wall - p_wall,
            "score_poses_device_ms_median": med(score_ms), "score_poses_launches": launches,
            "best_rank": [int(x[0]["rank"]) for x in cands], "best_fit": [float(x[0]["fit"]["fit"]) for x in cands],
            "fields_equal_plain": same, "fits_equal_score_poses": fits_match, "gpu": gpu}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeat", type=int, default=20, help="timed frame calls and serial rounds per K (after one warm-up each)")
    ap.add_argument("--verify", action="store_true", help="time the verified frame call and b200ppf_score_poses instead")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.out is None:
        args.out = os.path.join(ROOT, "profiles", "r5_verify.jsonl" if args.verify else "r4_cv_frame.jsonl")
    if args.repeat < 1:
        ap.error("--repeat must be at least 1")
    from yolo_ppf_pose_estimation_b200 import capi
    c = capi.Context(0)
    gpu = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for name, scene, boxes, leaf in frames(c):
            for K in ((1, 8) if args.verify else (1, 2, 4, 8)):
                line = json.dumps((bench_verify if args.verify else bench)(c, name, scene, boxes, leaf, K, args.repeat, gpu))
                print(line, flush=True)
                f.write(line + "\n")


if __name__ == "__main__":
    main()
