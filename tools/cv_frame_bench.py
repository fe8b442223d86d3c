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

--verify-depth: what verification against the depth image adds, on synth.synth_library_depth (1024 x 1024, the scene cloud
from b200ppf_cloud_from_depth, library boxes and detectors as above, leaf 0.005).  For K = 1, 2, 4, 8 boxes and both match
steps (match_S2B and Matching): --repeat b200cv_match_frame, _verified and _verified_depth calls, alternated after one warm-up
of each, medians of the wall time; b200ppf_score_poses_depth against b200ppf_score_poses on the depth-verified call's
candidates (CUDA events on the context's stream); the instances each call finds within 1 cm / 5 degrees and the best fits.
Once per run: b200ppf_cloud_from_depth on the 1 Mi-pixel image (CUDA events, median of --repeat).

--screen: what screening the pose clusters before ICP adds and recovers.  On the synthetic 1Mi frame b200cv_match_frame_screened
against b200cv_match_frame_verified, and on synth.synth_library_depth the _depth pair, for K = 1 and 8 boxes, both match steps,
icp_poses 5 and 1 and screen_poses = 0 (every cluster): --repeat calls of each, alternated after one warm-up of each, medians
of the wall time; the device time of the screen alone (score_poses / score_poses_depth on every cluster of the boxes, each
box's object cloud from b200cv_match_object and its clusters from CvDetector.match_cloud; CUDA events on the context's
stream); the instances each call finds within 1 cm / 5 degrees (of the model axis, as the tests judge the library's surfaces of
revolution, and of the whole rotation, as --verify-depth reports), the best fits, per box the clusters screened and the ranks
of the kept candidates, and the clusters within 1 cm / 5 degrees (axis) of the truth before ICP (or the nearest one) with
their screen fit and their position in the screen's order; for the depth screen the z-buffer slab it holds (8 bytes a pixel of every screened pose's splat
rectangle, restated on the host from the rule in include/b200ppf.h), the whole call's and the largest box's.

usage: python tools/cv_frame_bench.py [--repeat 20] [--verify | --verify-depth | --screen]
                                      [--out profiles/r4_cv_frame.jsonl | profiles/r5_verify.jsonl | profiles/r7_verify_depth.jsonl |
                                             profiles/r8_screen.jsonl]"""
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


def _event_ms(c, fn, repeat):
    """median device time of fn() on the context's stream (CUDA events), after one warm-up"""
    import torch
    stream = torch.cuda.ExternalStream(c.stream)
    fn()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(repeat)]
    for e0, e1 in ev:
        e0.record(stream)
        fn()
        e1.record(stream)
    torch.cuda.synchronize()
    return float(np.median([e0.elapsed_time(e1) for e0, e1 in ev]))


def _axis_angle_deg(A, B):
    R = A[:3, :3].T @ B[:3, :3]
    return float(np.degrees(np.arccos(np.clip((np.trace(R) - 1) / 2, -1.0, 1.0))))


def _model_axis_deg(A, B):
    """the angle between the models' z axes: the library models are surfaces of revolution about z, so the axis is what a
    pose fixes (tests/test_gpu_frame.py judges the library instances by it)"""
    return float(np.degrees(np.arccos(np.clip(A[:3, 2] @ B[:3, 2], -1.0, 1.0))))


def depth_frame(c):
    from yolo_ppf_pose_estimation_b200 import capi, synth
    f = synth.synth_library_depth()
    dimg = c.upload_depth(f["depth"], f["K"])
    boxes = []
    for k in range(8):
        m = synth.synth_model(2000, 10 + k, k).astype(np.float32)
        boxes.append((library_box(m, k), capi.CvDetector(c, SAMPLING_STEP, DISTANCE_STEP).train_model(m), c.upload_cloud(m)))
    return f, dimg, c.cloud_from_depth(dimg), boxes


def bench_verify_depth(c, dimg, scene, boxes, K, use_edges, repeat, gpu):
    from yolo_ppf_pose_estimation_b200 import synth
    cors = np.stack([b[0] for b in boxes[:K]])
    dets, mods = [b[1] for b in boxes[:K]], [b[2] for b in boxes[:K]]
    over = dict(leaf=0.005, use_edges=use_edges, relative_scene_sample_step=0.05 if use_edges else 1.0 / 14.0)
    calls = {"plain": lambda: c.cv_match_frame(scene, cors, dets, mods, **over),
             "verified": lambda: c.cv_match_frame_verified(scene, cors, dets, mods, **over),
             "depth_verified": lambda: c.cv_match_frame_verified_depth(scene, dimg, cors, dets, mods, **over)}
    wall = {n: [] for n in calls}
    out = {}
    for fn in calls.values():
        fn()  # warm-up
    for _ in range(repeat):
        for n, fn in calls.items():
            t0 = time.perf_counter()
            out[n] = fn()
            wall[n].append(1e3 * (time.perf_counter() - t0))
    for n, o in out.items():
        assert o[1].tolist() == [0] * K, (n, o[1])

    def found(res):
        return [k for k in range(K) if np.linalg.norm(res[k]["pose"][:3, 3] - synth.library_pose(k)[:3, 3]) < 0.01 and
                _axis_angle_deg(res[k]["pose"], synth.library_pose(k)) < 5.0]
    cands = out["depth_verified"][2]
    objects = [c.cv_match_object(dets[k], scene, cors[k], mods[k], **over)[1] for k in range(K)]
    jobs = [(mods[k], objects[k], np.stack([x["pose"] for x in cands[k]])) for k in range(K)]
    dfits = c.score_poses_depth(jobs, dimg)
    fits_match = all(f == x["fit"] for k in range(K) for f, x in zip(dfits[k], cands[k]))
    med = lambda v: float(np.median(v))  # noqa: E731
    return {"frame": "synth_library_depth 1024x1024", "boxes": K, "match": "match_S2B" if use_edges else "Matching", "calls": repeat,
            "leaf": 0.005, "verify": {"inlier_dist": 0.01, "normal_angle_deg": 30.0}, "candidates": int(sum(len(x) for x in cands)),
            "wall_ms_median": {n: med(w) for n, w in wall.items()},
            "score_poses_depth_device_ms_median": _event_ms(c, lambda: c.score_poses_depth(jobs, dimg), repeat),
            "score_poses_device_ms_median": _event_ms(c, lambda: c.score_poses(jobs), repeat),
            "found_1cm_5deg": {n: found(o[0]) for n, o in out.items()},
            "best_fit": {"verified": [round(float(x[0]["fit"]["fit"]), 4) for x in out["verified"][2]],
                         "depth_verified": [round(float(x[0]["fit"]["fit"]), 4) for x in cands]},
            "depth_best": [{k: int(v) if k not in ("fit", "rms") else round(float(v), 4) for k, v in x[0]["fit"].items()} for x in cands],
            "fits_equal_score_poses_depth": fits_match, "gpu": gpu}


def _zbuf_slab_bytes(model_rows, poses, dimg_host, K, tau=0.01):
    """the z-buffer bytes b200ppf_score_poses_depth holds for these poses: 8 bytes a pixel of each pose's clipped splat rectangle"""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from verify_depth_reference import project, splat_half
    total = 0
    m = model_rows[:, :3].astype(np.float64)
    for T in poses:
        p = m @ T[:3, :3].T + T[:3, 3]
        u, v, ok, _, _ = project(p, K, dimg_host.shape)
        if not ok.any():
            continue
        h = splat_half(p[ok, 2], float(K[0]), tau)
        u, v = u[ok], v[ok]
        rows, cols = dimg_host.shape
        w = min(int((u + h).max()), cols - 1) - max(int((u - h).min()), 0) + 1
        hh = min(int((v + h).max()), rows - 1) - max(int((v - h).min()), 0) + 1
        total += 8 * w * hh
    return total


def bench_screen(c, frame, scene, boxes, K, use_edges, icp_poses, repeat, gpu, depth=None):
    """frame: name; depth: None or (device image, host image, K4) for the _depth pair"""
    from yolo_ppf_pose_estimation_b200 import synth
    cors = np.stack([b[0] for b in boxes[:K]])
    dets, mods = [b[1] for b in boxes[:K]], [b[2] for b in boxes[:K]]
    over = dict(leaf=0.005, use_edges=use_edges, icp_poses=icp_poses, relative_scene_sample_step=0.05 if use_edges else 1.0 / 14.0)
    if depth is None:
        calls = {"verified": lambda: c.cv_match_frame_verified(scene, cors, dets, mods, **over),
                 "screened": lambda: c.cv_match_frame_screened(scene, cors, dets, mods, screen_poses=0, **over)}
    else:
        calls = {"verified": lambda: c.cv_match_frame_verified_depth(scene, depth[0], cors, dets, mods, **over),
                 "screened": lambda: c.cv_match_frame_screened_depth(scene, depth[0], cors, dets, mods, screen_poses=0, **over)}
    wall = {n: [] for n in calls}
    out = {}
    for fn in calls.values():
        fn()  # warm-up
    for _ in range(repeat):
        for n, fn in calls.items():
            t0 = time.perf_counter()
            out[n] = fn()
            wall[n].append(1e3 * (time.perf_counter() - t0))
    for n, o in out.items():
        assert o[1].tolist() == [0] * K, (n, o[1])

    def found(res, angle):
        return [k for k in range(K) if np.linalg.norm(res[k]["pose"][:3, 3] - synth.library_pose(k)[:3, 3]) < 0.01 and
                angle(res[k]["pose"], synth.library_pose(k)) < 5.0]
    # the screen alone: every cluster of every box, scored unrefined in one call
    jobs = []
    for k in range(K):
        _, obj, edges = c.cv_match_object(dets[k], scene, cors[k], mods[k], **over)
        top, n = dets[k].match_cloud(obj, edges if use_edges else None, over["relative_scene_sample_step"], 0.05, max_poses=obj.size)
        jobs.append((mods[k], obj, np.stack([t["pose"].reshape(4, 4) for t in top]).astype(np.float64)))
    if depth is None:
        screen_ms = _event_ms(c, lambda: c.score_poses(jobs), repeat)
        slab = None
    else:
        screen_ms = _event_ms(c, lambda: c.score_poses_depth(jobs, depth[0]), repeat)
        per_box = [_zbuf_slab_bytes(m.download(), P, depth[1], depth[2]) for m, _, P in jobs]
        slab = {"call_bytes": int(sum(per_box)), "largest_box_bytes": int(max(per_box))}
    # the clusters within 1 cm / 5 degrees (axis) of the truth before ICP, or the nearest one: rank and screen-fit position
    fits = c.score_poses(jobs) if depth is None else c.score_poses_depth(jobs, depth[0])
    truth = []
    for k, ((_, _, P), f) in enumerate(zip(jobs, fits)):
        T = synth.library_pose(k)
        pos = {r: i for i, r in enumerate(sorted(range(len(f)), key=lambda r: (-f[r]["fit"], r)))}
        dt = [float(np.linalg.norm(Q[:3, 3] - T[:3, 3])) for Q in P]
        near = [r for r in range(len(P)) if dt[r] < 0.01 and _model_axis_deg(P[r], T) < 5.0] or [int(np.argmin(dt))]
        truth.append([{"rank": r, "within": dt[r] < 0.01 and _model_axis_deg(P[r], T) < 5.0, "dt_mm": round(1e3 * dt[r], 1),
                       "axis_deg": round(_model_axis_deg(P[r], T), 1), "screen_fit": round(float(f[r]["fit"]), 4),
                       "screen_position": pos[r]} for r in near])
    med = lambda v: float(np.median(v))  # noqa: E731
    sres, _, scands = out["screened"]
    line = {"frame": frame, "boxes": K, "match": "match_S2B" if use_edges else "Matching", "icp_poses": icp_poses, "screen_poses": 0,
            "calls": repeat, "leaf": 0.005, "verify": {"inlier_dist": 0.01, "normal_angle_deg": 30.0},
            "wall_ms_median": {n: med(w) for n, w in wall.items()},
            "added_wall_ms": med(wall["screened"]) - med(wall["verified"]),
            "screen_device_ms_median": screen_ms, "clusters_screened": [int(x["n_poses"]) for x in sres],
            "kept_ranks": [sorted(int(x["rank"]) for x in cs) for cs in scands],
            "found_1cm_5deg_axis": {n: found(o[0], _model_axis_deg) for n, o in out.items()},
            "found_1cm_5deg_rotation": {n: found(o[0], _axis_angle_deg) for n, o in out.items()},
            "truth_clusters_before_icp": truth,
            "best_fit": {n: [round(float(x[0]["fit"]["fit"]), 4) for x in o[2]] for n, o in out.items()},
            "best_rank": {n: [int(x[0]["rank"]) for x in o[2]] for n, o in out.items()}, "gpu": gpu}
    if slab is not None:
        line["depth_screen_zbuf_slab"] = slab
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeat", type=int, default=20, help="timed frame calls and serial rounds per K (after one warm-up each)")
    ap.add_argument("--verify", action="store_true", help="time the verified frame call and b200ppf_score_poses instead")
    ap.add_argument("--verify-depth", action="store_true", help="time the depth-verified frame call and b200ppf_score_poses_depth")
    ap.add_argument("--screen", action="store_true", help="compare the screened frame calls with the verified ones")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.out is None:
        args.out = os.path.join(ROOT, "profiles", "r8_screen.jsonl" if args.screen else "r7_verify_depth.jsonl" if args.verify_depth else
                                "r5_verify.jsonl" if args.verify else "r4_cv_frame.jsonl")
    if args.repeat < 1:
        ap.error("--repeat must be at least 1")
    from yolo_ppf_pose_estimation_b200 import capi
    c = capi.Context(0)
    gpu = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        if args.screen:
            lib_scene, lib_boxes = frames(c)[0][1:3]
            fr, dimg, dscene, dboxes = depth_frame(c)
            for frame, scene, boxes, depth in (("synthetic 1Mi frame", lib_scene, lib_boxes, None),
                                                ("synth_library_depth 1024x1024", dscene, dboxes, (dimg, fr["depth"], fr["K"]))):
                for use_edges in (1, 0):
                    for icp_poses in (5, 1):
                        for K in (1, 8):
                            line = json.dumps(bench_screen(c, frame, scene, boxes, K, use_edges, icp_poses, args.repeat, gpu, depth))
                            print(line, flush=True)
                            f.write(line + "\n")
            return
        if args.verify_depth:
            fr, dimg, scene, boxes = depth_frame(c)
            line = json.dumps({"frame": "synth_library_depth 1024x1024", "measured_pixels": int(scene.size),
                               "cloud_from_depth_device_ms_median": _event_ms(c, lambda: c.cloud_from_depth(dimg), args.repeat),
                               "calls": args.repeat, "gpu": gpu})
            print(line, flush=True)
            f.write(line + "\n")
            for use_edges in (1, 0):
                for K in (1, 2, 4, 8):
                    line = json.dumps(bench_verify_depth(c, dimg, scene, boxes, K, use_edges, args.repeat, gpu))
                    print(line, flush=True)
                    f.write(line + "\n")
            return
        for name, scene, boxes, leaf in frames(c):
            for K in ((1, 8) if args.verify else (1, 2, 4, 8)):
                line = json.dumps((bench_verify if args.verify else bench)(c, name, scene, boxes, leaf, K, args.repeat, gpu))
                print(line, flush=True)
                f.write(line + "\n")


if __name__ == "__main__":
    main()
