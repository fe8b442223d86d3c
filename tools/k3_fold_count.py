#!/usr/bin/env python3
"""Counts, on the CPU, the table words the K3 voting kernel walks for a workload's sample reference points: one walk of the
whole bucket per in-radius scene pair (before folding), against folded walks (k3_vote.cu phase D: the constant-shift
ranges of the pairs that share a bucket and a shift walked once) at three scopes — the whole task, flushes of 8 192 pairs
and flushes of the candidate queue (2 048 pairs).  Buckets come from the oracle's table (unsliced; slicing divides every
bucket alike), each phase cell counted as 1/16 of its bucket; the pair's own cell is walked per pair either way.  Flushes
take the pairs in the order the kernel sweeps them (the 9 rows of the 27 grid cells around the reference point, cells of
the radius, points of a cell in scene order), which the kernel follows up to the order warps append to the queue.

    python tools/k3_fold_count.py --workload c3 --points 24 [--out profiles/r3_k3_fold_count.jsonl]

Prints one line per point and writes one JSON line with the totals.  No GPU needed."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CELLS = 16
CAND_CAP = 2048


def sweep_order(scene, s_r, idx, radius, lo):
    """positions of the pairs idx in the kernel's sweep: (row of the 27 cells, cell x, scene order)"""
    c = np.floor((scene[idx, :3] - lo) / radius).astype(np.int64)
    cr = np.floor((scene[s_r, :3] - lo) / radius).astype(np.int64)
    row = (c[:, 1] - cr[1] + 1) + 3 * (c[:, 2] - cr[2] + 1)
    return np.lexsort((idx, c[:, 0], row))


def walked(keys, q, cell, length, n_turn, scope):
    """(words walked with one walk per pair, words walked folded) over pairs in sweep order, folding within chunks of
    `scope` pairs (None: the whole task)"""
    per_pair = float(length.sum())
    own = float(length.sum()) / CELLS
    folded = own
    n = len(keys)
    step = n if scope is None else scope
    for b in range(0, max(n, 1), max(step, 1)):
        sl = slice(b, b + step)
        groups = {}  # (key, s) -> per-cell multiplier
        for k, qq, c, ln in zip(keys[sl].tolist(), q[sl].tolist(), cell[sl].tolist(), length[sl].tolist()):
            hi = groups.setdefault((k, qq), [0] * CELLS + [ln])
            for j in range(c + 1, CELLS):
                hi[j] += 1
            lo = groups.setdefault((k, (qq + 1) % n_turn), [0] * CELLS + [ln])
            for j in range(c):
                lo[j] += 1
        for m in groups.values():
            folded += sum(1 for j in range(CELLS) if m[j]) * m[CELLS] / CELLS
    return per_pair, folded


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--workload", default="c3")
    ap.add_argument("--points", type=int, default=24, help="the first N points of bench.sample_list")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_k3_fold_count.jsonl"))
    args = ap.parse_args()
    from yolo_ppf_pose_estimation_b200 import workloads
    import bench
    from oracle import binding as ob
    ob.build()
    wl = workloads.load(args.workload)
    t0 = time.time()
    _, hm = bench.oracle_table(wl)
    build_s = time.time() - t0
    dkeys, dlen = hm.dump_keys()
    bucket = {tuple(k): int(n) for k, n in zip(dkeys.tolist(), dlen.tolist())}
    step = float(wl.angle_step)
    T = 2.0 * np.pi / step
    n_turn = int(round(T))
    radius = 0.5 * hm.model_diameter
    scene = wl.scene.astype(np.float32)
    lo = scene[:, :3].min(axis=0)
    scopes = {"task": None, "8192": 8192, "2048": CAND_CAP}
    rows, tot = [], {"votes": 0.0, **{s: [0.0, 0.0] for s in scopes}}
    for s_r in bench.sample_list(wl)[:args.points]:
        inr, d, a = hm.scene_pairs(scene, s_r)
        idx = np.flatnonzero(inr)
        length = np.array([bucket.get(tuple(x), 0) for x in d[idx].tolist()], np.float64)
        keep = length > 0
        idx, length = idx[keep], length[keep]
        order = sweep_order(scene, s_r, idx, radius, lo)
        idx, length = idx[order], length[order]
        u = np.mod(a[idx].astype(np.float64) / step, T)
        q = np.minimum(np.floor(u).astype(np.int64), n_turn - 1)
        cell = np.minimum(np.floor((u - np.floor(u)) * CELLS).astype(np.int64), CELLS - 1)
        kid = {k: i for i, k in enumerate(sorted(set(map(tuple, d[idx].tolist()))))}
        keys = np.array([kid[tuple(x)] for x in d[idx].tolist()], np.int64)
        row = {"ref": int(s_r), "pairs": int(inr.sum()), "votes": float(length.sum())}
        for name, sc in scopes.items():
            pp, fo = walked(keys, q, cell, length, n_turn, sc)
            row[f"ratio_{name}"] = round(pp / fo, 3) if fo else 1.0
            tot[name][0] += pp
            tot[name][1] += fo
        tot["votes"] += row["votes"]
        rows.append(row)
        print(json.dumps(row), flush=True)
    line = {"tool": "k3_fold_count", "workload": args.workload, "points": len(rows), "table_entries": hm.num_entries,
            "table_keys": hm.num_keys, "oracle_build_s": round(build_s, 1), "votes": tot["votes"],
            "words_walked_per_pair": tot["task"][0],
            **{f"words_walked_folded_{s}": tot[s][1] for s in scopes},
            **{f"ratio_{s}": round(tot[s][0] / tot[s][1], 3) for s in scopes if tot[s][1]},
            "per_point": rows}
    with open(args.out, "w") as fh:
        fh.write(json.dumps(line) + "\n")
    print(json.dumps({k: v for k, v in line.items() if k != "per_point"}))


if __name__ == "__main__":
    main()
