#!/usr/bin/env python3
"""Counts, on the CPU, the table words the K3 voting kernel walks for a workload's sample reference points: one walk of the
whole bucket per in-radius scene pair (before folding), against folded walks (k3_vote.cu phase D: the constant-shift
ranges of the pairs that share a bucket and a shift walked once) under the kernel's flush boundaries and gates:

  flush  each flush of the candidate queue folds on its own, when it holds FOLD_MIN_PAIRS+ candidates (the kernel up to
         the fold buffer);
  scope  the kernel now: a task folds every flush when it flushes more than once or its one flush holds FOLD_MIN_PAIRS+
         candidates; its fold codes (one per pair with a non-empty bucket; the pairs within a guard band of a phase-cell
         edge, which leave none, are not modelled) collect across flushes and are folded once more than
         FOLD_SCOPE - CAND_CAP are buffered after a flush, and at the end of the task;
  task   the whole task folded at once, under the same gate (the bound of the scope form).

The flush model follows the kernel's sweep: the 9 rows of the 27 grid cells around the reference point (cells of edge
radius x 1.001 from the scene's bounding-box minimum, as scene_grid_params places them; the coarsening of very large
grids is ignored), cells in x order, points of a cell in scene order, blocks of THREADS points; after each block the
queue flushes when the 27 cells hold more than CAND_CAP points and more than CAND_CAP - THREADS candidates are buffered.
The kernel follows this order up to the order in which warps append to the queue.  Buckets come from the oracle's table
(unsliced; slicing divides every bucket alike), each phase cell counted as 1/16 of its bucket; the pair's own cell is
walked per pair in every form.

    python tools/k3_fold_count.py --workload c3 --points 24 [--out profiles/r6_k3_fold_count.jsonl]

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
THREADS = 1024  # the launch shape of the sliced tables that fold
FOLD_MIN_PAIRS = 1024
FOLD_SCOPE = 8192


def sweep_flushes(scene, s_r, in_radius, radius, threads=THREADS, cand_cap=CAND_CAP):
    """The kernel's flushes of reference point s_r: (27 cells overflow the queue, [candidate indices of each flush in
    sweep order]).  in_radius: per scene point, whether it passes the radius test against s_r."""
    lo = scene[:, :3].min(axis=0)
    cid = np.floor((scene[:, :3] - lo) / (radius * 1.001)).astype(np.int64)
    c0 = cid[s_r]
    near = np.flatnonzero(np.all(np.abs(cid - c0) <= 1, axis=1))
    run = (cid[near, 1] - c0[1] + 1) + 3 * (cid[near, 2] - c0[2] + 1)
    order = np.lexsort((near, cid[near, 0], run))
    near, run = near[order], run[order]
    many = len(near) > cand_cap
    flushes, cur = [], []
    for r in range(9):
        pts = near[run == r]
        for b in range(0, len(pts), threads):
            cur += [int(s) for s in pts[b:b + threads] if s != s_r and in_radius[s]]
            if many and len(cur) > cand_cap - threads:
                flushes.append(cur)
                cur = []
    flushes.append(cur)
    return many, flushes


def fold_scopes(flush_cands, flush_codes, fold_min=FOLD_MIN_PAIRS, scope=FOLD_SCOPE, cand_cap=CAND_CAP):
    """The kernel's fold scopes: lists of flush indices whose codes phase D folds together (empty: the task does not
    fold).  flush_cands: candidates per flush (the gate); flush_codes: fold codes per flush (where a scope ends)."""
    if not (len(flush_cands) > 1 or flush_cands[0] >= fold_min):
        return []
    scopes, cur, n = [], [], 0
    for i, c in enumerate(flush_codes):
        cur.append(i)
        n += c
        if n > scope - cand_cap or i + 1 == len(flush_codes):
            scopes.append(cur)
            cur, n = [], 0
    return scopes


def fold_words(keys, q, cell, length, n_turn):
    """words the folded constant-shift walks of these pairs touch (own cells not included)"""
    groups = {}  # (key, s) -> per-cell multiplier
    for k, qq, c, ln in zip(keys, q, cell, length):
        hi = groups.setdefault((k, qq), [0] * CELLS + [ln])
        for j in range(c + 1, CELLS):
            hi[j] += 1
        lo = groups.setdefault((k, (qq + 1) % n_turn), [0] * CELLS + [ln])
        for j in range(c):
            lo[j] += 1
    return sum(sum(1 for j in range(CELLS) if m[j]) * m[CELLS] / CELLS for m in groups.values())


def walked(flushes, code, n_turn):
    """words walked per form: {"per_pair", "flush", "scope", "task"}.  flushes: candidate indices per flush; code: index ->
    (key, q, cell, bucket length) for candidates with a non-empty bucket."""
    per = [[code[s] for s in f if s in code] for f in flushes]
    allc = [x for f in per for x in f]
    total = float(sum(x[3] for x in allc))
    own = total / CELLS
    unfolded = lambda cs: sum(x[3] for x in cs) * (CELLS - 1) / CELLS
    folded = lambda cs: fold_words(*zip(*cs), n_turn) if cs else 0.0
    out = {"per_pair": total}
    out["flush"] = own + sum(folded(cs) if len(f) >= FOLD_MIN_PAIRS else unfolded(cs) for f, cs in zip(flushes, per))
    scopes = fold_scopes([len(f) for f in flushes], [len(cs) for cs in per])
    out["scope"] = own + (sum(folded([x for i in sc for x in per[i]]) for sc in scopes) if scopes else unfolded(allc))
    out["task"] = own + (folded(allc) if scopes else unfolded(allc))
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--workload", default="c3")
    ap.add_argument("--points", type=int, default=24, help="the first N points of bench.sample_list")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r6_k3_fold_count.jsonl"))
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
    forms = ("per_pair", "flush", "scope", "task")
    rows, tot = [], {f: 0.0 for f in forms}
    for s_r in bench.sample_list(wl)[:args.points]:
        inr, d, a = hm.scene_pairs(scene, s_r)
        _, flushes = sweep_flushes(scene, s_r, inr, radius)
        code = {}
        for s in (x for f in flushes for x in f):
            ln = bucket.get(tuple(d[s].tolist()), 0)
            if ln:
                u = np.mod(float(a[s]) / step, T)
                qq = min(int(np.floor(u)), n_turn - 1)
                code[s] = (tuple(d[s].tolist()), qq, min(int((u - np.floor(u)) * CELLS), CELLS - 1), float(ln))
        w = walked(flushes, code, n_turn)
        row = {"ref": int(s_r), "pairs": len(code), "flushes": [len(f) for f in flushes], "votes": w["per_pair"],
               **{f"ratio_{f}": round(w["per_pair"] / w[f], 3) if w[f] else 1.0 for f in forms[1:]}}
        for f in forms:
            tot[f] += w[f]
        rows.append(row)
        print(json.dumps(row), flush=True)
    line = {"tool": "k3_fold_count", "workload": args.workload, "points": len(rows), "table_entries": hm.num_entries,
            "table_keys": hm.num_keys, "oracle_build_s": round(build_s, 1), "threads": THREADS, "cand_cap": CAND_CAP,
            "fold_min_pairs": FOLD_MIN_PAIRS, "fold_scope": FOLD_SCOPE, "words_walked_per_pair": tot["per_pair"],
            **{f"words_walked_folded_{f}": tot[f] for f in forms[1:]},
            **{f"ratio_{f}": round(tot["per_pair"] / tot[f], 3) for f in forms[1:] if tot[f]},
            "per_point": rows}
    with open(args.out, "w") as fh:
        fh.write(json.dumps(line) + "\n")
    print(json.dumps({k: v for k, v in line.items() if k != "per_point"}))


if __name__ == "__main__":
    main()
