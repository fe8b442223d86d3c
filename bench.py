#!/usr/bin/env python
"""bench.py — scene point-pairs voted per second (and ms per 6-D pose) of the PPF hot path.

    python bench.py --gpus N --steps K --warmup W [--workload c3] [--impl reference]

Default workload = c3, the configuration BASELINE.json's metric and target are quoted on ("10k-point model vs
100k-point scene, every scene point as reference, sharded across 1/2/4/8 B200"; north_star: ">= 50x the host-CPU
PCL PPFRegistration throughput on a 100k-point scene at 1 B200"); it fits one GPU.  --workload c1 | c2 | c2_5mm |
c3s | c4 | c4s select the other BASELINE configurations (workloads.py); c2 is the reference's own fixture.

A step is one PPFRegistration::align of the workload's scene against its (pre-built, resident)
model table: K3 voting over this rank's shard of scene reference points, K3b pose assembly, the
all-gather of 64-byte hypotheses (N > 1, NCCL), K4 clustering.  Building the model table is the
reference's *offline* training step (include/CloudProcessing.h:222-261 / :106-121) and is reported
separately (table_build_ms), not inside the step.

  value     in-radius scene point pairs (PCL's inner-loop trip count, "pairs voted") per second,
            scene + table resident in HBM, per-step CUDA events on the context stream, max over ranks
  e2e       the same through the host-buffer C ABI: every step uploads the scene from pinned host
            memory, runs align and reads the poses back
  roofline  the voting kernel against what binds it — the SM's L1 data pipe: one shared-memory reduction per vote.
            achieved = votes / s inside the kernel (CUDA events on the context stream), peak = the rate of the same
            loop shape (one coalesced 4-byte gather + one red.shared per vote) with conflict-free addresses, measured
            live by csrc/microbench.cu; HBM bytes per launch (ncu) are reported as `traffic`, L2 bandwidth beside it
  cpu_baseline  the CPU oracle (port of PCL's loop) on a fixed, bounded sample of reference points, all host cores

--impl reference times the CPU oracle with every host core on the same workload: each step votes on the next few
entries of a FIXED list of 64 evenly spread reference points (the same points on every box and at every --gpus)
and clusters them.  The oracle is test infrastructure: it is only ever the baseline here.

--dump-outputs DIR writes what the last timed step returned to its caller, the best poses and their votes of every
model, as DIR/poses.npy (float32, K x 4 x 4) and DIR/votes.npy (float64: exact for the uint32 counts); with a model
library, DIR/poses_model<k>.npy and DIR/votes_model<k>.npy.  The inputs are fixed files and seeded synthetic clouds,
so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "scene_point_pairs_voted_per_sec"
UNIT = "pairs/s"


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region.

    NVML is polled from a thread every 50 ms (a polling `nvidia-smi -lms` process was measured to
    slow this launch-heavy step by ~20 %: its queries contend with kernel launches for driver locks);
    nvidia-smi is only the fallback when pynvml is unavailable."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device, self.proc, self.path = device, None, None
        self.thread, self.stop_flag, self.samples = None, False, []

    def _nvml_loop(self, nv, handle):
        while not self.stop_flag:
            try:
                sm = nv.nvmlDeviceGetClockInfo(handle, nv.NVML_CLOCK_SM)
                try:
                    reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(handle)
                except Exception:
                    reasons = nv.nvmlDeviceGetCurrentClocksThrottleReasons(handle)
                self.samples.append((sm, reasons))
            except Exception:
                pass
            time.sleep(0.05)

    def start(self):
        try:
            import threading
            import pynvml as nv
            nv.nvmlInit()
            # NVML enumerates physical devices; honour CUDA_VISIBLE_DEVICES when it is a plain index list
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            idx = self.device
            if vis and all(x.strip().isdigit() for x in vis.split(",")):
                idx = int(vis.split(",")[self.device])
            h = nv.nvmlDeviceGetHandleByIndex(idx)
            self.nv, self.handle = nv, h
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            self.thread = threading.Thread(target=self._nvml_loop, args=(nv, h), daemon=True)
            self.thread.start()
            return
        except Exception:
            self.thread = None
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "500"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "source": None}
        if self.thread:
            self.stop_flag = True
            self.thread.join(timeout=2)
            nv = self.nv
            names = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                     "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                     "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                     "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
            if self.samples:
                seen = set()
                for _, r in self.samples:
                    for n, bit in names.items():
                        if r & bit:
                            seen.add(n)
                out.update(sm_mhz=float(np.median([s for s, _ in self.samples])), sm_max_mhz=float(self.max_mhz),
                           reasons=sorted(seen), samples=len(self.samples), source="nvml thread, 50 ms")
            return out
        if not self.proc:
            return out
        time.sleep(0.6)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                p = [x.strip() for x in line.split(",")]
                if len(p) < 9:
                    continue
                try:
                    sm.append(float(p[1]))
                    mx.append(float(p[2]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm),
                       source="nvidia-smi -lms 500")
        return out


def oracle_table(wl, model=None):
    from oracle import binding as ob  # loads the library build() made: the benchmark compiles nothing into the tree
    th = host_threads()  # the container is built sharded by key over the host cores: same buckets, seconds instead of minutes
    feats = ob.ppf_estimation(wl.model if model is None else model, n_threads=th)
    hm = ob.HashMap(wl.angle_step, wl.dist_step).set_input_feature_cloud(feats, n_threads=th)
    return ob, hm


def host_threads():
    """Cores this process may run on.  Not omp_get_max_threads(): torchrun exports OMP_NUM_THREADS=1."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


SAMPLE_SLOTS = 64


def sample_list(wl):
    """The fixed CPU sample of a workload: 64 reference slots spread evenly over the scene (slot k sits in the middle
    of the k-th 64th), listed in bit-reversed order so that every prefix — and every run of consecutive entries — is
    itself evenly spread.  The synthetic scenes are stored in a fixed pseudo-random order, so an even spread is a uniform
    random sample of the surfaces (object, ground, walls, clutter), the same on every box.  Returns reference-point
    indices into the scene."""
    n = min(SAMPLE_SLOTS, wl.n_ref)
    bits = max(1, (n - 1).bit_length())
    order = [int(format(k, f"0{bits}b")[::-1], 2) for k in range(1 << bits)]
    order = [k for k in order if k < n]
    return [int((k + 0.5) * wl.n_ref / n) * wl.ref_rate for k in order]


# votes one reference point costs on average (measured on the B200 arm; only used to size a CPU step)
VOTES_PER_REF = {"c1": 1.0e5, "c2": 1.7e5, "c2_5mm": 2.2e6, "c3": 8.1e7, "c3s": 1.3e6, "c4": 8.1e6, "c4s": 8.1e6}


def refs_per_cpu_step(wl, threads, requested, models=1, seconds=4.0):
    """reference points one CPU step votes on: about `seconds` of work at ~1.1e6 votes/s per thread, 1 .. 64"""
    if requested:
        return max(1, min(requested, SAMPLE_SLOTS, wl.n_ref))
    per_ref = VOTES_PER_REF.get(wl.name, 1e6) * models / (1.1e6 * threads)
    return int(max(1, min(SAMPLE_SLOTS, wl.n_ref, round(seconds / per_ref))))


def vote_refs(hm, wl, model, refs, threads):
    """the oracle's voting loop on an explicit list of reference points -> (hypotheses, counters)"""
    return hm.vote_refs(model, wl.scene, refs, n_threads=threads)


def dump_outputs(out_dir, results, n_models):
    """results: {model index: (poses, votes)} of one align.  At most 3 poses per model: a few KB for every workload."""
    os.makedirs(out_dir, exist_ok=True)
    for k, (poses, votes) in results.items():
        suffix = f"_model{k}" if n_models > 1 else ""
        np.save(os.path.join(out_dir, f"poses{suffix}.npy"), np.asarray(poses, np.float32).reshape(-1, 4, 4))
        np.save(os.path.join(out_dir, f"votes{suffix}.npy"), np.asarray(votes, np.float64))


def workload_config(wl, gpus):
    """`config` of the JSON line: the workload only — identical in the B200 arm and the reference arm"""
    m = wl.library()[0]
    return {"workload": f"{wl.name}: {wl.description}", "n_model": int(m.shape[0]), "models": len(wl.library()),
            "n_scene": int(wl.scene.shape[0]), "n_ref": int(wl.n_ref), "ref_rate": int(wl.ref_rate), "angle_step_deg": 12,
            "dist_step": float(wl.dist_step), "alpha_columns": "ceil(2*pi/step) = 30 (current PCL)", "gpus": int(gpus),
            "l2": "B200 arm: 256 MiB memset between steps, outside the per-step CUDA-event brackets; CPU arm: n/a"}


def run_reference(args, wl):
    """The reference arm: CPU oracle, all host cores, a fixed rotating sample of reference points."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    library = wl.library()
    tables = [oracle_table(wl, m) for m in library]
    ob = tables[0][0]
    threads = host_threads()
    refs_all = sample_list(wl)
    per_step = refs_per_cpu_step(wl, threads, args.cpu_sample, len(library))
    times, pairs, votes, used = [], 0, 0, []
    for k in range(args.warmup + args.steps):
        refs = [refs_all[(k * per_step + j) % len(refs_all)] for j in range(per_step)]
        t0 = time.perf_counter()
        step_pairs = step_votes = 0
        results = {}
        for k_m, (m, (_, hm_k)) in enumerate(zip(library, tables)):
            hyps, st = vote_refs(hm_k, wl, m, refs, threads)
            results[k_m] = ob.cluster(hyps, wl.pos_thr, wl.rot_thr)[:2]
            step_pairs += st["pairs_in_radius"]
            step_votes += st["votes"]
        dt = time.perf_counter() - t0
        if k >= args.warmup:
            times.append(dt)
            pairs += step_pairs
            votes += step_votes
            used += refs
    total_s = float(np.sum(times))
    ms = 1e3 * total_s / args.steps
    value = pairs / total_s
    n_used = len(set(used))
    sample = (f"{per_step} reference point(s) per step from a fixed list of {len(refs_all)} evenly spread ones (bit-reversed order, "
              f"{n_used} distinct points over the {args.steps} timed steps), full scene, vote + cluster"
              + (f", for each of the {len(library)} models" if len(library) > 1 else ""))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": wl.data, "config": workload_config(wl, args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "sample_refs": sorted(set(used)),
        "sample_work": {"pairs_in_radius": pairs, "votes": votes, "votes_per_pair": votes / max(1, pairs)},
        "ms_per_pose_extrapolated": 1e3 * total_s / max(1, len(used)) * wl.n_ref,
        "votes_per_sec": votes / total_s,  # the sample-independent rate (pairs differ in cost by orders of magnitude)
    }
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, results, len(library))
    print(json.dumps(line), flush=True)


def run_b200(args, wl):
    import torch
    import torch.distributed as dist
    from yolo_ppf_pose_estimation_b200 import capi, sharding

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the B200 path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG", "WARN")              # no "NCCL version ..." banner
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    ctx = capi.Context(local)
    stream = torch.cuda.ExternalStream(ctx.stream, device=dev)

    n_ref = wl.n_ref
    library = wl.library()
    lib_mode = len(library) > 1
    lib_sharded = lib_mode and args.c4_mode == "refs" and world > 1
    if lib_sharded:
        # model library (c4), second partitioning: every rank holds all tables, the reference points of every model's
        # align are shared by all ranks (the group's queue) — one align per model, each over all GPUs
        my_models = list(range(len(library)))
        first, step, count = sharding.shard(n_ref, rank, world)
        chunk = sharding.chunk_size(n_ref, world)
    elif lib_mode:
        # model library (c4): model-parallel — rank r aligns models r, r + world, ... against the replicated scene,
        # every reference point each; no hypothesis exchange, only the final poses are gathered
        my_models = [k for k in range(len(library)) if k % world == rank]
        first, step, count = 0, 1, n_ref
        chunk = n_ref
    else:
        my_models = [0]
        first, step, count = sharding.shard(n_ref, rank, world)
        chunk = sharding.chunk_size(n_ref, world)
    with torch.cuda.stream(stream):
        local_buf = torch.zeros((chunk, 16), dtype=torch.float32, device=dev)
        flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    # ---- offline stage: model upload + table build (reported, not part of the step) ---------------
    dms = [ctx.upload_cloud(library[k]) for k in my_models]
    ctx.table_build_from_cloud(dms[0], wl.angle_step, wl.dist_step).free()  # untimed: first use loads the kernels
    t0 = time.perf_counter()
    tables = [ctx.table_build_from_cloud(dm, wl.angle_step, wl.dist_step) for dm in dms]
    table_build_ms = 1e3 * (time.perf_counter() - t0)
    tim = ctx.timings()
    info = tables[0].info if tables else None
    ds_resident = ctx.upload_cloud(wl.scene)
    scene_pinned = torch.from_numpy(np.ascontiguousarray(wl.scene, np.float32)).pin_memory()
    n_s = wl.scene.shape[0]

    # ---- several GPUs: b200ppf_group_* — the record exchange is fused into the vote epilogue (NVLink peer stores), the
    # per-step barrier is a flag the peers' kernels raise and a one-thread kernel awaits: no torch.distributed call in a step
    p2p = world > 1 and (not lib_mode or lib_sharded) and args.exchange == "p2p"
    group = None
    if p2p:
        group = capi.Group(ctx, rank, world, chunk * world)
        handles = [None] * world
        dist.all_gather_object(handles, group.handles.tobytes())   # bootstrap only: 192 bytes per rank, once
        group.connect([np.frombuffer(h, np.uint8) for h in handles])

    def align(ds, collect=None):
        """vote (this rank's shard) -> exchange -> cluster, once per model of this rank; returns {model: (poses, votes)}."""
        results = {}
        for k_m, dm, table in zip(my_models, dms, tables):
            if p2p:
                group.vote(dm, table, ds, wl.ref_rate)
            else:
                ctx.vote_device(dm, table, ds, first * wl.ref_rate, step * wl.ref_rate, count, local_buf.data_ptr())
            if collect is not None:  # untimed bookkeeping pass: work counters and kernel time of every model
                st = ctx.vote_stats()
                for k, v in st.items():
                    collect[k] = collect.get(k, 0) + v
                collect["vote_ms"] = collect.get("vote_ms", 0.0) + ctx.timings()["vote_ms"]
            if p2p:
                results[k_m] = group.cluster(dm, table, ds, wl.ref_rate, wl.pos_thr, wl.rot_thr)
            elif world > 1 and (not lib_mode or lib_sharded):
                with torch.cuda.stream(stream):
                    ordered = sharding.all_gather_hypotheses(local_buf, n_ref, world, dist)
                results[k_m] = ctx.cluster(None, wl.pos_thr, wl.rot_thr, device_ptr=ordered.data_ptr(), n=n_ref)
                del ordered
            else:
                results[k_m] = ctx.cluster(None, wl.pos_thr, wl.rot_thr, device_ptr=local_buf.data_ptr(), n=n_ref)
        return results

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_steps(make_scene, k_steps):
        """per-step CUDA events on the context stream; L2 flushed between steps outside the brackets"""
        total, vote_ms, launches = 0.0, [], 0
        for _ in range(k_steps):
            with torch.cuda.stream(stream):
                flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            l0 = ctx.launch_count
            e0.record(stream)
            results = align(make_scene())
            e1.record(stream)
            e1.synchronize()
            total += e0.elapsed_time(e1)
            launches += ctx.launch_count - l0
            if not lib_mode:
                vote_ms.append(ctx.timings()["vote_ms"])
        return total, vote_ms, launches, results

    # ---- resident-input measurement ---------------------------------------------------------------
    sampler = ClockSampler(local)
    if rank == 0 and os.environ.get("BENCH_CLOCKS", "1") != "0":
        sampler.start()  # NVML is initialised here, outside the timed region; only the samples of the timed region are kept
    barrier()
    timed_steps(lambda: ds_resident, args.warmup)
    stats = {}
    align(ds_resident, collect=stats)
    for k in ("pairs_in_radius", "votes", "pairs_examined", "nonempty_lookups", "vote_ms"):
        stats.setdefault(k, 0)
    barrier()
    sampler.samples.clear()
    total_ms, vote_ms, launches, results = timed_steps(lambda: ds_resident, args.steps)
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    poses, votes = results[my_models[-1]]
    # model-parallel ranks each hold their own models' results; otherwise every rank holds the same ones
    if args.dump_outputs and (rank == 0 or (lib_mode and not lib_sharded)):
        dump_outputs(args.dump_outputs, results, len(library))

    # ---- end to end through the host-buffer API: H2D scene every step, poses read back -------------
    def upload():
        return ctx.upload_cloud((scene_pinned.data_ptr(), n_s), stride=6, normal_offset=3)
    timed_steps(upload, min(args.warmup, 3))
    barrier()
    e2e_total_ms, _, _, _ = timed_steps(upload, args.steps)
    barrier()

    # whole-job numbers: max over ranks of the time, sum over ranks of the work
    if lib_mode:
        vote_ms = [stats["vote_ms"]]
    t = torch.tensor([total_ms, e2e_total_ms, float(np.mean(vote_ms)) if vote_ms else 0.0], dtype=torch.float64, device=dev)
    w = torch.tensor([stats["pairs_in_radius"], stats["votes"], stats["pairs_examined"], stats["nonempty_lookups"]],
                     dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(w, op=dist.ReduceOp.SUM)
    total_ms, e2e_total_ms, vote_kernel_ms = (float(x) for x in t.cpu())
    pairs, nvotes, examined, nonempty = (float(x) for x in w.cpu())

    if rank == 0:
        ms_per_step = total_ms / args.steps
        value = pairs / (ms_per_step * 1e-3)
        e2e_ms = e2e_total_ms / args.steps
        hbm_peak, hbm_src = measured_peaks()
        # algorithmic bytes of one voting launch on one rank (DESIGN.md "K3 roofline"):
        #   4 B gathered per vote (the hot word; the 1/16 of votes in the scene phase's own cell gather 8 B: 4.25 B mean);
        #   per in-radius pair and slice 16 B of CSR offsets + 32 B of point/normal;
        #   16 B per scene point per resident wave of CTAs for the position sweep
        my_pairs, my_votes = stats["pairs_in_radius"], stats["votes"]
        ctas = count * info.n_slices * len(my_models)
        waves = max(1, -(-ctas // (148 * 2)))
        per_vote = 4.0 + 4.0 / max(1, info.phase_cells) if info.phase_cells > 1 else 8.0
        alg_bytes = per_vote * my_votes + 48.0 * my_pairs * info.n_slices + 16.0 * n_s * waves
        k3_ms = float(np.mean(vote_ms))
        votes_per_s = my_votes / (k3_ms * 1e-3)
        # The roof: the SM's L1 data pipe.  Measured live (csrc/microbench.cu) in the voting loop's own shape — one
        # coalesced 4-byte gather from an L2-resident table + one red.shared.add per vote, eight gathers in flight per
        # lane — with conflict-free addresses; +8 = the 1024-thread x 1 CTA/SM launch shape of sliced tables.
        shape = 8 if info.n_slices > 1 else 0
        peak_cf = max(ctx.microbench_atoms(5 + shape) for _ in range(2))
        peak_2way = max(ctx.microbench_atoms(7 + shape) for _ in range(2))
        peak_random = max(ctx.microbench_atoms(6 + shape) for _ in range(2))
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "k3_dram_traffic.json")
        if os.path.exists(tpath):
            with open(tpath) as f:
                traffic = json.load(f).get(wl.name)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": wl.data,
            "config": workload_config(wl, world),
            "run": {"table_entries": int(info.n_entries), "accumulator_slices": int(info.n_slices),
                    "alpha_columns": int(info.n_alpha), "phase_cells": int(info.phase_cells),
                    "sharding": (f"model-parallel: {len(library)} models over {world} rank(s), scene replicated" if lib_mode and not lib_sharded
                                 else ((f"b200ppf_group: {world} ranks draw (reference point, slice) tasks from one queue over NVLink, "
                                        f"table + scene replicated, 8-byte peaks merged into every rank's array by system-scope atomicMax, "
                                        f"device-side flags" if p2p else
                                        f"reference points interleaved over {world} rank(s), table + scene replicated, 64 B hypotheses "
                                        f"exchanged by an NCCL all-gather")) if world > 1 else "single GPU")},
            "ms_per_pose": ms_per_step / len(library),
            "votes_per_sec": nvotes / (ms_per_step * 1e-3),
            "pairs_examined_per_sec": examined / (ms_per_step * 1e-3),
            "work_per_step": {"pairs_in_radius": pairs, "votes": nvotes, "pairs_examined": examined},
            "result": {"votes": [int(v) for v in votes], "translation": [float(x) for x in poses[0][:3, 3]] if len(poses) else None},
            "table_build_ms": table_build_ms,
            "table_build_stage_ms": {k: tim[k] for k in ("keys_ms", "sort_ms", "csr_ms")},
            "e2e": {"value": pairs / (e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": int(2 * 16 * n_s), "d2h_bytes_per_step": int(3 * 16 * 4 + 8 * 4 + 8)},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"kernel": "ppf_vote_kernel", "bound": "shared_atomic", "achieved": votes_per_s, "peak": peak_cf,
                         "unit": "shared-memory reductions/s", "frac": votes_per_s / peak_cf,
                         "peak_source": "measured in this run: b200ppf_microbench_atoms, the voting loop's shape (coalesced 4-byte "
                                        "gather + red.shared per vote, 8 in flight per lane), conflict-free addresses",
                         "peak_two_lanes_per_bank": peak_2way, "peak_random_words": peak_random,
                         "frac_of_random_words_peak": votes_per_s / peak_random,
                         "traffic": traffic["dram_bytes_per_launch"] if traffic else None,
                         "traffic_source": traffic["source"] if traffic else None,
                         "kernel_ms": k3_ms, "kernel_ms_max_over_ranks": vote_kernel_ms,
                         "kernel_share_of_step": k3_ms / ms_per_step,
                         "hbm": {"algorithmic_bytes_per_launch": alg_bytes, "algorithmic_gbs": alg_bytes / (k3_ms * 1e-3) / 1e9,
                                 "peak_gbs": hbm_peak, "peak_source": hbm_src,
                                 "note": "the gathered table words are served by L2/L1, not HBM (DRAM traffic = table + scene "
                                         "once per launch): an HBM fraction of the algorithmic bytes is not a bound"},
                         "l2": {"gathered_gbs": per_vote * my_votes / (k3_ms * 1e-3) / 1e9,
                                "note": "hot words gathered per second, an upper bound on the L2 -> L1 traffic (part hits L1)"}},
        }
        if world == 1 and not args.no_cpu and not lib_mode:
            ob, hm = oracle_table(wl)
            threads = host_threads()
            refs = sample_list(wl)[:refs_per_cpu_step(wl, threads, args.cpu_sample, 1, seconds=20.0)]
            t0 = time.perf_counter()
            _, cst = vote_refs(hm, wl, wl.model, refs, threads)
            dt = time.perf_counter() - t0
            line["cpu_baseline"] = {"value": cst["pairs_in_radius"] / dt, "unit": UNIT, "cores": threads, "kind": "port",
                                    "sample": f"the first {len(refs)} of the fixed list of {SAMPLE_SLOTS} evenly spread reference "
                                              f"points (bench.py sample_list), full scene, voting loop only, {dt:.1f} s",
                                    "votes_per_sec": cst["votes"] / dt,
                                    "sample_votes_per_pair": cst["votes"] / max(1, cst["pairs_in_radius"]),
                                    "workload_votes_per_pair": nvotes / max(1.0, pairs)}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c3", help="c1 | c2 | c2_5mm | c3 (default) | c3s | c4 | c4s (workloads.py)")
    ap.add_argument("--cpu-sample", type=int, default=0,
                    help="reference points per CPU step, taken in order from the fixed 64-point list (0 = sized for ~4 s per step)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--c4-mode", default="models", choices=["models", "refs"],
                    help="model library on several GPUs: one model per GPU (default) or every table on every GPU with the "
                         "reference points of each align shared by all GPUs")
    ap.add_argument("--exchange", default="p2p", choices=["p2p", "nccl"],
                    help="several GPUs: records written into every peer's buffer by the vote epilogue (default) or NCCL all-gather")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the poses and votes the last timed step returned as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    from yolo_ppf_pose_estimation_b200 import workloads
    wl = workloads.load(args.workload)
    if args.impl == "reference":
        run_reference(args, wl)
    else:
        run_b200(args, wl)


if __name__ == "__main__":
    main()
