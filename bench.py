#!/usr/bin/env python
"""Benchmark of the scan-to-map registration hot path (BASELINE.json config[1]: 100k-pt scan vs 5M-pt map, 1xB200).

A step = one synthetic Livox scan through the whole per-scan path (ll_scan_to_pose): feature extraction (K1-K3),
VoxelGrid x2 per feature class (K4), then the ICP loop against the HBM-resident map: transform + exact 5-NN + residual
blocks (K6-K7), robust LM solve x2 with inlier selection (K8-K10).  The map index (K5) is built once, outside the steps.

  value : scans/s with the raw scans already resident in HBM, timed with CUDA events on the context's stream.
  e2e   : scans/s through the same C-ABI call with the raw scan in pinned HOST memory (H2D inside the timed region,
          pose read back to the host), host wall clock around the call.
L2 is flushed (256 MiB write) between timed steps, outside the timed regions.

`--impl reference` times the CPU restatement of the reference (oracle/) on the host cores instead (no GPU used).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark leaves the tree it runs from as it found it (which may be read-only)

from loam_livox_b200 import synthetic as S  # noqa: E402

WORKLOADS = {"c2": "C2: 100k-pt Livox scan vs 5M-pt map (0.5M corner + 4.5M surface), extract + VoxelGrid + 5-NN + LM registration",
             "c4": "C4: 100k-pt Livox scan vs 20M-pt map (2M corner + 18M surface), extract + VoxelGrid + 5-NN + LM registration"}
WORKLOAD = WORKLOADS["c2"]
N_SCAN = 100_000
N_MAP_CORNER, N_MAP_SURF = 500_000, 4_500_000
N_MAP_CORNER_C4, N_MAP_SURF_C4 = 2_000_000, 18_000_000
# leaves scaled from the precision YAML (0.1 / 0.4 m on a ~0.2 m map) to this map's ~0.02 m point spacing
PIPE = dict(pieces=3, use_piece=0, extractor_leaf_corner=0.01, extractor_leaf_surf=0.01, mapping_leaf_corner=0.01, mapping_leaf_surf=0.02, whole_frame=1)
N_DISTINCT_SCANS = 6


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f)["hbm_gbs"], "measured"
    return 6650.0, "fallback"


def source_sha(name):
    """sha1 of a kernel source file: ncu summaries under profiles/ are stamped with it, so a stale capture is never quoted."""
    import hashlib
    with open(os.path.join(ROOT, "loam_livox_b200", "csrc", name), "rb") as f:
        return hashlib.sha1(f.read()).hexdigest()


def ncu_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` from the committed `ncu --set full` capture of this same command
    (profiles/ncu_<kernel>_r2.json, written by profiles/summarize.py together with the sha1 of the kernel's source file).  None when the capture is
    absent or was taken from a different version of the source."""
    src = {"knn_blocks_kernel": "knn.cu", "lm_solve_kernel": "solve.cu"}[kernel]
    p = os.path.join(ROOT, "profiles", f"ncu_{kernel}_r2.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        if d.get("source_sha1") == source_sha(src):
            return d.get("traffic_bytes_per_launch")
    return None


def depth_levels(n):
    return int(np.ceil(np.log2(max(n, 16) / 15.0)))


def knn_algorithmic_bytes(qc, qs, nmc, nms):
    """SURVEY.md §8(d): per query 16 (query) + 16*D(N) (root-to-leaf path) + 240 (home leaf)."""
    return qc * (16 * depth_levels(nmc) + 256) + qs * (16 * depth_levels(nms) + 256)


def solve_algorithmic_bytes(blocks, evals_per_launch):
    """SURVEY.md §8(d): K7+K8 64 B per residual block per evaluation, K10 8 B read + 1 B write per block, per launch (= per ICP iteration)."""
    return blocks * (64.0 * evals_per_launch + 9.0)


class ClockSampler:
    """One `nvidia-smi -lms 50` process for the duration of the timed regions (clocks + throttle reasons under load)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, device=0):
        self.device = device
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.device}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        rows = []
        if self.proc is not None:
            self.proc.terminate()
            try:
                out, _ = self.proc.communicate(timeout=5)
                rows = [[c.strip() for c in ln.split(",")] for ln in out.strip().splitlines() if ln.strip()]
            except Exception:
                self.proc.kill()
        sm = [float(r[0]) for r in rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            for k, nme in enumerate(names):
                if len(r) > 3 + k and r[3 + k].lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


def workload_sizes(name):
    return {"c2": (N_MAP_CORNER, N_MAP_SURF), "c4": (N_MAP_CORNER_C4, N_MAP_SURF_C4)}[name]


def make_inputs(rank=0, workload="c2", maps=None):
    """Map + a few distinct scans (different sensor poses) + perturbed initial guesses, all seeded.  Every rank of the replicated mode gets its own
    scans (seeded by rank); tests/test_bench_inputs.py runs all of them through the oracle without a GPU."""
    nmc, nms = workload_sizes(workload)
    mc, ms = maps if maps is not None else S.make_map(nmc, nms)
    rng = np.random.default_rng(S.SEED + 100 + rank)
    scans, guesses, truths = [], [], []
    for k in range(N_DISTINCT_SCANS):
        pose = S.Pose(S.quat_from_euler(0.01 * k, -0.02, 0.05 + 0.03 * k), np.array([0.3 + 0.5 * k, 0.2 - 0.1 * k, 0.1]))
        scans.append(S.make_scan(N_SCAN, pose, seed=S.SEED + 1000 * rank + k))
        guesses.append(S.perturb_pose(pose, rng))
        truths.append(pose)
    return mc, ms, scans, guesses, truths


# ------------------------------------------------------------------------------------------------ CPU arm
def oracle_step(O, ex, trees, mc, ms, raw, guess, threads):
    """The same per-scan path on the host: oracle extractor -> VoxelGrid x2 -> registration."""
    ex.extract(raw, 100.0)
    c, s, _ = ex.get_features(0.0, 1.0)
    c = O.voxel_grid(O.voxel_grid(c, PIPE["extractor_leaf_corner"]), PIPE["mapping_leaf_corner"])
    s = O.voxel_grid(O.voxel_grid(s, PIPE["extractor_leaf_surf"]), PIPE["mapping_leaf_surf"])
    p = O.default_params(q_w_last=guess.q, t_w_last=guess.t, q_w_curr=guess.q, t_w_curr=guess.t, num_threads=threads)
    st, res = O.register(mc, trees[0], ms, trees[1], c, s, p)
    return st, res, c.shape[0], s.shape[0]


def host_threads():
    """Host threads this process may use -- NOT omp_get_max_threads(): torchrun exports OMP_NUM_THREADS=1, which made every multi-GPU CPU arm of
    round 1 single-threaded.  The oracle takes its team size as an explicit argument (num_threads clause)."""
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def cpu_baseline(threads, n_scans, inputs, trees=None, warmup=1, in_flight=1):
    """`in_flight` > 1 = the reference's throughput mode (maximum_parallel_thread scans registered concurrently, each by a `threads`-thread team;
    /root/reference/source/laser_mapping.hpp:1737-1742): scans/s of the whole pool."""
    from oracle import oracle as O
    mc, ms, scans, guesses, _ = inputs
    t0 = time.perf_counter()
    if trees is None:
        trees = (O.KdTree(mc), O.KdTree(ms))
        cpu_baseline.t_build = time.perf_counter() - t0
    t_build = getattr(cpu_baseline, "t_build", 0.0)
    exs = [O.Extractor() for _ in range(in_flight)]
    for w in range(max(1, warmup)):
        oracle_step(O, exs[0], trees, mc, ms, scans[w % len(scans)], guesses[w % len(scans)], threads)
    last = {}
    if in_flight == 1:
        t0 = time.perf_counter()
        for k in range(n_scans):
            st, res, nc, ns = oracle_step(O, exs[0], trees, mc, ms, scans[k % len(scans)], guesses[k % len(scans)], threads)
        total = time.perf_counter() - t0
        last = dict(res=res, nc=nc, ns=ns)
    else:
        def worker(w):
            for k in range(w, n_scans, in_flight):
                st, res, nc, ns = oracle_step(O, exs[w], trees, mc, ms, scans[k % len(scans)], guesses[k % len(scans)], threads)
                last.update(res=res, nc=nc, ns=ns)
        ths = [threading.Thread(target=worker, args=(w,)) for w in range(in_flight)]
        t0 = time.perf_counter()
        for t in ths:
            t.start()
        for t in ths:
            t.join()
        total = time.perf_counter() - t0
    per = total / n_scans
    return {"value": 1.0 / per, "unit": "scans/s", "cores": threads * in_flight, "kind": "port",
            "sample": f"{n_scans} scans of the same workload (oracle/ = CPU restatement of the reference; PCL/Ceres/Eigen are not installed), "
                      f"{threads} thread(s) per scan x {in_flight} scan(s) in flight, map index build {t_build:.1f} s not included", "ms_per_scan": per * 1e3, "index_build_s": t_build,
            "features": [last["nc"], last["ns"]], "icp_iterations": last["res"].icp_iterations}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as O
    hw = host_threads()
    wl = "c4" if args.mode == "sharded" else "c2"
    inputs = make_inputs(0, wl)
    t0 = time.perf_counter()
    mc, ms = inputs[0], inputs[1]
    trees = (O.KdTree(mc), O.KdTree(ms))
    cpu_baseline.t_build = time.perf_counter() - t0
    in_flight = max(1, args.contexts)
    # "all the host threads it can use": more threads than the path can use make it slower (128 threads: 0.24 scans/s, 16 threads: 11 scans/s on the
    # same box), so the arm takes the best of a few team sizes, each tried on two scans
    cands = sorted({c for c in (hw, 64, 32, 16, 8, 4, 2, 1) if c * in_flight <= hw} or {1}, reverse=True)
    trial = {c: cpu_baseline(c, 2 * in_flight, inputs, trees=trees, in_flight=in_flight)["value"] for c in cands}
    best = max(trial, key=trial.get)
    # the requested steps and warm-up, unless that would take longer than the time budget (then as many as fit, and the line says so)
    budget_s = 150.0
    per = 1.0 / trial[best]
    n = int(max(min(args.steps, budget_s / per), min(args.steps, 4)))
    w = int(max(1, min(args.warmup, 0.1 * budget_s / per)))
    cb = cpu_baseline(best, n, inputs, trees=trees, warmup=w, in_flight=in_flight)
    cb["sample"] += (f"; team size chosen among {cands} of {hw} host threads (scans/s on two scans each: " + ", ".join(f"{c}: {trial[c]:.2f}" for c in cands) + ")"
                     + ("" if n == args.steps else f"; {n} of the requested {args.steps} steps fit the {budget_s:.0f} s budget"))
    line = {"impl": "reference", "metric": "scans_per_sec", "value": cb["value"], "unit": "scans/s", "n_gpus": args.gpus, "steps": n, "warmup": w,
            "ms_per_step": cb["ms_per_scan"], "higher_is_better": True, "scaling": "strong" if args.mode == "sharded" else "weak", "vs_baseline": None, "dtype": "f32 kNN / f64 solve", "data": "synthetic",
            "config": config_block(wl, args, [float(cb["features"][0]), float(cb["features"][1])], 1, None),
            "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": cb["value"], "unit": "scans/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0,
            "wall_s": time.perf_counter() - t0}
    print(json.dumps(line))


def config_block(wl, args, feats, world, t_index_ms):
    """Same keys in both arms (the driver compares the two config dicts)."""
    if args.mode == "sharded":
        par = f"ONE scan registered by {world} GPU(s): map sharded by spatial cell (owner cells + 1.42 m / 7.07 m halo), features processed by the owner of their cell, " \
              "29 normal-equation sums all-reduced inside the solver kernel over NVLink peer memory"
    elif args.contexts > 1:
        par = f"throughput mode: {args.contexts} scans in flight per GPU ({args.contexts} contexts / host threads, one shared map snapshot), x{world} GPU(s)"
    else:
        par = f"scan-parallel x{world} (one map replica per GPU, no data-path collective)" if world > 1 else "1 GPU"
    return {"workload": WORKLOADS[wl], "pipeline": PIPE, "features_per_scan": feats, "l2": "flushed (256 MiB write) between timed steps, outside the timed regions",
            "parallelism": par, "map_index_build_ms": t_index_ms}


# ------------------------------------------------------------------------------------------------ GPU arm
def check_against_oracle(step, inputs, world_note=""):
    """The bar of the timed work: every distinct scan of this rank through the library AND through the oracle (checker) -- same feature counts, same
    ICP iteration count, pose within north_star's 1e-4 m / 1e-4 rad.  Returns the largest deviations (m, rad)."""
    from oracle import oracle as O
    mc, ms, scans, guesses, _ = inputs
    trees = (O.KdTree(mc), O.KdTree(ms))
    ex = O.Extractor()
    worst_t, worst_a = 0.0, 0.0
    for k in range(len(scans)):
        res, nc, ns = step(k)
        ost, ores, onc, ons = oracle_step(O, ex, trees, mc, ms, scans[k], guesses[k], 1)
        dt = float(np.linalg.norm(np.array(res.t_w_curr) - np.array(ores.t_w_curr)))
        da = float(S.quat_angle(np.array(res.q_w_curr), np.array(ores.q_w_curr)))
        assert res.status == ost == 1 and res.registered == 1, (k, res.status, ost, world_note)
        assert (nc, ns) == (onc, ons) and res.icp_iterations == ores.icp_iterations, (k, nc, ns, onc, ons, res.icp_iterations, ores.icp_iterations, world_note)
        assert dt < 1e-4 and da < 1e-4, (k, dt, da, world_note)
        worst_t, worst_a = max(worst_t, dt), max(worst_a, da)
    return worst_t, worst_a


def dump_outputs(out_dir, ctx, res, nc, ns):
    """What the caller of ll_scan_to_pose receives from the last timed step (pose, increment, costs and counts of the ll_reg_result, feature counts),
    plus the scan-frame feature clouds that registration matched (x, y, z, intensity), one DIR/<name>.npy each.  The inputs are seeded, so two
    builds run with the same arguments can be compared file by file."""
    from loam_livox_b200.registration import features_to_pointcloud2
    out = {"q_w_curr": np.array(res.q_w_curr), "t_w_curr": np.array(res.t_w_curr), "q_w_incre": np.array(res.q_w_incre), "t_w_incre": np.array(res.t_w_incre),
           "costs": np.array([res.initial_cost, res.final_cost, res.inlier_threshold, res.angular_diff, res.t_diff]),
           "counts": np.array([res.status, res.registered, res.num_residual_blocks, res.icp_iterations, res.corner_used, res.surf_used,
                               res.total_lm_iterations, res.total_evaluations, nc, ns], np.float64),
           "corner_features": np.frombuffer(features_to_pointcloud2(ctx, 0), np.float32).reshape(-1, 4),
           "surface_features": np.frombuffer(features_to_pointcloud2(ctx, 1), np.float32).reshape(-1, 4)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_gpu(args):
    import ctypes as C
    import torch
    import torch.distributed as dist
    from loam_livox_b200 import capi
    from loam_livox_b200.registration import Context, Map, scan_to_pose

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    sharded = args.mode == "sharded"
    wl = "c4" if sharded else "c2"
    nmc, nms = workload_sizes(wl)
    inputs = make_inputs(0 if sharded else rank, wl)      # sharded: every rank registers the SAME scans, together
    mc, ms, scans, guesses, truths = inputs
    K = max(1, args.contexts)
    ctxs = [Context(local, max_scan_points=N_SCAN, max_features=N_SCAN) for _ in range(K)]
    ctx = ctxs[0]
    if sharded and world > 1:
        from loam_livox_b200.distributed import connect
        connect(ctx, rank, world, dist)
    def build_map():
        if sharded and world > 1:
            return Map(ctx, mc, ms, rank=rank, world=world, cell_size=2.0)
        return Map(ctx, mc, ms)
    t0 = time.perf_counter()
    m = build_map()
    t_index = time.perf_counter() - t0
    t0 = time.perf_counter()
    m2 = build_map()
    t_index = min(t_index, time.perf_counter() - t0)
    m2.release()
    shard = None
    if sharded and world > 1:
        info, _ = m.shard_info()
        sz = torch.tensor([info.kept_corner, info.kept_surf], dtype=torch.int64, device="cuda")
        allsz = [torch.zeros_like(sz) for _ in range(world)]
        dist.all_gather(allsz, sz)
        shard = {"cell_size_m": 2.0, "halo_m": [2.0 ** 0.5, 50.0 ** 0.5], "total_points": [int(info.total_corner), int(info.total_surf)],
                 "kept_points_per_rank": [[int(v) for v in t.tolist()] for t in allsz]}
    pc = capi.PipelineCfg(**PIPE)
    states = [capi.default_reg_state(q_w_last=g.q, t_w_last=g.t, q_w_curr=g.q, t_w_curr=g.t) for g in guesses]
    streams = [torch.cuda.ExternalStream(c.stream(), device=local) for c in ctxs]
    stream = streams[0]
    dev_scans = [torch.from_numpy(s).cuda() for s in scans]
    pin_scans = [torch.from_numpy(s).pin_memory() for s in scans]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()

    def step_dev(k, c=None):
        return scan_to_pose(c or ctx, m, dev_scans[k].data_ptr(), 100.0 + 0.1 * k, pc, states[k], where=capi.LL_DEVICE, n=N_SCAN, fmt=capi.LL_FMT_XYZI16)

    def step_host(k, c=None):
        c = c or ctx
        res = capi.RegResult()
        nc, ns = C.c_int(), C.c_int()
        c.check(c._lib.ll_scan_to_pose(c.h, m.h, pin_scans[k].data_ptr(), N_SCAN, capi.LL_FMT_XYZI16, capi.LL_HOST, 100.0 + 0.1 * k, C.byref(pc), C.byref(states[k]),
                                       C.byref(res), C.byref(nc), C.byref(ns)))
        return res, nc.value, ns.value

    def do_flush():
        with torch.cuda.stream(stream):
            flush.zero_()

    nd = len(scans)
    for c in ctxs:
        for w in range(args.warmup):
            step_dev(w % nd, c)
            step_host(w % nd, c)
    # ---- the bar: the timed work equals the oracle's (pose, ICP iterations, feature counts) on every distinct scan of this rank
    if args.no_cpu:
        for k in range(nd):
            res, nc, ns = step_dev(k)
            assert res.status == 1 and res.registered == 1, (k, res.status)
        dev = torch.tensor([float("nan"), float("nan")], dtype=torch.float64, device="cuda")
    else:
        if sharded and world > 1:
            # the ranks must step through the scans in lock-step (the registration is collective); the oracle runs beside it on every rank
            wt, wa = check_against_oracle(step_dev, inputs, f"sharded x{world} rank {rank}")
        else:
            wt, wa = check_against_oracle(step_dev, inputs, f"rank {rank}")
        dev = torch.tensor([wt, wa], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(dev, op=dist.ReduceOp.MAX)
        dist.barrier()
    torch.cuda.synchronize()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    # ---- value: device-resident inputs, CUDA events on the context streams
    l0 = sum(c.launches() for c in ctxs)
    icp_iters, knn_ms, knn_all_ms, solve_all_ms, sel_all_ms, reg_ms, feats, blocks, evals = [], [], [], [], [], [], [], [], []

    def note(res, nc, ns):
        icp_iters.append(res.icp_iterations); knn_ms.append(res.gpu_ms_knn); reg_ms.append(res.gpu_ms_total); feats.append((nc, ns))
        knn_all_ms.append(res.gpu_ms_knn_all); solve_all_ms.append(res.gpu_ms_solve_all); sel_all_ms.append(res.gpu_ms_select_all)
        blocks.append(res.corner_used + res.surf_used); evals.append(res.total_evaluations)

    if K == 1:
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        for i in range(args.steps):
            k = i % nd
            do_flush()
            ev[i][0].record(stream)
            res, nc, ns = step_dev(k)
            ev[i][1].record(stream)
            note(res, nc, ns)
        torch.cuda.synchronize()
        total_ms = float(np.sum([a.elapsed_time(b) for a, b in ev]))
        last, last_ctx = (res, nc, ns), ctx
    else:
        # throughput mode: K host threads, one context each, all on the shared map; the device time is the span from the first start event to the
        # last end event (events of different streams of one device share a clock); the L2 cannot be flushed between steps of concurrent streams,
        # so each thread cycles through inputs + map (> 126 MB) instead
        starts = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
        ends = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
        results = [[] for _ in range(K)]
        bar = threading.Barrier(K)

        def worker(w):
            torch.cuda.set_device(local)
            bar.wait()
            starts[w].record(streams[w])
            for i in range(w, args.steps, K):
                results[w].append(step_dev(i % nd, ctxs[w]))
            ends[w].record(streams[w])
        do_flush()
        torch.cuda.synchronize()
        ths = [threading.Thread(target=worker, args=(w,)) for w in range(K)]
        for t in ths:
            t.start()
        for t in ths:
            t.join()
        torch.cuda.synchronize()
        first = min(range(K), key=lambda w: starts[0].elapsed_time(starts[w]))
        total_ms = max(starts[first].elapsed_time(e) for e in ends)
        for r in results:
            for (res, nc, ns) in r:
                note(res, nc, ns)
        w = (args.steps - 1) % K
        last, last_ctx = results[w][-1], ctxs[w]
    launches = sum(c.launches() for c in ctxs) - l0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last_ctx, *last)
    # ---- e2e: pinned host inputs through the same public call, host wall clock, H2D + result D2H inside
    if K == 1:
        e2e_s = 0.0
        for i in range(args.steps):
            k = i % nd
            do_flush()
            torch.cuda.synchronize()
            if sharded and world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            step_host(k)
            e2e_s += time.perf_counter() - t0
    else:
        bar = threading.Barrier(K + 1)

        def hworker(w):
            torch.cuda.set_device(local)
            bar.wait()
            for i in range(w, args.steps, K):
                step_host(i % nd, ctxs[w])
        ths = [threading.Thread(target=hworker, args=(w,)) for w in range(K)]
        for t in ths:
            t.start()
        do_flush()
        torch.cuda.synchronize()
        bar.wait()
        t0 = time.perf_counter()
        for t in ths:
            t.join()
        e2e_s = time.perf_counter() - t0
    torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else None
    cyc = np.zeros(16, np.int64)
    ctx.check(ctx._lib.ll_debug_solver_cycles(ctx.h, cyc.ctypes.data))
    t = torch.tensor([total_ms, e2e_s * 1e3], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, e2e_ms = float(t[0]), float(t[1])
    if rank == 0:
        peak, peak_src = peaks()
        qc = float(np.mean([f[0] for f in feats])); qs = float(np.mean([f[1] for f in feats]))
        n_iter = float(np.sum(icp_iters))
        scans_done = args.steps * (1 if sharded else world)
        # ---- roofline of the two hot kernels; the headline `roofline` is the one that takes more of the step
        knn_ms_launch = float(np.sum(knn_all_ms)) / n_iter
        solve_ms_launch = float(np.sum(solve_all_ms)) / n_iter
        q_share = 1.0 / world if (sharded and world > 1) else 1.0   # a rank of the sharded mode searches only the features it owns
        alg_knn = knn_algorithmic_bytes(qc, qs, nmc, nms) * q_share
        alg_solve = solve_algorithmic_bytes(float(np.mean(blocks)), float(np.sum(evals)) / n_iter)
        roofs = {}
        for name, alg, ms_l, what in (("knn_blocks_kernel", alg_knn, knn_ms_launch, "transform + exact 5-NN + residual blocks; one launch per ICP iteration"),
                                      ("lm_solve_kernel", alg_solve, solve_ms_launch, "solve #1 + inlier selection + solve #2 + pose; one launch per ICP iteration")):
            ach = alg / (ms_l * 1e-3) / 1e9 if ms_l > 0 else 0.0
            roofs[name] = {"bound": "hbm", "kernel": f"{name} ({what})", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": ncu_traffic(name),
                           "peak_source": peak_src, "algorithmic_bytes_per_launch": alg, "kernel_ms": ms_l, "launches_per_step": n_iter / len(icp_iters),
                           "share_of_step": ms_l * n_iter / (total_ms * (K if K > 1 else 1))}
        dominant = max(roofs, key=lambda k: roofs[k]["kernel_ms"])
        other = [k for k in roofs if k != dominant][0]
        line = {
            "metric": "scans_per_sec", "value": scans_done / (total_ms * 1e-3), "unit": "scans/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "strong" if sharded else "weak", "vs_baseline": None, "dtype": "f32 kNN / f64 solve", "data": "synthetic",
            "config": config_block(wl, args, [qc, qs], world, t_index * 1e3),
            "ms_per_icp_iter": float(np.sum(reg_ms) / max(1, n_iter)), "icp_iterations_mean": float(np.mean(icp_iters)),
            "pose_vs_oracle_max": None if args.no_cpu else {"translation_m": float(dev[0]), "rotation_rad": float(dev[1]), "bar": "1e-4 m / 1e-4 rad, same ICP iteration and feature counts, every distinct scan of every rank"},
            "clocks": clocks,
            "e2e": {"value": scans_done / (e2e_ms * 1e-3), "unit": "scans/s", "h2d_bytes_per_step": N_SCAN * 16, "d2h_bytes_per_step": int(round((np.mean(icp_iters) + 1) * ctx._lib.ll_state_snapshot_bytes() + 44)),
                    "ms_per_step": e2e_ms / args.steps},
            "gpu_launches": int(launches),
            "roofline": roofs[dominant], "roofline_other": roofs[other],
            "kernel_ms_per_step": {"knn_first_iteration": float(np.mean(knn_ms)), "knn_all": float(np.mean(knn_all_ms)), "solve_all": float(np.mean(solve_all_ms)),
                                   "select_exchange_all": float(np.mean(sel_all_ms)), "registration_total": float(np.mean(reg_ms))},
        }
        if K > 1:
            line["contexts"] = K
        if shard is not None:
            line["shard"] = shard
            ev_n = max(1, int(cyc[5]))
            mhz = (clocks or {}).get("sm_mhz") or 1965.0
            line["exchange"] = {"in_kernel_allreduce_plus_grid_reduce_us_per_evaluation": float(cyc[2]) / ev_n / mhz, "evaluations_last_registration": ev_n,
                                "l1_exchange_plus_select_us_per_icp_iteration": 1e3 * float(np.sum(sel_all_ms)) / n_iter,
                                "note": "cycle counters of the solver's master CTA over the last registration (ll_debug_solver_cycles); the all-reduce is 29 doubles per rank pushed into every peer's staging slot + one flag"}
        if not args.no_cpu:
            cb = cpu_baseline(1, args.cpu_scans, inputs)
            line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------ C3: streaming odometry (not the default line)
def run_stream(args):
    """BASELINE.json configs[2]: a synthetic sequence (stationary for the first init_accumulate_frames + 1 scans, then ~0.3 m/s with sinusoidal yaw)
    through the device mapper (ll_mapper_process_scan): features, match-map refresh (--matching-mode 0: the sliding window of the last 400 feature
    clouds, the shipped YAMLs' mode; 1: radius + FOV select from the growing cell map, per-cell VoxelGrid), whole-map VoxelGrid, index build,
    registration, append.  Raw scans come from pinned host memory; host wall clock around each call (this IS the end-to-end path).
    Leaves 0.05 / 0.1 m (denser than the precision YAML's 0.1 / 0.4 so that a scan carries several thousand features and the map grows into the
    hundreds of thousands of points).  The oracle runs the first scans of the same sequence beside it: its drift is printed next to the GPU's."""
    import torch
    from loam_livox_b200 import capi
    from loam_livox_b200.registration import Context, Laser_mapping
    n_total = args.steps + args.warmup
    init = 50 if n_total > 200 else 3                # mapping/init_accumulate_frames (50 in both YAMLs); short smoke runs start registering earlier
    LINE, PLANE = 0.05, 0.1
    poses = S.trajectory(n_scans=n_total, n_static=init + 1, speed=1.0, zero_mean_yaw=True, y0=-1.6)   # stays inside the room and between the pillar rows for all 1000 scans
    ctx = Context(0, max_scan_points=N_SCAN, max_features=N_SCAN)
    pipe = capi.PipelineCfg(pieces=3, use_piece=0, extractor_leaf_corner=LINE, extractor_leaf_surf=PLANE / 2, mapping_leaf_corner=LINE, mapping_leaf_surf=PLANE, whole_frame=1)
    gm = Laser_mapping(ctx, reg=capi.default_reg_state(mapping_init_accumulate_frames=init), pipeline=pipe, line_resolution=LINE, plane_resolution=PLANE,
                       matching_mode=args.matching_mode, maximum_history_size=400,
                       reserve_map_points=1 << 22, reserve_store_points=1 << 23)   # sized for the whole sequence: no reallocation inside the timed calls
    pin = [torch.empty((N_SCAN, 4), dtype=torch.float32).pin_memory() for _ in range(2)]
    sampler = ClockSampler(0); sampler.start()
    times, stats_last, l0, phases, checkpoints, track = [], None, 0, [], {}, []
    R0, t0w = poses[0].R(), poses[0].t
    n_cpu = 0 if args.no_cpu else min(n_total, init + 30)
    for k in range(n_total):
        raw = S.make_scan(N_SCAN, poses[k], seed=S.SEED + k)          # generated outside the timed call
        pin[k & 1].copy_(torch.from_numpy(raw))
        if k == args.warmup:
            l0 = ctx.launches()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        try:
            res, st = gm.process_new_scan(pin[k & 1].numpy(), 100.0 + 0.1 * k)   # pinned host buffer, H2D inside the call
        except Exception:
            ls = stats_last
            print(f"c3: scan {k} failed; pose {poses[k].t}; last stats: " + (f"features {ls.n_corner}+{ls.n_surf}, map {ls.map_corner}+{ls.map_surf}, appended {ls.appended_corner}+{ls.appended_surf}" if ls else "none"), file=sys.stderr)
            raise
        dt = time.perf_counter() - t0
        if k >= args.warmup:
            times.append(dt)
            phases.append((st.ms_front_end, st.ms_refresh, st.ms_register, st.ms_append))
        stats_last = st
        if args.dump_poses:
            q, t, f = gm.pose(); track.append([float(x) for x in q] + [float(x) for x in t])
        if k + 1 in (n_cpu, n_total):
            q, t, f = gm.pose()
            checkpoints[k + 1] = float(np.linalg.norm(t - R0.T @ (poses[k].t - t0w)))
            final_pose = {"scan": k + 1, "q_wxyz": [float(x) for x in q], "t": [float(x) for x in t]}
    clocks = sampler.stop()
    if args.dump_poses:
        np.save(args.dump_poses, np.array(track))
    line = {"metric": "scans_per_sec", "value": len(times) / float(np.sum(times)), "unit": "scans/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * float(np.mean(times)), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 kNN / f64 solve", "data": "synthetic",
            "config": {"workload": f"C3: streaming sequence of {n_total} 100k-pt scans, matching_mode {args.matching_mode} "
                                   f"({'history window of 400 feature clouds' if args.matching_mode == 0 else 'growing device cell map, radius + FOV select'}), match map re-indexed after every scan; leaves {LINE}/{PLANE} m",
                       "final_map_points": [stats_last.map_corner, stats_last.map_surf], "features_per_scan": [stats_last.n_corner, stats_last.n_surf],
                       "final_position_error_m": checkpoints.get(n_total), "position_error_m_at_scan": checkpoints,
                       "final_pose": final_pose, "reserved_points": {"map": 1 << 22, "store": 1 << 23}, "calls_over_20ms": int(np.sum(np.array(times) > 0.02))},
            "clocks": clocks, "e2e": {"value": len(times) / float(np.sum(times)), "unit": "scans/s", "h2d_bytes_per_step": N_SCAN * 16, "d2h_bytes_per_step": 1400},
            "gpu_launches": int(ctx.launches() - l0), "p50_ms": 1e3 * float(np.median(times)), "p99_ms": 1e3 * float(np.quantile(times, 0.99)),
            "phase_ms_median": dict(zip(("front_end", "refresh", "register", "append"), [float(x) for x in np.median(np.array(phases), axis=0)])),
            "slowest": [(int(i), round(1e3 * times[i], 2), [round(float(x), 2) for x in phases[i]]) for i in np.argsort(times)[-4:]]}
    if n_cpu:
        from oracle import oracle
        om = oracle.Mapper(oracle.default_params(mapping_init_accumulate_frames=init, num_threads=1), threads=1, line_resolution=LINE, plane_resolution=PLANE,
                           extractor_leaf_corner=LINE, extractor_leaf_surf=PLANE / 2, matching_mode=args.matching_mode, maximum_history_size=400)
        t_reg = 0.0
        for k in range(n_cpu):
            raw = S.make_scan(N_SCAN, poses[k], seed=S.SEED + k)
            t0 = time.perf_counter()
            st_o, q_o, t_o = om.process_scan(raw, 100.0 + 0.1 * k)
            if k > init:
                t_reg += time.perf_counter() - t0
        err_o = float(np.linalg.norm(t_o - R0.T @ (poses[n_cpu - 1].t - t0w)))
        line["cpu_baseline"] = {"value": max(1, n_cpu - init - 1) / max(t_reg, 1e-9), "unit": "scans/s", "cores": 1, "kind": "port",
                                "sample": f"the registered scans among the first {n_cpu} of the same sequence through oracle.Mapper (1 thread, same leaves and matching mode)"}
        line["config"]["oracle_position_error_m_at_scan"] = {n_cpu: err_o}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ C5: Mid-100 triple-lidar frames (not the default line)
def run_c5(args):
    """BASELINE.json configs[4]: 300k-pt Mid-100 frames (three Mid-40 heads yawed -25 / 0 / +25 degrees), precision-YAML resolutions (line 0.1 m, plane 0.4 m:
    extractor leaves 0.1 / 0.2, mapping leaves 0.1 / 0.4), the 20M-point map, scan-parallel over the GPUs given (one map replica each).  A step = one frame
    through ll_frame_to_pose: ONE extractor over the three heads, feature clouds summed (laser_feature_extractor.hpp:339-389), four VoxelGrids, registration.
    Inputs are resident in HBM for `value`; `e2e` passes the three heads from pinned host memory."""
    import ctypes as C
    import torch
    import torch.distributed as dist
    from loam_livox_b200 import capi
    from loam_livox_b200.registration import Context, Map, frame_to_pose
    world, rank, local = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    N_FRAME = 300_000
    mc, ms = S.make_map(N_MAP_CORNER_C4, N_MAP_SURF_C4)
    rng = np.random.default_rng(S.SEED + 500 + rank)
    frames, guesses = [], []
    for k in range(4):
        pose = S.Pose(S.quat_from_euler(0.01 * k, -0.02, 0.05 + 0.03 * k), np.array([0.3 + 0.5 * k, 0.2 - 0.1 * k, 0.1]))
        frames.append(S.make_triple_scan(N_FRAME, pose, seed=S.SEED + 1000 * rank + 10 * k))
        guesses.append(S.perturb_pose(pose, rng, dt=0.05, dang_deg=1.0))
    ctx = Context(local, max_scan_points=N_FRAME, max_features=N_FRAME)
    m = Map(ctx, mc, ms)
    pipe = dict(pieces=2, use_piece=0, extractor_leaf_corner=0.1, extractor_leaf_surf=0.2, mapping_leaf_corner=0.1, mapping_leaf_surf=0.4, whole_frame=1)
    pc = capi.PipelineCfg(**pipe)
    states = [capi.default_reg_state(q_w_last=g.q, t_w_last=g.t, q_w_curr=g.q, t_w_curr=g.t) for g in guesses]
    dev = [[torch.from_numpy(h).cuda() for h in f] for f in frames]
    pin = [[torch.from_numpy(h).pin_memory() for h in f] for f in frames]
    stream = torch.cuda.ExternalStream(ctx.stream(), device=local)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    stamps = lambda k: [100.0 + 0.1 * k + 1e-3 * h for h in range(3)]

    def step(k, host=False):
        if host:   # the three heads from pinned host memory: H2D inside the call
            return frame_to_pose(ctx, m, [t.numpy() for t in pin[k]], stamps(k), pc, states[k])
        return frame_to_pose(ctx, m, [t.data_ptr() for t in dev[k]], stamps(k), pc, states[k], where=capi.LL_DEVICE, ns=[t.shape[0] for t in dev[k]], fmt=capi.LL_FMT_XYZI16)
    nd = len(frames)
    for w in range(args.warmup):
        step(w % nd); step(w % nd, True)
    worst = [0.0, 0.0]
    if not args.no_cpu:   # the bar: same features, ICP iterations and pose as the oracle's staged flow, every distinct frame of this rank
        from oracle import oracle as O
        trees = (O.KdTree(mc), O.KdTree(ms))
        for k in range(nd):
            res, nc, ns = step(k)
            ex = O.Extractor(); oc, os_ = [], []
            for h, st_ in zip(frames[k], stamps(k)):
                ex.extract(h, st_); c, s_, _ = ex.get_features(0.0, 1.0); oc.append(c); os_.append(s_)
            fc = O.voxel_grid(O.voxel_grid(np.concatenate(oc), 0.1), 0.1); fs = O.voxel_grid(O.voxel_grid(np.concatenate(os_), 0.2), 0.4)
            ost, ores = O.register(mc, trees[0], ms, trees[1], fc, fs, O.default_params(q_w_last=guesses[k].q, t_w_last=guesses[k].t, q_w_curr=guesses[k].q, t_w_curr=guesses[k].t, num_threads=host_threads()))
            dt = float(np.linalg.norm(np.array(res.t_w_curr) - np.array(ores.t_w_curr))); da = float(S.quat_angle(np.array(res.q_w_curr), np.array(ores.q_w_curr)))
            assert (nc, ns) == (fc.shape[0], fs.shape[0]) and res.status == ost and res.icp_iterations == ores.icp_iterations and dt < 1e-4 and da < 1e-4, (k, nc, ns, dt, da)
            worst = [max(worst[0], dt), max(worst[1], da)]
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = ctx.launches()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    feats, iters = [], []
    for i in range(args.steps):
        with torch.cuda.stream(stream):
            flush.zero_()
        ev[i][0].record(stream)
        res, nc, ns = step(i % nd)
        ev[i][1].record(stream)
        feats.append((nc, ns)); iters.append(res.icp_iterations)
    torch.cuda.synchronize()
    total_ms = float(np.sum([a.elapsed_time(b) for a, b in ev]))
    launches = ctx.launches() - l0
    e2e_s = 0.0
    for i in range(args.steps):
        with torch.cuda.stream(stream):
            flush.zero_()
        torch.cuda.synchronize()
        t0 = time.perf_counter(); step(i % nd, True); e2e_s += time.perf_counter() - t0
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([total_ms, e2e_s * 1e3, worst[0], worst[1]], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    if rank == 0:
        line = {"metric": "scans_per_sec", "value": world * args.steps / (float(t[0]) * 1e-3), "unit": "scans/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": float(t[0]) / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 kNN / f64 solve", "data": "synthetic",
                "config": {"workload": "C5: Mid-100 triple-LiDAR 300k-pt frame (3 heads) vs 20M-pt map, precision-YAML resolutions (0.1 / 0.4 m)", "pipeline": pipe,
                           "features_per_scan": [float(np.mean([f[0] for f in feats])), float(np.mean([f[1] for f in feats]))], "l2": "flushed (256 MiB write) between timed steps",
                           "parallelism": f"scan-parallel x{world} (one map replica per GPU, no data-path collective)"},
                "icp_iterations_mean": float(np.mean(iters)), "pose_vs_oracle_max": None if args.no_cpu else {"translation_m": float(t[2]), "rotation_rad": float(t[3])},
                "clocks": clocks, "e2e": {"value": world * args.steps / (float(t[1]) * 1e-3), "unit": "scans/s", "h2d_bytes_per_step": N_FRAME * 16, "d2h_bytes_per_step": int((np.mean(iters) + 1) * 1400)},
                "gpu_launches": int(launches)}
        print(json.dumps(line))
    if world > 1:
        dist.barrier(); dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="c2", choices=["c2", "c3", "c5"], help="c2 = the headline line (default); c3 = streaming odometry through the device mapper; c5 = Mid-100 triple-lidar 300k-pt frames vs the 20M map")
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default="replicas", choices=["replicas", "sharded"], help="replicas = every GPU registers its own scans against its own map (default, weak scaling); "
                    "sharded = config C4: ONE scan registered by all GPUs together against the 20M-point map sharded by spatial cell (strong scaling)")
    ap.add_argument("--contexts", type=int, default=1, help="scans in flight per GPU (throughput mode: K contexts on K host threads sharing one map; the reference runs maximum_parallel_thread of them)")
    ap.add_argument("--matching-mode", type=int, default=0, choices=[0, 1], help="c3 only: mapping/matching_mode (0 = history window, the shipped YAMLs' mode; 1 = cell map)")
    ap.add_argument("--dump-poses", default=None, help="c3 only: write the pose after every scan (q_wxyz, t) to this .npy (diagnostics: first scan at which GPU and oracle part)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--cpu-scans", type=int, default=5)
    ap.add_argument("--dump-outputs", default=None, metavar="DIR", help="--workload c2 (either --mode) only: after the timed steps, write what "
                    "the last one returned (pose, increment, costs, counts, feature clouds) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.workload != "c2"):
        ap.error("--dump-outputs writes the outputs of the GPU registration path (--impl ours, --workload c2)")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "c3":
        run_stream(args)
    elif args.workload == "c5":
        run_c5(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
