#!/usr/bin/env python
"""bench.py -- headline benchmark of the BoundPlanner geometry core on B200.

Workload (BASELINE.json configs[1], "C2"): synthetic 1k random box obstacles,
256 seeds per GPU, set inflation (find_set_around_point, fixed_mid=True,
optimize=True) + all-pairs set-graph build (tol 0.01).  One "step" = one pass of
that hot path over the seed batch.  Metric: convex sets built per second
(whole job), with set-pair checks/s alongside.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

N > 1 is launched by torchrun (one rank per GPU): every rank builds its own 256
seeds over the replicated scene (weak scaling), the sets are exchanged by peer
stores over NVLink and the global pair matrix is split in balanced row blocks.

Besides the headline line's contract keys (value, e2e, roofline, cpu_baseline,
clocks, gpu_launches) the line carries
  stages_ms   per-stage device time of one step (max over ranks at N > 1)
  saturated   the same set build with 2048 seeds in one launch (chip filled)
  c3 / c4 / c5  the other BASELINE configs: batched planning queries (queries/s,
              p50/p95 latency over ALL queries), the 10k-obstacle / 2048-seed graph
              (strong scaling over the ranks), the MPC step geometry (us per step)
  adjacency_equals_single_rank   (N > 1) the exchanged global graph re-tested by
              rank 0 alone, outside the timed region

--dump-outputs DIR saves the results of the last timed step as .npy files.  The
inputs are seeded, so two builds run with the same arguments can be compared
output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_OBS = 1000
N_SEEDS = 256           # per GPU
TOL = 0.01
METRIC = "convex_sets_built_per_sec"
UNIT = "sets/s"
WORKLOAD = ("C2: 1000 random box obstacles (edge U[0.02,0.08], inflate 0.01), 256 seeds/GPU, IRIS loop fixed_mid + "
            "all-pairs set graph tol 0.01")
PAIRS_PER_SET = (N_SEEDS - 1) / 2.0        # 32 640 pairs / 256 sets on one GPU


def config_dict(world):
    """the same dict in both arms (the driver compares them)"""
    return {"workload": WORKLOAD, "n_obstacles": N_OBS, "seeds_per_gpu": N_SEEDS,
            "pairs_per_set": PAIRS_PER_SET if world == 1 else (N_SEEDS * world - 1) / 2.0,
            "l2": "flushed between timed steps (256 MiB fill)"}


# ----------------------------------------------------------------------------
# clocks sampler (nvidia-smi during the timed region)
# ----------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu_index = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                 "-i", str(self.gpu_index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for nm, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------
# CPU arm: the oracle port of the reference's Python path on a persistent process pool
# ----------------------------------------------------------------------------
_FINDER = None


def _pool_init(boxes, inflate, ws_min, ws_max):
    """runs once in every worker: the scene is ingested here, outside any timed region"""
    global _FINDER
    from oracle.convex_set_finder import ConvexSetFinder
    from oracle.obstacles import obstacle_reps

    obs_sets, pts, _ = obstacle_reps(boxes, inflate)
    _FINDER = ConvexSetFinder(obs_sets, pts, ws_max, ws_min, max_rows=None)


def _pool_build(seed):
    """find_set_around_point (ConvexSetFinder.py:190-240) for one seed; None when the reference would raise"""
    try:
        A, b, _, _ = _FINDER.find_set_around_point(seed, fixed_mid=True, optimize=True)
        return [A, b]
    except (RuntimeError, ValueError):
        return None


def _pool_pairs(chunk):
    """the reference's set_intersection call (BoundPlanner.py:774-787) for a chunk of set pairs"""
    from oracle.set_graph import set_intersection

    return [bool(set_intersection(s1, s2, TOL)[2]) for s1, s2 in chunk]


class CpuArm:
    """The reference's CPU path (oracle port: vectorised NumPy closest points + barrier MVIE, SciPy/HiGHS pair
    LPs) over `cores` persistent worker processes.  One step = `n_seeds` sets built + the GPU arm's ratio of
    pair checks per set (127.5 at one GPU), against the sets built before."""

    def __init__(self, cores):
        import multiprocessing as mp

        from boundplanner_b200 import scenes

        self.cores = cores
        self.boxes, self.inflate, self.seeds, self.ws_min, self.ws_max = scenes.config_c2(N_OBS, N_SEEDS)
        self.pool = mp.get_context("fork").Pool(cores, initializer=_pool_init,
                                                initargs=(self.boxes, self.inflate, self.ws_min, self.ws_max)) if cores > 1 else None
        if self.pool is None:
            _pool_init(self.boxes, self.inflate, self.ws_min, self.ws_max)
        self.sets = []              # every set built so far (pair partners)
        self.cursor = 0

    def step(self, n_seeds):
        """returns (seconds, sets built, pair checks)"""
        sel = [self.seeds[(self.cursor + k) % N_SEEDS] for k in range(n_seeds)]
        self.cursor += n_seeds
        t0 = time.perf_counter()
        built = self.pool.map(_pool_build, sel, chunksize=1) if self.pool else [_pool_build(s) for s in sel]
        built = [s for s in built if s is not None]
        want = int(round(len(built) * PAIRS_PER_SET))
        pairs = []
        partners = self.sets + built
        for a, s in enumerate(built):                # newest sets first, like add_edges walks the graph's nodes
            me = len(self.sets) + a
            for j in range(me - 1, -1, -1):
                if len(pairs) >= (a + 1) * want // max(len(built), 1):
                    break
                pairs.append((s, partners[j]))
        if self.pool:
            n_chunks = self.cores * 4
            chunks = [pairs[k::n_chunks] for k in range(n_chunks) if pairs[k::n_chunks]]
            res = self.pool.map(_pool_pairs, chunks, chunksize=1)
        else:
            res = [_pool_pairs(pairs)]
        dt = time.perf_counter() - t0
        self.sets.extend(built)
        return dt, len(built), sum(len(r) for r in res)

    def close(self):
        if self.pool:
            self.pool.close()
            self.pool.join()


def cpu_measure(cores, n_seeds, steps, warmup, partner_sets=None):
    arm = CpuArm(cores)
    # partners for the pair checks: enough sets that the first timed step already finds 127.5 per new set
    # (untimed: sets handed in by the caller, else built here)
    need = int(PAIRS_PER_SET) + 1
    if partner_sets:
        arm.sets.extend(partner_sets[:need])
    while len(arm.sets) < need:
        arm.step(min(n_seeds, need))
    for _ in range(warmup):
        arm.step(n_seeds)
    tot_t = tot_sets = tot_pairs = 0
    for _ in range(steps):
        t, ns, npairs = arm.step(n_seeds)
        tot_t += t
        tot_sets += ns
        tot_pairs += npairs
    arm.close()
    return tot_t, tot_sets, tot_pairs


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path.  The true reference cannot run here
    (casadi / cvxpy / cdd / pinocchio absent, no network), so this is the oracle port (kind "port") on all host
    cores, a bounded sample of the same workload per step: 2 seeds per core + 127.5 pair checks per set."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = min(os.cpu_count() or 1, 32)
    per_step = 2 * cores
    tot_t, tot_sets, tot_pairs = cpu_measure(cores, per_step, args.steps, min(args.warmup, 2))
    value = tot_sets / tot_t
    sample = (f"{per_step} of the {N_SEEDS} C2 seeds + {int(round(per_step * PAIRS_PER_SET))} pair checks per step "
              f"(the GPU arm's {PAIRS_PER_SET} pairs per set), oracle port (vectorised NumPy + barrier MVIE, "
              f"scipy linprog/HiGHS per pair) on a persistent pool of {cores} processes; scene ingest and pool "
              "start outside the timed region")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_dict(1),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "pair_checks_per_sec": tot_pairs / tot_t, "sets_timed": tot_sets, "pairs_timed": tot_pairs,
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------
def run_gpu(args):
    import torch
    import torch.distributed as dist

    from boundplanner_b200 import _lib, distributed as bpd, geometry as geo, scenes

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    _lib.load()

    # same scene on every rank, per-rank seeds (weak scaling: 256 seeds per GPU)
    boxes, inflate, seeds0, ws_min, ws_max = scenes.config_c2(N_OBS, N_SEEDS)
    if rank == 0:
        seeds = seeds0
    else:
        seeds = scenes.free_points(N_SEEDS, boxes, inflate, np.random.default_rng(100 + rank), ws_min, ws_max)
    scene = geo.Scene(boxes, inflate)
    seeds_host = torch.as_tensor(seeds).pin_memory()
    seeds_dev = seeds_host.cuda()
    S_total = N_SEEDS * world

    def pair_fn(A, b, m, tol, r0, r1):
        return geo.pair_feasible(A, b, m, tol, r0, r1)

    # single GPU: static buffers + one CUDA graph per step (boundplanner_b200/pipeline.py);
    # multi GPU: one CUDA graph per rank with the exchange by peer stores (or the NCCL all-gather pipeline)
    pipe = None
    if world == 1 and not args.no_cuda_graph:
        from boundplanner_b200.pipeline import SetGraphPipeline

        pipe = SetGraphPipeline(scene, N_SEEDS, ws_min, ws_max, fixed_mid=True, optimize=True, tol=TOL)
        pipe.seeds_dev.copy_(seeds_dev)

    spipe = None
    peer_note = None
    if world > 1 and not args.no_cuda_graph:
        from boundplanner_b200.pipeline import PeerSetGraphPipeline, ShardedSetGraphPipeline

        if os.environ.get("BPGEO_PEER", "1") != "0":
            try:
                spipe = PeerSetGraphPipeline(scene, N_SEEDS, ws_min, ws_max, fixed_mid=True, optimize=True, tol=TOL)
            except Exception as e:  # noqa: BLE001
                peer_note = f"symmetric memory unavailable ({type(e).__name__}): NCCL pipeline"
                spipe = None
        if spipe is None:
            spipe = ShardedSetGraphPipeline(scene, N_SEEDS, ws_min, ws_max, fixed_mid=True, optimize=True, tol=TOL)
        spipe.seeds_dev.copy_(seeds_dev)
    is_peer = type(spipe).__name__ == "PeerSetGraphPipeline"

    def step_device(seeds_d):
        if pipe is not None:
            return pipe.run_device()
        if spipe is not None:
            if seeds_d is not spipe.seeds_dev and seeds_d is not seeds_dev:
                spipe.seeds_dev.copy_(seeds_d)
            return spipe.run_device()
        out = geo.build_sets_point(scene, seeds_d, ws_min, ws_max, fixed_mid=True, optimize=True)
        bits, _ = bpd.sharded_adjacency(out.A, out.b, out.m, pair_fn, TOL)
        return out, bits

    e2e_host = []

    def step_e2e():
        if pipe is not None:
            return pipe.run(seeds_host)                              # H2D seeds, graph replay, D2H results
        sd = seeds_host.cuda(non_blocking=True)                      # H2D of the step's inputs
        out, bits = step_device(sd)
        srcs = (out.A, out.b, out.m, out.q_ellipse, out.p_mid, out.status, bits)
        if not e2e_host:                                             # pinned mirrors, allocated once
            e2e_host.extend(torch.empty(t.shape, dtype=t.dtype, pin_memory=True) for t in srcs)
        for h, t in zip(e2e_host, srcs):                             # D2H of every result, one synchronize
            h.copy_(t, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return e2e_host

    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device="cuda")   # 256 MiB > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    warm = max(args.warmup, 3)
    for _ in range(warm):
        out, bits = step_device(seeds_dev)
    barrier()

    # ---- timed region: K steps, device-resident inputs, L2 flushed between steps
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    for k in range(args.steps):
        flush.fill_(float(k))
        ev[k][0].record()
        out, bits = step_device(seeds_dev)
        ev[k][1].record()
    barrier()
    dev_ms = sum(a.elapsed_time(b) for a, b in ev)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        # before the end-to-end and per-stage runs below, which write into the same buffers
        dump_outputs(args.dump_outputs, out, spipe.adjacency_bits() if spipe is not None else bits, S_total, geo,
                     world, rank, dist)

    # ---- end to end through the public API with host buffers
    for _ in range(2):
        step_e2e()
    e2e_depth = 1
    if pipe is not None and os.environ.get("BPGEO_E2E_DEPTH", "2") != "1":
        # two pipeline objects used round-robin: every step still copies its seeds in and all its results out, but
        # the D2H of step k (copy stream) overlaps step k+1 and the host does not synchronize per step
        from boundplanner_b200.pipeline import PipelinedSetGraph

        e2e_depth = 2
        ps = PipelinedSetGraph(scene, N_SEEDS, ws_min, ws_max, depth=e2e_depth, fixed_mid=True, optimize=True, tol=TOL)
        for _ in range(4):
            ps.take()
            ps.put(seeds_host)
        ps.drain()
        barrier()
        t0 = time.perf_counter()
        for k in range(args.steps):
            got = ps.take()                      # results of step k - 2, delivered in pinned host memory
            if got is not None:
                res = got
            ps.put(seeds_host)
        res = ps.drain()[-1]
        barrier()
        e2e_s = time.perf_counter() - t0
    else:
        barrier()
        t0 = time.perf_counter()
        for k in range(args.steps):
            res = step_e2e()
        barrier()
        e2e_s = time.perf_counter() - t0
    h2d = seeds_host.numel() * 8
    d2h = sum(t.numel() * t.element_size() for t in res)

    # ---- per-stage breakdown of one step (eager launches, CUDA events between the stages; outside the timed region)
    stages = None
    if pipe is not None or is_peer:
        stages = (pipe or spipe).stage_times(reps=7)
        if world > 1:
            keys = sorted(stages)
            tt = torch.tensor([stages[k] for k in keys], dtype=torch.float64, device="cuda")
            tmax, tmin = tt.clone(), tt.clone()
            dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
            dist.all_reduce(tmin, op=dist.ReduceOp.MIN)
            stages = {k: {"max": tmax[i].item(), "min": tmin[i].item()} for i, k in enumerate(keys)}

    # ---- N > 1: the exchanged global graph, re-tested by rank 0 alone from the global set tables
    adj_equal = None
    if world > 1 and spipe is not None:
        gbits = spipe.adjacency_bits().clone()
        if is_peer:
            Ag, bg, mg = spipe.Ag, spipe.bg, spipe.mg
        else:
            Ag, bg, mg = spipe.Ag, spipe.bg, spipe.mg
        if rank == 0:
            single = geo.pair_feasible(Ag, bg, mg, TOL)
            adj_equal = bool(torch.equal(single, gbits))
        # every rank's local sets are what the global table holds at its slot
        own = torch.equal(Ag[rank * N_SEEDS: (rank + 1) * N_SEEDS], out.A)
        flag = torch.tensor([1.0 if own else 0.0], device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if rank == 0:
            adj_equal = adj_equal and bool(flag.item() == 1.0)

    # ---- per-kernel timing of the dominant kernels (roofline), CUDA events on the launch stream
    prof = kernel_profile(geo, scene, seeds_dev, ws_min, ws_max, out, torch) if rank == 0 else None

    # ---- the other BASELINE configs (outside the headline's timed region)
    extras = {}
    if not args.no_extras:
        extras["c3"] = bench_c3(args, world, rank, dist, torch)
        extras["c4"] = bench_c4(args, world, rank, dist, torch, geo, scenes)
        if rank == 0:
            extras["c5"] = bench_c5(torch, geo, scenes)

    if world > 1:
        tt = torch.tensor([dev_ms, e2e_s], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dev_ms, e2e_s = tt[0].item(), tt[1].item()
    status = out.status.cpu().numpy()
    mrows = out.m.cpu().numpy()
    n_pairs = S_total * (S_total - 1) // 2
    value = S_total * args.steps / (dev_ms * 1e-3)
    fused = os.environ.get("BPGEO_FUSED", "1") != "0"
    # fused: k_iris_fused (boxes and peer stores in its epilogue) + filter + lp;  else state_init, 5x(poly,mvie),
    # final mvie, export, aabb + filter + lp
    launches_per_step = (1 + 2) if fused else (1 + 5 * 2 + 1 + 1 + 3)
    if is_peer:
        launches_per_step += 1 if fused else 2      # the adjacency-row scatter (+ the set scatter when not fused)
    tail_mode = bool(getattr(pipe if pipe is not None else spipe, "tail", False))
    if tail_mode:
        launches_per_step = 3                       # k_step_begin, k_step_epoch, k_iris_fused (build + exchange + pairs)
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        which = "measured" if "hbm_gbs" in peaks else "fallback"
        launch = (("one CUDA graph per step; pair tests in the tail of the set-build kernel" if tail_mode else
                   "one CUDA graph per step") if pipe is not None else
                  ("one CUDA graph per step and rank: set build, exchange by peer stores + per-set arrival flags over "
                   "NVLink and pair tests in ONE kernel, one signal-pad barrier per step (no NCCL on the data path)"
                   + ("" if getattr(spipe, "_graph", None) is not None else " [eager: capture refused]"))
                  if is_peer and tail_mode else
                  ("one CUDA graph per step; sets and adjacency rows exchanged by peer stores over NVLink + two "
                   "signal-pad barriers (no NCCL on the data path)"
                   + ("" if getattr(spipe, "_graph", None) is not None else " [eager: capture refused]"))
                  if is_peer else
                  "two CUDA graphs + two NCCL all-gathers per step" if spipe is not None else "eager launches")
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": warm, "ms_per_step": dev_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_dict(world),
            "run": {"pairs": n_pairs, "launch": launch, "peer_note": peer_note,
                    "frac_sets_over_20_rows": float((mrows > 20).mean()),
                    "frac_status_ok": float((status == 0).mean()),
                    "adjacency_density": float(geo.unpack_adjacency(
                        spipe.adjacency_bits() if spipe is not None else bits, S_total).sum().item())
                    / max(n_pairs, 1)},
            "pair_checks_per_sec": n_pairs * args.steps / (dev_ms * 1e-3),
            "e2e": {"value": S_total * args.steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "steps_in_flight": e2e_depth},
            "gpu_launches": launches_per_step * args.steps,
            "clocks": clocks,
            "stages_ms": stages,
            "roofline": prof["roofline"](),
            "roofline_fk": prof["roofline_fk"](hbm_peak, which),
            "saturated": prof["saturated"],
            "kernels": prof["kernels"],
        }
        if adj_equal is not None:
            line["adjacency_equals_single_rank"] = adj_equal
        line.update(extras)
        if world == 1 and not args.no_plan_latency:
            line["plan_latency"] = plan_latency(not args.no_cpu_baseline)
        # CPU baseline on a bounded sample of the same workload (rank 0, N=1 only): the reference arm's routine
        if world == 1 and not args.no_cpu_baseline:
            cores = min(os.cpu_count() or 1, 32)
            per_step = 2 * cores
            gsets = [[a.copy(), b.copy()] for a, b in out.to_sets()]      # pair partners (untimed)
            t, ns, npairs = cpu_measure(cores, per_step, 6, 1, gsets)
            line["cpu_baseline"] = {
                "value": ns / t, "unit": UNIT, "cores": cores, "kind": "port",
                "sample": f"6 steps of {per_step} C2 seeds + {int(round(per_step * PAIRS_PER_SET))} pair checks each "
                          f"({ns} sets, {npairs} pairs), oracle port on a persistent pool of {cores} processes "
                          "(the routine of --impl reference)"}
            t1, ns1, np1 = cpu_measure(1, 6, 1, 0, gsets)
            line["cpu_baseline"]["one_core_sets_per_sec"] = ns1 / t1
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


DUMP_LIMIT = 64_000_000      # bytes, all files written by --dump-outputs together


def dump_outputs(out_dir, out, bits, S_total, geo, world, rank, dist):
    """What the last timed step handed its callers, one .npy per array: the sets of every rank's seeds in rank
    order (halfspaces padded to m_max rows, row counts, ellipsoids, centres, status) and the global adjacency
    matrix (upper triangle, 0/1).  Integer arrays are stored as float64, which holds them exactly.  When the dense
    adjacency would take the files over DUMP_LIMIT, a fixed, seeded sample of its rows is stored instead and
    adjacency_rows.npy lists their indices.  Every rank calls this (the sets are gathered); rank 0 writes."""
    import torch

    arrays = {}
    for name in ("A", "b", "m", "q_ellipse", "p_mid", "status"):
        t = getattr(out, name).contiguous()
        if world > 1:
            parts = [torch.empty_like(t) for _ in range(world)]
            dist.all_gather(parts, t)
            t = torch.cat(parts)
        arrays[name] = t.cpu().numpy().astype(np.float64)
    if rank != 0:
        return
    adj = geo.unpack_adjacency(bits, S_total)
    room = DUMP_LIMIT - sum(a.nbytes for a in arrays.values()) - 8 * 4096       # 4 KiB per file for .npy headers
    if S_total * S_total * 4 > room:
        rows = np.sort(np.random.default_rng(0).choice(S_total, room // (S_total * 4 + 8), replace=False))
        arrays["adjacency_rows"] = rows.astype(np.float64)
        adj = adj[torch.as_tensor(rows, device=adj.device)]
    arrays["adjacency"] = adj.cpu().numpy().astype(np.float32)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


# ----------------------------------------------------------------------------
# C3: batched planning queries (BASELINE configs[2]) -- queries sharded over the ranks, no communication
# ----------------------------------------------------------------------------
def bench_c3(args, world, rank, dist, torch):
    from scipy.spatial.transform import Rotation as R

    from boundplanner_b200 import scenes
    from boundplanner_b200.planner import plan_batch
    from boundplanner_b200.planner_native import NativePlanner

    nq = args.c3_queries
    r0 = R.from_euler("XYZ", [0, 90, 0], degrees=True).as_matrix()
    ids = list(range(rank * nq, (rank + 1) * nq))
    queries = []
    for i in ids:
        ob, infl, st, en, wmin, wmax = scenes.config_c3_query(i)
        queries.append(dict(obstacles=ob, start=st, end=en, r0=r0, r1=r0))
    wmin, wmax = list(wmin), list(wmax)
    # the native lock-step driver (bp_plan_run): per-query loop in C++, one kernel chain per round
    NativePlanner(queries[:8], 0.01, wmax, wmin).run(ids[:8])               # warm-up (module load, pinned arenas)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    planner = NativePlanner(queries, 0.01, wmax, wmin)                      # scene batch upload + device tables
    results, stats = planner.run(ids)
    torch.cuda.synchronize()
    dt_ingest = time.perf_counter() - t0
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    results, stats = planner.run(ids)                                       # scenes resident in HBM
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    lat = np.asarray(stats["finish_ms"], float)
    ok = np.array([not isinstance(r, Exception) for r in results])
    # the Python lock-step driver over the same kernels on the first queries of this rank: speed and equality
    n_py = min(32, nq)
    plan_batch(queries[:4], 0.01, wmax, wmin, rng_seeds=ids[:4])
    t0 = time.perf_counter()
    want, _ = plan_batch(queries[:n_py], 0.01, wmax, wmin, rng_seeds=ids[:n_py])
    dt_py = time.perf_counter() - t0
    same = 0
    for w, g in zip(want, results[:n_py]):
        if isinstance(w, Exception):
            same += int(isinstance(g, Exception) and type(g) is type(w))
        else:
            same += int((not isinstance(g, Exception)) and g["path"] == w["path"] and g["set_ids"] == w["set_ids"] and
                        float(np.abs(g["p_via"] - w["p_via"]).max()) < 1e-9)
    if world > 1:
        tt = torch.tensor([dt, dt_ingest], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt, dt_ingest = tt[0].item(), tt[1].item()
        lat_all = [torch.zeros(nq, dtype=torch.float64, device="cuda") for _ in range(world)]
        dist.all_gather(lat_all, torch.as_tensor(lat, device="cuda"))
        lat = torch.cat(lat_all).cpu().numpy()
        okc = torch.tensor([float(ok.sum()), float(same)], dtype=torch.float64, device="cuda")
        dist.all_reduce(okc)
        n_ok, same = int(okc[0].item()), int(okc[1].item())
    else:
        n_ok = int(ok.sum())
    return {"what": "C3: independent planning queries over 200-obstacle scenes, plan_convex_set_path up to the planned "
                    "set sequence; native lock-step driver (bp_plan_run: per-query loop in C++, one kernel chain + one "
                    "H2D + one D2H per round); queries sharded over the ranks, no communication",
            "queries_per_gpu": nq, "queries": nq * world, "plan_queries_per_sec": nq * world / dt, "seconds": dt,
            "plan_queries_per_sec_incl_scene_ingest": nq * world / dt_ingest,
            "latency_ms_p50": float(np.percentile(lat, 50)), "latency_ms_p95": float(np.percentile(lat, 95)),
            "latency_over": "all queries incl. the reference's error exits (completion time inside the lock-step batch)",
            "success_fraction": n_ok / (nq * world), "rounds_rank0": stats["rounds"],
            "kernel_chains_rank0": stats["kernel_chains"], "device_wait_ms_rank0": stats["device_wait_ms"],
            "python_driver": {"what": "planner.plan_batch (Python generators, same kernels) on the first queries of "
                                      "every rank", "queries_per_rank": n_py, "queries_per_sec_one_gpu": n_py / dt_py,
                              "results_identical_to_native": f"{same} of {n_py * world}"}}


# ----------------------------------------------------------------------------
# C4: 10k obstacles, 2048 seeds, full intersection graph (BASELINE configs[3]); strong scaling over the ranks
# ----------------------------------------------------------------------------
def bench_c4(args, world, rank, dist, torch, geo, scenes):
    boxes, inflate, seeds, ws_min, ws_max = scenes.config_c4()
    S = seeds.shape[0]
    scene = geo.Scene(boxes, inflate)
    reps = 5
    if world == 1:
        from boundplanner_b200.pipeline import SetGraphPipeline

        pipe = SetGraphPipeline(scene, S, ws_min, ws_max, fixed_mid=True, optimize=True, tol=TOL)
        pipe.seeds_dev.copy_(torch.as_tensor(seeds).cuda())
        run = pipe.run_device
        st_fn = pipe.stage_times
        mode = "one CUDA graph"
    else:
        from boundplanner_b200.pipeline import PeerSetGraphPipeline

        s_loc = S // world
        pipe = PeerSetGraphPipeline(scene, s_loc, ws_min, ws_max, fixed_mid=True, optimize=True, tol=TOL)
        pipe.seeds_dev.copy_(torch.as_tensor(seeds[rank * s_loc: (rank + 1) * s_loc]).cuda())
        run = pipe.run_device
        st_fn = pipe.stage_times
        mode = "one CUDA graph per rank, peer stores over NVLink"
    for _ in range(3):
        run()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if world > 1:
            dist.barrier()
        a.record()
        run()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    ms = statistics.median(ts)
    stages = st_fn(reps=3)
    if world > 1:
        tt = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms = tt.item()
        keys = sorted(stages)
        sv = torch.tensor([stages[k] for k in keys], dtype=torch.float64, device="cuda")
        dist.all_reduce(sv, op=dist.ReduceOp.MAX)
        stages = {k: sv[i].item() for i, k in enumerate(keys)}
        bits = pipe.adjacency_bits()
        status = pipe.batch.status
        mrows = pipe.batch.m
    else:
        bits = pipe.bits
        status = pipe.batch.status
        mrows = pipe.batch.m
    n_pairs = S * (S - 1) // 2
    edges = int(geo.unpack_adjacency(bits, S).sum().item())
    return {"what": "C4: 10 000 obstacles (shelf plates + clutter), 2048 seeds, full 2 096 128-pair graph; the seeds are "
                    "split over the ranks (strong scaling), sets exchanged into the global graph",
            "n_obstacles": int(boxes.shape[0]), "seeds": S, "ms_per_step": ms, "sets_per_sec": S / (ms * 1e-3),
            "pair_checks_per_sec": n_pairs / (ms * 1e-3), "stages_ms": stages, "launch": mode,
            "edges": edges, "frac_status_ok_rank0": float((status == 0).double().mean().item()),
            "frac_over_20_rows_rank0": float((mrows > 20).double().mean().item())}


# ----------------------------------------------------------------------------
# C5: the geometry of one MPC step (BASELINE configs[4]): 12 FK evaluations + 6 line sets (BoundMPC.py:480-496)
# plus the loop's own forward_kinematics(q, dq) (MPCNode.py:118)
# ----------------------------------------------------------------------------
def bench_c5(torch, geo, scenes):
    import boundplanner_b200 as bp
    from boundplanner_b200 import mpc_geometry

    boxes, ws_min, ws_max, _ = scenes.example_scene()
    scene = geo.Scene(boxes, 0.0)                                   # obs_size_increase = 0.0 in the MPC (BoundMPC.py:265)
    q_a = np.array([0, 0, 0, -np.pi / 2, 0, np.pi / 2, 0.0])        # boundplanner_with_mpc_example.py:20-26
    q_b = q_a + np.array([0.6, 0.4, -0.3, 0.5, 0.2, -0.4, 0.3])
    n = 200
    traj = [q_a + (q_b - q_a) * 0.5 * (1 - np.cos(np.pi * k / (n - 1))) for k in range(n + 10)]
    model = bp.RobotModel()
    for k in range(5):
        mpc_geometry.collision_sets(scene, traj[k], traj[k + 10], ws_min, ws_max)
        model.forward_kinematics(traj[k], traj[k + 1] - traj[k])
    torch.cuda.synchronize()
    lat = []
    for k in range(n):
        t0 = time.perf_counter()
        p_lie, jac, djac = model.forward_kinematics(traj[k], (traj[k + 1] - traj[k]) / 0.1)       # MPCNode.py:118
        a_sets, b_sets, coll = mpc_geometry.collision_sets(scene, traj[k], traj[k + 10], ws_min, ws_max)
        lat.append((time.perf_counter() - t0) * 1e6)
    # the same geometry for a whole horizon sweep in one batch (T = 200 (q0, qf) pairs): device-side rate
    q0 = np.array(traj[:n])
    qf = np.array(traj[10: n + 10])
    mpc_geometry.collision_sets(scene, q0, qf, ws_min, ws_max)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(5):
        mpc_geometry.collision_sets(scene, q0, qf, ws_min, ws_max)
    torch.cuda.synchronize()
    batched_us = (time.perf_counter() - t0) / 5 / n * 1e6
    # the replanning call of the receding-horizon loop (plan_convex_set_path(replanning=True, p_horizon=...),
    # BoundPlanner.py:231-276) up to the planned set sequence, from points along the first plan
    from scipy.spatial.transform import Rotation as R

    from boundplanner_b200.planner import GpuBackend, SetSequencePlanner

    boxes_p, wmin_p, wmax_p, infl_p = scenes.example_scene()
    r0 = R.from_euler("XYZ", [0, 90, 0], degrees=True).as_matrix()
    p0, p1 = np.array([0.3, 0.0, 0.7]), np.array([0.45, -0.5, 0.2])
    pl = SetSequencePlanner(boxes_p, infl_p, list(wmax_p), list(wmin_p), rng=np.random.default_rng(0),
                            backend=GpuBackend(boxes_p, infl_p, list(wmax_p), list(wmin_p)))
    first = pl.plan_set_sequence(p0.copy(), p1.copy(), r0, r0)
    pv = first["p_via"]
    replan_ms = []
    for frac in (0.02, 0.1, 0.2, 0.3, 0.4, 0.5):
        start = pv[0] + frac * (pv[1] - pv[0])
        horizon = np.array([start + ti * (pv[1] - start) for ti in np.linspace(0.05, 0.6, 8)])
        t0 = time.perf_counter()
        try:
            pl.plan_set_sequence(start.copy(), p1.copy(), r0, r0, replanning=True, p_horizon=horizon)
        except (RuntimeError, ValueError):
            pass
        replan_ms.append((time.perf_counter() - t0) * 1e3)
    # per-call latency of the drop-ins an UNCHANGED planner would hit one call at a time (host arrays in, host
    # arrays out): ConvexSetFinder.find_set_around_point / find_set_collision_avoidance, set_intersection, fk_pos_col
    from boundplanner_b200.planner import obstacle_sets
    from boundplanner_b200.utils import obstacle_points_sets

    obs_sets = obstacle_sets(boxes_p, infl_p)
    finder = bp.ConvexSetFinder(obs_sets, obstacle_points_sets(obs_sets), list(wmax_p), list(wmin_p))
    pts = scenes.free_points(24, boxes_p, infl_p, np.random.default_rng(3), wmin_p + 0.05, wmax_p - 0.05)

    def p50_us(fn, n):
        fn(0)
        ts = []
        for k in range(n):
            t0 = time.perf_counter()
            fn(k)
            ts.append((time.perf_counter() - t0) * 1e6)
        return float(np.percentile(ts, 50))

    sets_h = [finder.find_set_around_point(pts[k], fixed_mid=True)[:2] for k in range(8)]
    dropin = {
        "find_set_around_point": p50_us(lambda k: finder.find_set_around_point(pts[k % 24], fixed_mid=True), 24),
        "find_set_collision_avoidance": p50_us(lambda k: finder.find_set_collision_avoidance(
            pts[k % 24], pts[k % 24] + np.array([0.03, -0.02, 0.02]), True), 24),
        "set_intersection": p50_us(lambda k: bp.set_intersection(sets_h[k % 8], sets_h[(k + 3) % 8], 0.01), 24),
        "fk_pos_col": p50_us(lambda k: model.fk_pos_col(traj[k % n], k % 6), 24),
    }
    return {"replan_ms_p50": float(np.percentile(replan_ms, 50)), "replans": len(replan_ms),
            "dropin_call_us_p50": dropin,
            "what": "C5: geometry of one MPC step through the drop-in API from host arrays -- forward_kinematics(q, dq) "
                    "+ 12 FK evaluations + 6 find_set_collision_avoidance(limit_space=True, e_max=0.7) over the 12 "
                    "example obstacles, results back on the host; replan_ms = plan_set_sequence(replanning=True, p_horizon) on "
                    "the C1 scene from points along the first plan",
            "steps": n, "us_per_mpc_step_p50": float(np.percentile(lat, 50)),
            "us_per_mpc_step_p95": float(np.percentile(lat, 95)),
            "us_per_mpc_step_batched_200": batched_us}


def plan_latency(with_cpu):
    """p50 plan latency (BASELINE.json metric, third part): SetSequencePlanner.plan_set_sequence -- the
    reference's plan_convex_set_path up to the planned set sequence -- one query at a time (every primitive a
    batch-of-one kernel call) on the C1 example and on the first 24 C3 queries, failures included."""
    from scipy.spatial.transform import Rotation as R

    from boundplanner_b200 import scenes
    from boundplanner_b200.planner import GpuBackend, SetSequencePlanner

    r0 = R.from_euler("XYZ", [0, 90, 0], degrees=True).as_matrix()

    def cases():
        boxes, ws_min, ws_max, inflate = scenes.example_scene()
        yield "C1", boxes, inflate, np.array([0.3, 0.0, 0.7]), np.array([0.45, -0.5, 0.2]), ws_min, ws_max, 0
        for i in range(24):
            ob, infl, st, en, wmin, wmax = scenes.config_c3_query(i)
            yield f"C3[{i}]", ob, infl, st, en, wmin, wmax, i

    def run(backend_factory, names=None, reps=2):
        lat = {}
        for name, ob, infl, st, en, wmin, wmax, seed in cases():
            if names is not None and name not in names:
                continue
            backend = backend_factory(ob, infl, list(wmax), list(wmin))
            for rep in range(reps):
                planner = SetSequencePlanner(ob, infl, list(wmax), list(wmin), backend=backend,
                                             rng=np.random.default_rng(seed))
                t0 = time.perf_counter()
                try:
                    res = planner.plan_set_sequence(st.copy(), en.copy(), r0, r0)
                    info = (len(res["set_ids"]), res["graph"].number_of_nodes(), True)
                except (RuntimeError, ValueError):
                    info = (0, 0, False)
                lat[name] = ((time.perf_counter() - t0) * 1e3,) + info
        return lat

    def run_native(reps=2):
        """The same queries one at a time through the native driver (bp_plan_run with a batch of one): the planner
        object (scene upload, device tables) is set up once per query, like the reference's BoundPlanner(...)."""
        from boundplanner_b200.planner_native import NativePlanner

        lat = {}
        for name, ob, infl, st, en, wmin, wmax, seed in cases():
            pl = NativePlanner([dict(obstacles=ob, start=st, end=en, r0=r0, r1=r0)], infl, list(wmax), list(wmin))
            for rep in range(reps):
                t0 = time.perf_counter()
                res, _ = pl.run([seed])
                ok = not isinstance(res[0], Exception)
                lat[name] = ((time.perf_counter() - t0) * 1e3, len(res[0]["set_ids"]) if ok else 0, 0, ok)
            pl.close()
        return lat

    gpu = run(GpuBackend)
    nat = run_native()
    vals = sorted(v[0] for v in nat.values())
    vals_ok = sorted(v[0] for v in nat.values() if v[3])
    pvals = sorted(v[0] for v in gpu.values())
    pvals_ok = sorted(v[0] for v in gpu.values() if v[3])
    same = sum(1 for k in gpu if gpu[k][3] == nat[k][3] and gpu[k][1] == nat[k][1])
    out = {"unit": "ms", "p50": statistics.median(vals), "p95": float(np.percentile(vals, 95)), "max": vals[-1],
           "p50_successful": statistics.median(vals_ok) if vals_ok else None,
           "queries": len(vals), "success_fraction": len(vals_ok) / len(vals),
           "c1_ms": nat["C1"][0],
           "what": "plan_convex_set_path up to the planned set sequence (no final Ipopt NLP), one query at a time "
                   "through the native driver (bp_plan_run, batch of one: one kernel chain per round); C1 + the "
                   "first 24 C3 queries, the reference's error exits included",
           "python_driver": {"p50": statistics.median(pvals), "p95": float(np.percentile(pvals, 95)),
                             "p50_successful": statistics.median(pvals_ok) if pvals_ok else None, "c1_ms": gpu["C1"][0],
                             "what": "the same queries through SetSequencePlanner.plan_set_sequence (Python generator, "
                                     "batch-of-one kernel calls)", "same_outcome_and_sequence_length": f"{same} of {len(gpu)}"}}
    if with_cpu:
        from tests.util import OracleBackend

        cpu = run(OracleBackend, names=("C1", "C3[7]"), reps=1)
        out["cpu_port_ms"] = {k: v[0] for k, v in cpu.items()}
    return out


def kernel_profile(geo, scene, seeds_dev, ws_min, ws_max, out, torch):
    """Time the kernels of one step in isolation (CUDA events on the launch stream,
    several back-to-back launches per measurement) and build the roofline entries."""
    import ctypes

    from boundplanner_b200 import _lib, scenes
    from boundplanner_b200.robot_model import Q_LIM_UPPER

    def timeit(fn, reps=5, inner=4):
        ts = []
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a.record()
            for _ in range(inner):
                fn()
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b) / inner)
        return statistics.median(ts)

    S = seeds_dev.shape[0]
    N = scene.n
    # one polyhedron pass (K3) with the initial sphere, one fixed-mid and one free MVIE (K4) on the built rows
    q0 = torch.eye(3, dtype=torch.float64, device="cuda").repeat(S, 1, 1)
    init_rows = torch.zeros((S, 6, 4), dtype=torch.float64, device="cuda")
    for i in range(3):
        init_rows[:, 2 * i, i] = 1.0
        init_rows[:, 2 * i, 3] = float(ws_max[i])
        init_rows[:, 2 * i + 1, i] = -1.0
        init_rows[:, 2 * i + 1, 3] = -float(ws_min[i])
    qi, qe = q0 * 1e-4, q0 * 1e4
    t_poly = timeit(lambda: geo.polyhedron(scene, seeds_dev, qi, qe, init_rows))
    t_mvie_fm = timeit(lambda: geo.mvie(out.A, out.b, out.m, seeds_dev, False))
    t_mvie_free = timeit(lambda: geo.mvie(out.A, out.b, out.m, seeds_dev, True))
    newton_free = float(geo.mvie(out.A, out.b, out.m, seeds_dev, True)[4].double().mean().item())
    newton_fm = float(geo.mvie(out.A, out.b, out.m, seeds_dev, False)[4].double().mean().item())
    t_pair = timeit(lambda: geo.pair_feasible(out.A, out.b, out.m, TOL))
    sb = geo.alloc_set_batch(S)
    t_build = timeit(lambda: geo.build_sets_point(scene, seeds_dev, ws_min, ws_max, fixed_mid=True, optimize=True,
                                                  out=sb))
    passes_mean = float(torch.clamp(sb.iters.double(), max=5).mean().item())
    m_mean = float(out.m.double().mean().item())

    # FP64 pipe peak of this part (dependent-free DFMA chains, full chip)
    lib = _lib.load()
    probe_out = torch.empty(296 * 256, dtype=torch.float64, device="cuda")
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    iters = 20000
    t_probe = timeit(lambda: lib.bp_probe_fp64(8, 296, 256, iters, ctypes.c_void_p(probe_out.data_ptr()), st),
                     reps=3, inner=1)
    fp64_peak_tflops = 296 * 256 * 8 * iters * 2 / (t_probe * 1e-3) / 1e12

    def algorithmic_flops(n_seeds, passes, rows, n_fm, n_free):
        # SURVEY 8(d) per-unit figures: per (seed, obstacle, pass) closest-point QP 1.1 kflop + 64 flop per picked
        # row and obstacle (exclusion test); per Newton iteration of an MVIE m*200 + 250 flop (DESIGN.md section 3)
        picks = max(rows - 6.0, 0.0)
        return n_seeds * (passes * N * (1100.0 + 64.0 * picks) + (passes * n_fm + n_free) * (rows * 200.0 + 250.0))

    # the chip filled: the same set build with 2048 seeds (8 x the headline batch) in ONE launch
    S_sat = 2048
    seeds_sat = scenes.free_points(S_sat, scenes.config_c2(N_OBS, 8)[0], 0.01, np.random.default_rng(7), ws_min, ws_max)
    seeds_sat_dev = torch.as_tensor(seeds_sat).cuda()
    sb_sat = geo.alloc_set_batch(S_sat)
    t_sat = timeit(lambda: geo.build_sets_point(scene, seeds_sat_dev, ws_min, ws_max, fixed_mid=True, optimize=True,
                                                out=sb_sat), reps=5, inner=2)
    passes_sat = float(torch.clamp(sb_sat.iters.double(), max=5).mean().item())
    rows_sat = float(sb_sat.m.double().mean().item())
    flops_sat = algorithmic_flops(S_sat, passes_sat, rows_sat, newton_fm, newton_free)
    saturated = {"what": "k_iris_fused on the C2 scene with 2048 seeds in one launch (all SMs occupied)",
                 "seeds": S_sat, "ms": t_sat, "sets_per_sec": S_sat / (t_sat * 1e-3),
                 "fp64_tflops_algorithmic": flops_sat / (t_sat * 1e-3) / 1e12,
                 "frac_of_fp64_peak": flops_sat / (t_sat * 1e-3) / 1e12 / fp64_peak_tflops}

    # K7 FK micro-benchmark (C5): B = 2^20 configurations, inputs larger than L2 are flushed between runs
    B = 1 << 20
    lim = torch.as_tensor(Q_LIM_UPPER, device="cuda")
    qq = (torch.rand((B, 7), dtype=torch.float64, device="cuda") * 2 - 1) * lim
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device="cuda")
    ts = []
    for k in range(8):
        flush.fill_(float(k))
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        geo.fk_iiwa14(qq)
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    t_fk = statistics.median(ts[2:])
    fk_bytes = B * (56 + 24 + 168)

    kernels = {
        "build_sets_point_ms": t_build, "iris_passes_mean": passes_mean,
        "k_poly_point_ms": t_poly, "k_mvie_fixed_mid_ms": t_mvie_fm, "k_mvie_free_ms": t_mvie_free,
        "pair_pipeline_ms": t_pair, "k_fk_1M_ms": t_fk, "newton_iters_fixed_mid": newton_fm,
        "newton_iters_free": newton_free, "mean_rows": m_mean, "fp64_peak_tflops_measured": fp64_peak_tflops,
    }

    def roofline():
        # Dominant kernel of the step: the set build (k_iris_fused: one launch = the whole IRIS loop of S seeds).
        # SURVEY 8(d): set build and pair LP are bound by the FP64 CUDA-core pipe, not by HBM (operands live in
        # shared memory / L2).  achieved = ALGORITHMIC flops per launch (the reference algorithm's work: N
        # closest-point QPs per pass although the kernel's lazy bounds skip most of them) / measured duration;
        # peak = this GPU's FP64 pipe measured by a DFMA probe in this run (MEASURED_PEAKS.json has no FP64 entry).
        flops = algorithmic_flops(S, passes_mean, m_mean, newton_fm, newton_free)
        ach = flops / (t_build * 1e-3) / 1e12
        bytes_alg = S * 24 + N * 48 + S * (m_mean * 32 + 12 * 8 + 12)
        return {"kernel": "k_iris_fused (set build: whole find_set_around_point loop, one CTA per seed)",
                "bound": "fp64", "achieved": ach, "peak": fp64_peak_tflops, "unit": "TFLOP/s",
                "frac": ach / fp64_peak_tflops, "traffic": 388608,
                "traffic_source": "ncu dram__bytes_read+write per launch (profiles/r02b_ncu_iris.txt: 388.6 KB read, 0 "
                                  f"written back before the kernel ends; algorithmic bytes {int(bytes_alg)}: scene + seeds "
                                  "in, one padded set out -- the rest is the kernel's 380 KB of instructions and the "
                                  "TMA-staged scene fetched once per SM instead of once per launch)",
                "peak_source": "bp_probe_fp64: independent DFMA chains on all SMs, measured in this run",
                "algorithmic_gflop_per_launch": flops / 1e9, "launch_ms": t_build,
                "note": "latency-bound at 256 seeds (one CTA per seed, 256 CTAs on 148 SMs); `saturated` gives the "
                        "same kernel with the chip filled; roofline_fk is the HBM-bound kernel of the path"}

    def roofline_fk(hbm_peak, which):
        ach = fk_bytes / (t_fk * 1e-3) / 1e9
        return {"kernel": "k_fk<false,false> (B = 2^20 configurations, 248 B each)", "bound": "hbm", "achieved": ach,
                "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak, "traffic": 202077184,
                "traffic_source": "ncu dram__bytes_read+write per launch (below the 260 MB algorithmic bytes: part "
                                  "of the output is still dirty in the 126 MB L2 at kernel end), profiles/",
                "peak_source": which, "poses_per_sec": B / (t_fk * 1e-3)}

    return {"kernels": kernels, "roofline": roofline, "roofline_fk": roofline_fk, "saturated": saturated}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--c3-queries", type=int, default=512, help="C3 planning queries per GPU (BASELINE: 4096 over 8)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-plan-latency", action="store_true")
    ap.add_argument("--no-cuda-graph", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the C3 / C4 / C5 measurements")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the results of the last timed step to DIR/<name>.npy (all sets and the global graph)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's results; the reference arm has none to write")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
