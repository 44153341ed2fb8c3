"""Corridor checks in an MPC loop with moving obstacles on one GPU: after every obstacle update, test the planned
queries' corridors (their sets_via_prev) against the new obstacles (NativePlanner.corridor_hits, bp_sets_obstacles)
and replan only the queries whose corridor is hit or whose last plan failed (run(active=), bp_plan_run_active),
against replanning every query (run()).

  1. `--queries` C3 queries (scenes.config_c3_query, 200 boxes each; --polytopes: config_c3_polytope_query, 200
     polytopes each) are planned once.
  2. `--steps` MPC steps as in tools/bench_moving_obstacles.py: every query's obstacles move (scenes.moved_obstacles:
     a quarter translated, 4 removed, 4 added), new_obs=True, planned queries replan with their sets_via_prev.
  3. Per step: update_obstacles, then corridor_hits on the planned queries' sets_via_prev -- its device time (CUDA
     events around the library call) and its wall time (packing, copies and the call); the fraction of planned
     corridors hit; run(active=hit or failed) and run() over all queries, wall time and device wait each (the step's
     inputs packed once before either run).  Every active result is compared with the full run's (bit for bit); the
     next step follows the full run.
Prints the card and its power limit, and one JSON line.

    python tools/bench_corridor_check.py [--polytopes] [--queries 512] [--steps 5]
"""
import argparse
import json
import os
import sys
import time
from concurrent.futures import ProcessPoolExecutor

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

from boundplanner_b200 import scenes  # noqa: E402
from tools.bench_c3_polytopes import _card, _polytope_query  # noqa: E402
from tools.bench_moving_obstacles import _next_queries, _same  # noqa: E402
from tools.bench_replan import _box_query  # noqa: E402

WMIN, WMAX = list(scenes.WORKSPACE_MIN), list(scenes.WORKSPACE_MAX)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--polytopes", action="store_true", help="C3 over 200 general convex polytopes per query")
    ap.add_argument("--queries", type=int, default=512)
    ap.add_argument("--steps", type=int, default=5)
    args = ap.parse_args()
    import torch

    from boundplanner_b200.planner_native import NativePlanner

    if not torch.cuda.is_available():
        raise SystemExit("bench_corridor_check needs a CUDA device")
    ids = list(range(args.queries))
    if args.polytopes:
        with ProcessPoolExecutor(max_workers=min(32, os.cpu_count() or 1)) as ex:     # (scipy's qhull per obstacle)
            queries = list(ex.map(_polytope_query, ids, chunksize=8))
    else:
        queries = [_box_query(i) for i in ids]
    name, power = _card()
    Q = len(queries)

    pl = NativePlanner(queries, 0.01, WMAX, WMIN)
    steps = []
    try:
        res, _ = pl.run(ids)
        for step in range(1, args.steps + 1):
            queries = _next_queries(queries, res, np.random.default_rng(100 + step), False)
            seeds = [1000 * step + i for i in ids]
            pl.update_obstacles(queries)
            corridors = [q["sets_via_prev"] if isinstance(r, dict) else None for q, r in zip(queries, res)]
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            hits = pl.corridor_hits(corridors)
            t1 = time.perf_counter()
            ev0, ev1 = pl.corridor_events
            hit = [h is not None and bool((h >= 0).any()) for h in hits]
            active = [h or c is None for h, c in zip(hit, corridors)]
            n_planned = sum(c is not None for c in corridors)
            pl.run(seeds, active=[False] * Q)      # packs the step's inputs once (PackedQueries): both runs reuse them
            torch.cuda.synchronize()
            t2 = time.perf_counter()
            sub, sst = pl.run(seeds, active=active)
            torch.cuda.synchronize()
            t3 = time.perf_counter()
            full, fst = pl.run(seeds)
            torch.cuda.synchronize()
            t4 = time.perf_counter()
            idx = [k for k in range(Q) if active[k]]
            same = sum(int(_same(sub[k], full[k])) for k in idx)
            steps.append({"step": step, "planned_corridors": n_planned,
                          "corridor_sets": int(sum(len(c) for c in corridors if c is not None)),
                          "corridors_hit": int(sum(hit)), "hit_fraction": sum(hit) / max(n_planned, 1),
                          "active": len(idx), "check_device_ms": ev0.elapsed_time(ev1), "check_wall_ms": 1e3 * (t1 - t0),
                          "run_active_ms": 1e3 * (t3 - t2), "run_active_device_wait_ms": sst["device_wait_ms"],
                          "run_all_ms": 1e3 * (t4 - t3), "run_all_device_wait_ms": fst["device_wait_ms"],
                          "active_identical_to_full": same})
            res = full
    finally:
        pl.close()

    kind = "200 general convex polytopes" if args.polytopes else "200 boxes"
    out = {"what": f"MPC loop with moving obstacles, C3 over {kind} per query, {Q} queries: corridor check + replan of "
                   f"the hit / failed queries vs replanning every query", "card": name,
           "power_limit_and_max_sm_clock": power, "steps": steps}
    print(f"card: {name}, power limit / max SM clock: {power}")
    for s in steps:
        print(f"step {s['step']}: check {s['check_device_ms']:.3f} ms device / {s['check_wall_ms']:.2f} ms wall over "
              f"{s['corridor_sets']} sets | hit {s['corridors_hit']}/{s['planned_corridors']} planned corridors "
              f"({100 * s['hit_fraction']:.1f} %) | run(active={s['active']}) {s['run_active_ms']:.1f} ms (wait "
              f"{s['run_active_device_wait_ms']:.1f}) vs run() {s['run_all_ms']:.1f} ms (wait "
              f"{s['run_all_device_wait_ms']:.1f}) | identical {s['active_identical_to_full']}/{s['active']}")
    print(json.dumps(out))
    bad = [s["step"] for s in steps if s["active_identical_to_full"] != s["active"]]
    if bad:
        raise SystemExit(f"active results differ from the full run's in steps {bad}")


if __name__ == "__main__":
    main()
