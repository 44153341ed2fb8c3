"""Moving obstacles in an MPC loop on one GPU: rewrite the resident scenes in place (NativePlanner.update_obstacles,
bp_scene_update_batch / bp_scene_update_polytopes_batch) against building a fresh NativePlanner every step.

  1. `--queries` C3 queries (scenes.config_c3_query, 200 boxes each; --polytopes: config_c3_polytope_query, 200
     polytopes each with their vertex lists; --enumerate: without them, enumerated on the device) are planned once.
  2. `--steps` MPC steps: every query's obstacles move (scenes.moved_obstacles: a quarter translated, 4 removed, 4
     added), new_obs=True, planned queries replan with the previous sets_via_prev, failed ones plan again.
  3. Per step: the update's device time (CUDA events around the library call: staging copy, kernels, the final
     synchronisation), its host packing time and its wall time,
     and the run after it; then a fresh NativePlanner on the same queries (its construction, scene ingest included,
     and its first run, arena allocations included).  Every result of the updated planner is compared with the fresh
     planner's (bit for bit); the next step follows the updated planner's results.
Prints the card and its power limit, and one JSON line.

    python tools/bench_moving_obstacles.py [--polytopes [--enumerate]] [--queries 512] [--steps 5]
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
from tools.bench_replan import _box_query, mpc_step  # noqa: E402

WMIN, WMAX = list(scenes.WORKSPACE_MIN), list(scenes.WORKSPACE_MAX)


def _moved(q, rng, enumerate_vertices):
    if "obs_sets" in q:
        sets, pts = scenes.moved_obstacles(q["obs_sets"], rng, obs_points=q.get("obs_points_sets"))
        return dict(q, obs_sets=sets, obs_points_sets=None if enumerate_vertices else pts)
    return dict(q, obstacles=scenes.moved_obstacles(np.asarray(q["obstacles"]), rng))


def _same(g, w):
    if isinstance(w, Exception):
        return isinstance(g, Exception) and type(g) is type(w) and str(g) == str(w)
    if isinstance(g, Exception) or g["path"] != w["path"] or g["set_ids"] != w["set_ids"]:
        return False
    if not np.array_equal(g["p_via"], w["p_via"]) or len(g["sets_via_prev"]) != len(w["sets_via_prev"]):
        return False
    return all(np.array_equal(a, c) and np.array_equal(b, d) for (a, b), (c, d) in zip(g["sets_via_prev"],
                                                                                       w["sets_via_prev"]))


def _next_queries(queries, res, rng, enumerate_vertices):
    out = []
    for q, r in zip(queries, res):
        q = _moved(q, rng, enumerate_vertices)
        out.append(dict(mpc_step(q, r), new_obs=True) if not isinstance(r, Exception)
                   else dict(q, replanning=False, new_obs=True))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--polytopes", action="store_true", help="C3 over 200 general convex polytopes per query")
    ap.add_argument("--enumerate", action="store_true", help="polytopes without vertex lists (enumerated on the device)")
    ap.add_argument("--queries", type=int, default=512)
    ap.add_argument("--steps", type=int, default=5)
    args = ap.parse_args()
    import torch

    from boundplanner_b200.planner_native import NativePlanner

    if not torch.cuda.is_available():
        raise SystemExit("bench_moving_obstacles needs a CUDA device")
    ids = list(range(args.queries))
    if args.polytopes:
        with ProcessPoolExecutor(max_workers=min(32, os.cpu_count() or 1)) as ex:     # (scipy's qhull per obstacle)
            queries = list(ex.map(_polytope_query, ids, chunksize=8))
        if args.enumerate:
            queries = [dict(q, obs_points_sets=None) for q in queries]
    else:
        queries = [_box_query(i) for i in ids]
    name, power = _card()
    Q = len(queries)

    pl = NativePlanner(queries, 0.01, WMAX, WMIN)
    steps = []
    try:
        res, _ = pl.run(ids)
        for step in range(1, args.steps + 1):
            queries = _next_queries(queries, res, np.random.default_rng(100 + step), args.enumerate)
            seeds = [1000 * step + i for i in ids]
            # update in place, then plan
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            pl.update_obstacles(queries)
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            ev0, ev1 = pl.scene.update_events
            res, st = pl.run(seeds)
            torch.cuda.synchronize()
            t2 = time.perf_counter()
            # the alternative: a fresh planner over the same queries
            fresh = NativePlanner(queries, 0.01, WMAX, WMIN)
            torch.cuda.synchronize()
            t3 = time.perf_counter()
            try:
                want, _ = fresh.run(seeds)
                torch.cuda.synchronize()
                t4 = time.perf_counter()
            finally:
                fresh.close()
            same = sum(int(_same(g, w)) for g, w in zip(res, want))
            upd, run_u, make, run_f = t1 - t0, t2 - t1, t3 - t2, t4 - t3
            steps.append({"step": step, "obstacles": int(sum(len(q["obs_sets"] if "obs_sets" in q else q["obstacles"])
                                                for q in queries)),
                          "update_device_ms": ev0.elapsed_time(ev1), "update_pack_ms": 1e3 * pl.scene.pack_seconds,
                          "update_wall_ms": 1e3 * upd, "run_after_update_ms": 1e3 * run_u,
                          "recreate_ms": 1e3 * make, "first_run_of_fresh_ms": 1e3 * run_f,
                          "update_plus_run_queries_per_sec": Q / (upd + run_u),
                          "recreate_plus_run_queries_per_sec": Q / (make + run_f),
                          "planned": int(sum(not isinstance(r, Exception) for r in res)), "rounds": st["rounds"],
                          "identical_to_fresh": same})
    finally:
        pl.close()

    kind = ("200 general convex polytopes" + (" (vertices enumerated on the device)" if args.enumerate else "")
            if args.polytopes else "200 boxes")
    out = {"what": f"MPC loop with moving obstacles, C3 over {kind} per query, {Q} queries: update in place vs a "
                   f"fresh NativePlanner per step", "card": name, "power_limit_and_max_sm_clock": power, "steps": steps}
    print(f"card: {name}, power limit / max SM clock: {power}")
    for s in steps:
        print(f"step {s['step']}: update {s['update_device_ms']:.2f} ms device / {s['update_pack_ms']:.1f} ms packing / "
              f"{s['update_wall_ms']:.1f} ms wall, run {s['run_after_update_ms']:.0f} ms | recreate "
              f"{s['recreate_ms']:.1f} ms, first run {s['first_run_of_fresh_ms']:.0f} ms | queries/s update+run "
              f"{s['update_plus_run_queries_per_sec']:.0f}, recreate+run {s['recreate_plus_run_queries_per_sec']:.0f} | "
              f"planned {s['planned']}, identical {s['identical_to_fresh']}/{Q}")
    print(json.dumps(out))


if __name__ == "__main__":
    main()
