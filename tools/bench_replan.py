"""Replanning on the native lock-step driver, one GPU: the call an MPC loop makes again and again
(BoundPlanner.plan_convex_set_path with replanning=True, :231-276) against the first plan of the same queries.

  1. `--queries` C3 queries (scenes.config_c3_query, 200 boxes each; --polytopes: config_c3_polytope_query, 200
     polytopes each) are planned natively, seeded.
  2. The planned ones become an MPC-style replanning batch: start 2 % along the first segment, a 10-point horizon
     along the path, sets_via_prev from the first result.
  3. First-plan batch and replanning batch of those queries on the same resident scenes (one NativePlanner), best of
     `--reps` each: queries/s, p50 / p95 completion, device wait, rounds.
  4. A 5-step MPC loop over the first `--loop` of them, sets_via_prev threaded forward (native results only).
  5. planner.plan_batch (Python lock-step driver, same kernels) on the first `--python` replanning queries as the
     equality reference.
Prints the card and its power limit, and one JSON line.

    python tools/bench_replan.py [--polytopes] [--queries 512] [--loop 64] [--python 32] [--reps 3]
"""
import argparse
import json
import os
import sys
import time
from concurrent.futures import ProcessPoolExecutor

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
from scipy.spatial.transform import Rotation as R  # noqa: E402

from boundplanner_b200 import scenes  # noqa: E402
from tools.bench_c3_polytopes import _card, _polytope_query, _summary  # noqa: E402

R0 = R.from_euler("XYZ", [0, 90, 0], degrees=True).as_matrix()
WMIN, WMAX = list(scenes.WORKSPACE_MIN), list(scenes.WORKSPACE_MAX)


def _box_query(i):
    ob, infl, st, en, _, _ = scenes.config_c3_query(i)
    return dict(obstacles=ob, start=st, end=en, r0=R0, r1=R0)


def mpc_step(q, res, frac=0.02, n_horizon=10):
    """The next MPC call after a planned result: start `frac` along the first segment, n_horizon points along the
    first 60 % of the remaining path, the result's sets_via_prev."""
    p_via = res["p_via"]
    start = p_via[0] + frac * (p_via[1] - p_via[0])
    pts = np.vstack((start, p_via[1:]))
    seg = np.cumsum(np.r_[0.0, np.linalg.norm(np.diff(pts, axis=0), axis=1)])
    s = np.linspace(0.0, 1.0, n_horizon + 1)[1:] * seg[-1] * 0.6
    horizon = np.stack([np.interp(s, seg, pts[:, k]) for k in range(3)], axis=1)
    return dict(q, start=start, replanning=True, p_horizon=horizon, sets_via_prev=res["sets_via_prev"])


def _best(pl, seeds, reps, queries=None):
    """(seconds, stats, results) of the best of `reps` timed runs after one warm-up."""
    import torch

    pl.run(seeds, queries=queries, want_nodes=False)
    torch.cuda.synchronize()
    best = None
    for _ in range(reps):
        t0 = time.perf_counter()
        res, st = pl.run(seeds, queries=queries, want_nodes=False)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if best is None or dt < best[0]:
            best = (dt, st, res)
    return best


def _same(g, w):
    if isinstance(w, Exception):
        return isinstance(g, Exception) and type(g) is type(w) and str(g).split("(")[0] == str(w).split("(")[0]
    return (not isinstance(g, Exception) and g["path"] == w["path"] and g["set_ids"] == w["set_ids"] and
            float(np.abs(g["p_via"] - w["p_via"]).max()) < 1e-9 and
            ("p_horizon_max" in g) == ("p_horizon_max" in w) and
            ("p_horizon_max" not in w or np.array_equal(g["p_horizon_max"], w["p_horizon_max"])))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--polytopes", action="store_true", help="C3 over 200 general convex polytopes per query")
    ap.add_argument("--queries", type=int, default=512)
    ap.add_argument("--loop", type=int, default=64, help="queries of the 5-step MPC loop")
    ap.add_argument("--python", type=int, default=32, help="replanning queries also planned by planner.plan_batch")
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    import torch

    from boundplanner_b200.planner import plan_batch
    from boundplanner_b200.planner_native import NativePlanner

    if not torch.cuda.is_available():
        raise SystemExit("bench_replan needs a CUDA device")
    ids = list(range(args.queries))
    t0 = time.perf_counter()
    if args.polytopes:
        with ProcessPoolExecutor(max_workers=min(32, os.cpu_count() or 1)) as ex:     # (scipy's qhull per obstacle)
            base = list(ex.map(_polytope_query, ids, chunksize=8))
    else:
        base = [_box_query(i) for i in ids]
    t_gen = time.perf_counter() - t0
    name, power = _card()

    # 1-2: first plans of all queries, the replanning batch of the planned ones
    pl = NativePlanner(base, 0.01, WMAX, WMIN)
    try:
        first, _ = pl.run(ids)
    finally:
        pl.close()
    ok = [i for i, r in enumerate(first) if not isinstance(r, Exception)]
    sub = [base[i] for i in ok]
    replan = [mpc_step(base[i], first[i]) for i in ok]
    seeds = list(range(len(ok)))

    # 3: first plans and replanning calls of the planned queries on the same resident scenes
    pl = NativePlanner(sub, 0.01, WMAX, WMIN)
    try:
        dt_f, st_f, res_f = _best(pl, seeds, args.reps)
        dt_r, st_r, res_r = _best(pl, seeds, args.reps, queries=replan)
    finally:
        pl.close()

    # 4: a 5-step MPC loop, sets threaded forward
    n_loop = min(args.loop, len(ok))
    pl = NativePlanner(sub[:n_loop], 0.01, WMAX, WMIN)
    loop = []
    try:
        queries = [mpc_step(sub[k], first[ok[k]]) for k in range(n_loop)]
        for step in range(5):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res, st = pl.run([100 * step + k for k in range(n_loop)], queries=queries)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            planned = [not isinstance(r, Exception) for r in res]
            loop.append({"step": step, "queries_per_sec": n_loop / dt, "rounds": st["rounds"],
                         "planned_fraction": float(np.mean(planned))})
            queries = [mpc_step(q, r) if not isinstance(r, Exception) else dict(q, replanning=False)
                       for q, r in zip(queries, res)]
    finally:
        pl.close()

    # 5: the Python lock-step driver on the first replanning queries (same seeds as the timed native runs)
    n_py = min(args.python, len(ok))
    t0 = time.perf_counter()
    want, _ = plan_batch(replan[:n_py], 0.01, WMAX, WMIN, rng_seeds=seeds[:n_py])
    dt_py = time.perf_counter() - t0
    same = sum(int(_same(g, w)) for g, w in zip(res_r[:n_py], want))

    kind = "200 general convex polytopes" if args.polytopes else "200 boxes"
    out = {"what": f"replanning vs first plans on the native lock-step driver, C3 over {kind} per query, "
                   f"best of {args.reps} runs after a warm-up, scenes resident",
           "card": name, "power_limit_and_max_sm_clock": power, "first_planned": len(ok), "of_queries": args.queries,
           "first_plan": _summary(len(ok), dt_f, st_f, res_f), "replanning": _summary(len(ok), dt_r, st_r, res_r),
           "mpc_loop": {"queries": n_loop, "steps": loop},
           "python_driver_replanning": {"queries": n_py, "plan_queries_per_sec": n_py / dt_py,
                                        "identical_to_native": same},
           "query_generation_s": t_gen}
    print(f"card: {name}, power limit / max SM clock: {power}")
    print(f"{len(ok)} of {args.queries} queries planned; on them:")
    for k in ("first_plan", "replanning"):
        s = out[k]
        print(f"{k:11s}: {s['plan_queries_per_sec']:.0f} queries/s, p50 {s['latency_ms_p50']:.1f} ms, p95 "
              f"{s['latency_ms_p95']:.1f} ms, device wait {s['device_wait_ms']:.1f} ms, rounds {s['rounds']}, "
              f"planned {s['success_fraction']:.2f}")
    for s in loop:
        print(f"MPC loop step {s['step']}: {n_loop} queries, {s['queries_per_sec']:.0f} queries/s, rounds {s['rounds']}, "
              f"planned {s['planned_fraction']:.2f}")
    print(f"python driver on {n_py} replanning queries: {n_py / dt_py:.1f} queries/s, identical to native: {same}/{n_py}")
    print(json.dumps(out))


if __name__ == "__main__":
    main()
