"""C3 over general convex polytope obstacles on one GPU: the native lock-step driver (bp_plan_run over a polytope scene
batch) on `--queries` queries of scenes.config_c3_polytope_query (200 polytopes each), the Python lock-step driver
(planner.plan_batch, same kernels) on the first `--python` of them as an equality and speed reference, and the box C3
queries (scenes.config_c3_query) through the native driver in the same process for comparison.  Prints the card and
its power limit, and one JSON line.

    python tools/bench_c3_polytopes.py [--queries 512] [--python 32] [--reps 3]
"""
import argparse
import json
import os
import subprocess
import sys
import time
from concurrent.futures import ProcessPoolExecutor

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
from scipy.spatial.transform import Rotation as R  # noqa: E402

from boundplanner_b200 import scenes  # noqa: E402

R0 = R.from_euler("XYZ", [0, 90, 0], degrees=True).as_matrix()


def _polytope_query(i):
    obs_sets, pts, infl, st, en, wmin, wmax = scenes.config_c3_polytope_query(i)
    return dict(obs_sets=obs_sets, obs_points_sets=pts, start=st, end=en, r0=R0, r1=R0)


def _card():
    import torch

    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = "nvidia-smi unavailable"
    return name, out


def _native(queries, ids, reps):
    """(best run: seconds, stats, results) of `reps` timed runs after one warm-up, scenes resident."""
    import torch

    from boundplanner_b200.planner_native import NativePlanner

    pl = NativePlanner(queries, 0.01, list(scenes.WORKSPACE_MAX), list(scenes.WORKSPACE_MIN))
    try:
        pl.run(ids)
        torch.cuda.synchronize()
        best = None
        for _ in range(reps):
            t0 = time.perf_counter()
            res, st = pl.run(ids, want_nodes=False)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            if best is None or dt < best[0]:
                best = (dt, st, res)
        return best
    finally:
        pl.close()


def _summary(nq, dt, st, res):
    lat = np.asarray(st["finish_ms"], float)
    return {"queries": nq, "plan_queries_per_sec": nq / dt, "seconds": dt,
            "latency_ms_p50": float(np.percentile(lat, 50)), "latency_ms_p95": float(np.percentile(lat, 95)),
            "device_wait_ms": st["device_wait_ms"], "rounds": st["rounds"], "kernel_chains": st["kernel_chains"],
            "set_requests": st["set_requests"], "pair_tests": st["pair_tests"], "projections": st["projections"],
            "success_fraction": float(np.mean([not isinstance(r, Exception) for r in res]))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--queries", type=int, default=512)
    ap.add_argument("--python", type=int, default=32, help="queries also planned by planner.plan_batch")
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    import torch

    from boundplanner_b200.planner import plan_batch

    if not torch.cuda.is_available():
        raise SystemExit("bench_c3_polytopes needs a CUDA device")
    nq = args.queries
    ids = list(range(nq))
    t0 = time.perf_counter()
    with ProcessPoolExecutor(max_workers=min(32, os.cpu_count() or 1)) as ex:       # (scipy's qhull per obstacle)
        poly = list(ex.map(_polytope_query, ids, chunksize=8))
    t_gen = time.perf_counter() - t0
    boxes = []
    for i in ids:
        ob, infl, st, en, _, _ = scenes.config_c3_query(i)
        boxes.append(dict(obstacles=ob, start=st, end=en, r0=R0, r1=R0))
    name, power = _card()

    dt_p, st_p, res_p = _native(poly, ids, args.reps)
    dt_b, st_b, res_b = _native(boxes, ids, args.reps)
    # the Python lock-step driver over the same kernels: speed and equality on the first queries
    n_py = min(args.python, nq)
    wmin, wmax = list(scenes.WORKSPACE_MIN), list(scenes.WORKSPACE_MAX)
    plan_batch(poly[:4], 0.01, wmax, wmin, rng_seeds=ids[:4])
    t0 = time.perf_counter()
    want, _ = plan_batch(poly[:n_py], 0.01, wmax, wmin, rng_seeds=ids[:n_py])
    dt_py = time.perf_counter() - t0
    same = 0
    for w, g in zip(want, res_p[:n_py]):
        if isinstance(w, Exception):
            same += int(isinstance(g, Exception) and type(g) is type(w))
        else:
            same += int((not isinstance(g, Exception)) and g["path"] == w["path"] and g["set_ids"] == w["set_ids"] and
                        float(np.abs(g["p_via"] - w["p_via"]).max()) < 1e-9)
    out = {"what": "C3 over 200 general convex polytopes per query (scenes.config_c3_polytope_query), native lock-step "
                   "driver, best of %d runs after a warm-up, scenes resident" % args.reps,
           "card": name, "power_limit_and_max_sm_clock": power,
           "polytopes": _summary(nq, dt_p, st_p, res_p), "boxes": _summary(nq, dt_b, st_b, res_b),
           "python_driver_polytopes": {"queries": n_py, "plan_queries_per_sec": n_py / dt_py,
                                       "identical_to_native": same},
           "query_generation_s": t_gen}
    print(f"card: {name}, power limit / max SM clock: {power}")
    for k in ("polytopes", "boxes"):
        s = out[k]
        print(f"{k:9s}: {s['plan_queries_per_sec']:.0f} queries/s, p50 {s['latency_ms_p50']:.1f} ms, p95 "
              f"{s['latency_ms_p95']:.1f} ms, device wait {s['device_wait_ms']:.1f} ms, rounds {s['rounds']}, "
              f"planned {s['success_fraction']:.2f}")
    print(f"python driver on {n_py} polytope queries: {n_py / dt_py:.1f} queries/s, identical to native: {same}/{n_py}")
    print(json.dumps(out))


if __name__ == "__main__":
    main()
