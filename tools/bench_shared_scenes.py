"""Many queries over shared scenes on one GPU: a NativePlanner whose queries share their scenes (``scenes=``,
bp_plan_create_mapped) against the same queries with one copy of their scene each.

Workloads, each at Q = 512 and 2048 queries:
  (a) one C2 scene (scenes.config_c2: 1000 boxes), start / end free and at least 0.3 m apart;
  (b) 8 C3 box scenes (scenes.config_c3_query 0..7, 200 boxes each), the queries spread over them in turn;
  (c) with --polytopes: one C3 polytope scene (scenes.config_c3_polytope_query(0), 200 polytopes with vertex lists).
Per workload, Q and form (shared / copies):
  - construction wall time: host packing of bp_plan_in (PackedQueries), scene ingest and bp_plan_create (the
    NativePlanner constructor), with a device synchronisation;
  - the device memory the planner takes (torch.cuda.mem_get_info before and after the constructor: the library
    allocates with cudaMalloc); node tables and lane workspaces are the same in both forms, the difference is the scenes;
  - run queries/s: best of 3 timed runs after one warm-up, each ending in a device synchronisation;
  - how many results of the shared planner are identical to the copies' (bit for bit).
Prints the card, its power limit and max SM clock, and one JSON line.

    python tools/bench_shared_scenes.py [--polytopes] [--queries 512 2048]
"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
from scipy.spatial.transform import Rotation  # noqa: E402

from boundplanner_b200 import scenes  # noqa: E402
from tools.bench_c3_polytopes import _card  # noqa: E402
from tools.bench_moving_obstacles import _same  # noqa: E402

WMIN, WMAX = scenes.WORKSPACE_MIN, scenes.WORKSPACE_MAX
R0 = Rotation.from_euler("XYZ", [0, 90, 0], degrees=True).as_matrix()


def _endpoints(scene, infl, rng):
    while True:
        if "obs_sets" in scene:
            pts = scenes.polytope_free_points(2, scene["obs_sets"], 0.06, rng, WMIN + 0.1, WMAX - 0.1)
        else:
            pts = scenes.free_points(2, scene["obstacles"], infl + 0.06, rng, WMIN + 0.1, WMAX - 0.1)
        if np.linalg.norm(pts[0] - pts[1]) >= 0.3:
            return pts[0], pts[1]


def workload(name):
    """(scene list, inflate) of a workload."""
    if name == "c2_one_scene":
        ob, infl, _, _, _ = scenes.config_c2()
        return [dict(obstacles=ob)], infl
    if name == "c3_eight_box_scenes":
        return [dict(obstacles=scenes.config_c3_query(i)[0]) for i in range(8)], 0.01
    obs_sets, pts, infl, _, _, _, _ = scenes.config_c3_polytope_query(0)
    return [dict(obs_sets=obs_sets, obs_points_sets=pts)], infl


def queries_of(scene_list, infl, Q):
    """(shared queries, copies): query k plans in scene k mod n_scenes; the copies carry that scene's obstacles."""
    shared, copies = [], []
    for k in range(Q):
        s = k % len(scene_list)
        st, en = _endpoints(scene_list[s], infl, np.random.default_rng(10_000 + k))
        q = dict(start=st, end=en, r0=R0, r1=R0)
        shared.append(dict(q, scene=s))
        copies.append(dict(q, **scene_list[s]))
    return shared, copies


def measure(queries, infl, scene_list, seeds, reps=3):
    import torch

    from boundplanner_b200 import planner_native as pn

    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    t0 = time.perf_counter()
    pk = pn.PackedQueries(queries, infl, WMAX, WMIN, seeds, scenes=scene_list)
    t1 = time.perf_counter()
    pl = pn.NativePlanner(queries, infl, WMAX, WMIN, scenes=scene_list)
    torch.cuda.synchronize()
    t2 = time.perf_counter()
    free1 = torch.cuda.mem_get_info()[0]
    del pk
    try:
        res, _ = pl.run(seeds)                           # warm-up (arenas, the packed inputs of these seeds)
        best, st = float("inf"), None
        for _ in range(reps):
            torch.cuda.synchronize()
            t = time.perf_counter()
            res, st = pl.run(seeds)
            torch.cuda.synchronize()
            best = min(best, time.perf_counter() - t)
    finally:
        pl.close()
    return dict(pack_ms=1e3 * (t1 - t0), create_ms=1e3 * (t2 - t1), construction_ms=1e3 * (t2 - t0),
                device_mb=(free0 - free1) / 2**20, run_queries_per_sec=len(queries) / best, rounds=st["rounds"],
                planned=int(sum(not isinstance(r, Exception) for r in res))), res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--polytopes", action="store_true", help="also (c): one C3 polytope scene")
    ap.add_argument("--queries", type=int, nargs="+", default=[512, 2048])
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench_shared_scenes needs a CUDA device")
    name, power = _card()
    names = ["c2_one_scene", "c3_eight_box_scenes"] + (["c3_one_polytope_scene"] if args.polytopes else [])
    rows = []
    for wl in names:
        scene_list, infl = workload(wl)
        for Q in args.queries:
            shared, copies = queries_of(scene_list, infl, Q)
            seeds = list(range(Q))
            m_sh, r_sh = measure(shared, infl, scene_list, seeds)
            m_cp, r_cp = measure(copies, infl, None, seeds)
            same = sum(int(_same(g, w)) for g, w in zip(r_sh, r_cp))
            rows.append(dict(workload=wl, queries=Q, scenes=len(scene_list), shared=m_sh, copies=m_cp,
                             identical=same))
            print(f"{wl} Q={Q}: construction {m_sh['construction_ms']:.1f} vs {m_cp['construction_ms']:.1f} ms "
                  f"(pack {m_sh['pack_ms']:.1f} vs {m_cp['pack_ms']:.1f}), device {m_sh['device_mb']:.1f} vs "
                  f"{m_cp['device_mb']:.1f} MB, run {m_sh['run_queries_per_sec']:.0f} vs "
                  f"{m_cp['run_queries_per_sec']:.0f} queries/s, planned {m_sh['planned']}, identical {same}/{Q}",
                  flush=True)
    print(f"card: {name}, power limit / max SM clock: {power}")
    print(json.dumps({"what": "shared scenes vs one copy per query (NativePlanner)", "card": name,
                      "power_limit_and_max_sm_clock": power, "rows": rows}))


if __name__ == "__main__":
    main()
