"""Many queries over shared scenes: the query -> scene map of the batched planners (bp_plan_create_mapped,
NativePlanner / plan_batch_native / plan_batch with ``scenes=``, BatchedGpuExecutor's query_scene) and of the MPC
joint sets (mpc_geometry.collision_sets with ``robot_scene``).

A query planned in a shared scene must give the results, bit for bit, of the same query holding a copy of that scene
of its own.  CPU: the native state machines in the host harness (hh_plan_batch_mapped against hh_plan_batch), every
request answered by the oracle, and the Python planner; the ValueErrors of malformed batches, raised without a device.
GPU: the native driver over shared scenes against one copy per query (boxes, polytopes, the 1000-box C2 scene, an MPC
loop with moving obstacles), plan_batch, the C entry point's errors and the MPC joint sets."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from boundplanner_b200 import planner_native as pn
from boundplanner_b200 import scenes
from boundplanner_b200.planner import plan_batch
from tests.util import (R0, MemoBackend, PolytopeOracleBackend, _same_sets, assert_same_result, mpc_step, python_plan,
                        run_native_with_oracle)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

WMIN, WMAX = scenes.WORKSPACE_MIN, scenes.WORKSPACE_MAX
_OUTPUTS = ("err_kind", "path", "path_len", "set_ids", "n_ids", "p_via", "n_via", "rng_out", "n_nodes", "n_inter",
            "n_edges", "finish_round", "node_A", "node_b", "node_m", "stats", "p_horizon_max")


# ---- scenes and queries ---------------------------------------------------------------------------------------
def _box_scene(i):
    ob, infl, _, _, _, _ = scenes.config_c3_query(i)
    return dict(obstacles=ob), infl


def _poly_scene(i):
    obs_sets, pts, infl, _, _, _, _ = scenes.config_c3_polytope_query(i)
    return dict(obs_sets=obs_sets, obs_points_sets=pts), infl


def _endpoints(scene, infl, rng):
    """A seeded free start / end of a scene, at least 0.3 m apart (as C3 draws them)."""
    while True:
        if "obs_sets" in scene:
            pts = scenes.polytope_free_points(2, scene["obs_sets"], 0.06, rng, WMIN + 0.1, WMAX - 0.1)
        else:
            pts = scenes.free_points(2, scene["obstacles"], infl + 0.06, rng, WMIN + 0.1, WMAX - 0.1)
        if np.linalg.norm(pts[0] - pts[1]) >= 0.3:
            return pts[0], pts[1]


def shared_form(queries, query_scene, scene_list=None):
    """(queries carrying ``scene`` instead of obstacles, scenes) of queries that carry their own obstacles: scene s
    holds the obstacles of the first query that query_scene maps to s (or is scene_list[s])."""
    keys = ("obstacles", "obs_sets", "obs_points_sets")
    if scene_list is None:
        scene_list = [None] * (int(max(query_scene)) + 1)
        for q, s in zip(queries, query_scene):
            if scene_list[s] is None:
                scene_list[s] = {k: q[k] for k in keys if k in q}
    shared = [dict({k: v for k, v in q.items() if k not in keys}, scene=int(s)) for q, s in zip(queries, query_scene)]
    return shared, scene_list


def _copies(scene_list, infl, query_scene, seed):
    """One query per entry of query_scene, each carrying a copy of its scene's obstacles (the same objects)."""
    out = []
    for k, s in enumerate(query_scene):
        st, en = _endpoints(scene_list[s], infl, np.random.default_rng(seed + 7919 * k))
        out.append(dict(scene_list[s], start=st, end=en, r0=R0, r1=R0))
    return out


def _assert_same_packed(got, want):
    """Every output of two host-harness runs, bit for bit (error messages included)."""
    assert got.err_msg.raw == want.err_msg.raw
    for k in _OUTPUTS:
        g, w = getattr(got, k), getattr(want, k)
        assert g.dtype == w.dtype and g.shape == w.shape and np.array_equal(g.view(np.uint8), w.view(np.uint8)), k


def _assert_same_plans(got, want, gst=None, wst=None):
    """Bit-identical results of two native runs (and the same round statistics)."""
    assert len(got) == len(want)
    for i, (g, w) in enumerate(zip(got, want)):
        if isinstance(w, Exception):
            assert type(g) is type(w) and str(g) == str(w), (i, g, w)
            continue
        assert not isinstance(g, Exception), (i, g)
        assert g["path"] == w["path"] and g["set_ids"] == w["set_ids"], i
        assert np.array_equal(g["p_via"], w["p_via"]), i
        assert (g["n_nodes"], g["n_inter"], g["n_edges"]) == (w["n_nodes"], w["n_inter"], w["n_edges"]), i
        _same_sets(g["sets_via"], w["sets_via"])
        _same_sets(g["sets_via_prev"], w["sets_via_prev"])
        assert ("p_horizon_max" in g) == ("p_horizon_max" in w)
        if "p_horizon_max" in w:
            assert np.array_equal(g["p_horizon_max"], w["p_horizon_max"]), i
    if wst is not None:
        for k in ("rounds", "set_requests", "pair_tests", "projections", "shortest_paths"):
            assert gst[k] == wst[k], k


def _assert_like_plan_batch(got, want):
    """bp_plan_run against planner.plan_batch (the comparison of the other native-driver tests)."""
    n_ok = 0
    for i, (w, g) in enumerate(zip(want, got)):
        if isinstance(w, Exception):
            assert isinstance(g, Exception) and type(g) is type(w), (i, g, w)
            assert str(g).split("(")[0] == str(w).split("(")[0], (i, g, w)
            continue
        n_ok += 1
        assert not isinstance(g, Exception), f"query {i}: {g!r}"
        assert g["path"] == w["path"] and g["set_ids"] == w["set_ids"], i
        assert np.abs(g["p_via"] - w["p_via"]).max() < 1e-9, i
        _same_sets(g["sets_via_prev"], w["sets_via_prev"], 1e-12)
        assert ("p_horizon_max" in g) == ("p_horizon_max" in w)
        if "p_horizon_max" in w:
            assert np.array_equal(g["p_horizon_max"], w["p_horizon_max"]), i
    return n_ok


# ---- CPU: host harness with the oracle answering ----------------------------------------------------------------
@pytest.fixture(scope="module")
def mapped_harness():
    """tests/host_harness_mapped.cpp: the host harness plus hh_plan_batch_mapped (g++, built like conftest's
    host_harness)."""
    build = os.path.join(ROOT, "tests", "_build")
    os.makedirs(build, exist_ok=True)
    so = os.path.join(build, "libbp_host_harness_mapped.so")
    src = os.path.join(ROOT, "tests", "host_harness_mapped.cpp")
    deps = [src, os.path.join(ROOT, "tests", "host_harness.cpp"), os.path.join(ROOT, "include", "bpgeo.h")] + [
        os.path.join(ROOT, "boundplanner_b200", "csrc", f)
        for f in ("bp_math.cuh", "bp_mvie.cuh", "bp_lp.cuh", "bp_fk.cuh", "bp_mvie_fixed_r.cuh", "bp_mvie_pd.cuh",
                  "bp_planner.h")]
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-pthread", "-ffp-contract=off", "-o", so,
                               src])
    return ctypes.CDLL(so)


class _SharedScenesHarness:
    """The mapped harness behind the one oracle runner (tests.util.run_native_with_oracle): the runner's
    hh_plan_batch call plans the batch over shared scenes instead -- the same queries in their shared form, packed by
    PackedQueries with ``scenes=`` (every scene once, the query -> scene map) -- through hh_plan_batch_mapped, with the
    runner's callbacks and into the runner's output buffers."""

    def __init__(self, lib, queries, query_scene, scene_list, inflate, ws_max, ws_min, seeds, sample_chunk=32):
        shared, scene_list = shared_form(queries, query_scene, scene_list)
        self.lib = lib
        self.packed = pn.PackedQueries(shared, inflate, ws_max, ws_min, seeds, sample_chunk, scenes=scene_list)

    def hh_plan_batch(self, inp, out, *callbacks_and_lanes):
        assert inp._obj.Q == self.packed.Q          # (the runner's per-query packing of the same batch)
        return self.lib.hh_plan_batch_mapped(ctypes.byref(self.packed.inp),
                                             self.packed.query_scene.ctypes.data_as(ctypes.POINTER(ctypes.c_int)), out,
                                             *callbacks_and_lanes)


def _run_both(harness, mapped_lib, queries, scene_list, infl, seeds, backends, query_scene, lanes=1):
    """(the driver on one scene copy per query, the driver over the shared scenes scene_list, the shared
    PackedQueries), both with every request answered by the oracle."""
    wmin, wmax = list(WMIN), list(WMAX)
    want = run_native_with_oracle(harness, queries, infl, wmax, wmin, seeds, backends, lanes=lanes)
    shared = _SharedScenesHarness(mapped_lib, queries, query_scene, scene_list, infl, wmax, wmin, seeds)
    got = run_native_with_oracle(shared, queries, infl, wmax, wmin, seeds, backends, lanes=lanes)
    return want, got, shared.packed


def _cpu_check(harness, mapped_lib, scene_list, infl, query_scene, backends_of_scene, lanes, seed):
    wmin, wmax = list(WMIN), list(WMAX)
    queries = _copies(scene_list, infl, query_scene, seed)
    backends = [backends_of_scene[s] for s in query_scene]
    seeds = [seed + k for k in range(len(queries))]
    want, got, packed = _run_both(harness, mapped_lib, queries, scene_list, infl, seeds, backends, query_scene, lanes)
    assert packed.box_off.shape[0] == len(scene_list) + 1 and want.box_off.shape[0] == len(queries) + 1
    _assert_same_packed(got, want)
    results = got.results()
    for i, q in enumerate(queries):
        w, pl = python_plan(q, infl, wmax, wmin, seeds[i], backends[i])
        assert_same_result(results[i], w, pl, i, exact=True)
        assert [int(v) for v in got.rng_out[i]] == pn.rng_state_words(pl.rng)
    return queries, results, seeds


@pytest.fixture(scope="module")
def box_scenes():
    sc = [_box_scene(i) for i in (0, 1)]
    infl = sc[0][1]
    wmin, wmax = list(WMIN), list(WMAX)
    return [s for s, _ in sc], infl, [MemoBackend(s["obstacles"], infl, wmax, wmin) for s, _ in sc]


@pytest.mark.parametrize("lanes", [1, 2])
def test_boxes_mapped_equals_copies_on_cpu(host_harness, mapped_harness, box_scenes, lanes):
    scene_list, infl, backends = box_scenes
    _cpu_check(host_harness, mapped_harness, scene_list, infl, [0, 1, 1, 0, 1, 0], backends, lanes, seed=40)


def test_polytopes_mapped_equals_copies_on_cpu(host_harness, mapped_harness):
    sc = [_poly_scene(i) for i in (0, 1)]
    infl = sc[0][1]
    scene_list = [s for s, _ in sc]
    backends = [PolytopeOracleBackend(s["obs_sets"], s["obs_points_sets"], list(WMAX), list(WMIN)) for s in scene_list]
    pk_queries, _, _ = _cpu_check(host_harness, mapped_harness, scene_list, infl, [1, 0, 0, 1], backends, 1, seed=60)
    assert all("obs_sets" in q for q in pk_queries)


def test_replanning_mapped_equals_copies_on_cpu(host_harness, mapped_harness, box_scenes):
    """One mpc_step replanning call per planned query (one of them with new_obs) over shared scenes."""
    scene_list, infl, backends_of_scene = box_scenes
    wmin, wmax = list(WMIN), list(WMAX)
    query_scene = [0, 1, 1, 0, 1, 0]
    queries, results, seeds = _cpu_check(host_harness, mapped_harness, scene_list, infl, query_scene,
                                         backends_of_scene, 1, seed=40)
    planned = [i for i, r in enumerate(results) if not isinstance(r, Exception)]
    assert planned, "no query of the batch planned"
    nxt = [mpc_step(queries[i], results[i]) for i in planned]
    nxt[-1] = dict(nxt[-1], new_obs=True)
    qs = [query_scene[i] for i in planned]
    backends = [backends_of_scene[s] for s in qs]
    seeds = [s + 100 for s in seeds[: len(nxt)]]
    want, got, packed = _run_both(host_harness, mapped_harness, nxt, scene_list, infl, seeds, backends, qs)
    assert packed.box_off.shape[0] == len(scene_list) + 1 and packed.replan is not None
    _assert_same_packed(got, want)
    res = got.results()
    for i, q in enumerate(nxt):
        w, pl = python_plan(q, infl, wmax, wmin, seeds[i], backends[i])
        assert_same_result(res[i], w, pl, i, exact=True)
    assert int(got.replan["replanning"].sum()) == len(nxt)


def test_malformed_shared_batches_raise_without_a_device():
    """Every ValueError of a malformed batch over shared scenes comes before anything touches the device."""
    b = scenes.random_box_scene(5, np.random.default_rng(0))
    poly, _ = scenes.random_polytope_scene(3, np.random.default_rng(1))
    base = dict(start=np.array([0.1, 0.0, 0.5]), end=np.array([0.4, 0.2, 0.6]), r0=R0, r1=R0)
    sc = [dict(obstacles=b), dict(obstacles=b + 0.1)]
    cases = [
        ([dict(base, scene=2)], sc, "out of range"),
        ([dict(base, scene=-1)], sc, "out of range"),
        ([dict(base, scene=1.0)], sc, "not an int"),
        ([dict(base, scene="0")], sc, "not an int"),
        ([dict(base, scene=0, obstacles=b)], sc, "both 'scene' and obstacles"),
        ([dict(base, scene=0, obs_sets=poly)], sc, "both 'scene' and obstacles"),
        ([dict(base)], sc, "no 'scene'"),
        ([dict(base, scene=0)], [dict(obstacles=b), dict(obs_sets=poly)], "mixes box and polytope scenes"),
        ([dict(base, scene=0)], [dict(obstacles=b, obs_sets=poly)], "scene 0 must carry either"),
        ([dict(base, scene=0)], None, "no scenes were given"),
        ([dict(base, scene=0)], [], "scenes is empty"),
    ]
    for queries, scene_list, msg in cases:
        with pytest.raises(ValueError, match=msg):
            pn.NativePlanner(queries, scenes=scene_list)
        with pytest.raises(ValueError, match=msg):
            pn.plan_batch_native(queries, scenes=scene_list)
        with pytest.raises(ValueError, match=msg):
            plan_batch(queries, scenes=scene_list)
        with pytest.raises(ValueError, match=msg):
            pn.PackedQueries(queries, 0.01, WMAX, WMIN, scenes=scene_list)
    # the shared form of a batch packs every scene once
    queries = [dict(base, obstacles=sc[s]["obstacles"]) for s in (1, 0, 1)]
    shared, sl = shared_form(queries, [1, 0, 1])
    pk = pn.PackedQueries(shared, 0.01, WMAX, WMIN, scenes=sl)
    assert pk.box_off.tolist() == [0, 5, 10] and pk.query_scene.tolist() == [1, 0, 1]
    assert np.array_equal(pk.boxes, np.vstack((b, b + 0.1)))


# ---- GPU ------------------------------------------------------------------------------------------------------
def _native(queries, infl, seeds, scene_list=None, query_scene=None):
    """NativePlanner over shared scenes (scene_list, query_scene) or over the queries' copies: (results, stats)."""
    if scene_list is not None:
        queries, scene_list = shared_form(queries, query_scene)
    pl = pn.NativePlanner(queries, infl, WMAX, WMIN, scenes=scene_list)
    try:
        return pl.run(seeds)
    finally:
        pl.close()


@pytest.mark.gpu
def test_native_boxes_shared_equals_copies():
    sc = [_box_scene(i) for i in range(4)]
    infl = sc[0][1]
    scene_list = [s for s, _ in sc]
    query_scene = [k % 4 for k in range(256)]
    queries = _copies(scene_list, infl, query_scene, seed=300)
    seeds = [500 + k for k in range(256)]
    got, gst = _native(queries, infl, seeds, scene_list, query_scene)
    want, wst = _native(queries, infl, seeds)
    _assert_same_plans(got, want, gst, wst)
    assert sum(not isinstance(r, Exception) for r in got) >= 16
    shared, sl = shared_form(queries[:24], query_scene[:24])
    py, _ = plan_batch(shared, infl, WMAX, WMIN, rng_seeds=seeds[:24], scenes=sl)
    assert _assert_like_plan_batch(got[:24], py) >= 2


@pytest.mark.gpu
@pytest.mark.parametrize("given", [True, False], ids=["vertices_given", "vertices_enumerated"])
def test_native_polytopes_shared_equals_copies(given):
    sc = [_poly_scene(i) for i in range(2)]
    infl = sc[0][1]
    scene_list = [s if given else dict(s, obs_points_sets=None) for s, _ in sc]
    query_scene = [(k // 3) % 2 for k in range(48)]
    queries = _copies(scene_list, infl, query_scene, seed=700)
    seeds = [900 + k for k in range(48)]
    got, gst = _native(queries, infl, seeds, scene_list, query_scene)
    want, wst = _native(queries, infl, seeds)
    _assert_same_plans(got, want, gst, wst)
    assert sum(not isinstance(r, Exception) for r in got) >= 4
    shared, sl = shared_form(queries[:12], query_scene[:12])
    py, _ = plan_batch(shared, infl, WMAX, WMIN, rng_seeds=seeds[:12], scenes=sl)
    _assert_like_plan_batch(got[:12], py)


@pytest.mark.gpu
def test_native_large_scene_shared_equals_copies():
    """64 queries in the 1000-box C2 scene."""
    ob, infl, _, _, _ = scenes.config_c2()
    scene_list = [dict(obstacles=ob)]
    query_scene = [0] * 64
    queries = _copies(scene_list, infl, query_scene, seed=1100)
    seeds = list(range(64))
    got, gst = _native(queries, infl, seeds, scene_list, query_scene)
    want, wst = _native(queries, infl, seeds)
    _assert_same_plans(got, want, gst, wst)


def _moved_scene(s, rng):
    if "obs_sets" in s:
        sets, pts = scenes.moved_obstacles(s["obs_sets"], rng, obs_points=s.get("obs_points_sets"))
        return dict(obs_sets=sets, obs_points_sets=pts)
    return dict(obstacles=scenes.moved_obstacles(np.asarray(s["obstacles"]), rng))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["boxes", "polytopes"])
def test_mpc_loop_over_shared_scenes(kind):
    """3 MPC steps of 24 queries over 3 shared scenes that move every step: update_obstacles(queries, scenes=...)
    then the replanning calls, each step equal to a fresh planner on one copy per query; failed updates raise and
    leave the planner as it was."""
    make = _box_scene if kind == "boxes" else _poly_scene
    sc = [make(i) for i in range(3)]
    infl = sc[0][1]
    scene_list = [s for s, _ in sc]
    query_scene = [k % 3 for k in range(24)]
    copies = _copies(scene_list, infl, query_scene, seed=1300)
    queries, _ = shared_form(copies, query_scene)
    pl = pn.NativePlanner(queries, infl, WMAX, WMIN, scenes=scene_list)
    n_rep = 0
    try:
        for step in range(3):
            seeds = [40 * step + i for i in range(24)]
            if step:
                pl.update_obstacles(queries, scenes=scene_list)
            got, gst = pl.run(seeds)
            want, wst = _native(copies, infl, seeds)
            _assert_same_plans(got, want, gst, wst)
            if step == 1:
                other = [make(i)[0] for i in range(3, 6)]
                other_kind = [_poly_scene(0)[0] if kind == "boxes" else _box_scene(0)[0]] * 3
                for bad, msg in ((scene_list[:2], "2 scenes for a planner of 3"), (other_kind, "scenes hold"),
                                 (None, "updated with scenes=")):
                    with pytest.raises(ValueError, match=msg):
                        pl.update_obstacles(queries, scenes=bad)
                shifted = [dict(q, scene=(q["scene"] + 1) % 3) for q in queries]
                with pytest.raises(ValueError, match="scene indices differ"):
                    pl.update_obstacles(shifted, scenes=other)
                with pytest.raises(ValueError, match="scene indices differ"):
                    pl.run(seeds, queries=shifted)
                with pytest.raises(ValueError, match="no 'scene'"):
                    pl.run(seeds, queries=copies)
                again, ast = pl.run(seeds)
                _assert_same_plans(again, got, ast, gst)
                again, ast = pl.run(seeds, queries=queries)
                _assert_same_plans(again, got, ast, gst)
            rng = np.random.default_rng(77 + step)
            scene_list = [_moved_scene(s, rng) for s in scene_list]
            nxt_q, nxt_c = [], []
            for q, c, g in zip(queries, copies, got):
                if isinstance(g, Exception):
                    nq = dict(q, replanning=False, new_obs=True)
                else:
                    nq = dict(mpc_step(q, g), new_obs=True)
                    n_rep += step > 0
                nxt_q.append(nq)
                nxt_c.append(dict({k: v for k, v in nq.items() if k != "scene"}, **scene_list[q["scene"]]))
            queries, copies = nxt_q, nxt_c
    finally:
        pl.close()
    assert n_rep >= 3


@pytest.mark.gpu
def test_mapped_plan_abi_errors():
    from boundplanner_b200 import _lib
    from boundplanner_b200 import geometry as geo

    lib = _lib.load()
    sc = [_box_scene(i)[0] for i in range(3)]
    infl = 0.01
    batch = geo.SceneBatch([s["obstacles"] for s in sc], infl)
    h = ctypes.c_void_p(0)
    ip = ctypes.POINTER(ctypes.c_int)
    try:
        bad = np.array([0, 2, 3, 1], np.int32)
        assert lib.bp_plan_create_mapped(batch._h, 4, bad.ctypes.data_as(ip), ctypes.byref(h)) != 0
        assert b"query 2 maps to scene 3, the batch has 3 scenes" in lib.bp_last_error_string()
        assert not h.value
        query_scene = [2, 0, 2, 1]
        queries, _ = shared_form(_copies(sc, infl, query_scene, seed=5), query_scene)
        mp = np.asarray(query_scene, np.int32)
        _lib.check(lib.bp_plan_create_mapped(batch._h, 4, mp.ctypes.data_as(ip), ctypes.byref(h)))
        # the input's scene 1 loses an obstacle: the call fails before any round runs
        short = [sc[0], dict(obstacles=sc[1]["obstacles"][:-1]), sc[2]]
        pk = pn.PackedQueries(queries, infl, WMAX, WMIN, list(range(4)), scenes=short)
        assert lib.bp_plan_run(h, ctypes.byref(pk.inp), ctypes.byref(pk.out), None) != 0
        assert b"scene 1 has 199 obstacles in the input, 200 in the plan's scene batch" in lib.bp_last_error_string()
        assert int(pk.stats[0]) == 0 and int(pk.n_nodes.sum()) == 0
    finally:
        if h.value:
            lib.bp_plan_destroy(h)
        batch.close()


@pytest.mark.gpu
def test_collision_sets_over_a_scene_batch():
    """collision_sets with robot_scene over a batch of 3 scenes equals the per-robot calls on the single scenes."""
    from boundplanner_b200 import geometry as geo
    from boundplanner_b200 import mpc_geometry as mg

    rng = np.random.default_rng(9)
    # (at most 6 + 8 rows per joint set: within the 15 rows the joint sets are padded to)
    boxes = [scenes.random_box_scene(8, rng, 0.1, 0.3) for _ in range(3)]
    batch = geo.SceneBatch(boxes, 0.0)
    singles = [geo.Scene(bx, 0.0) for bx in boxes]
    robot_scene = np.array([2, 0, 1, 2, 0, 1, 1])
    q_start = np.array([0, 0, 0, -np.pi / 2, 0, np.pi / 2, 0.0])
    q0 = q_start[None] + rng.uniform(-0.4, 0.4, (7, 7))
    qf = q0 + rng.uniform(-0.05, 0.05, (7, 7))
    try:
        A, b, coll = mg.collision_sets(batch, q0, qf, WMIN, WMAX, robot_scene=robot_scene)
        for t, s in enumerate(robot_scene):
            a1, b1, c1 = mg.collision_sets(singles[s], q0[t], qf[t], WMIN, WMAX)
            assert np.array_equal(A[t].view(np.uint8), a1[0].view(np.uint8)), t
            assert np.array_equal(b[t].view(np.uint8), b1[0].view(np.uint8)), t
            assert np.array_equal(coll[t], c1[0]), t
        with pytest.raises(ValueError, match="robot_scene has 6 entries for 7 robots"):
            mg.collision_sets(batch, q0, qf, WMIN, WMAX, robot_scene=robot_scene[:6])
    finally:
        batch.close()
        for s in singles:
            s.close()
