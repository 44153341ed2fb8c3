"""Replanning in the batched planner drivers: the replanning branch of plan_convex_set_path (:231-276) and the
start-in-collision fallbacks (:296-324), as an MPC loop calls the planner again and again with the previous call's
sets (``sets_via_prev``).

CPU: the native driver's state machines (csrc/bp_planner.h) in the host harness, the oracle answering their requests,
against SetSequencePlanner.plan_set_sequence with the same answers -- boxes and polytopes, the C1 replanning scenario,
3-step MPC sequences and every fallback -- and planner.plan_batch with an oracle executor on the same sequences:
paths, set sequences, via points (bit for bit), graph sizes, p_horizon_max, the returned sets_via_prev, exception
type and message and the generator state afterwards.
GPU: bp_plan_run against planner.plan_batch over the kernels (and both against plan_set_sequence on the GpuBackend),
a 5-step MPC loop, and batches without replanning inputs against batches with all of them zero."""
import ctypes

import numpy as np
import pytest

from boundplanner_b200 import planner_native as pn
from boundplanner_b200 import scenes
from boundplanner_b200.planner import SetSequencePlanner, plan_batch
from tests.util import (ERRORS, R0, MemoBackend, OracleLockstepExecutor, _backend, _c3, _c3_poly, _dp, _ip, _is_poly,
                        _same_sets, assert_same_result, mpc_step, python_plan, run_native_with_oracle)

P0 = np.array([0.3, 0.0, 0.7])                  # boundplanner_example.py:89-92
P1 = np.array([0.45, -0.5, 0.2])


# ---- the two sides, the oracle answering both -------------------------------------------------------------------
def check_native(harness, queries, inflate, ws_max, ws_min, seeds):
    """plan_set_sequence, the native state machines and plan_batch (oracle executor) on one batch: identical."""
    backends = [_backend(q, inflate, ws_max, ws_min) for q in queries]
    want = [python_plan(q, inflate, ws_max, ws_min, s, be) for q, s, be in zip(queries, seeds, backends)]
    pk = run_native_with_oracle(harness, queries, inflate, ws_max, ws_min, seeds, backends)
    got = pk.results()
    for i, ((w, pl), g) in enumerate(zip(want, got)):
        assert_same_result(g, w, pl, i)
        assert [int(v) for v in pk.rng_out[i]] == pn.rng_state_words(pl.rng), f"query {i}: generator state"
    ex = OracleLockstepExecutor(backends)
    res, stats = plan_batch(queries, inflate, ws_max, ws_min, rng_seeds=seeds, executor=ex)
    assert stats["rounds"] == ex.calls
    for i, ((w, pl), g) in enumerate(zip(want, res)):
        assert_same_result(g, w, pl, i)
    return want, got


# ---- queries -------------------------------------------------------------------------------------------------
def _inside_point(q, away_from):
    """A point inside one of the query's inflated obstacles, 0.15 m or more from `away_from`."""
    if _is_poly(q):
        centres = [v.mean(axis=0) for v in q["obs_points_sets"]]
    else:
        centres = [0.5 * (b[:3] + b[3:]) for b in np.asarray(q["obstacles"], float)]
    return next(c for c in centres if np.linalg.norm(c - away_from) > 0.15)


def fallback_queries(q, prev_sets):
    """A start segment that runs into an obstacle, with every fallback of :296-324 and a horizon too short."""
    through = _inside_point(q, q["start"])
    hz = np.array([q["start"], through])
    return [dict(q, replanning=True, p_horizon=hz),                                     # IndexError (first plan)
            dict(q, replanning=True, p_horizon=hz, sets_via_prev=prev_sets),            # previous end set reused
            dict(q, replanning=True, p_horizon=hz, new_obs=True),                       # rebuilt around start
            dict(q, start=through, replanning=True, p_horizon=np.array([through, q["start"]]),
                 new_obs=True),                                                         # AttributeError (Q12)
            dict(q, replanning=True, p_horizon=hz[:1], new_obs=True),                   # horizon too short
            dict(q, replanning=True, p_horizon=np.zeros((0, 3)), sets_via_prev=prev_sets)]


# ---- CPU ------------------------------------------------------------------------------------------------------
def test_c1_replanning_and_fallbacks_native_equals_python(host_harness):
    """The C1 scenario of the sequential driver's replanning test, and every fallback, in one lock-step batch."""
    boxes, ws_min, ws_max, inflate = scenes.example_scene()
    ws_min, ws_max = list(ws_min), list(ws_max)
    base = dict(obstacles=boxes, start=P0, end=P1, r0=R0, r1=R0)
    first, pl0 = python_plan(base, inflate, ws_max, ws_min, 0, MemoBackend(boxes, inflate, ws_max, ws_min))
    prev = [[a.copy(), b.copy()] for a, b in pl0.sets_via_prev]
    p_via = first["p_via"]
    horizon = np.array([p_via[0] + t * (p_via[1] - p_via[0]) for t in np.linspace(0.05, 0.6, 8)])
    start = p_via[0] + 0.02 * (p_via[1] - p_via[0])
    below = np.array([0.0, -0.6, 0.53 - inflate - 0.03])        # its tool tip lies in obstacle 5: the tip segment collides
    queries = [base,
               dict(base, start=start, replanning=True, p_horizon=horizon, sets_via_prev=prev),
               dict(base, start=start, replanning=True, p_horizon=horizon, sets_via_prev=prev, new_obs=True),
               dict(base, start=below),                                                   # IndexError
               dict(base, start=below, sets_via_prev=prev),                               # previous end set reused
               dict(base, start=below, new_obs=True)]                                     # rebuilt around start
    queries += fallback_queries(base, prev)
    want, got = check_native(host_harness, queries, inflate, ws_max, ws_min, list(range(len(queries))))
    kinds = [type(w).__name__ if isinstance(w, Exception) else "planned" for w, _ in want]
    assert kinds[:3] == ["planned"] * 3 and kinds[3] == "IndexError" and kinds[4:6] == ["planned"] * 2, kinds
    assert kinds[6:] == ["IndexError", "planned", "planned", "AttributeError", "IndexError", "IndexError"], kinds
    assert str(want[10][0]) == "index 1 is out of bounds for axis 0 with size 1"
    assert str(want[11][0]) == "index -1 is out of bounds for axis 0 with size 0"       # start in a previous set
    # the reused end set: node 0 is reduce_ineqs of the previous last set, q_ellipse = I
    g0 = want[4][0]["graph"].nodes[0]
    assert np.array_equal(g0["q_ellipse"], np.eye(3)) and np.array_equal(g0["p_mid"], below)
    assert got[1]["p_horizon_max"] is not None and "p_horizon_max" not in got[0]


@pytest.mark.parametrize("kind", ["boxes", "polytopes"])
def test_mpc_sequences_native_equals_python(host_harness, kind):
    """3-step MPC sequences on six C3 queries: every step's batch mixes replanning queries (the planned ones, their
    sets threaded forward) with first plans (the failed ones, which keep the caller's sets) and fallbacks."""
    make = _c3 if kind == "boxes" else _c3_poly
    base, infl, wmin, wmax = [], None, None, None
    for i in (0, 1, 5, 7, 8, 11) if kind == "boxes" else range(6):
        q, infl, wmin, wmax = make(i)
        base.append(q)
    queries, seeds = list(base), list(range(len(base)))
    n_replanned = 0
    for step in range(3):
        want, _ = check_native(host_harness, queries, infl, wmax, wmin, seeds)
        nxt = []
        for q, (w, pl) in zip(queries, want):
            if isinstance(w, Exception):
                nxt.append(dict(q, replanning=False, sets_via_prev=[[a.copy(), b.copy()] for a, b in pl.sets_via_prev]))
            else:
                w["sets_via_prev"] = pl.sets_via_prev
                nxt.append(mpc_step(q, w))
                n_replanned += 1
        if step == 0:                                                   # the fallbacks, once, on the first query
            ok = next(w for w, _ in want if not isinstance(w, Exception))
            nxt += fallback_queries(base[0], ok["sets_via_prev"])
        queries, seeds = nxt, [s + 100 for s in range(len(nxt))]
    assert n_replanned >= 6


def test_native_driver_rejects_malformed_replanning_inputs(host_harness):
    q, infl, wmin, wmax = _c3(0)
    good = [[np.eye(3), np.ones(3)]]
    with pytest.raises(ValueError, match="previous sets"):
        pn.PackedQueries([dict(q, sets_via_prev=good * 65)], infl, wmax, wmin, [0])
    for bad in ([[np.zeros((0, 3)), np.zeros(0)]], [[np.ones((49, 3)), np.ones(49)]], [[np.ones((4, 3)), np.ones(3)]]):
        with pytest.raises(ValueError, match="rows"):
            pn.PackedQueries([dict(q, sets_via_prev=bad)], infl, wmax, wmin, [0])
    # the C side checks the same (and the offsets) before any round: hand-made arrays
    cases = [("prev_off", np.array([0, 65], np.int32), "65 previous sets"),
             ("prev_off", np.array([1, 1], np.int32), "prev_off[0]"),
             ("horizon_off", np.array([0, -1], np.int32), "horizon_off decreases"),
             ("prev_row_off", np.array([0, 49], np.int32), "49 rows")]
    for field, arr, msg in cases:
        pk = pn.PackedQueries([dict(q, replanning=True, p_horizon=[q["start"]], sets_via_prev=good)], infl, wmax, wmin, [0])
        setattr(pk.inp, field, arr.ctypes.data_as(_ip))
        pk.keep = arr
        rows = np.zeros((65, 4))
        pk.inp.prev_rows = rows.ctypes.data_as(_dp)
        pk.keep_rows = rows
        assert host_harness.hh_plan_batch(ctypes.byref(pk.inp), ctypes.byref(pk.out), None, None, None, None,
                                          None, 1) == 3
        assert msg in pk.err_msg.value.decode(), (field, pk.err_msg.value)
    pk = pn.PackedQueries([dict(q, replanning=True)], infl, wmax, wmin, [0])
    pk.inp.horizon_off = None
    assert host_harness.hh_plan_batch(ctypes.byref(pk.inp), ctypes.byref(pk.out), None, None, None, None,
                                      None, 1) == 3
    assert b"without horizon_off" in pk.err_msg.value


def test_horizon_index_uses_the_element_wise_rows():
    """replanning_horizon_index decides every threshold on (a0 x0 + a1 x1) + a2 x2 - b, element by element."""
    from boundplanner_b200.planner import _rows_minus_b

    rng = np.random.default_rng(3)
    for _ in range(20):
        sets = [[rng.normal(size=(7, 3)), rng.uniform(0.2, 1.0, 7)] for _ in range(3)]
        start = rng.normal(scale=0.05, size=3)
        horizon = start + np.cumsum(rng.normal(scale=0.1, size=(6, 3)), axis=0)
        pl = SetSequencePlanner(())
        pl.sets_via_prev = sets
        want = 1
        for a, b in sets:
            start_in = _rows_minus_b(a, b, start).max() < 1e-8
            out = [k for k, h in enumerate(horizon) if not _rows_minus_b(a, b, h).max() < 1e-8]
            if out:
                if out[0] != 0 and start_in:
                    want = max(want, out[0] - 1)
            elif start_in:
                want = len(horizon) - 1
                break
        assert pl.replanning_horizon_index(start, horizon) == want
        assert pl.replanning_horizon_index(start, horizon, new_obs=True) == 1


# ---- GPU ------------------------------------------------------------------------------------------------------
def _replan_batch(make, ids):
    """First plans of queries `ids` on the native driver, then the MPC replanning batch built from them: planned
    queries move on (mpc_step), failed ones are planned again from scratch, and every fourth planned query is
    turned into one of the fallbacks."""
    base, infl, wmin, wmax = [], None, None, None
    for i in ids:
        q, infl, wmin, wmax = make(i)
        base.append(q)
    first, _ = pn.plan_batch_native(base, infl, wmax, wmin, rng_seeds=list(ids))
    queries = []
    for k, (q, r) in enumerate(zip(base, first)):
        if isinstance(r, Exception):
            queries.append(q)
        elif k % 4 == 3:
            queries.append(fallback_queries(q, r["sets_via_prev"])[(k // 4) % 6])
        else:
            queries.append(mpc_step(q, r))
    return base, queries, infl, wmin, wmax


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["boxes", "polytopes"])
def test_native_replanning_equals_python_plan_batch_on_gpu(kind):
    """bp_plan_run == planner.plan_batch over the kernels on 24 C3 replanning queries incl. fallbacks; a few of them
    also == plan_set_sequence on the GpuBackend."""
    from boundplanner_b200.planner import GpuBackend

    ids = list(range(24))
    base, queries, infl, wmin, wmax = _replan_batch(_c3 if kind == "boxes" else _c3_poly, ids)
    seeds = [100 + i for i in ids]
    want, _ = plan_batch(queries, infl, wmax, wmin, rng_seeds=seeds)
    npl = pn.NativePlanner(base, infl, wmax, wmin)
    try:
        got, stats = npl.run(seeds, queries=queries)
    finally:
        npl.close()
    assert stats["kernel_chains"] <= stats["rounds"] * stats["lanes"]
    n_ok = n_rep = 0
    for i, (w, g) in enumerate(zip(want, got)):
        if isinstance(w, Exception):
            assert isinstance(g, Exception) and type(g) is type(w), (i, g, w)
            assert str(g).split("(")[0] == str(w).split("(")[0], (i, g, w)
            continue
        n_ok += 1
        n_rep += "p_horizon_max" in w
        assert not isinstance(g, Exception), f"query {i}: {g!r}"
        assert g["path"] == w["path"] and g["set_ids"] == w["set_ids"], i
        assert np.abs(g["p_via"] - w["p_via"]).max() < 1e-9, i
        assert g["n_nodes"] == w["graph"].number_of_nodes() and g["n_inter"] == w["inter_graph"].number_of_nodes()
        _same_sets(g["sets_via_prev"], w["sets_via_prev"], 1e-12)
        assert ("p_horizon_max" in g) == ("p_horizon_max" in w)
        if "p_horizon_max" in w:
            assert np.array_equal(g["p_horizon_max"], w["p_horizon_max"]), i
    assert n_ok >= 6 and n_rep >= 4
    for i in ids[:6]:                                         # the sequential driver on the GpuBackend
        q = queries[i]
        pl = SetSequencePlanner(() if _is_poly(q) else q["obstacles"], infl, wmax, wmin, rng=np.random.default_rng(seeds[i]),
                                obs_sets=q.get("obs_sets"), obs_points_sets=q.get("obs_points_sets"))
        pl.sets_via_prev = [[np.array(a), np.array(b)] for a, b in q.get("sets_via_prev", ())]
        try:
            res = pl.plan_set_sequence(q["start"].copy(), q["end"].copy(), R0, R0, None, q.get("replanning", False),
                                       q.get("p_horizon", ()), q.get("new_obs", False))
        except ERRORS as e:
            res = e
        assert isinstance(pl.backend, GpuBackend)
        assert_same_result(want[i], res, pl, i, exact=False)
        assert_same_result(got[i], res, pl, i, exact=False)


@pytest.mark.gpu
def test_mpc_loop_threads_sets_forward_on_gpu():
    """A 5-step MPC loop of 8 queries on one NativePlanner (run(queries=...) over the same scenes): every step equals
    plan_batch on the same inputs, and the native results' sets_via_prev feed the next step."""
    ids = list(range(8))
    base = [_c3(i)[0] for i in ids]
    _, infl, wmin, wmax = _c3(0)
    npl = pn.NativePlanner(base, infl, wmax, wmin)
    try:
        queries, n_rep = base, 0
        for step in range(5):
            seeds = [10 * step + i for i in ids]
            got, _ = npl.run(seeds, queries=queries)
            want, _ = plan_batch(queries, infl, wmax, wmin, rng_seeds=seeds)
            nxt = []
            for i, (q, g, w) in enumerate(zip(queries, got, want)):
                if isinstance(w, Exception):
                    assert type(g) is type(w), (step, i, g, w)
                    nxt.append(dict(q, replanning=False))
                    continue
                assert g["path"] == w["path"] and g["set_ids"] == w["set_ids"], (step, i)
                assert np.abs(g["p_via"] - w["p_via"]).max() < 1e-9
                _same_sets(g["sets_via_prev"], w["sets_via_prev"], 1e-12)
                n_rep += step > 0 and "p_horizon_max" in g
                nxt.append(mpc_step(q, g))
            queries = nxt
        assert n_rep >= 8
        with pytest.raises(ValueError, match="obstacles differ"):
            npl.run([0] * 8, queries=[_c3(i + 1)[0] for i in ids])
    finally:
        npl.close()


@pytest.mark.gpu
def test_null_and_zero_replanning_fields_plan_like_before():
    """24 C3 first plans: the replanning fields NULL (a batch without the keys) and all zero give the same bits, the
    same rounds and one kernel chain per lane round."""
    ids = list(range(24))
    base = [_c3(i)[0] for i in ids]
    _, infl, wmin, wmax = _c3(0)
    npl = pn.NativePlanner(base, infl, wmax, wmin)
    try:
        a, sa = npl.run(ids)
        assert npl._packed[next(iter(npl._packed))].replan is None
        zeros = [dict(q, replanning=False, new_obs=False, p_horizon=np.zeros((0, 3)), sets_via_prev=[]) for q in base]
        b, sb = npl.run(ids, queries=zeros)
    finally:
        npl.close()
    assert sa["rounds"] == sb["rounds"] and sa["kernel_chains"] == sb["kernel_chains"]
    assert sa["set_requests"] == sb["set_requests"] and sa["pair_tests"] == sb["pair_tests"]
    for x, y in zip(a, b):
        if isinstance(x, Exception):
            assert type(x) is type(y) and str(x) == str(y)
            continue
        assert x["path"] == y["path"] and x["set_ids"] == y["set_ids"] and np.array_equal(x["p_via"], y["p_via"])
        _same_sets(x["sets_via"], y["sets_via"])
        assert "p_horizon_max" not in x and "p_horizon_max" not in y
