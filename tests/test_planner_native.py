"""The native lock-step planner driver (csrc/bp_planner.h: per-query state machines + numpy's PCG64 stream in C++)
against the Python planner loop (boundplanner_b200/planner.py).  CPU: the driver is compiled into the host harness
with its requests answered by callbacks into the oracle -- the same answers the Python planner gets -- so paths, set
sequences, via points, graph sizes, error exits and the generator state after the query must agree exactly.
GPU: ``bp_plan_batch`` (requests answered by the kernels) against ``planner.plan_batch`` on the same kernels."""
import ctypes

import numpy as np
import pytest
from scipy.spatial.transform import Rotation as R

from boundplanner_b200 import planner_native as pn
from boundplanner_b200 import scenes
from tests.util import (R0, EdgeAns, MemoBackend, Node, ProjAns, ReduceReq, SetAns, SetReq, _dp, assert_same_result,
                        python_plan, run_native_with_oracle)

R1 = R.from_euler("XYZ", [20, 70, -30], degrees=True).as_matrix()


def test_struct_layouts(host_harness):
    """The ctypes mirrors have the sizes of the C records (hh_sizeof), and the last fields of bp_plan_in / bp_plan_out
    end their records."""
    for k, t in enumerate((SetReq, SetAns, Node, EdgeAns, ProjAns, ReduceReq, pn.BpPlanIn, pn.BpPlanOut)):
        assert host_harness.hh_sizeof(k) == ctypes.sizeof(t), t.__name__
    assert pn.BpPlanIn.prev_rows.offset + ctypes.sizeof(_dp) == ctypes.sizeof(pn.BpPlanIn)
    assert pn.BpPlanOut.p_horizon_max.offset + ctypes.sizeof(_dp) == ctypes.sizeof(pn.BpPlanOut)


def test_pcg64_stream_is_numpys(host_harness):
    lo, hi = np.array([-1.0, -1.0, 0.0]), np.array([1.0, 1.0, 1.2])
    for seed in (0, 7, 123456789):
        g = np.random.default_rng(seed)
        st = np.array(pn.rng_state_words(g), np.uint64)
        want = g.uniform(lo, hi, (40, 3))
        got = np.zeros((40, 3))
        host_harness.hh_pcg64_uniform3(st.ctypes.data_as(ctypes.POINTER(ctypes.c_ulonglong)), lo.ctypes.data_as(_dp),
                                       hi.ctypes.data_as(_dp), 40, got.ctypes.data_as(_dp))
        assert np.array_equal(got, want)
        assert [int(v) for v in st] == pn.rng_state_words(g)          # and the state afterwards
        # one at a time == in one call (what the driver's rewind relies on)
        g2 = np.random.default_rng(seed)
        assert np.array_equal(np.array([g2.uniform(lo, hi, 3) for _ in range(40)]), want)


def test_native_driver_equals_python_planner_on_cpu(host_harness):
    """Mixed batch in lock step: the C1 example scene (with and without first_sample, different end rotation) and
    C3 queries that plan, hit the 20-row cap (ValueError) or stop early."""
    boxes, ws_min, ws_max, inflate = scenes.example_scene()
    p0, p1 = np.array([0.3, 0.0, 0.7]), np.array([0.45, -0.5, 0.2])
    ws_min, ws_max = list(ws_min), list(ws_max)
    queries = [dict(obstacles=boxes, start=p0, end=p1, r0=R0, r1=R0),
               dict(obstacles=boxes, start=p0, end=p1, r0=R0, r1=R1, first_sample=np.array([0.5, -0.2, 0.6]))]
    seeds = [3, 1]
    pk = _check(host_harness, queries, inflate, ws_max, ws_min, seeds, chunk=5)
    assert pk.err_kind.sum() == 0 and pk.stats[0] > 5
    queries, seeds = [], []
    for i in (0, 1, 5, 7, 8, 11):
        ob, infl, st, en, wmin, wmax = scenes.config_c3_query(i)
        queries.append(dict(obstacles=ob, start=st, end=en, r0=R0, r1=R0))
        seeds.append(i)
    pk = _check(host_harness, queries, infl, list(wmax), list(wmin), seeds, chunk=32)
    assert (pk.err_kind != 0).sum() >= 1 and (pk.err_kind == 0).sum() >= 2
    # two and three independent lock-step lanes (query i -> lane i mod L), the state machines of a round resumed
    # by a pool of three host threads: the same answers per query
    import os

    os.environ["BPGEO_PLAN_THREADS"], os.environ["BPGEO_PLAN_POOL_MIN"] = "3", "1"
    for lanes in (2, 3):
        pk2 = _check(host_harness, queries, infl, list(wmax), list(wmin), seeds, chunk=32, lanes=lanes, backends=pk.backends)
        assert np.array_equal(pk2.err_kind, pk.err_kind) and pk2.stats[0] <= pk.stats[0]
    del os.environ["BPGEO_PLAN_THREADS"], os.environ["BPGEO_PLAN_POOL_MIN"]


def _check(host_harness, queries, inflate, ws_max, ws_min, seeds, chunk, lanes=1, backends=None):
    if backends is None:
        backends = [MemoBackend(q["obstacles"], inflate, ws_max, ws_min) for q in queries]
    want = [python_plan(q, inflate, ws_max, ws_min, s, be) for q, s, be in zip(queries, seeds, backends)]
    pk = run_native_with_oracle(host_harness, queries, inflate, ws_max, ws_min, seeds, backends, sample_chunk=chunk,
                                lanes=lanes)
    pk.backends = backends
    for i, ((w, pl), g) in enumerate(zip(want, pk.results())):
        assert_same_result(g, w, pl, i)
        assert [int(v) for v in pk.rng_out[i]] == pn.rng_state_words(pl.rng), f"query {i}: generator state"
    return pk


@pytest.mark.gpu
def test_native_plan_batch_equals_python_plan_batch_on_gpu():
    """bp_plan_batch (kernels answer the requests, tables on the device) == planner.plan_batch (Python lock-step
    driver over the same kernels) on 24 C3 queries incl. the error exits, and on the C1 scene."""
    from boundplanner_b200.planner import plan_batch

    ids = list(range(24))
    queries = []
    for i in ids:
        ob, infl, st, en, wmin, wmax = scenes.config_c3_query(i)
        queries.append(dict(obstacles=ob, start=st, end=en, r0=R0, r1=R0))
    want, _ = plan_batch(queries, infl, list(wmax), list(wmin), rng_seeds=ids)
    got, stats = pn.plan_batch_native(queries, infl, list(wmax), list(wmin), rng_seeds=ids)
    assert stats["rounds"] > 10
    n_ok = 0
    for i, (w, g) in enumerate(zip(want, got)):
        if isinstance(w, Exception):
            assert isinstance(g, Exception) and type(g) is type(w), (i, g, w)
            assert str(g).split("(")[0] == str(w).split("(")[0], (i, g, w)
            continue
        n_ok += 1
        assert not isinstance(g, Exception), f"query {i}: {g!r}"
        assert g["path"] == w["path"] and g["set_ids"] == w["set_ids"], i
        assert np.abs(g["p_via"] - w["p_via"]).max() < 1e-9
        assert g["n_nodes"] == w["graph"].number_of_nodes() and g["n_inter"] == w["inter_graph"].number_of_nodes()
        for (ga, gb), (wa, wb) in zip(g["sets_via"], w["sets_via"]):
            assert ga.shape == wa.shape and np.abs(ga - wa).max() < 1e-12 and np.abs(gb - wb).max() < 1e-12
    assert n_ok >= 6
    boxes, ws_min, ws_max, inflate = scenes.example_scene()
    q1 = [dict(obstacles=boxes, start=np.array([0.3, 0.0, 0.7]), end=np.array([0.45, -0.5, 0.2]), r0=R0, r1=R1,
               first_sample=np.array([0.5, -0.2, 0.6]))]
    want, _ = plan_batch(q1, inflate, list(ws_max), list(ws_min), rng_seeds=[1])
    got, _ = pn.plan_batch_native(q1, inflate, list(ws_max), list(ws_min), rng_seeds=[1])
    assert got[0]["path"] == want[0]["path"] and got[0]["set_ids"] == want[0]["set_ids"]
    assert np.abs(got[0]["p_via"] - want[0]["p_via"]).max() < 1e-9
