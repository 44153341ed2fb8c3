"""Planning over general convex polytope obstacles (obs_sets of up to 15 rows, as ConvexSetFinder takes them).

CPU: the native driver's state machines (csrc/bp_planner.h, general-row push-out of `end`) in the host harness with
the oracle answering their requests, against SetSequencePlanner with the same answers; the host-side push-out of
`end` (:199-204) on general rows against the reference's literal loop, and against the box arithmetic for boxes;
the new_obs start-in-collision quirk.
GPU: bp_plan_run over a polytope scene batch against planner.plan_batch; plan_set_sequence on the GPU backend
against the oracle backend; boxes handed over as polytopes against the same boxes; the kind checks."""
import ctypes

import numpy as np
import pytest

from boundplanner_b200 import planner_native as pn
from boundplanner_b200 import scenes
from boundplanner_b200.planner import SetSequencePlanner
from tests.util import R0, PolytopeOracleBackend, _c3_poly, assert_same_result, python_plan, run_native_with_oracle

ORDER_TOL = 1e-15          # general push-out vs the reference's `@` (BLAS may fuse): last bits only


def _literal_push_out(obs_sets, end, r):
    """BoundPlanner.py:199-204 verbatim."""
    end = np.array(end, float)
    for ob in obs_sets:
        viol = ob[0] @ end - ob[1]
        if not np.any(viol > 0):
            idx = np.argmax(viol)
            end -= (viol[idx] - r) * ob[0][idx, :]
    return end


def _padded(A, b):
    a_pad, b_pad = np.zeros((15, 3)), np.full(15, 10.0)
    a_pad[: len(A)], b_pad[: len(A)] = A, b
    return [a_pad, b_pad]


def _box_rows(lo, hi, cut=None):
    """[I; -I] rows of the box lo..hi, plus an optional extra (redundant) row that makes it a general polytope."""
    A = np.concatenate((np.eye(3), -np.eye(3)))
    b = np.concatenate((np.asarray(hi, float), -np.asarray(lo, float)))
    if cut is not None:
        A, b = np.vstack((A, cut[0])), np.append(b, cut[1])
    return _padded(A, b)


# ---- CPU: the native driver's state machines against the Python planner, the oracle answering both -----------
def test_native_driver_equals_python_planner_over_polytopes_on_cpu(host_harness):
    """Six C3 polytope queries (one with its `end` inside an obstacle) through the native state machines and through
    SetSequencePlanner, the oracle answering both: the same paths, set ids, via points (bit for bit), graph sizes,
    sets, error exits and generator states."""
    queries, seeds, backends = [], [], []
    for i in range(6):
        q, infl, wmin, wmax = _c3_poly(i)
        queries.append(q)
        seeds.append(i)
        backends.append(PolytopeOracleBackend(q["obs_sets"], q["obs_points_sets"], wmax, wmin))
    # query 2: `end` at the centroid of an obstacle that lies 0.3 m or more from `start` -- pushed out on the host
    q = queries[2]
    far = [k for k, v in enumerate(q["obs_points_sets"]) if np.linalg.norm(v.mean(axis=0) - q["start"]) > 0.3]
    q["end"] = q["obs_points_sets"][far[0]].mean(axis=0)
    pl = SetSequencePlanner((), infl, wmax, wmin, obs_sets=q["obs_sets"])
    assert pl.polytopes and pl._in_collision(q["end"])
    assert not np.array_equal(pl._push_out_general(q["end"].copy()), q["end"])

    want = [python_plan(q, infl, wmax, wmin, s, be) for q, s, be in zip(queries, seeds, backends)]
    pk = run_native_with_oracle(host_harness, queries, infl, wmax, wmin, seeds, backends)
    assert pk.kind == "polytopes" and pk.boxes is None
    for i, ((w, pl), g) in enumerate(zip(want, pk.results())):
        assert_same_result(g, w, pl, i)
        assert [int(v) for v in pk.rng_out[i]] == pn.rng_state_words(pl.rng), f"query {i}: generator state"
    assert (pk.err_kind != 0).sum() >= 1 and (pk.err_kind == 0).sum() >= 2, pk.err_kind


# ---- CPU: the push-out of `end` on general rows ----------------------------------------------------------------
def _planner(obs_sets, r=0.01):
    return SetSequencePlanner((), r, obs_sets=obs_sets)


def test_push_out_cases_match_the_reference_loop():
    r = 0.01
    cut = (np.array([1.0, 1.0, 1.0]) / np.sqrt(3.0), 5.0)                       # redundant row: a general polytope
    cases = []
    # inside one polytope (a random one of the C3 polytope scene, at its centroid)
    q, *_ = _c3_poly(0)
    cases.append((q["obs_sets"], q["obs_points_sets"][7].mean(axis=0), "inside one"))
    # two overlapping polytopes: pushed out of the first through x = 0.1; the moved `end` (not the given one) lies in
    # the second, which pushes it out through y = 0.045
    two = [_box_rows([0, 0, 0], [0.1, 0.1, 0.1], cut), _box_rows([0.1, 0.045, 0], [0.3, 0.1, 0.1], cut)]
    cases.append((two, np.array([0.09, 0.05, 0.05]), "two overlapping"))
    # exactly on a face: viol = 0 counts as inside
    half = [_box_rows([0, 0, 0], [0.5, 0.5, 0.5], cut)]
    cases.append((half, np.array([0.5, 0.25, 0.25]), "on a face"))
    # a two-face tie (x+ and y+ at viol 0): the first row wins
    cases.append((half, np.array([0.5, 0.5, 0.25]), "two-face tie"))
    for obs_sets, end, tag in cases:
        pl = _planner(obs_sets, r)
        assert pl.polytopes, tag
        got = pl._push_out_general(end.copy())
        want = _literal_push_out(obs_sets, end, r)
        assert np.abs(got - want).max() <= ORDER_TOL, tag
        assert not np.array_equal(got, end), tag
    def pushed(obs_sets, end):
        return _planner(obs_sets, r)._push_out_general(np.array(end, float))

    # the second obstacle of the overlapping pair saw the moved `end` (x = 0.11)
    assert np.allclose(pushed(two[:1], [0.09, 0.05, 0.05]), [0.11, 0.05, 0.05], rtol=0, atol=1e-15)
    assert np.allclose(pushed(two[1:], [0.09, 0.05, 0.05]), [0.09, 0.05, 0.05], rtol=0, atol=0)
    assert np.allclose(pushed(two, [0.09, 0.05, 0.05]), [0.11, 0.035, 0.05], rtol=0, atol=1e-15)
    assert np.array_equal(pushed(half, [0.5, 0.25, 0.25]), [0.5 + r, 0.25, 0.25])      # on the x+ face
    assert np.array_equal(pushed(half, [0.5, 0.5, 0.25]), [0.5 + r, 0.5, 0.25])        # x+ and y+ tie: x+ wins


def test_push_out_general_rows_equal_the_box_path_on_boxes():
    """Box obstacles (add_obstacle_reps rows): the general form, forced by one far-away non-box obstacle after them,
    gives the box path's `end` bit for bit -- for ends at box centres, on faces, corners and in free space."""
    from oracle.obstacles import obstacle_reps

    far = _box_rows([5, 5, 5], [5.1, 5.1, 5.1], (np.array([0.6, 0.0, 0.8]), 10.0))
    rng = np.random.default_rng(4)
    n_moved = 0
    for i in range(4):
        boxes, infl, st, en, *_ = scenes.config_c3_query(i)
        obs_sets, _, _ = obstacle_reps(boxes, infl)
        box_pl, gen_pl = _planner(obs_sets, infl), _planner(obs_sets + [far], infl)
        assert not box_pl.polytopes and gen_pl.polytopes
        lo, hi = boxes[:, :3] - infl, boxes[:, 3:] + infl
        ends = [en, 0.5 * (boxes[0, :3] + boxes[0, 3:]), hi[1], np.array([hi[2, 0], 0.5 * (lo[2, 1] + hi[2, 1]), lo[2, 2]])]
        ends += list(rng.uniform(scenes.WORKSPACE_MIN, scenes.WORKSPACE_MAX, (40, 3)))
        for e in ends:
            want = box_pl._push_out_boxes(np.array(e, float))
            got = gen_pl._push_out_general(np.array(e, float))
            assert np.array_equal(got, want), (i, e, got, want)
            n_moved += not np.array_equal(want, e)
    assert n_moved >= 8


def test_new_obs_with_start_inside_a_polytope_raises_attribute_error():
    """Quirk Q12 on polytopes: with new_obs, a start inside an inflated obstacle ends in the reference's
    AttributeError (`ob.A()` on a list), as on boxes."""
    q, infl, wmin, wmax = _c3_poly(1)
    backend = PolytopeOracleBackend(q["obs_sets"], q["obs_points_sets"], wmax, wmin)
    inside = q["obs_points_sets"][3].mean(axis=0)
    pl = SetSequencePlanner((), infl, wmax, wmin, backend=backend, rng=np.random.default_rng(0), obs_sets=q["obs_sets"])
    assert pl.polytopes and pl._in_collision(inside)
    with pytest.raises(AttributeError):
        pl.plan_set_sequence(inside.copy(), q["end"].copy(), R0, R0, replanning=True,
                             p_horizon=np.array([inside, q["start"]]), new_obs=True)


def test_mixed_batches_raise_value_error():
    q, infl, wmin, wmax = _c3_poly(0)
    boxes, _, st, en, *_ = scenes.config_c3_query(0)
    qb = dict(obstacles=boxes, start=st, end=en, r0=R0, r1=R0)
    assert pn.query_kind([q, q]) == "polytopes" and pn.query_kind([qb]) == "boxes"
    with pytest.raises(ValueError, match="mixes"):
        pn.PackedQueries([qb, q], infl, wmax, wmin)
    with pytest.raises(ValueError, match="either"):
        pn.PackedQueries([dict(q, obstacles=boxes)], infl, wmax, wmin)
    with pytest.raises(ValueError, match="mixes"):
        pn.plan_batch_native([q, qb], infl, wmax, wmin)
    from boundplanner_b200.planner import plan_batch

    with pytest.raises(ValueError, match="mixes"):
        plan_batch([qb, q], infl, wmax, wmin)
    pk = pn.PackedQueries([q], infl, wmax, wmin, [0])
    assert pk.obs_rows.shape == (200, 15, 4) and np.array_equal(pk.box_off, [0, 200])
    assert np.array_equal(pk.obs_rows[:, :, :3], np.stack([s[0] for s in q["obs_sets"]]))
    assert np.array_equal(pk.obs_rows[:, :, 3], np.stack([s[1] for s in q["obs_sets"]]))


# ---- GPU ---------------------------------------------------------------------------------------------------
def _same(g, w, i, via_tol):
    if isinstance(w, Exception):
        assert isinstance(g, Exception) and type(g) is type(w), (i, g, w)
        assert str(g).split("(")[0] == str(w).split("(")[0], (i, g, w)
        return False
    assert not isinstance(g, Exception), f"query {i}: {g!r}"
    assert g["path"] == w["path"] and g["set_ids"] == w["set_ids"], i
    assert np.abs(g["p_via"] - w["p_via"]).max() < via_tol, i
    return True


def _n_nodes(res):
    return res["n_nodes"] if "n_nodes" in res else res["graph"].number_of_nodes()    # native | Python driver


@pytest.mark.gpu
def test_native_plan_batch_equals_python_plan_batch_over_polytopes_on_gpu():
    """bp_plan_run over a polytope scene batch == planner.plan_batch over the same kernels, 24 C3 polytope queries."""
    from boundplanner_b200.planner import plan_batch

    ids = list(range(24))
    queries = []
    for i in ids:
        q, infl, wmin, wmax = _c3_poly(i)
        queries.append(q)
    want, _ = plan_batch(queries, infl, wmax, wmin, rng_seeds=ids)
    got, stats = pn.plan_batch_native(queries, infl, wmax, wmin, rng_seeds=ids)
    assert stats["rounds"] > 10
    n_ok = 0
    for i, (w, g) in enumerate(zip(want, got)):
        if not _same(g, w, i, 1e-9):
            continue
        n_ok += 1
        assert g["n_nodes"] == w["graph"].number_of_nodes() and g["n_inter"] == w["inter_graph"].number_of_nodes()
        for (ga, gb), (wa, wb) in zip(g["sets_via"], w["sets_via"]):
            assert ga.shape == wa.shape and np.abs(ga - wa).max() < 1e-12 and np.abs(gb - wb).max() < 1e-12
    assert n_ok >= 6


@pytest.mark.gpu
def test_polytope_queries_gpu_backend_matches_oracle_sequence():
    """plan_set_sequence on the GPU backend (the default backend of a polytope planner) == the oracle backend."""
    n_ok = 0
    for i in range(8):
        q, infl, wmin, wmax = _c3_poly(i)
        out = []
        for backend in (None, PolytopeOracleBackend(q["obs_sets"], q["obs_points_sets"], wmax, wmin)):
            pl = SetSequencePlanner((), infl, wmax, wmin, backend=backend, rng=np.random.default_rng(i),
                                    obs_sets=q["obs_sets"], obs_points_sets=q["obs_points_sets"])
            try:
                out.append(pl.plan_set_sequence(q["start"].copy(), q["end"].copy(), R0, R0))
            except (RuntimeError, ValueError) as e:
                out.append(e)
            if backend is None:
                from boundplanner_b200.planner import GpuBackend

                assert isinstance(pl.backend, GpuBackend) and pl.backend._bx.scene.__class__.__name__ == "PolytopeSceneBatch"
        n_ok += _same(out[0], out[1], i, 1e-6)
    assert n_ok >= 3


@pytest.mark.gpu
def test_boxes_handed_over_as_polytopes_plan_like_boxes():
    """The 24 C3 box queries given as obs_sets (add_obstacle_reps rows + corners) through both drivers: the answers
    of the same queries given as boxes."""
    from boundplanner_b200.planner import plan_batch
    from oracle.obstacles import obstacle_reps

    ids = list(range(24))
    qb, qp = [], []
    for i in ids:
        ob, infl, st, en, wmin, wmax = scenes.config_c3_query(i)
        qb.append(dict(obstacles=ob, start=st, end=en, r0=R0, r1=R0))
        obs_sets, pts, _ = obstacle_reps(ob, infl)
        qp.append(dict(obs_sets=obs_sets, obs_points_sets=pts, start=st, end=en, r0=R0, r1=R0))
    wmin, wmax = list(wmin), list(wmax)
    for driver in (pn.plan_batch_native, plan_batch):
        want, _ = driver(qb, infl, wmax, wmin, rng_seeds=ids)
        got, _ = driver(qp, infl, wmax, wmin, rng_seeds=ids)
        n_ok = 0
        for i, (w, g) in enumerate(zip(want, got)):
            if not _same(g, w, i, 1e-7):
                continue
            n_ok += 1
            assert _n_nodes(g) == _n_nodes(w), i
            for (ga, gb), (wa, wb) in zip(g["sets_via"], w["sets_via"]):
                assert ga.shape == wa.shape and np.abs(ga - wa).max() < 1e-9 and np.abs(gb - wb).max() < 1e-9
        assert n_ok >= 6, driver.__name__


@pytest.mark.gpu
def test_bp_plan_run_refuses_the_other_obstacle_kind():
    """bp_plan_run fails, without planning, when the input's obstacle kind or counts are not the scene batch's."""
    from boundplanner_b200 import _lib

    q, infl, wmin, wmax = _c3_poly(0)
    ob, _, st, en, *_ = scenes.config_c3_query(0)
    qb = dict(obstacles=ob, start=st, end=en, r0=R0, r1=R0)
    lib = _lib.load()
    import torch

    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    poly = pn.NativePlanner([q], infl, wmax, wmin)
    box = pn.NativePlanner([qb], infl, wmax, wmin)
    try:
        for plan, other in ((poly, qb), (box, q)):
            pk = pn.PackedQueries([other], infl, wmax, wmin, [0])
            assert lib.bp_plan_run(plan._h, ctypes.byref(pk.inp), ctypes.byref(pk.out), stream) != 0
            assert b"the plan's scene batch holds" in lib.bp_last_error_string()
            assert pk.stats[0] == 0 and pk.finish_round[0] == -1                  # nothing planned
        short = dict(q, obs_sets=q["obs_sets"][:199])                             # one obstacle fewer than the scene
        pk = pn.PackedQueries([short], infl, wmax, wmin, [0])
        assert lib.bp_plan_run(poly._h, ctypes.byref(pk.inp), ctypes.byref(pk.out), stream) != 0
        assert b"has 199 obstacles, its scene 200" in lib.bp_last_error_string()
        res, _ = poly.run([0])                                                     # the plan itself is unharmed
        assert len(res) == 1
    finally:
        poly.close()
        box.close()
