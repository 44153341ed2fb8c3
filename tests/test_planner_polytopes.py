"""Planning over general convex polytope obstacles (obs_sets of up to 15 rows, as ConvexSetFinder takes them).

CPU: the native driver's state machines (csrc/bp_planner.h, general-row push-out of `end`) in the host harness with
the oracle answering their requests, against SetSequencePlanner with the same answers; the host-side push-out of
`end` (:199-204) on general rows against the reference's literal loop, and against the box arithmetic for boxes;
the new_obs start-in-collision quirk.
GPU: bp_plan_run over a polytope scene batch against planner.plan_batch; plan_set_sequence on the GPU backend
against the oracle backend; boxes handed over as polytopes against the same boxes; the kind checks."""
import ctypes

import networkx as nx
import numpy as np
import pytest
from scipy.spatial.transform import Rotation as R

from boundplanner_b200 import planner_native as pn
from boundplanner_b200 import scenes
from boundplanner_b200.planner import SetSequencePlanner
from tests.test_planner_native import (CB_EDGES, CB_PATH, CB_PROJECT, CB_SET, MemoBackend, _error_status, _fill_set,
                                       _node_set)

R0 = R.from_euler("XYZ", [0, 90, 0], degrees=True).as_matrix()
ORDER_TOL = 1e-15          # general push-out vs the reference's `@` (BLAS may fuse): last bits only


class PolytopeOracleBackend(MemoBackend):
    """The oracle's ConvexSetFinder over polytope obstacles (obs_sets + obs_points_sets), answers memoised."""

    def __init__(self, obs_sets, obs_points_sets, workspace_max, workspace_min):
        from oracle.convex_set_finder import ConvexSetFinder as OracleFinder

        self.obs_sets = obs_sets
        self.set_finder = OracleFinder(obs_sets, obs_points_sets, list(workspace_max), list(workspace_min))
        self.memo = {}


def _polytope_query(i):
    obs_sets, pts, infl, st, en, wmin, wmax = scenes.config_c3_polytope_query(i)
    return dict(obs_sets=obs_sets, obs_points_sets=pts, start=st, end=en, r0=R0, r1=R0), infl, list(wmin), list(wmax)


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
def run_native_with_oracle(host_harness, queries, inflate, ws_max, ws_min, seeds, backends, sample_chunk=32):
    """tests.test_planner_native.run_native_with_oracle for polytope queries (obs_sets instead of obstacles)."""
    pk = pn.PackedQueries(queries, inflate, ws_max, ws_min, seeds, sample_chunk)
    assert pk.kind == "polytopes" and pk.boxes is None
    helpers = [SetSequencePlanner((), inflate, list(ws_max), list(ws_min), backend=backends[i], obs_sets=q["obs_sets"])
               for i, q in enumerate(queries)]
    ee = []
    for q in queries:
        omega = R.from_matrix(q["r1"] @ q["r0"].T).as_rotvec()
        on = np.linalg.norm(omega)
        ee.append((q["r0"] @ np.array([-0.05, 0, 0]), omega / on if on > 1e-6 else np.array([0, 0, 1.0]), on))
    errors = []

    def in_safe(nodes, n, x):
        return any(np.max(_node_set(nodes[k])[0] @ x - _node_set(nodes[k])[1]) < 1e-3 for k in range(n))

    def dvertex(nodes, n, Q, p):
        if n == 0:
            return np.inf
        return min(np.linalg.norm(np.array(nodes[k].Q[:]).reshape(3, 3) - Q) + np.linalg.norm(np.array(nodes[k].P[:]) - p)
                   for k in range(n))

    def cb_set(qid, req, n_nodes, nodes, out):
        try:
            r, o = req.contents, out.contents
            o.first, o.dv, o.collision = 0, np.inf, 0
            p0 = np.array(r.p0[:])
            if r.kind == 1:
                try:
                    _fill_set(o, backends[qid].execute(("set_line", p0, np.array(r.p1[:]))), True)
                except (RuntimeError, ValueError) as e:
                    _error_status(e, o)
                return 0
            if r.kind == 2:
                cand = np.ctypeslib.as_array(r.cand, shape=(r.n_cand, 3)).copy()
                o.first = -1
                for i, c in enumerate(cand):
                    if not helpers[qid]._in_collision(c) and not in_safe(nodes, n_nodes, c):
                        o.first, p0 = i, c
                        break
                if o.first < 0:
                    return 0
            try:
                ans = backends[qid].execute(("set_point", p0, bool(r.fixed_mid), bool(r.optimize)))
            except (RuntimeError, ValueError) as e:
                _error_status(e, o)
                return 0
            _fill_set(o, ans, False)
            if r.with_dv:
                o.dv = dvertex(nodes, n_nodes, ans[2], ans[3])
            return 0
        except Exception as e:                               # noqa: BLE001 -- surfaces in the test below
            errors.append(e)
            return 7

    def cb_edges(qid, id_new, n_nodes, nodes, has_target, xd, out):
        try:
            others = [_node_set(nodes[k]) for k in range(id_new)]
            new = _node_set(nodes[id_new])
            res = backends[qid].execute(("edges", others, new, 0.01, ee[qid]))
            for k, (x, ok, fits, via) in enumerate(res):
                out[k].ok, out[k].fits, out[k].proj_ok = int(bool(ok)), int(bool(fits)), 0
                if ok:
                    out[k].x[:] = np.asarray(x).tolist()
                    out[k].omega = float(via[3]) if fits else -1.0
                    if has_target[k]:
                        pr = backends[qid].execute(("project", np.concatenate((others[k][0], new[0])),
                                                    np.concatenate((others[k][1], new[1])),
                                                    np.array([xd[3 * k], xd[3 * k + 1], xd[3 * k + 2]])))
                        out[k].proj[:] = np.asarray(pr).tolist()
                        out[k].proj_ok = 1
            return 0
        except Exception as e:                               # noqa: BLE001
            errors.append(e)
            return 7

    def cb_project(qid, id0, id1, xd, n_nodes, nodes, out):
        try:
            s0, s1 = _node_set(nodes[id0]), _node_set(nodes[id1])
            x = backends[qid].execute(("project", np.concatenate((s0[0], s1[0])), np.concatenate((s0[1], s1[1])),
                                       np.array([xd[0], xd[1], xd[2]])))
            out.contents.x[:] = np.asarray(x).tolist()
            return 0
        except Exception as e:                               # noqa: BLE001
            errors.append(e)
            return 7

    def cb_path(qid, n, edge_off, edge_dst, edge_w, path_out, path_len):
        try:
            g = nx.Graph()
            g.add_nodes_from(range(n))
            for v in range(n):
                for e in range(edge_off[v], edge_off[v + 1]):
                    g._adj[v][edge_dst[e]] = {"weight": edge_w[e]}
            p = nx.shortest_path(g, 0, 1, weight="weight")
            path_len[0] = len(p)
            for k, v in enumerate(p[: pn.MAX_PATH]):
                path_out[k] = v
            return 0
        except Exception as e:                               # noqa: BLE001
            errors.append(e)
            return 7

    cbs = (CB_SET(cb_set), CB_EDGES(cb_edges), CB_PROJECT(cb_project), CB_PATH(cb_path))
    host_harness.hh_plan_batch.restype = ctypes.c_int
    rc = host_harness.hh_plan_batch(ctypes.byref(pk.inp), ctypes.byref(pk.out), *cbs, 1)
    assert not errors, errors[0]
    assert rc == 0
    return pk


def test_native_driver_equals_python_planner_over_polytopes_on_cpu(host_harness):
    """Six C3 polytope queries (one with its `end` inside an obstacle) through the native state machines and through
    SetSequencePlanner, the oracle answering both: the same paths, set ids, via points (bit for bit), graph sizes,
    sets, error exits and generator states."""
    queries, seeds, backends = [], [], []
    for i in range(6):
        q, infl, wmin, wmax = _polytope_query(i)
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

    want = []
    for q, s, be in zip(queries, seeds, backends):
        pl = SetSequencePlanner((), infl, wmax, wmin, backend=be, rng=np.random.default_rng(s), obs_sets=q["obs_sets"])
        try:
            res = pl.plan_set_sequence(q["start"].copy(), q["end"].copy(), q["r0"], q["r1"])
        except (RuntimeError, ValueError) as e:
            res = e
        want.append((res, pl))
    pk = run_native_with_oracle(host_harness, queries, infl, wmax, wmin, seeds, backends)
    got = pk.results()
    for i, ((w, pl), g) in enumerate(zip(want, got)):
        if isinstance(w, Exception):
            assert isinstance(g, Exception), f"query {i}: native planned, python raised {w!r}"
            assert type(g) is type(w) and str(g).split("(")[0] == str(w).split("(")[0], (i, g, w)
        else:
            assert not isinstance(g, Exception), f"query {i}: {g!r}"
            assert g["path"] == w["path"] and g["set_ids"] == w["set_ids"], i
            assert np.array_equal(g["p_via"], w["p_via"]), i
            assert g["n_nodes"] == w["graph"].number_of_nodes() and g["n_inter"] == w["inter_graph"].number_of_nodes()
            assert g["n_edges"] == w["inter_graph"].number_of_edges()
            for (ga, gb), (wa, wb) in zip(g["sets_via"], w["sets_via"]):
                assert np.array_equal(ga, wa) and np.array_equal(gb, wb)
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
    q, *_ = _polytope_query(0)
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
    q, infl, wmin, wmax = _polytope_query(1)
    backend = PolytopeOracleBackend(q["obs_sets"], q["obs_points_sets"], wmax, wmin)
    inside = q["obs_points_sets"][3].mean(axis=0)
    pl = SetSequencePlanner((), infl, wmax, wmin, backend=backend, rng=np.random.default_rng(0), obs_sets=q["obs_sets"])
    assert pl.polytopes and pl._in_collision(inside)
    with pytest.raises(AttributeError):
        pl.plan_set_sequence(inside.copy(), q["end"].copy(), R0, R0, replanning=True,
                             p_horizon=np.array([inside, q["start"]]), new_obs=True)


def test_mixed_batches_raise_value_error():
    q, infl, wmin, wmax = _polytope_query(0)
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
        q, infl, wmin, wmax = _polytope_query(i)
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
        q, infl, wmin, wmax = _polytope_query(i)
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

    q, infl, wmin, wmax = _polytope_query(0)
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
