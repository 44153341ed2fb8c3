"""Moving obstacles: a resident scene batch rewritten in place (bp_scene_update_batch,
bp_scene_update_polytopes_batch; SceneBatch / PolytopeSceneBatch.update_scenes; NativePlanner.update_obstacles).

CPU: the vectorised polytope packing against a literal restatement of PolytopeScene's per-obstacle loop.
GPU: an updated batch against a freshly created one of the same obstacles (sample filter flags, point and line set
builds, bit for bit; growth past capacity, shrinking, empty box scenes, box scenes past the shared-memory staging size,
polytope vmax up and down, vertices given and enumerated on the device); an updated NativePlanner against a fresh one
and plan_batch; a 4-step MPC loop with obstacles that move every step; failed updates that leave the planner as it
was."""
import numpy as np
import pytest

from boundplanner_b200 import geometry as geo
from boundplanner_b200 import planner_native as pn
from boundplanner_b200 import scenes
from boundplanner_b200.planner import plan_batch
from tests.util import _c3, _c3_poly, _same_sets, mpc_step

WMIN, WMAX = scenes.WORKSPACE_MIN, scenes.WORKSPACE_MAX


# ---- CPU -------------------------------------------------------------------------------------------------------
def _loop_rows(obs_sets):
    """PolytopeScene.__init__'s loop, restated: rows of nonzero norm in order, padded with (0, 0, 0, 10)."""
    n = len(obs_sets)
    rows = np.zeros((n, 15, 4))
    rows[:, :, 3] = 10.0
    nrows = np.zeros(n, np.int32)
    for j, (a_set, b_set) in enumerate(obs_sets):
        a_set = np.asarray(a_set, float).reshape(-1, 3)
        b_set = np.asarray(b_set, float).reshape(-1)
        nz = np.linalg.norm(a_set, axis=1) > 0
        k = int(nz.sum())
        rows[j, :k, :3], rows[j, :k, 3] = a_set[nz], b_set[nz]
        nrows[j] = k
    return rows, nrows


def _odd_sets(rng):
    """Obstacles with interior zero rows, a single row, 15 rows (and zero rows around them), plus C3 polytopes."""
    sets, _ = scenes.random_polytope_scene(12, rng, 0.05, 0.2)
    a = rng.normal(size=(15, 3))
    sets.append([a, rng.uniform(0.1, 1.0, 15)])                                       # 15 rows
    sets.append([np.vstack((a[:20], np.zeros((3, 3)))), np.r_[rng.uniform(size=15), 10, 10, 10]])
    sets.append([a[:1], np.array([0.5])])                                              # 1 row
    z = a[:7].copy()
    z[[1, 4]] = 0.0                                                                    # interior zero rows
    sets.append([z, rng.uniform(size=7)])
    sets.append([np.vstack((np.zeros((2, 3)), a[:3], np.zeros((1, 3)), a[3:5])), rng.uniform(size=8)])
    sets.append([np.zeros((0, 3)), np.zeros(0)])                                       # no row at all
    return sets


def test_vectorised_polytope_packing_equals_the_loop():
    rng = np.random.default_rng(7)
    sets = _odd_sets(rng)
    rows, nrows = geo.pack_polytope_rows(sets)
    want_rows, want_nrows = _loop_rows(sets)
    assert rows.dtype == want_rows.dtype and np.array_equal(rows, want_rows)
    assert nrows.dtype == np.int32 and np.array_equal(nrows, want_nrows)
    assert {1, 15, 5, 0} <= set(nrows.tolist())
    with pytest.raises(ValueError, match="more than 15 rows"):
        geo.pack_polytope_rows(sets + [[rng.normal(size=(16, 3)), np.ones(16)]])
    pts = [rng.normal(size=(k, 3)) for k in (4, 9, 1, 12)]
    verts, nverts, vmax = geo.pack_vertices(pts)
    assert vmax == 12 and nverts.tolist() == [4, 9, 1, 12]
    want = np.zeros((4, 12, 3))
    for j, v in enumerate(pts):
        want[j, : v.shape[0]] = v
    assert np.array_equal(verts, want)


def test_moved_obstacles_is_seeded():
    boxes = scenes.random_box_scene(50, np.random.default_rng(0))
    a = scenes.moved_obstacles(boxes, np.random.default_rng(1))
    b = scenes.moved_obstacles(boxes, np.random.default_rng(1))
    assert np.array_equal(a, b) and a.shape == (50, 6)
    assert 0 < int((~np.isin(boxes, a).all(axis=1)).sum()) < 50


# ---- GPU -------------------------------------------------------------------------------------------------------
def _probe(scene, n_scenes, seed=3):
    """Every scene of a batch through the sample filter (flags on a jittered 4x4x4 grid), the point set build (4 fixed
    seeds) and the line set build (2 fixed segments): host arrays of everything they return."""
    import torch

    rng = np.random.default_rng(seed)
    g = (np.arange(4) + 0.5) / 4
    grid = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
    cand = WMIN + (WMAX - WMIN) * (grid[None] + rng.uniform(-0.1, 0.1, (n_scenes, 64, 3)))
    first, flags = geo.sample_filter(scene, cand, item_scene=np.arange(n_scenes), want_flags=True)
    seeds = rng.uniform(WMIN + 0.1, WMAX - 0.1, (n_scenes * 4, 3))
    pt = geo.build_sets_point(scene, seeds, WMIN, WMAX, fixed_mid=True, item_scene=np.repeat(np.arange(n_scenes), 4))
    p0 = rng.uniform(WMIN + 0.1, WMAX - 0.1, (n_scenes * 2, 3))
    p1 = p0 + rng.uniform(-0.2, 0.2, p0.shape)
    ln = geo.build_sets_line(scene, p0, p1, WMIN, WMAX, item_scene=np.repeat(np.arange(n_scenes), 2))
    torch.cuda.synchronize()
    out = dict(first=first, flags=flags)
    for k in ("A", "b", "m", "q_ellipse", "p_mid", "status", "iters"):
        out["point_" + k] = getattr(pt, k)
    for k in ("A", "b", "m", "status", "collision"):
        out["line_" + k] = getattr(ln, k)
    return {k: v.cpu().numpy() for k, v in out.items()}


def _assert_same_probe(got, want):
    assert got.keys() == want.keys()
    for k in want:
        assert got[k].dtype == want[k].dtype and got[k].shape == want[k].shape, k
        assert np.array_equal(got[k].view(np.uint8), want[k].view(np.uint8)), k


def _box_batches():
    rng = np.random.default_rng(11)
    a = [scenes.random_box_scene(200, rng, 0.05, 0.2) for _ in range(5)]
    b = [scenes.random_box_scene(1500, rng, 0.02, 0.06),       # past capacity, past the shared-memory staging size
         scenes.random_box_scene(40, rng, 0.05, 0.2),          # shrinks
         np.zeros((0, 6)),                                      # drops to 0
         scenes.moved_obstacles(a[3], rng),
         scenes.random_box_scene(260, rng, 0.05, 0.2)]
    c = [scenes.random_box_scene(30, rng, 0.05, 0.2) for _ in range(5)]   # everything shrinks, no reallocation
    c[4] = np.zeros((0, 6))
    return [a, b, c]


@pytest.mark.gpu
def test_box_batch_update_equals_a_fresh_batch():
    steps = _box_batches()
    sc = geo.SceneBatch(steps[0], 0.01)
    try:
        for boxes in steps[1:] + steps[:1]:
            sc.update_scenes(boxes)
            fresh = geo.SceneBatch(boxes, 0.01)
            assert sc.n == fresh.n
            _assert_same_probe(_probe(sc, 5), _probe(fresh, 5))
            fresh.close()
    finally:
        sc.close()


def _box_polytope(rng, n):
    """n axis-aligned boxes as 6-row polytopes (8 vertices each)."""
    sets = []
    for bx in scenes.random_box_scene(n, rng, 0.05, 0.2):
        a = np.vstack((np.eye(3), -np.eye(3)))
        sets.append([np.vstack((a, np.zeros((9, 3)))), np.r_[bx[3:], -bx[:3], np.full(9, 10.0)]])
    return sets


def _poly_batches():
    rng = np.random.default_rng(12)
    a = [_box_polytope(rng, 30) for _ in range(4)]                                    # vmax 8
    b = [scenes.random_polytope_scene(n, rng, 0.05, 0.2)[0] for n in (120, 25, 1, 60)]   # more vertices, growth
    for a_set, b_set in _box_polytope(rng, 3):                                         # interior zero rows
        order = [0, 1, 6, 2, 3, 7, 4, 5]
        b[2].append([a_set[order], b_set[order]])
    c = [_box_polytope(rng, n) for n in (10, 3, 12, 1)]                                # shrink, vmax 8 again
    return [a, b, c]


@pytest.mark.gpu
@pytest.mark.parametrize("given", [True, False], ids=["vertices_given", "vertices_enumerated"])
def test_polytope_batch_update_equals_a_fresh_batch(given):
    from boundplanner_b200.utils import obstacle_points_sets

    steps = _poly_batches()

    def scenes_of(sets_list):
        return [(s, obstacle_points_sets(s) if given else None) for s in sets_list]

    sc = geo.PolytopeSceneBatch(scenes_of(steps[0]))
    vmaxes = []
    try:
        for sets_list in steps[1:] + steps[:1]:
            sc.update_scenes(scenes_of(sets_list))
            fresh = geo.PolytopeSceneBatch(scenes_of(sets_list))
            assert sc.n == fresh.n
            vmaxes.append(max(len(v) for s in sets_list for v in obstacle_points_sets(s)))
            _assert_same_probe(_probe(sc, 4), _probe(fresh, 4))
            fresh.close()
    finally:
        sc.close()
    assert vmaxes[0] > 8 and vmaxes[1] == 8


def _assert_same_plans(got, want, gst=None, wst=None):
    """Bit-identical results of two native runs (and the same round statistics)."""
    for i, (g, w) in enumerate(zip(got, want)):
        if isinstance(w, Exception):
            assert type(g) is type(w) and str(g) == str(w), (i, g, w)
            continue
        assert not isinstance(g, Exception), (i, g)
        assert g["path"] == w["path"] and g["set_ids"] == w["set_ids"], i
        assert np.array_equal(g["p_via"], w["p_via"]), i
        _same_sets(g["sets_via_prev"], w["sets_via_prev"])
        assert ("p_horizon_max" in g) == ("p_horizon_max" in w)
        if "p_horizon_max" in w:
            assert np.array_equal(g["p_horizon_max"], w["p_horizon_max"]), i
    if wst is not None:
        for k in ("rounds", "set_requests", "pair_tests"):
            assert gst[k] == wst[k], k


def _assert_like_plan_batch(got, want):
    """The comparison of the replanning tests between bp_plan_run and planner.plan_batch."""
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


def _queries(kind, ids):
    make = _c3 if kind == "boxes" else _c3_poly
    out = [make(i) for i in ids]
    return [q for q, *_ in out], out[0][1], out[0][2], out[0][3]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["boxes", "polytopes"])
def test_planner_after_an_update_equals_a_fresh_planner(kind):
    qa, infl, wmin, wmax = _queries(kind, range(24))
    qb, _, _, _ = _queries(kind, range(24, 48))
    seeds = [200 + i for i in range(24)]
    pl = pn.NativePlanner(qa, infl, wmax, wmin)
    fresh = pn.NativePlanner(qb, infl, wmax, wmin)
    try:
        pl.run(seeds)
        pl.update_obstacles(qb)
        assert pl.queries is qb
        got, gst = pl.run(seeds)
        want, wst = fresh.run(seeds)
        # run(queries=...) now checks against the new obstacles
        again, _ = pl.run(seeds, queries=qb)
        with pytest.raises(ValueError, match="obstacles differ"):
            pl.run(seeds, queries=qa)
    finally:
        pl.close()
        fresh.close()
    _assert_same_plans(got, want, gst, wst)
    _assert_same_plans(again, want)
    py, _ = plan_batch(qb, infl, wmax, wmin, rng_seeds=seeds)
    assert _assert_like_plan_batch(got, py) >= 4


def _moved(q, rng, step, enumerate_vertices):
    if "obs_sets" in q:
        sets, pts = scenes.moved_obstacles(q["obs_sets"], rng, obs_points=q.get("obs_points_sets"))
        if enumerate_vertices:
            return dict(q, obs_sets=sets, obs_points_sets=None)
        if pts is None:
            from boundplanner_b200.utils import obstacle_points_sets

            pts = obstacle_points_sets(sets)
        return dict(q, obs_sets=sets, obs_points_sets=pts)
    return dict(q, obstacles=scenes.moved_obstacles(np.asarray(q["obstacles"]), rng))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["boxes", "polytopes"])
def test_mpc_loop_with_moving_obstacles(kind):
    """4 MPC steps of 12 queries, the obstacles moving every step (new_obs=True, sets_via_prev threaded forward):
    every step of the updated planner equals a fresh planner bit for bit and plan_batch."""
    queries, infl, wmin, wmax = _queries(kind, range(12))
    pl = pn.NativePlanner(queries, infl, wmax, wmin)
    n_rep = n_err = 0
    try:
        for step in range(4):
            seeds = [50 * step + i for i in range(12)]
            if step:
                pl.update_obstacles(queries)
            got, gst = pl.run(seeds)
            fresh = pn.NativePlanner(queries, infl, wmax, wmin)
            try:
                want, wst = fresh.run(seeds)
            finally:
                fresh.close()
            _assert_same_plans(got, want, gst, wst)
            py, _ = plan_batch(queries, infl, wmax, wmin, rng_seeds=seeds)
            _assert_like_plan_batch(got, py)
            rng = np.random.default_rng(1000 + step)
            nxt = []
            for i, (q, g) in enumerate(zip(queries, got)):
                q = _moved(q, rng, step, enumerate_vertices=(kind == "polytopes" and step % 2 == 0))
                if isinstance(g, Exception):
                    n_err += 1
                    nxt.append(dict(q, replanning=False, new_obs=True))
                else:
                    n_rep += step > 0 and "p_horizon_max" in g
                    nxt.append(dict(mpc_step(q, g), new_obs=True))
            queries = nxt
    finally:
        pl.close()
    assert n_rep >= 3


@pytest.mark.gpu
def test_failed_updates_leave_the_planner_as_it_was():
    from boundplanner_b200 import _lib

    qb, infl, wmin, wmax = _queries("boxes", range(8))
    qp, _, _, _ = _queries("polytopes", range(8))
    seeds = list(range(8))
    pb = pn.NativePlanner(qb, infl, wmax, wmin)
    pp = pn.NativePlanner(qp, infl, wmax, wmin)
    try:
        want_b, st_b = pb.run(seeds)
        want_p, st_p = pp.run(seeds)
        with pytest.raises(ValueError, match="hold boxes"):
            pb.update_obstacles(qp)                                        # kind change
        with pytest.raises(ValueError, match="7 queries"):
            pb.update_obstacles(qb[1:])                                     # number of queries
        big = [dict(q) for q in qp]
        box = [np.vstack((np.eye(3), -np.eye(3))), np.r_[0.1, 0.1, 0.1, 0.0, 0.0, 0.0]]
        big[3] = dict(qp[3], obs_sets=[box] * 16385, obs_points_sets=None)
        with pytest.raises(ValueError, match="at most 16384"):
            pp.update_obstacles(big)                                        # above the per-scene limit
        open_ = [dict(q, obs_points_sets=None) for q in qp]
        open_[5] = dict(open_[5], obs_sets=open_[5]["obs_sets"][:7] + [[box[0][:5], box[1][:5]]])
        with pytest.raises(_lib.BpGeoError, match="scene 5, obstacle 7: Polyhedron is not a polytope"):
            pp.update_obstacles(open_)                                      # not a polytope, found on the device
        assert pb.queries is qb and pp.queries is qp
        got_b, gst_b = pb.run(seeds)
        got_p, gst_p = pp.run(seeds)
    finally:
        pb.close()
        pp.close()
    _assert_same_plans(got_b, want_b, gst_b, st_b)
    _assert_same_plans(got_p, want_p, gst_p, st_p)


@pytest.mark.gpu
def test_batch_update_rejects_malformed_inputs():
    """The C entry points: wrong kind, another number of scenes, decreasing offsets, obstacles without 1..15 rows;
    the batch stays usable and unchanged."""
    import ctypes

    from boundplanner_b200 import _lib

    lib = _lib.load()
    rng = np.random.default_rng(5)
    boxes = [scenes.random_box_scene(20, rng) for _ in range(3)]
    sc = geo.SceneBatch(boxes, 0.01)
    ps = geo.PolytopeSceneBatch([(_box_polytope(rng, 4), None) for _ in range(3)])
    ip = ctypes.POINTER(ctypes.c_int)
    dp = ctypes.POINTER(ctypes.c_double)
    try:
        before = _probe(sc, 3)
        bx = np.ascontiguousarray(np.vstack(boxes))
        for offs, n, msg in (([0, 20, 40], 2, "2 scenes for a batch of 3"), ([0, 30, 20, 60], 3, "non-decreasing")):
            o = np.asarray(offs, np.int32)
            assert lib.bp_scene_update_batch(sc._h, bx.ctypes.data_as(dp), o.ctypes.data_as(ip), n, 0.01, None) != 0
            assert msg in lib.bp_last_error_string().decode()
        o = np.asarray([0, 1, 2, 3], np.int32)
        rows = np.zeros((3, 15, 4))
        nrows = np.array([6, 0, 6], np.int32)
        assert lib.bp_scene_update_polytopes_batch(sc._h, rows.ctypes.data_as(dp), nrows.ctypes.data_as(ip), None,
                                                   None, o.ctypes.data_as(ip), 3, 0, None) != 0
        assert "holds boxes" in lib.bp_last_error_string().decode()
        assert lib.bp_scene_update_polytopes_batch(ps._h, rows.ctypes.data_as(dp), nrows.ctypes.data_as(ip), None,
                                                   None, o.ctypes.data_as(ip), 3, 0, None) != 0
        assert "scene 1, obstacle 0 needs 1..15 rows" in lib.bp_last_error_string().decode()
        assert lib.bp_scene_update_batch(ps._h, bx.ctypes.data_as(dp), o.ctypes.data_as(ip), 3, 0.01, None) != 0
        assert "holds polytopes" in lib.bp_last_error_string().decode()
        _assert_same_probe(_probe(sc, 3), before)
    finally:
        sc.close()
        ps.close()
