"""Corridor checks of an MPC loop with moving obstacles: the set-obstacle hit test (bp_sets_obstacles,
geometry.sets_obstacle_hits, NativePlanner.corridor_hits) and planning a subset of a batch (bp_plan_run_active,
``run(active=)``, ``plan_batch(active=)``).

A set is hit by an obstacle when set_intersection([A_s, b_s], [A_o, b_o], tol) succeeds: both shrunk by tol share a
point.  An active query of a subset run must get, bit for bit, what a run of the whole batch gives it.
CPU: the native state machines in the host harness (hh_plan_batch_active against hh_plan_batch) with the oracle
answering, the Python driver's subset, the packing and the ValueErrors of corridor_hits.  GPU: exact margins, the
oracle after moved obstacles, the C2 golden sets, edge cases, and subset runs of the native planner."""
import ctypes
import os
import subprocess
from fractions import Fraction as Fr

import numpy as np
import pytest

from boundplanner_b200 import planner_native as pn
from boundplanner_b200 import scenes
from boundplanner_b200.planner import plan_batch
from tests.test_shared_scenes import _assert_same_plans, _box_scene, _copies, _moved_scene, _poly_scene, shared_form
from tests.util import (MemoBackend, OracleLockstepExecutor, PolytopeOracleBackend, _same_sets, mpc_step,
                        run_native_with_oracle)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WMIN, WMAX = scenes.WORKSPACE_MIN, scenes.WORKSPACE_MAX
_IP = ctypes.POINTER(ctypes.c_int)
# every output of bp_plan_out, with its bytes per query
_OUTPUTS = ("err_kind", "path", "path_len", "set_ids", "n_ids", "p_via", "n_via", "rng_out", "n_nodes", "n_inter",
            "n_edges", "finish_round", "node_A", "node_b", "node_m", "p_horizon_max")
SENTINEL = 0x5A


# ---- CPU: the host harness with the oracle answering -----------------------------------------------------------
@pytest.fixture(scope="module")
def active_harness():
    """tests/host_harness_active.cpp: the host harness plus hh_plan_batch_active (g++, built like conftest's
    host_harness)."""
    build = os.path.join(ROOT, "tests", "_build")
    os.makedirs(build, exist_ok=True)
    so = os.path.join(build, "libbp_host_harness_active.so")
    src = os.path.join(ROOT, "tests", "host_harness_active.cpp")
    deps = [src, os.path.join(ROOT, "tests", "host_harness.cpp"), os.path.join(ROOT, "include", "bpgeo.h")] + [
        os.path.join(ROOT, "boundplanner_b200", "csrc", f)
        for f in ("bp_math.cuh", "bp_mvie.cuh", "bp_lp.cuh", "bp_fk.cuh", "bp_mvie_fixed_r.cuh", "bp_mvie_pd.cuh",
                  "bp_planner.h")]
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-pthread", "-ffp-contract=off", "-o", so,
                               src])
    return ctypes.CDLL(so)


class _ActiveHarness:
    """The active harness behind the one oracle runner (tests.util.run_native_with_oracle): the runner's hh_plan_batch
    call plans only the active queries (hh_plan_batch_active), over the queries' own scenes or, with ``packed``, over
    shared scenes (PackedQueries with ``scenes=``), into the runner's output buffers -- which are first filled with
    SENTINEL bytes, so that what a skipped query's entries hold afterwards shows whether anything wrote them.  The full
    runs go through the same filling (``plain``: hh_plan_batch itself), so that the bytes no run writes compare equal."""

    def __init__(self, lib, active, packed=None, plain=False):
        # plain: hh_plan_batch itself (the full run); active None: hh_plan_batch_active without a mask
        self.lib, self.packed, self.plain = lib, packed, plain
        self.active = None if active is None else np.asarray(active, np.int32)

    def hh_plan_batch(self, inp, out, *callbacks_and_lanes):
        pk_out = out._obj
        Q = inp._obj.Q
        err_msg = ctypes.c_void_p.from_buffer(pk_out, pn.BpPlanOut.err_msg.offset).value
        ctypes.memset(err_msg, SENTINEL, 160 * Q)
        for name, _ in pn.BpPlanOut._fields_:
            ptr = getattr(pk_out, name)
            if name in ("err_msg", "stats", "finish_ms") or not ptr:
                continue
            ctypes.memset(ptr, SENTINEL, self.sizes[name] * Q)
        if self.plain:
            return self.lib.hh_plan_batch(inp, out, *callbacks_and_lanes)
        in_ref = inp if self.packed is None else ctypes.byref(self.packed.inp)
        qs = None if self.packed is None else self.packed.query_scene.ctypes.data_as(_IP)
        act = None if self.active is None else self.active.ctypes.data_as(_IP)
        return self.lib.hh_plan_batch_active(in_ref, qs, act, out, *callbacks_and_lanes)

    sizes = dict(err_kind=4, path=4 * 64, path_len=4, set_ids=4 * 64, n_ids=4, p_via=8 * 66 * 3, n_via=4, rng_out=32,
                 n_nodes=4, n_inter=4, n_edges=4, finish_round=4, node_A=8 * 64 * 24 * 3, node_b=8 * 64 * 24,
                 node_m=4 * 64, p_horizon_max=24)


def _check_subset(full, sub, active):
    """Active queries: every output equal to the full run's, bit for bit; skipped ones: sentinel bytes everywhere,
    finish_round -1."""
    Q = len(active)
    for q in range(Q):
        if active[q]:
            # (the message up to its terminating zero: the bytes after it are the buffer's own)
            msg = [pk.err_msg.raw[160 * q: 160 * (q + 1)].split(b"\0", 1)[0] for pk in (full, sub)]
            assert msg[0] == msg[1], q
        else:
            assert set(sub.err_msg.raw[160 * q: 160 * (q + 1)]) == {SENTINEL}, q
        for k in _OUTPUTS:
            g, w = getattr(sub, k)[q: q + 1], getattr(full, k)[q: q + 1]
            if k == "finish_round" and not active[q]:
                assert int(g[0]) == -1, q
            elif active[q]:
                assert np.array_equal(g.view(np.uint8), w.view(np.uint8)), (q, k)
            else:
                assert set(g.reshape(-1).view(np.uint8).tolist()) == {SENTINEL}, (q, k)
    assert sub.stats[1] < full.stats[1]          # set requests of the active queries only


def _scene_backends(kind, n):
    make = _box_scene if kind == "boxes" else _poly_scene
    sc = [make(i) for i in range(n)]
    infl = sc[0][1]
    scene_list = [s for s, _ in sc]
    if kind == "boxes":
        backends = [MemoBackend(s["obstacles"], infl, list(WMAX), list(WMIN)) for s in scene_list]
    else:
        backends = [PolytopeOracleBackend(s["obs_sets"], s["obs_points_sets"], list(WMAX), list(WMIN))
                    for s in scene_list]
    return scene_list, infl, backends


@pytest.fixture(scope="module")
def cpu_batches():
    """Module-wide scenes, oracle backends (memoised: the subset runs ask questions the full run has answered) and
    the full runs of every case, keyed by (case, lanes)."""
    return dict(boxes=_scene_backends("boxes", 2), polytopes=_scene_backends("polytopes", 2), runs={})


def _full_run(harness, cpu_batches, case, lanes):
    key = (case, lanes)
    if key in cpu_batches["runs"]:
        return cpu_batches["runs"][key]
    kind = "polytopes" if case == "polytopes" else "boxes"
    scene_list, infl, backends_of_scene = cpu_batches[kind]
    query_scene = [0, 1, 1, 0, 1, 0] if kind == "boxes" else [1, 0, 0, 1]
    queries = _copies(scene_list, infl, query_scene, seed=40 if kind == "boxes" else 60)
    seeds = [40 + k for k in range(len(queries))]
    if case == "replanning":
        first_queries, first = _full_run(harness, cpu_batches, "boxes", lanes)[:2]
        res = first.results()
        planned = [i for i, r in enumerate(res) if not isinstance(r, Exception)]
        assert len(planned) >= 3, "too few planned queries to replan"
        queries = [mpc_step(first_queries[i], res[i]) for i in planned]
        queries[-1] = dict(queries[-1], new_obs=True)
        query_scene = [query_scene[i] for i in planned]
        seeds = [140 + k for k in range(len(queries))]
    backends = [backends_of_scene[s] for s in query_scene]
    full = run_native_with_oracle(_ActiveHarness(harness, None, plain=True), queries, infl, list(WMAX), list(WMIN), seeds,
                                  backends, lanes=lanes)
    out = (queries, full, query_scene, seeds, backends, scene_list, infl)
    cpu_batches["runs"][key] = out
    return out


@pytest.mark.parametrize("lanes", [1, 2])
@pytest.mark.parametrize("case", ["boxes", "polytopes", "replanning", "shared"])
def test_active_subset_equals_full_run_on_cpu(active_harness, cpu_batches, case, lanes):
    queries, full, query_scene, seeds, backends, scene_list, infl = _full_run(
        active_harness, cpu_batches, "boxes" if case == "shared" else case, lanes)
    Q = len(queries)
    active = [(k * 7 + 3) % 5 < 3 for k in range(Q)]
    active[0], active[-1] = True, False
    packed = None
    if case == "shared":
        shared, sl = shared_form(queries, query_scene, scene_list)
        packed = pn.PackedQueries(shared, infl, list(WMAX), list(WMIN), seeds, scenes=sl)
    hh = _ActiveHarness(active_harness, active, packed)
    sub = run_native_with_oracle(hh, queries, infl, list(WMAX), list(WMIN), seeds, backends, lanes=lanes)
    _check_subset(full, sub, active)
    res = sub.results(pn.active_mask(active, Q))
    assert [r is None for r in res] == [not a for a in active]
    if case == "replanning":
        assert sub.replan is not None and any(isinstance(r, dict) and "p_horizon_max" in r for r in res)


def test_active_none_and_all_equal_the_full_run_on_cpu(active_harness, cpu_batches):
    queries, full, _, seeds, backends, _, infl = _full_run(active_harness, cpu_batches, "boxes", 1)
    for active in (None, [1] * len(queries)):
        got = run_native_with_oracle(_ActiveHarness(active_harness, active), queries, infl, list(WMAX), list(WMIN),
                                     seeds, backends)
        assert got.err_msg.raw == full.err_msg.raw
        for k in _OUTPUTS + ("stats",):
            assert np.array_equal(getattr(got, k).view(np.uint8), getattr(full, k).view(np.uint8)), k


def _same_python_results(got, want):
    for i, (g, w) in enumerate(zip(got, want)):
        if isinstance(w, Exception):
            assert type(g) is type(w) and str(g) == str(w), (i, g, w)
            continue
        assert g["path"] == w["path"] and g["set_ids"] == w["set_ids"], i
        assert np.array_equal(g["p_via"], w["p_via"]), i
        _same_sets(g["sets_via_prev"], w["sets_via_prev"])


def test_plan_batch_active_on_cpu(cpu_batches):
    scene_list, infl, backends_of_scene = cpu_batches["boxes"]
    query_scene = [0, 1, 1, 0]
    queries = _copies(scene_list, infl, query_scene, seed=40)
    backends = [backends_of_scene[s] for s in query_scene]
    seeds = [40 + k for k in range(4)]
    full, _ = plan_batch(queries, infl, WMAX, WMIN, rng_seeds=seeds, executor=OracleLockstepExecutor(backends))
    active = [False, True, True, False]
    sub, _ = plan_batch(queries, infl, WMAX, WMIN, rng_seeds=seeds, executor=OracleLockstepExecutor(backends),
                        active=active)
    assert sub[0] is None and sub[3] is None
    _same_python_results(sub[1:3], full[1:3])
    with pytest.raises(ValueError, match="active has 3 entries for 4 queries"):
        plan_batch(queries, infl, WMAX, WMIN, rng_seeds=seeds, executor=OracleLockstepExecutor(backends),
                   active=[1, 1, 1])
    with pytest.raises(ValueError, match="active has 5 entries for 4 queries"):
        pn.plan_batch_native(queries, infl, WMAX, WMIN, active=[1] * 5)


def test_corridor_packing_and_errors():
    rng = np.random.default_rng(3)

    def rset(m):
        return [rng.normal(size=(m, 3)), rng.uniform(0.1, 1.0, m)]

    padded = [np.vstack((rset(6)[0], np.zeros((9, 3)))), np.r_[rng.uniform(0.1, 1, 6), np.full(9, 10.0)]]
    sets = [[rset(6), rset(48)], None, [], [padded, rset(1)]]
    for qmap in (None, np.array([2, 0, 1, 2], np.int32)):
        buf, offs, S, m_max, spans = pn.pack_corridors(sets, qmap)
        assert (S, m_max) == (4, 48) and spans == [(0, 2), None, (2, 0), (2, 2)]
        A = buf[offs[0]:].view(np.float64)[: S * m_max * 3].reshape(S, m_max, 3)
        b = buf[offs[1]:].view(np.float64)[: S * m_max].reshape(S, m_max)
        m = buf[offs[2]:].view(np.int32)[:S]
        sc = buf[offs[3]:].view(np.int32)[:S]
        assert m.tolist() == [6, 48, 15, 1]
        assert sc.tolist() == ([0, 0, 3, 3] if qmap is None else [2, 2, 2, 2])
        assert np.array_equal(A[1], sets[0][1][0]) and np.array_equal(b[1], sets[0][1][1])
        assert np.array_equal(A[2, :15], padded[0]) and np.array_equal(b[2, :15], padded[1])
        assert np.all(A[0, 6:] == 0.0) and np.all(b[0, 6:] == 10.0) and np.all(b[3, 1:] == 10.0)
    assert pn.pack_corridors([None, []], None)[2] == 0
    # the planner's checks come before anything touches the device (no device here: a planner without one)
    pl = pn.NativePlanner.__new__(pn.NativePlanner)
    pl.queries, pl.query_scene = [{}] * 3, None
    for bad, msg in (([[rset(2)]] * 2, "2 corridors for a planner of 3"),
                     ([None, [rset(49)], None], "49 rows"),
                     ([None, None, [[np.zeros((0, 3)), np.zeros(0)]]], "0 rows"),
                     ([None, [[np.zeros((4, 3)), np.zeros(3)]], None], "one b each")):
        with pytest.raises(ValueError, match=msg):
            pl.corridor_hits(bad)


# ---- GPU: the hit test --------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def geo():
    import torch

    from boundplanner_b200 import geometry

    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return geometry


def _pack_sets(sets, m_max=48):
    S = len(sets)
    A = np.zeros((S, m_max, 3))
    b = np.full((S, m_max), 10.0)
    m = np.zeros(S, np.int32)
    for k, (a, bb) in enumerate(sets):
        A[k, : a.shape[0]], b[k, : a.shape[0]], m[k] = a, bb, a.shape[0]
    return A, b, m


def _hits(geo, scene, sets, set_scene=None, tol=1e-3):
    A, b, m = _pack_sets(sets)
    return geo.sets_obstacle_hits(scene, A, b, m, set_scene, tol).cpu().numpy()


def _box_rows(box, inflate):
    """The reference's make_box + obs_size_increase rows of one box."""
    lo, hi = np.asarray(box[:3], float) - inflate, np.asarray(box[3:], float) + inflate
    return [np.vstack((np.eye(3), -np.eye(3))), np.r_[hi, -lo]]


# exact margins: set rows and obstacle rows whose deciding margin is exact in rational arithmetic
ASSERTED = (1e-3, 1e-6, 1e-8, 1e-9)


def _far(rng, n, centre):
    """n redundant rows at least 1.6 from centre (scaled by powers of two, so that they stay exact)."""
    u = rng.normal(size=(n, 3))
    u /= np.linalg.norm(u, axis=1)[:, None]
    s = 2.0 ** rng.integers(-2, 3, n)
    return u * s[:, None], (u @ centre + rng.uniform(1.6, 2.6, n)) * s


def _arrange_last(rng, A, b, dec, n_total, centre):
    """Pad to n_total rows with far rows, deciding rows last."""
    Af, bf = _far(rng, n_total - A.shape[0], centre)
    A, b = np.vstack((A, Af)), np.r_[b, bf]
    rest = [r for r in range(n_total) if r not in dec]
    order = list(rng.permutation(rest)) + list(dec)
    return np.ascontiguousarray(A[order]), np.ascontiguousarray(b[order])


def _signed_perm(rng):
    return np.eye(3)[rng.permutation(3)] * rng.choice([-1.0, 1.0], 3)[:, None]


def _box_cases(rng, tol, m_total):
    """(kind, margin, set [A, b], box [lo | hi] with inflate 0, exact margin): face to face (the set's top row 2^k e_z
    against the box's bottom face) and vertex to face (a pyramid's apex against the bottom face), the set padded to
    m_total rows with its deciding rows last, the whole configuration turned by a signed axis permutation (exact)."""
    from tests.test_pair_boundary import _cramer

    out = []
    for delta in [s * d for d in ASSERTED for s in (1.0, -1.0)]:
        # face to face: set {2^k z <= b, z >= z0 - 0.3} with five lateral rows; box row -z <= -lz, c2 = fl(-lz - tol)
        z0, k = rng.uniform(-0.2, 0.2), int(rng.integers(-2, 3))
        th = 2 * np.pi * (np.arange(5) + rng.uniform(-0.2, 0.2, 5)) / 5
        A1 = np.vstack(([0.0, 0.0, 2.0 ** k], [0.0, 0.0, -1.0], np.c_[np.cos(th), np.sin(th), np.zeros(5)]))
        b1 = np.r_[(z0 + 0.3) * 2.0 ** k, -(z0 - 0.3), np.full(5, 0.3)]
        top = Fr(float(b1[0] - tol)) / Fr(2.0 ** k)      # the shrunk set reaches z = top, exactly
        lz = float(top - Fr(delta)) - tol
        exact = top + Fr(float(-lz - tol))
        box = np.r_[-0.5, -0.5, lz, 0.5, 0.5, lz + 0.5]
        out.append(("face", delta, A1, b1, [0], box, exact, np.array([0.0, 0.0, z0 + 0.3])))
        # vertex to face: a pyramid below its apex (rows n.x <= n.apex, n_z > 0) and a bottom row
        h = rng.uniform(-0.2, 0.2)
        apex = np.array([0.0, 0.0, h])
        th = 2 * np.pi * (np.arange(3) + rng.uniform(-0.15, 0.15, 3)) / 3
        N = np.c_[np.cos(th), np.sin(th), rng.uniform(0.4, 1.0, 3)] * (2.0 ** rng.integers(-2, 3, 3))[:, None]
        A1 = np.vstack((N, [0.0, 0.0, -1.0]))
        b1 = np.r_[N @ apex, -(h - 0.5)]
        xa = _cramer(A1[:3], [float(v) - tol for v in b1[:3]])     # the shrunk apex, exactly
        lz = float(xa[2] - Fr(delta)) - tol
        exact = xa[2] + Fr(float(-lz - tol))
        x0, y0 = float(xa[0]), float(xa[1])
        box = np.r_[x0 - 0.6, y0 - 0.6, lz, x0 + 0.6, y0 + 0.6, lz + 0.5]
        out.append(("vertex", delta, A1, b1, [0, 1, 2], box, exact, apex))
    cases = []
    for kind, delta, A1, b1, dec, box, exact, centre in out:
        A1, b1 = _arrange_last(rng, A1, b1, dec, m_total, centre)
        P = _signed_perm(rng)                             # rows a -> P a, box corners -> P corner
        c = np.array([box[:3], box[3:]]) @ P.T
        cases.append((kind, delta, [A1 @ P.T, b1], np.r_[c.min(axis=0), c.max(axis=0)], exact))
    return cases


def _poly_cases(rng, tol, m_total):
    """(set, obstacle [A, b] of <= 15 rows, exact margin) from the face-to-face and vertex-to-face constructions of
    test_pair_boundary (random rotations, mixed row scales), the set padded to m_total rows, deciding rows last."""
    from tests import test_pair_boundary as tpb

    assert tpb.TOL == tol
    out = []
    for delta in [s * d for d in ASSERTED for s in (1.0, -1.0)]:
        for make in (tpb._face_to_face, tpb._vertex_to_face):
            case = make(rng, delta, aligned=False, dominant=bool(rng.integers(2)))
            n2 = case.A2.shape[0]
            A1, b1, pos1 = tpb._arrange(rng, case.A1, case.b1, case.dec1, m_total, case.centre, case.dominant, True)
            A2, b2, pos2 = tpb._arrange(rng, case.A2, case.b2, case.dec2, min(15, n2 + int(rng.integers(0, 4))),
                                        case.centre, case.dominant, True)
            tpb._certify(case, A1, b1, pos1, A2, b2, pos2)
            out.append((case.kind, delta, [A1, b1], [A2, b2], case.exact))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("m_total", [20, 48], ids=["le32_rows", "33_63_rows"])
def test_exact_margins(geo, m_total):
    """Box obstacles (6 rows: 26 or 54 stacked) and polytopes of <= 15 rows (<= 32 or 33 .. 63 stacked), the set's
    deciding rows last (up to index 47), margins +-1e-3 .. +-1e-9; every set against a scene of its own obstacle."""
    rng = np.random.default_rng(7 + m_total)
    tol = 0.01
    n_dec = 0
    for _ in range(2):
        cases = _box_cases(rng, tol, m_total)
        batch = geo.SceneBatch([c[3][None] for c in cases], 0.0)
        try:
            got = _hits(geo, batch, [c[2] for c in cases], np.arange(len(cases), dtype=np.int32), tol)
        finally:
            batch.close()
        for (kind, delta, s, _, exact), g in zip(cases, got):
            assert (s[0].shape[0] + 6 > 32) == (m_total == 48)
            assert g == (0 if exact > 0 else -1), (kind, delta, float(exact), g)
            n_dec += 1
        pcases = _poly_cases(rng, tol, m_total)
        batch = geo.PolytopeSceneBatch([([c[3]], None) for c in pcases])
        try:
            got = _hits(geo, batch, [c[2] for c in pcases], np.arange(len(pcases), dtype=np.int32), tol)
        finally:
            batch.close()
        for (kind, delta, s, o, exact), g in zip(pcases, got):
            rows = s[0].shape[0] + o[0].shape[0]
            assert (rows > 32) if m_total == 48 else (rows <= 32)
            assert g == (0 if exact > 0 else -1), (kind, delta, float(exact), g)
            n_dec += 1
    assert n_dec == 2 * (16 + 16)


def _oracle_first_hits(sets, obstacles, obs_boxes, set_boxes, tol):
    """The lowest obstacle index for which the oracle's set_intersection succeeds, per set; only pairs whose
    boxes overlap are asked (disjoint boxes cannot intersect)."""
    from oracle.set_graph import set_intersection

    out, calls = [], 0
    for s, bx in zip(sets, set_boxes):
        hit = -1
        near = np.nonzero(np.all(obs_boxes[:, :3] <= bx[3:] + 1e-6, axis=1) &
                          np.all(obs_boxes[:, 3:] >= bx[:3] - 1e-6, axis=1))[0]
        for o in near:
            calls += 1
            if set_intersection(s, obstacles[o], tol)[2]:
                hit = int(o)
                break
        out.append(hit)
    return np.array(out, np.int32), calls


def _set_boxes(geo, sets):
    import torch

    A, b, m = _pack_sets(sets)
    return geo.set_aabb(geo._dev(A), geo._dev(b), geo._dev(m, torch.int32)).cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["boxes", "polytopes"])
def test_corridor_hits_against_the_oracle(geo, kind):
    """64 C3 box queries (48 polytope queries) planned, their obstacles moved, every corridor set checked."""
    from oracle.obstacles import obstacle_reps

    Q = 64 if kind == "boxes" else 48
    make = _box_scene if kind == "boxes" else _poly_scene
    sc = [make(i) for i in range(Q)]
    infl = sc[0][1]
    queries = _copies([s for s, _ in sc], infl, list(range(Q)), seed=3100)
    pl = pn.NativePlanner(queries, infl, WMAX, WMIN)
    try:
        res, _ = pl.run(list(range(Q)))
        rng = np.random.default_rng(5)
        moved = [dict(q, **_moved_scene(q, rng)) for q in queries]
        pl.update_obstacles(moved)
        corridors = [r["sets_via_prev"] if isinstance(r, dict) else None for r in res]
        hits = pl.corridor_hits(corridors, tol=1e-3)
        ev = pl.corridor_events
    finally:
        pl.close()
    n_sets = n_hit = n_calls = 0
    for q, (c, h) in enumerate(zip(corridors, hits)):
        if c is None:
            assert h is None
            continue
        if kind == "boxes":
            ob = np.asarray(moved[q]["obstacles"])
            obstacles, _, _ = obstacle_reps(ob, infl)
            obs_boxes = np.c_[ob[:, :3] - infl, ob[:, 3:] + infl]
        else:
            obstacles = moved[q]["obs_sets"]
            obs_boxes = np.array([np.r_[p.min(axis=0), p.max(axis=0)] for p in moved[q]["obs_points_sets"]])
        want, calls = _oracle_first_hits(c, obstacles, obs_boxes, _set_boxes(geo, c), 1e-3)
        assert np.array_equal(h, want), (q, h, want)
        n_sets += len(c)
        n_hit += int((h >= 0).sum())
        n_calls += calls
    assert ev[0].elapsed_time(ev[1]) >= 0.0
    print(f"\n{kind}: {n_sets} corridor sets, {n_hit} hit, {n_calls} oracle calls")
    assert n_sets >= 32 and 0 < n_hit < n_sets


def _c2_golden_sets():
    g = np.load(os.path.join(ROOT, "tests", "golden", "c2_graph_golden.npz"))
    off = np.r_[0, np.cumsum(g["m"])]
    rows = g["rows"]
    return [[rows[off[s]: off[s + 1], :3].copy(), rows[off[s]: off[s + 1], 3].copy()] for s in range(len(g["m"]))
            if g["status"][s] == 0]


@pytest.mark.gpu
@pytest.mark.parametrize("inflate", [0.01, 0.03])
def test_c2_golden_sets(geo, inflate):
    """The C2 golden sets against the C2 scene (the inflation they were built with: no hit expected) and against the
    same scene inflated further."""
    from oracle.obstacles import obstacle_reps

    ob, infl, _, _, _ = scenes.config_c2()
    sets = _c2_golden_sets()
    sc = geo.Scene(ob, inflate)
    try:
        got = _hits(geo, sc, sets)
    finally:
        sc.close()
    obstacles, _, _ = obstacle_reps(ob, inflate)
    obs_boxes = np.c_[ob[:, :3] - inflate, ob[:, 3:] + inflate]
    want, calls = _oracle_first_hits(sets, obstacles, obs_boxes, _set_boxes(geo, sets), 1e-3)
    assert np.array_equal(got, want)
    print(f"\nC2 golden sets at inflate {inflate}: {len(sets)} sets, {int((got >= 0).sum())} hit, {calls} oracle calls")
    if inflate == infl:
        assert (got == -1).all()
    else:
        assert (got >= 0).any()


@pytest.mark.gpu
def test_edge_cases(geo):
    from boundplanner_b200 import _lib

    # a unit-ish set around the origin; obstacles 0 and 2 far, 1, 3 and 4 hitting it: the lowest index (1) wins
    s = _box_rows([-0.1, -0.1, -0.1, 0.1, 0.1, 0.1], 0.0)
    boxes = np.array([[0.5, 0.5, 0.5, 0.6, 0.6, 0.6], [0.05, 0.0, 0.0, 0.3, 0.1, 0.1], [-0.9, -0.9, -0.9, -0.8, -0.8, -0.8],
                      [-0.3, -0.05, -0.05, 0.0, 0.05, 0.05], [-0.05, -0.05, -0.05, 0.05, 0.05, 0.05]])
    padded = [np.vstack((s[0], np.zeros((7, 3)))), np.r_[s[1], np.full(7, 10.0)]]
    sc = geo.Scene(boxes, 0.0)
    try:
        assert _hits(geo, sc, [s, padded]).tolist() == [1, 1]
        assert _hits(geo, sc, [s], tol=0.2).tolist() == [-1]          # shrunk by 0.2 the set is empty
        one = geo.Scene(np.array([[0.0995, -0.1, -0.1, 0.3, 0.1, 0.1]]), 0.0)   # overlaps s by 5e-4 < 2 tol
        try:
            assert _hits(geo, one, [s]).tolist() == [-1]
            assert _hits(geo, one, [s], tol=0.0).tolist() == [0]
        finally:
            one.close()
        A, b, m = _pack_sets([s])
        for bad_tol in (-1e-3, float("nan"), float("inf")):
            with pytest.raises(_lib.BpGeoError, match="tol must be finite"):
                geo.sets_obstacle_hits(sc, A, b, m, tol=bad_tol)
        with pytest.raises(_lib.BpGeoError, match="m_max"):
            geo.sets_obstacle_hits(sc, np.zeros((1, 49, 3)), np.ones((1, 49)), np.array([6]))
    finally:
        sc.close()
    # a batch with an empty scene, a shared-scene map and out-of-range scene indices
    batch = geo.SceneBatch([boxes[::-1], np.zeros((0, 6)), boxes[:2]], 0.0)
    try:
        got = _hits(geo, batch, [s, s, s, s, s, padded], np.array([0, 1, 2, 3, -1, 2], np.int32))
        assert got.tolist() == [0, -1, 1, -2, -2, 1]
        assert _hits(geo, batch, [s]).tolist() == [0]                # set_scene None: scene 0
    finally:
        batch.close()
    poly = [_box_rows(bx, 0.0) for bx in boxes]
    pb = geo.PolytopeSceneBatch([(poly[:3], None), (poly[3:], None)])
    try:
        got = _hits(geo, pb, [s, s, padded], np.array([0, 1, 1], np.int32))
        assert got.tolist() == [1, 0, 0]
    finally:
        pb.close()


# ---- GPU: subset runs of the native planner --------------------------------------------------------------------
def _rng_words(pl):
    return next(iter(pl._packed.values())).rng_out


def _mpc_subset_loop(kind, shared):
    Q = 32
    make = _box_scene if kind == "boxes" else _poly_scene
    n_sc = 4 if shared else Q
    sc = [make(i) for i in range(n_sc)]
    infl = sc[0][1]
    scene_list = [s for s, _ in sc]
    query_scene = [k % n_sc for k in range(Q)]
    copies = _copies(scene_list, infl, query_scene, seed=4100)
    queries, _ = shared_form(copies, query_scene) if shared else (copies, None)
    pl = pn.NativePlanner(queries, infl, WMAX, WMIN, scenes=scene_list if shared else None)
    n_active = n_checked = 0
    try:
        seeds = list(range(Q))
        res, _ = pl.run(seeds)
        for step in range(2):
            rng = np.random.default_rng(90 + step)
            nxt = []
            for q, r in zip(queries, res):
                nq = dict(mpc_step(q, r), new_obs=True) if isinstance(r, dict) else dict(q, replanning=False)
                nxt.append(nq)
            if shared:
                scene_list = [_moved_scene(s, rng) for s in scene_list]
                pl.update_obstacles(nxt, scenes=scene_list)
            else:
                nxt = [dict(q, **_moved_scene(q, rng)) for q in nxt]
                pl.update_obstacles(nxt)
            queries = nxt
            hits = pl.corridor_hits([q.get("sets_via_prev") for q in queries])
            active = [h is None or bool((h >= 0).any()) or k % 5 == 0 for k, h in enumerate(hits)]
            active[1] = False
            seeds = [100 * (step + 1) + k for k in range(Q)]
            full, fst = pl.run(seeds)
            rng_full = _rng_words(pl).copy()
            _rng_words(pl)[:] = 0
            sub, sst = pl.run(seeds, active=active)
            rng_sub = _rng_words(pl)
            assert [r is None for r in sub] == [not a for a in active]
            idx = [k for k in range(Q) if active[k]]
            _assert_same_plans([sub[k] for k in idx], [full[k] for k in idx])
            assert np.array_equal(rng_sub[idx], rng_full[idx])
            assert np.all(rng_sub[[k for k in range(Q) if not active[k]]] == 0)
            assert sst["set_requests"] <= fst["set_requests"]
            assert all(int(sst["finish_round"][k]) == -1 for k in range(Q) if not active[k])
            n_active += len(idx)
            n_checked += sum(isinstance(full[k], dict) for k in idx)
            res = full
    finally:
        pl.close()
    assert n_checked >= 4 and n_active < 2 * Q


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["boxes", "polytopes"])
def test_native_active_equals_full_run(kind):
    _mpc_subset_loop(kind, shared=False)


@pytest.mark.gpu
def test_native_active_over_shared_scenes():
    _mpc_subset_loop("boxes", shared=True)


@pytest.mark.gpu
def test_plan_batch_active_equals_native():
    sc = [_box_scene(i) for i in range(8)]
    infl = sc[0][1]
    queries = _copies([s for s, _ in sc], infl, list(range(8)), seed=5100)
    seeds = list(range(8))
    active = [True, False, True, True, False, True, False, True]
    nat, _ = pn.plan_batch_native(queries, infl, WMAX, WMIN, rng_seeds=seeds, active=active)
    py, _ = plan_batch(queries, infl, WMAX, WMIN, rng_seeds=seeds, active=active)
    assert [r is None for r in nat] == [r is None for r in py] == [not a for a in active]
    for i, (g, w) in enumerate(zip(nat, py)):
        if w is None:
            continue
        if isinstance(w, Exception):
            assert type(g) is type(w), (i, g, w)
            continue
        assert g["path"] == w["path"] and g["set_ids"] == w["set_ids"], i
        assert np.abs(g["p_via"] - w["p_via"]).max() < 1e-9, i
