"""Shared helpers for the parity tests."""
import ctypes
import re

import networkx as nx
import numpy as np
from scipy.spatial.transform import Rotation as R

from boundplanner_b200 import planner_native as pn
from boundplanner_b200 import scenes
from boundplanner_b200.planner import SetSequencePlanner
from oracle.convex_set_finder import ConvexSetFinder as OracleFinder
from oracle.obstacles import obstacle_reps

# north_star: halfspace coefficients agree within 1e-6 relative (fp64)
RTOL = 1e-6
R0 = R.from_euler("XYZ", [0, 90, 0], degrees=True).as_matrix()
ERRORS = (RuntimeError, ValueError, IndexError, AttributeError)     # what plan_set_sequence may raise for a query


def oracle_finder(boxes, inflate, ws_min, ws_max, max_rows=None):
    obs_sets, pts, _ = obstacle_reps(boxes, inflate)
    return OracleFinder(obs_sets, pts, ws_max, ws_min, max_rows=max_rows)


REORDERED = []      # (tag) of every comparison that only matched up to a permutation of the picked rows


def assert_rows_close(A, b, Ao, bo, tag=""):
    """Rows agree within RTOL, in order.  The picked rows (index >= 6) may come in a different ORDER when the
    greedy loop met a numerical tie: the obstacles an inscribed ellipsoid touches are all at distance exactly 1 in
    its metric (ConvexSetFinder.py:429-431), so which of them np.argmin returns first is decided by the last bits
    of the MVIE solve -- in the reference (OSQP / Clarabel tolerances) as much as here.  Such a permutation is
    accepted and recorded in REORDERED; the set of halfspaces must still be the same."""
    assert A.shape == Ao.shape, f"{tag}: row count {A.shape[0]} vs oracle {Ao.shape[0]}"
    scale = max(1.0, np.abs(bo).max())
    if np.abs(A - Ao).max() <= RTOL and np.abs(b - bo).max() <= RTOL * scale:
        return
    assert np.abs(A[:6] - Ao[:6]).max() <= RTOL and np.abs(b[:6] - bo[:6]).max() <= RTOL * scale, f"{tag}: init rows"
    free = list(range(6, Ao.shape[0]))
    for r in range(6, A.shape[0]):
        d = [max(np.abs(A[r] - Ao[k]).max(), abs(b[r] - bo[k]) / scale) for k in free]
        k = int(np.argmin(d))
        assert d[k] <= RTOL, f"{tag}: row {r} has no counterpart in the oracle's set (closest differs by {d[k]})"
        free.pop(k)
    REORDERED.append(tag)


class OracleBackend:
    """Planner-loop primitives served by the oracle (same interface as planner.GpuBackend)."""

    def __init__(self, obstacles, obs_size_increase, workspace_max, workspace_min):
        from oracle.obstacles import obstacle_reps

        self.obs_sets, pts, _ = obstacle_reps(obstacles, obs_size_increase)
        self.set_finder = OracleFinder(self.obs_sets, pts, list(workspace_max), list(workspace_min))

    def find_set_around_point(self, p, fixed_mid, optimize):
        return self.set_finder.find_set_around_point(p, fixed_mid=fixed_mid, optimize=optimize)

    def find_set_collision_avoidance(self, p0, p1, compute_ellipsoid):
        return self.set_finder.find_set_collision_avoidance(p0, p1, compute_ellipsoid)

    def reduce_ineqs(self, a_set, b_set):
        from oracle.reduce_ineqs import reduce_ineqs

        return reduce_ineqs(a_set, b_set)

    def set_intersection(self, set1, set2, tol):
        from oracle.set_graph import set_intersection

        return set_intersection(set1, set2, tol)

    def check_intersection(self, a_set, b_set, l_ee, sample, omega_normed, omega_norm):
        from oracle.planner_graph import check_intersection

        return check_intersection(a_set, b_set, l_ee, sample, omega_normed, omega_norm)

    def project(self, a_set, b_set, x_d, x0=None):
        from oracle.planner_graph import project_point

        return project_point(a_set, b_set, x_d)

    def execute(self, req):
        """Request protocol of boundplanner_b200/planner.py, answered by the oracle."""
        kind = req[0]
        if kind == "set_point":
            A, b, Q, p = self.find_set_around_point(req[1], req[2], req[3])
            Ar, br = self.reduce_ineqs(A, b)
            return A, b, Q, p, Ar, br
        if kind == "set_line":
            A, b, Q, p, coll = self.find_set_collision_avoidance(req[1], req[2], True)
            Ar, br = self.reduce_ineqs(A, b)
            return A, b, Q, p, coll, Ar, br
        if kind == "edges":
            l_ee, omega_normed, omega_norm = req[4]
            out = []
            for setc in req[1]:
                x, _, ok = self.set_intersection(setc, req[2], req[3])
                fits, via = False, None
                if ok:
                    a_set = np.concatenate((setc[0], req[2][0]))
                    b_set = np.concatenate((setc[1], req[2][1]))
                    fits, via = self.check_intersection(a_set, b_set, l_ee, x, omega_normed, omega_norm)
                out.append((x, ok, fits, via))
            return out
        if kind == "intersect_many":
            out = []
            for setc in req[1]:
                x, _, ok = self.set_intersection(setc, req[2], req[3])
                out.append((x, ok))
            return out
        if kind == "fit_many":
            l_ee, omega_normed, omega_norm = req[2]
            return [self.check_intersection(a, b, l_ee, s, omega_normed, omega_norm) for a, b, s in req[1]]
        if kind == "project":
            return self.project(req[1], req[2], req[3])
        if kind == "reduce":
            return self.reduce_ineqs(req[1], req[2])
        raise ValueError(kind)


class OracleDeviceLoopBackend(OracleBackend):
    """OracleBackend that also answers the device-loop requests of the planner (sample_set, shortest_path, set_point
    with the planner attached) -- with the REFERENCE'S host loops, so that the planner-side protocol (candidates
    drawn ahead in chunks, generator rewind) can be checked against the plain host loop without a GPU."""

    device_loop = True

    def execute(self, req):
        kind = req[0]
        if kind == "sample_set":
            cand, optimize, pl = np.asarray(req[1], float).reshape(-1, 3), req[2], req[3]
            for i, c in enumerate(cand):                      # BoundPlanner.py:459-478, one candidate at a time
                if not pl._in_collision(c) and not pl._in_safe(c):
                    try:
                        A, b, Q, p = self.find_set_around_point(c, True, optimize)
                    except (RuntimeError, ValueError) as e:
                        return i, e
                    Ar, br = self.reduce_ineqs(A, b)
                    return i, (A, b, Q, p, Ar, br, pl._min_node_distance(Q, p))
            return -1, None
        if kind == "shortest_path":
            return nx.shortest_path(req[1], 0, 1, weight="weight")
        if kind == "set_point" and len(req) > 4:
            out = super().execute(req[:4])
            return out + (req[4]._min_node_distance(out[2], out[3]),)
        return super().execute(req)


class MemoBackend(OracleBackend):
    """OracleBackend with its answers memoised by request content: the Python planner and the native driver ask
    the same questions, the oracle answers each once."""

    def __init__(self, *a):
        super().__init__(*a)
        self.memo = {}

    @staticmethod
    def _key(x):
        if isinstance(x, np.ndarray):
            return x.tobytes()
        if isinstance(x, (list, tuple)):
            return tuple(MemoBackend._key(v) for v in x)
        if isinstance(x, (float, np.floating)):
            return float(x)
        return x

    def execute(self, req):
        k = self._key(req)
        if k not in self.memo:
            try:
                self.memo[k] = super().execute(req)
            except (RuntimeError, ValueError) as e:
                self.memo[k] = e
        ans = self.memo[k]
        if isinstance(ans, Exception):
            raise ans
        return ans


class PolytopeOracleBackend(MemoBackend):
    """The oracle's ConvexSetFinder over polytope obstacles (obs_sets + obs_points_sets), answers memoised."""

    def __init__(self, obs_sets, obs_points_sets, workspace_max, workspace_min):
        self.obs_sets = obs_sets
        self.set_finder = OracleFinder(obs_sets, obs_points_sets, list(workspace_max), list(workspace_min))
        self.memo = {}


class OracleLockstepExecutor:
    """CPU stand-in for planner.BatchedGpuExecutor: every pending request answered by the query's oracle backend."""

    def __init__(self, backends):
        self.backends = backends
        self.calls = 0

    def execute(self, pending):
        out = {}
        self.calls += 1
        for qid, req in pending.items():
            try:
                out[qid] = self.backends[qid].execute(req)
            except (RuntimeError, ValueError) as e:
                out[qid] = e
        return out


# ---- the native lock-step driver in the host harness (tests/host_harness.cpp: hh_plan_batch) -------------------
# ctypes mirrors of its request and answer records (csrc/bp_planner.h) and of its callbacks
_dp = ctypes.POINTER(ctypes.c_double)
_ip = ctypes.POINTER(ctypes.c_int)


class SetReq(ctypes.Structure):
    _fields_ = [("qid", ctypes.c_int), ("kind", ctypes.c_int), ("fixed_mid", ctypes.c_int), ("optimize", ctypes.c_int),
                ("with_dv", ctypes.c_int), ("n_cand", ctypes.c_int), ("p0", ctypes.c_double * 3),
                ("p1", ctypes.c_double * 3), ("cand", _dp)]


class SetAns(ctypes.Structure):
    _fields_ = [("status", ctypes.c_int), ("rows_peak", ctypes.c_int), ("m", ctypes.c_int), ("m_red", ctypes.c_int),
                ("collision", ctypes.c_int), ("first", ctypes.c_int), ("dv", ctypes.c_double),
                ("A", ctypes.c_double * (pn.SET_ROWS * 3)), ("b", ctypes.c_double * pn.SET_ROWS),
                ("Ar", ctypes.c_double * (pn.SET_ROWS * 3)), ("br", ctypes.c_double * pn.SET_ROWS),
                ("Q", ctypes.c_double * 9), ("P", ctypes.c_double * 3)]


class Node(ctypes.Structure):
    _fields_ = [("m", ctypes.c_int), ("A", ctypes.c_double * (pn.NODE_ROWS * 3)), ("b", ctypes.c_double * pn.NODE_ROWS),
                ("Q", ctypes.c_double * 9), ("P", ctypes.c_double * 3), ("size", ctypes.c_double),
                ("c_size", ctypes.c_double)]


class EdgeAns(ctypes.Structure):
    _fields_ = [("ok", ctypes.c_int), ("fits", ctypes.c_int), ("x", ctypes.c_double * 3), ("omega", ctypes.c_double),
                ("proj_ok", ctypes.c_int), ("proj", ctypes.c_double * 3)]


class ProjAns(ctypes.Structure):
    _fields_ = [("x", ctypes.c_double * 3), ("status", ctypes.c_int)]


class ReduceReq(ctypes.Structure):
    _fields_ = [("qid", ctypes.c_int), ("m", ctypes.c_int), ("rows", _dp)]


CB_SET = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_int, ctypes.POINTER(SetReq), ctypes.c_int, ctypes.POINTER(Node),
                          ctypes.POINTER(SetAns))
CB_EDGES = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.POINTER(Node), _ip, _dp,
                            ctypes.POINTER(EdgeAns))
CB_PROJECT = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, _dp, ctypes.c_int,
                              ctypes.POINTER(Node), ctypes.POINTER(ProjAns))
CB_PATH = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_int, ctypes.c_int, _ip, _ip, _dp, _ip, _ip)
CB_REDUCE = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_int, ctypes.POINTER(ReduceReq), ctypes.POINTER(SetAns))


def _node_set(nd):
    m = nd.m
    return [np.array(nd.A[: 3 * m]).reshape(m, 3), np.array(nd.b[:m])]


def _fill_set(out, ans, with_line):
    if with_line:
        A, b, Q, p, coll, Ar, br = ans
        out.collision = int(bool(coll))
    else:
        A, b, Q, p, Ar, br = ans[:6]
    m, mr = A.shape[0], Ar.shape[0]
    assert m <= pn.SET_ROWS
    out.status, out.m, out.m_red, out.rows_peak = 0, m, mr, m
    out.A[: 3 * m] = A.reshape(-1).tolist()
    out.b[:m] = b.tolist()
    out.Ar[: 3 * mr] = Ar.reshape(-1).tolist()
    out.br[:mr] = br.tolist()
    out.Q[:] = np.asarray(Q).reshape(-1).tolist()
    out.P[:] = np.asarray(p).reshape(-1).tolist()


def _error_status(e, out):
    msg = str(e)
    if "Ellipse violates" in msg:
        out.status = 1
    elif "could not broadcast" in msg:
        out.status, out.rows_peak, out.m = 5, int(re.search(r"shape \((\d+),\)", msg).group(1)), 0
        out.m = out.rows_peak
    else:
        raise e


def _is_poly(q):
    return q.get("obs_sets") is not None


def _backend(q, inflate, ws_max, ws_min):
    if _is_poly(q):
        return PolytopeOracleBackend(q["obs_sets"], q["obs_points_sets"], ws_max, ws_min)
    return MemoBackend(q["obstacles"], inflate, ws_max, ws_min)


def _planner(q, inflate, ws_max, ws_min, backend, seed=None):
    return SetSequencePlanner(() if _is_poly(q) else q["obstacles"], inflate, list(ws_max), list(ws_min),
                              backend=backend, rng=np.random.default_rng(seed),
                              obs_sets=q["obs_sets"] if _is_poly(q) else backend.obs_sets)


def python_plan(q, inflate, ws_max, ws_min, seed, backend):
    """The sequential driver on one query, its planner holding the query's previous sets."""
    pl = _planner(q, inflate, ws_max, ws_min, backend, seed)
    pl.sets_via_prev = [[np.array(a, float), np.array(b, float)] for a, b in q.get("sets_via_prev", ())]
    try:
        res = pl.plan_set_sequence(q["start"].copy(), q["end"].copy(), q["r0"], q["r1"], q.get("first_sample"),
                                   q.get("replanning", False), q.get("p_horizon", ()), q.get("new_obs", False))
    except ERRORS as e:
        res = e
    return res, pl


def run_native_with_oracle(harness, queries, inflate, ws_max, ws_min, seeds, backends, sample_chunk=32, lanes=1):
    """The native state machines (hh_plan_batch) with every request answered by the queries' oracle backends -- the
    same answers the Python planner gets from them; boxes or polytopes.  Returns the PackedQueries."""
    pk = pn.PackedQueries(queries, inflate, ws_max, ws_min, seeds, sample_chunk)
    helpers = [_planner(q, inflate, ws_max, ws_min, backends[i]) for i, q in enumerate(queries)]
    ee = []
    for q in queries:
        omega = R.from_matrix(q["r1"] @ q["r0"].T).as_rotvec()
        on = np.linalg.norm(omega)
        ee.append((q["r0"] @ np.array([-0.05, 0, 0]), omega / on if on > 1e-6 else np.array([0, 0, 1.0]), on))
    errors = []

    def guarded(fn):
        def call(*a):
            try:
                return fn(*a)
            except Exception as e:                           # noqa: BLE001 -- surfaces in the assert below
                errors.append(e)
                return 7
        return call

    @guarded
    def cb_set(qid, req, n_nodes, nodes, out):
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
                safe = any(np.max(_node_set(nodes[k])[0] @ c - _node_set(nodes[k])[1]) < 1e-3 for k in range(n_nodes))
                if not helpers[qid]._in_collision(c) and not safe:
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
            o.dv = min((np.linalg.norm(np.array(nodes[k].Q[:]).reshape(3, 3) - ans[2]) +
                        np.linalg.norm(np.array(nodes[k].P[:]) - ans[3]) for k in range(n_nodes)), default=np.inf)
        return 0

    @guarded
    def cb_edges(qid, id_new, n_nodes, nodes, has_target, xd, out):
        others = [_node_set(nodes[k]) for k in range(id_new)]
        new = _node_set(nodes[id_new])
        res = backends[qid].execute(("edges", others, new, 0.01, ee[qid]))
        for k, (x, ok, fits, via) in enumerate(res):
            out[k].ok, out[k].fits, out[k].proj_ok = int(bool(ok)), int(bool(fits)), 0
            if ok:
                out[k].x[:] = np.asarray(x).tolist()
                out[k].omega = float(via[3]) if fits else -1.0
                if has_target[k]:                             # the hit's projection, asked for with the edges
                    pr = backends[qid].execute(("project", np.concatenate((others[k][0], new[0])),
                                                np.concatenate((others[k][1], new[1])),
                                                np.array([xd[3 * k], xd[3 * k + 1], xd[3 * k + 2]])))
                    out[k].proj[:] = np.asarray(pr).tolist()
                    out[k].proj_ok = 1
        return 0

    @guarded
    def cb_project(qid, id0, id1, xd, n_nodes, nodes, out):
        s0, s1 = _node_set(nodes[id0]), _node_set(nodes[id1])
        x = backends[qid].execute(("project", np.concatenate((s0[0], s1[0])), np.concatenate((s0[1], s1[1])),
                                   np.array([xd[0], xd[1], xd[2]])))
        out.contents.x[:] = np.asarray(x).tolist()
        return 0

    @guarded
    def cb_path(qid, n, edge_off, edge_dst, edge_w, path_out, path_len):
        g = nx.Graph()
        g.add_nodes_from(range(n))
        for v in range(n):                                    # adjacency dicts in the driver's insertion order
            for e in range(edge_off[v], edge_off[v + 1]):
                g._adj[v][edge_dst[e]] = {"weight": edge_w[e]}
        p = nx.shortest_path(g, 0, 1, weight="weight")
        path_len[0] = len(p)
        for k, v in enumerate(p[: pn.MAX_PATH]):
            path_out[k] = v
        return 0

    @guarded
    def cb_reduce(qid, req, out):
        r, o = req.contents, out.contents
        rows = np.ctypeslib.as_array(r.rows, shape=(r.m, 4)).copy()
        Ar, br = backends[qid].execute(("reduce", rows[:, :3].copy(), rows[:, 3].copy()))
        mr = Ar.shape[0]
        o.status, o.m, o.m_red = 0, r.m, mr
        o.Ar[: 3 * mr] = Ar.reshape(-1).tolist()
        o.br[:mr] = br.tolist()
        return 0

    cbs = (CB_SET(cb_set), CB_EDGES(cb_edges), CB_PROJECT(cb_project), CB_PATH(cb_path), CB_REDUCE(cb_reduce))
    rc = harness.hh_plan_batch(ctypes.byref(pk.inp), ctypes.byref(pk.out), *cbs, int(lanes))
    assert not errors, errors[0]
    assert rc == 0
    return pk


def _same_sets(got, want, tol=0.0):
    assert len(got) == len(want)
    for (ga, gb), (wa, wb) in zip(got, want):
        ga, gb, wa, wb = (np.asarray(v, float) for v in (ga, gb, wa, wb))
        assert ga.shape == wa.shape and gb.shape == wb.shape
        assert np.abs(ga - wa).max(initial=0.0) <= tol and np.abs(gb - wb).max(initial=0.0) <= tol


def assert_same_result(g, w, pl, i, exact=True):
    """g: a batched driver's result; w, pl: plan_set_sequence's result and planner."""
    if isinstance(w, Exception):
        assert isinstance(g, Exception), f"query {i}: planned, plan_set_sequence raised {w!r}"
        assert type(g) is type(w), (i, g, w)
        if exact:
            assert str(g) == str(w), (i, g, w)
        else:
            assert str(g).split("(")[0] == str(w).split("(")[0], (i, g, w)
        return False
    assert not isinstance(g, Exception), f"query {i}: {g!r}"
    assert g["path"] == w["path"] and g["set_ids"] == w["set_ids"], i
    tol = 0.0 if exact else 1e-9
    assert g["p_via"].shape == w["p_via"].shape and np.abs(g["p_via"] - w["p_via"]).max() <= tol, i
    n_nodes = g["n_nodes"] if "n_nodes" in g else g["graph"].number_of_nodes()
    n_inter = g["n_inter"] if "n_inter" in g else g["inter_graph"].number_of_nodes()
    assert n_nodes == w["graph"].number_of_nodes() and n_inter == w["inter_graph"].number_of_nodes(), i
    if "n_edges" in g:
        assert g["n_edges"] == w["inter_graph"].number_of_edges(), i
    set_tol = 0.0 if exact else 1e-9
    _same_sets(g["sets_via"], w["sets_via"], set_tol)
    _same_sets(g["sets_via_prev"], pl.sets_via_prev, set_tol)
    assert ("p_horizon_max" in g) == pl.replanning, i
    if pl.replanning:
        assert np.array_equal(g["p_horizon_max"], pl.p_horizon_max), i
    return True


# ---- queries -------------------------------------------------------------------------------------------------
def _c3(i):
    ob, infl, st, en, wmin, wmax = scenes.config_c3_query(i)
    return dict(obstacles=ob, start=st, end=en, r0=R0, r1=R0), infl, list(wmin), list(wmax)


def _c3_poly(i):
    obs_sets, pts, infl, st, en, wmin, wmax = scenes.config_c3_polytope_query(i)
    return dict(obs_sets=obs_sets, obs_points_sets=pts, start=st, end=en, r0=R0, r1=R0), infl, list(wmin), list(wmax)


def mpc_step(q, res, frac=0.02, n_horizon=10):
    """The next MPC call after a planned result: start `frac` along the first segment, a horizon of n_horizon
    points along the path from there, the result's sets_via_prev."""
    p_via = res["p_via"]
    start = p_via[0] + frac * (p_via[1] - p_via[0])
    t = np.linspace(0.0, 1.0, n_horizon + 1)[1:]
    pts = np.vstack((start, p_via[1:]))
    seg = np.cumsum(np.r_[0.0, np.linalg.norm(np.diff(pts, axis=0), axis=1)])
    s = t * seg[-1] * 0.6
    horizon = np.stack([np.interp(s, seg, pts[:, k]) for k in range(3)], axis=1)
    return dict(q, start=start, replanning=True, p_horizon=horizon, sets_via_prev=res["sets_via_prev"])
