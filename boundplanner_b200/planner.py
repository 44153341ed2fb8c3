"""Set-sequence planner: the reference's ``plan_convex_set_path`` up to the planned
set sequence, with every geometric primitive served by the GPU kernels.

Restates the control flow of bound_planner/BoundPlanner/BoundPlanner.py:

  plan_convex_set_path  :174-584   start / end sets (incl. the replanning branch :231-276 and the
                                   start-in-collision fallbacks :296-324), sampling loop, dedupe, convergence test
  compute_via_points    :586-743   with_rot=False branch (the via points are the p_proj's)
  add_edges             :789-896   intersection nodes, projection points, edge costs (quirk Q6)

What is NOT here: the final via-point NLP with rotations (Ipopt, :540-555) and, with it, the backwards
extension of the first segment when replanning (:706-729) -- they stay with the reference.  The output is what
precedes them: the shortest path through the intersection graph, the sets it visits ("planned set sequence") and
the position via points; ``sets_via_prev`` is kept for the next (re)planning call like the reference does
(:372, :556).

The loop is written ONCE, as a generator that yields *requests* for geometric
primitives and receives their results:

  ("set_point", p, fixed_mid, optimize) -> (A, b, q_ellipse, p_mid, A_red, b_red)   find_set_around_point + reduce_ineqs
  ("set_line", p0, p1)                  -> (A, b, q_ellipse, p_mid, collision, A_red, b_red)
  ("edges", sets, set_new, tol, ee)     -> [(point | None, ok, fits, via), ...]      set_intersection of the new set with
                                           every existing set + check_intersection of every hit (one device round:
                                           the fit check starts from the LP's point and never leaves the GPU)
  ("project", A, b, x_d)                -> x                                         projection QP of add_edges
  ("reduce", A, b)                      -> (A_red, b_red)                            reduce_ineqs of a given set
  with ``device_loop`` (backends that keep every query's known sets and node ellipsoids in device tables):
  ("sample_set", cand[C,3], optimize, planner) -> (first, (A, b, q, p, A_red, b_red, dvertex) | Exception)
                                           the rejection loop of :459-478 over C pre-drawn candidates (first accepted
                                           one, in draw order), find_set_around_point at it, reduce_ineqs and the
                                           duplicate-set distance of :505-512 -- one device round, nothing on the host
  ("set_point", p, fixed_mid, optimize, planner) -> (..., dvertex)                   the same for a given point
  ("shortest_path", inter_graph)        -> [node ids]                                nx.shortest_path(..., 0, 1) (:434)

Drivers: ``plan_set_sequence`` answers every request at once through a backend
(batch-of-one kernel calls; the parity tests plug the oracle in here), and
``plan_batch`` advances many queries in lock step, answering the pending
requests of ALL queries with one batched kernel call per primitive and round
(BASELINE config C3: thousands of independent queries, one scene each).
The intersections / fit checks of one add_edges call are independent of the
graph state that call mutates, so they are requested up front; the graph
bookkeeping then runs in the reference's order.
"""
from __future__ import annotations

import math

import networkx as nx
import numpy as np
from scipy.spatial.transform import Rotation as R

REFERENCE_MAX_ROWS = 20

try:                                   # np.linalg.det minus ~35 us of argument checking per call
    _det = np.linalg._umath_linalg.det
except AttributeError:                 # pragma: no cover
    _det = np.linalg.det


def _set_errors(status, rows):
    """Exception the reference would raise for a per-seed status (ConvexSetFinder.py:438, :516)."""
    if status == 1:
        return RuntimeError("Ellipse violates constraints")
    if status == 2:
        return ValueError("convex set needs more rows than the kernels hold")
    if status == 5 or (status == 0 and rows is not None and rows > REFERENCE_MAX_ROWS):
        return ValueError(f"could not broadcast input array from shape ({rows},) into shape ({REFERENCE_MAX_ROWS},)")
    if status in (3, 4):
        return RuntimeError(f"MVIE failed (status {status})")
    return None


class GpuBackend:
    """Answers planner requests one at a time: a batch of one through the same executor the lock-step driver
    uses, so every request is one chain of kernels on the device and one read-back.  Obstacles: boxes
    (``obstacles`` [N,6], inflated by obs_size_increase) or, with ``obs_sets``, inflated convex polytopes (vertex
    lists from ``obs_points_sets``, enumerated on the device when missing)."""

    device_loop = True       # sampling / duplicate test / shortest path on the device (K11-K13)

    def __init__(self, obstacles, obs_size_increase, workspace_max, workspace_min, obs_sets=None, obs_points_sets=None):
        if obs_sets is not None:
            self.obs_sets = obs_sets
            self._bx = BatchedGpuExecutor(None, obs_size_increase, workspace_max, workspace_min,
                                          polytope_scenes=[(obs_sets, obs_points_sets)])
            return
        self.obs_sets = obstacle_sets(obstacles, obs_size_increase)
        self._bx = BatchedGpuExecutor([np.asarray(obstacles, float).reshape(-1, 6)], obs_size_increase, workspace_max,
                                      workspace_min)

    def execute(self, req):
        ans = self._bx.execute({0: req})[0]
        if isinstance(ans, Exception):
            raise ans
        return ans


def obstacle_sets(obstacles, obs_size_increase):
    """add_obstacle_reps (:131-152): inflated boxes as [A (15x3), b (15)] padded like normalize_set_size."""
    boxes = np.asarray(obstacles, float).reshape(-1, 6)
    n = boxes.shape[0]
    a_all = np.zeros((n, 15, 3))
    a_all[:, :6] = np.concatenate((np.eye(3), -np.eye(3)))
    b_all = np.full((n, 15), 10.0)
    b_all[:, :3] = boxes[:, 3:] + obs_size_increase
    b_all[:, 3:6] = -boxes[:, :3] + obs_size_increase
    return [[a_all[i], b_all[i]] for i in range(n)]


_BOX_ROWS = np.concatenate((np.eye(3), -np.eye(3)))


def is_box_obstacle(a_set):
    """The rows of an axis-aligned box as add_obstacle_reps builds them (A = [I; -I], zero padding): the test of
    convex_set_finder.boxes_from_obs_sets."""
    a_set = np.asarray(a_set, float)
    return a_set.shape[0] >= 6 and np.array_equal(a_set[:6], _BOX_ROWS) and not np.any(a_set[6:] != 0.0)


def _rows_minus_b(A, b, x):
    """A x - b over stacked padded rows (A [..., 15, 3], b [..., 15]) as (a0 x0 + a1 x1) + a2 x2 - b, element by
    element: no BLAS, no fused multiply-add, the operation order of the native driver's push-out (bp_planner.h).  It
    differs from the reference's ob[0] @ x in the last bits only, and is exact for box rows."""
    return (A[..., 0] * x[0] + A[..., 1] * x[1]) + A[..., 2] * x[2] - b


class SetSequencePlanner:
    def __init__(self, obstacles=(), obs_size_increase=0.08, workspace_max=(1.0, 1.0, 1.2),
                 workspace_min=(-1.0, -1.0, 0.0), backend=None, rng=None, obs_sets=None, device_loop=None,
                 obs_points_sets=None):
        # device_loop: sampling / duplicate test / shortest path answered by the backend's kernels (K11-K13)
        # instead of the host loops below; default: whatever the backend offers
        self.device_loop = bool(getattr(backend, "device_loop", False)) if device_loop is None else bool(device_loop)
        self.sample_chunk = 32               # candidates drawn ahead per sampling request
        self.obs_size_increase = obs_size_increase
        self.workspace_max = list(workspace_max)
        self.workspace_min = list(workspace_min)
        # :47-58
        self.w_size = 0.1
        self.c_fit = 1.0
        self.w_bias = 0.01
        self.max_set_size = 20
        self.length_ee = 0.05
        self.max_iters = 20
        self.nr_optimized = 10
        self.nr_free_mid = 5
        self.max_samples = 500
        self.sets_via_prev = []              # :37; set by every successful plan (:372, :556)
        self.rng = rng if rng is not None else np.random.default_rng()      # unseeded in the reference (quirk Q4)
        self.backend = backend
        if obs_sets is not None:
            self.obs_sets = obs_sets
        elif backend is not None and hasattr(backend, "obs_sets"):
            self.obs_sets = backend.obs_sets
        else:
            self.obs_sets = obstacle_sets(obstacles, obs_size_increase)
        self._obstacles = obstacles
        self.obs_points_sets = obs_points_sets
        # general convex polytopes (any obstacle that is not a box): the host tests run on all 15 rows of every
        # obstacle (_rows_minus_b); box-shaped obs_sets keep the vectorised box forms below
        self.polytopes = not all(is_box_obstacle(ob[0]) for ob in self.obs_sets)
        if self.polytopes:
            n = len(self.obs_sets)
            self._obs_A = np.zeros((n, 15, 3))
            self._obs_b = np.full((n, 15), 10.0)
            for k, (a_set, b_set) in enumerate(self.obs_sets):
                a_set = np.asarray(a_set, float).reshape(-1, 3)
                self._obs_A[k, : a_set.shape[0]] = a_set
                self._obs_b[k, : a_set.shape[0]] = np.asarray(b_set, float).reshape(-1)
        # inflated box bounds for the vectorised form of the "sample in collision" test (:467-471): for a box
        # row (+-e_k) the reference's A x - b is exactly x_k - ub_k / lb_k - x_k, padded rows give -10
        ob_b = (np.zeros((len(self.obs_sets), 6)) if self.polytopes else       # (polytopes: not used)
                np.array([ob[1][:6] for ob in self.obs_sets]).reshape(-1, 6))
        self._ub, self._lb = ob_b[:, :3], -ob_b[:, 3:]
        self._b6 = np.ascontiguousarray(ob_b)                 # b of the rows [I; -I]: A x - b = [x; -x] - b6

    # ---- known sets, stacked (vectorised forms of the per-node loops of :472-476 and :505-512) ----
    def _nodes_reset(self):
        self._plan_epoch = getattr(self, "_plan_epoch", 0) + 1     # a new plan: device tables of the old one are stale
        self._rows_a = np.empty((0, 3))
        self._rows_b = np.empty(0)
        self._row_start = []                 # first stacked row of every node
        self._node_q = np.empty((0, 9))
        self._node_p = np.empty((0, 3))

    def _nodes_add(self, a_set, b_set, q_ellipse, p_mid):
        self._row_start.append(self._rows_a.shape[0])
        self._rows_a = np.concatenate((self._rows_a, np.asarray(a_set, float).reshape(-1, 3)))
        self._rows_b = np.concatenate((self._rows_b, np.asarray(b_set, float).reshape(-1)))
        self._node_q = np.concatenate((self._node_q, np.asarray(q_ellipse, float).reshape(1, 9)))
        self._node_p = np.concatenate((self._node_p, np.asarray(p_mid, float).reshape(1, 3)))

    def _in_safe(self, sample):
        """any node with max(a_set @ sample - b_set) < 1e-3  (:472-476)."""
        if not self._row_start:
            return False
        viol = self._rows_a @ sample - self._rows_b
        return bool((np.maximum.reduceat(viol, self._row_start) < 1e-3).any())

    def _min_node_distance(self, q_ellipse, p_mid):
        """min over nodes of ||q_ellipse - Q_v||_F + ||p_mid - p_v||  (:505-510)."""
        if self._node_q.shape[0] == 0:
            return np.inf
        dq = self._node_q - np.asarray(q_ellipse, float).reshape(1, 9)
        dp = self._node_p - np.asarray(p_mid, float).reshape(1, 3)
        return float((np.sqrt((dq * dq).sum(axis=1)) + np.sqrt((dp * dp).sum(axis=1))).min())

    def _in_collision(self, sample):
        if self._ub.shape[0] == 0:
            return False
        if self.polytopes:                                    # max over all 15 rows < 1e-3 (sample_flags)
            return bool((_rows_minus_b(self._obs_A, self._obs_b, sample).max(axis=1) < 1e-3).any())
        s6 = np.concatenate((sample, -sample))                # x - ub and lb - x = (-x) - (-lb), exactly
        return bool(((s6 - self._b6).max(axis=1) < 1e-3).any())

    def _push_out_boxes(self, end):
        """:199-204 over box obstacles, in place: obstacle by obstacle in order; the scan for the next obstacle that
        contains `end` is vectorised (box rows: A x - b is x_k - ub_k / lb_k - x_k; the padded rows give -10 and never
        decide)."""
        cursor = 0
        while cursor < len(self.obs_sets):
            inside = np.flatnonzero((np.maximum(end - self._ub[cursor:], self._lb[cursor:] - end) <= 0).all(axis=1))
            if inside.size == 0:
                break
            ob = self.obs_sets[cursor + int(inside[0])]
            viol = ob[0] @ end - ob[1]
            if not np.any(viol > 0):
                idx = np.argmax(viol)
                end -= (viol[idx] - self.obs_size_increase) * ob[0][idx, :]
            cursor += int(inside[0]) + 1
        return end

    def _push_out_general(self, end):
        """:199-204 over general polytope rows, in place: obstacle by obstacle in order, each tested with `end` as
        already moved; one without a positive A x - b over its 15 rows (padding included) pushes `end` out along its
        first row of largest A x - b (np.argmax).  The scan for the next such obstacle is vectorised; every A x - b
        is the element-wise form of _rows_minus_b."""
        cursor = 0
        while cursor < len(self.obs_sets):
            viol = _rows_minus_b(self._obs_A[cursor:], self._obs_b[cursor:], end)
            inside = np.flatnonzero(~(viol > 0).any(axis=1))
            if inside.size == 0:
                break
            k = int(inside[0])
            idx = int(np.argmax(viol[k]))
            end -= (viol[k, idx] - self.obs_size_increase) * self._obs_A[cursor + k, idx]
            cursor += k + 1
        return end

    # ---- :459-478 on the device ---------------------------------------------------
    def _sample_set_on_device(self, optimize):
        """The rejection loop with the candidates drawn ahead in chunks: the backend returns the first accepted
        candidate of a chunk (draw order) together with the convex set built around it.  Afterwards the generator is
        rewound to exactly the number of draws the reference's one-at-a-time loop would have consumed
        (rng.uniform(lo, hi, (n, 3)) is n successive rng.uniform(lo, hi, 3) draws of the same bit stream)."""
        lo, hi = self.workspace_min, self.workspace_max
        state = self.rng.bit_generator.state
        drawn, n, first, cand, payload = 0, 0, -1, None, None
        while drawn < self.max_samples + 1:
            c = min(self.sample_chunk, self.max_samples + 1 - drawn)
            cand = self.rng.uniform(lo, hi, (c, 3))
            first, payload = yield ("sample_set", cand, optimize, self)
            if first >= 0:
                n = drawn + first + 1
                break
            drawn += c
            n = drawn
        self.rng.bit_generator.state = state
        if n:
            self.rng.uniform(lo, hi, (n, 3))
        if first < 0 or n >= self.max_samples:                    # :477-478
            raise RuntimeError("(PosPath) Could not find collision-free sample")
        return cand[first].copy(), payload

    # ---- :789-896 -----------------------------------------------------------
    def _add_edges(self, id_new, graph, inter_graph, end, start):
        connected = False
        # (graph._node / inter_graph._node are networkx's own node -> attribute dicts: same objects the NodeView
        # hands out, without the view indirection on every access of this doubly nested loop)
        gnodes, inodes = graph._node, inter_graph._node
        set_new = gnodes[id_new]["cset"]
        others = [(vid, vdata) for vid, vdata in gnodes.items() if vid != id_new]
        if not others:
            return connected
        res = yield ("edges", [v["cset"] for _, v in others], set_new, 0.01,
                     (self.l_ee, self.omega_normed, self.omega_norm))
        hits = []
        for (vid, vdata), (p_intersect, ok, fits, via) in zip(others, res):
            if ok:
                set_inter = [np.concatenate((vdata["cset"][0], set_new[0])), np.concatenate((vdata["cset"][1], set_new[1]))]
                hits.append((vid, vdata, p_intersect, set_inter, fits, via))
        if not hits:
            return connected
        for vid, vdata, p_intersect, set_inter, fits, via in hits:
            self.id_inter += 1
            inter_graph.add_node(self.id_inter, cset=set_inter, id0=vid, id1=id_new, conn_to_start=False,
                                 conn_to_end=False, p_proj=None, p_via=via, fits=fits)
            self.nr_inter_set += 2
            me = inodes[self.id_inter]
            # the reference walks ALL intersection nodes in insertion order and keeps those that share a set with the
            # new one (:827-841); an index set -> its intersection nodes gives the same nodes in the same order
            # (intersection ids grow with insertion)
            by_node = self._inter_by_node
            by_node.setdefault(vid, []).append(self.id_inter)
            if id_new != vid:
                by_node.setdefault(id_new, []).append(self.id_inter)
            cand = by_node[vid] if id_new == vid else sorted(set(by_node[vid]) | set(by_node[id_new]))
            for eid in cand:
                edata = inodes[eid]
                v0, v1 = edata["id0"], edata["id1"]
                cond1 = v0 == vid or v1 == vid
                cond2 = v0 == id_new or v1 == id_new
                if cond1:
                    size = vdata["size"]
                elif cond2:
                    size = gnodes[id_new]["size"]
                if self.id_inter != eid and (cond1 or cond2):
                    self.nr_edges += 2
                    p_proj = edata["p_proj"]
                    if p_proj is None:
                        p_proj = end
                    if me["p_proj"] is None:
                        me["p_proj"] = yield ("project", set_inter[0], set_inter[1], np.array(p_proj, float))
                    dvec = me["p_proj"] - p_proj
                    dist = math.sqrt(float(dvec.dot(dvec)))            # == np.linalg.norm of a 1-D vector
                    conn_to_start = me["conn_to_start"] or edata["conn_to_start"]
                    conn_to_end = me["conn_to_end"] or edata["conn_to_end"]
                    me["conn_to_start"] = conn_to_start
                    me["conn_to_end"] = conn_to_end
                    edata["conn_to_start"] = conn_to_start
                    edata["conn_to_end"] = conn_to_end
                    connected = bool(conn_to_start and conn_to_end)          # last edge wins (quirk Q6)
                    c_size = float(np.tanh(0.25 - np.cbrt(size)))
                    cost = dist * (1 + self.w_size * c_size) + self.w_bias
                    if not fits:
                        cost += self.c_fit
                    inter_graph.add_edge(self.id_inter, eid, weight=cost)
        return connected

    # ---- :586-743 (with_rot=False) ---------------------------------------------
    def compute_via_points(self, path, start, end, graph, inter_graph):
        x0 = np.empty(0)
        sets_inter = []
        for edge in path[1:-1]:
            sets_inter.append(inter_graph.nodes[edge]["cset"])
            x0 = np.concatenate((x0, inter_graph.nodes[edge]["p_proj"], [0.5]))
            idx = np.linalg.norm(sets_inter[-1][0], axis=1) > 1e-4
            sets_inter[-1][1][idx] -= 0.001                    # in-place, every call (quirk Q7)
        sets, seq = [], []
        last_id = None
        for i in range(len(path)):
            node = inter_graph.nodes[path[i]]
            if i == 0:
                last_id = node["id0"]
            else:
                id0, id1 = node["id0"], node["id1"]
                if id0 != last_id:
                    last_id = id0
                elif id1 != last_id:
                    last_id = id1
            sets.append(graph.nodes[last_id]["cset"])
            seq.append(last_id)
        sets_via, seq_via = [], []
        p_via = [start]
        for i in range(len(sets_inter)):
            p_via_opt = x0[4 * i: 4 * i + 3]
            if np.linalg.norm(p_via_opt - p_via[-1]) > 1e-4:
                p_via.append(p_via_opt)
                sets_via.append(sets[i])
                seq_via.append(seq[i])
        p_via.append(end)
        sets_via.append(sets[-1])
        seq_via.append(seq[-1])
        return np.array(p_via), p_via, sets_via, seq_via

    # ---- :174-534 -------------------------------------------------------------
    def replanning_horizon_index(self, start, p_horizon, new_obs=False):
        """:231-266: how far along the MPC horizon the previous plan's sets still hold.  Walks ``sets_via_prev`` in
        order; a set that contains ``start`` extends the index to the last horizon point before the first one
        outside it (the whole horizon: stop); ``new_obs`` resets it to 1.  Every A x - b is the element-wise form of
        _rows_minus_b, as in the native driver: the thresholds are decided on the same bits (the reference's `@`
        differs from it in the last bits only)."""
        p_horizon = np.asarray(p_horizon, float).reshape(-1, 3)
        start = np.asarray(start, float)
        max_horizon_idx = 1
        for s in self.sets_via_prev:
            a_set, b_set = np.asarray(s[0], float), np.asarray(s[1], float)
            dist_start = _rows_minus_b(a_set, b_set, start)
            dist_horizon = _rows_minus_b(a_set[None], b_set[None], p_horizon.T[:, :, None])      # [H, m]
            start_in = np.max(dist_start) < 1e-8
            horizon_idx = np.where(np.logical_not(np.max(dist_horizon, axis=1) < 1e-8))[0]
            if horizon_idx.shape[0] > 0:
                if horizon_idx[0] != 0 and start_in:
                    max_horizon_idx = int(np.max((max_horizon_idx, horizon_idx[0] - 1)))
            elif start_in:
                max_horizon_idx = len(p_horizon) - 1
                break
        if new_obs:
            max_horizon_idx = 1
        return max_horizon_idx

    def plan_gen(self, start, end, r0, r1, first_sample=None, replanning=False, p_horizon=(), new_obs=False):
        """Generator form of the planner loop (see the module docstring for the request protocol)."""
        start = np.array(start, float)
        end = np.array(end, float)
        sampled_first = False
        if self.polytopes:                                        # :199-204
            self._push_out_general(end)
        else:
            self._push_out_boxes(end)
        self.omega = R.from_matrix(r1 @ r0.T).as_rotvec()        # :207-219
        self.omega_norm = np.linalg.norm(self.omega)
        self.omega_normed = self.omega / self.omega_norm if self.omega_norm > 1e-6 else np.array([0, 0, 1.0])
        self.l_ee = r0 @ np.array([-self.length_ee, 0, 0])
        self.l_ee_end = r1 @ np.array([-self.length_ee, 0, 0])
        graph, inter_graph = nx.Graph(), nx.Graph()
        self.nr_sets = self.nr_edges = self.nr_inter_set = 0
        self._nodes_reset()
        self._inter_by_node = {}

        self.replanning = bool(replanning)
        if replanning:                                            # :231-276
            self.p_horizon = np.asarray(p_horizon, float).reshape(-1, 3)
            self.p_horizon_max = self.p_horizon[self.replanning_horizon_index(start, self.p_horizon, new_obs)]
            a_set, b_set, q_start, p_mid_start, collision, a_red, b_red = yield ("set_line", start, self.p_horizon_max)
        else:
            a_set, b_set, q_start, p_mid_start, a_red, b_red = yield ("set_point", start, True, True)     # :278-283
            collision = False
            if np.max(a_set @ (start + self.l_ee) - b_set) > 1e-8:
                a_set, b_set, q_start, p_mid_start, collision, a_red, b_red = yield ("set_line", start, start + self.l_ee)
        if collision:                                             # :296-324
            if new_obs:
                # the reference pushes `start` out of every inflated obstacle that contains it -- through
                # `ob.A()[idx, :]` on a list (:311), i.e. it raises AttributeError as soon as one does (quirk Q12);
                # without such an obstacle the loop does nothing and the start set is built around `start`
                if self.polytopes and not (_rows_minus_b(self._obs_A, self._obs_b, start) > 0).any(axis=1).all():
                    raise AttributeError("'list' object has no attribute 'A'")
                for k in range(0 if self.polytopes else len(self.obs_sets)):
                    if not np.any(np.concatenate((start, -start)) - self._b6[k] > 0):
                        raise AttributeError("'list' object has no attribute 'A'")
                a_set, b_set, q_start, p_mid_start, a_red, b_red = yield ("set_point", start, True, True)
            else:
                # "Could not find start set, reusing old end set": IndexError on a first plan, like the reference
                prev = self.sets_via_prev[-1]
                a_prev, b_prev = np.array(prev[0], float), np.array(prev[1], float)
                a_red, b_red = yield ("reduce", a_prev, b_prev)
                p_mid_start = start
                q_start = np.eye(3)
        a_set, b_set = a_red, b_red                               # reduce_ineqs (:327)
        set_start = [a_set, b_set]
        self.id_inter = 0
        self.id_graph = 0
        graph.add_node(0, cset=set_start, size=1 / float(_det(q_start)), q_ellipse=q_start, p_mid=p_mid_start,
                       a_set=np.array(a_set), b_set=np.array(b_set))
        self._nodes_add(a_set, b_set, q_start, p_mid_start)
        inter_graph.add_node(0, cset=set_start, id0=0, id1=0, conn_to_start=True, conn_to_end=False, p_proj=start,
                             p_via=np.concatenate((start, [0.0])), fits=True)
        self._inter_by_node.setdefault(0, []).append(0)
        self.nr_sets += 1
        connected = yield from self._add_edges(0, graph, inter_graph, end, start)
        if np.max(a_set @ end - b_set) < 1e-8 and np.max(a_set @ (end + self.l_ee_end) - b_set) < 1e-8:   # :361-375
            from .utils import normalize_set_size

            self.sets_via_prev = normalize_set_size([[set_start[0], set_start[1]]], 15).copy()                          # :371-372
            return dict(path=[0], set_ids=[0], sets_via=[set_start], p_via=np.array([start, end]), graph=graph,
                        inter_graph=inter_graph)
        _, _, q_end, p_mid_end, collision, a_set, b_set = yield ("set_line", end, end + self.l_ee_end)  # :381-390
        set_end = [a_set, b_set]
        self.id_graph += 1
        self.id_inter += 1
        graph.add_node(1, cset=set_end, size=1 / float(_det(q_end)), q_ellipse=q_end, p_mid=p_mid_end,
                       a_set=np.array(a_set), b_set=np.array(b_set))
        self._nodes_add(a_set, b_set, q_end, p_mid_end)
        inter_graph.add_node(1, cset=set_end, id0=1, id1=1, conn_to_start=False, conn_to_end=True, p_proj=end,
                             p_via=np.concatenate((end, [1.0])), fits=True)
        self._inter_by_node.setdefault(1, []).append(1)
        self.nr_sets += 1
        conn = yield from self._add_edges(1, graph, inter_graph, end, start)
        connected = conn or connected

        j = 0
        nr_samples = 0
        p_via_old = None
        path = None
        while True:                                               # :430-534
            pre_answers = None
            if connected:
                if self.device_loop:
                    path = yield ("shortest_path", inter_graph)
                else:
                    path = nx.shortest_path(inter_graph, 0, 1, weight="weight")
                p_via, p_via_list, sets_via, seq_via = self.compute_via_points(path, start, end, graph, inter_graph)
                if p_via_old is not None and p_via_old.shape == p_via.shape and \
                        np.linalg.norm(p_via_old - p_via) < 1e-4:
                    break                                         # "Found path solution"
                samples = p_via_list[1:-1]
                p_via_old = np.copy(p_via)
            elif not sampled_first and first_sample is not None:
                samples = [first_sample]
            elif self.device_loop:
                sample, pre = yield from self._sample_set_on_device(not (nr_samples + 1 >= self.nr_optimized))
                samples, pre_answers = [sample], [pre]
                nr_samples += 1
                if nr_samples > self.max_iters:
                    raise RuntimeError("(PosPath) Exceeded max iterations")
            else:
                in_collision = in_safe = True
                nr_sampled = 0
                while (in_collision or in_safe) and nr_sampled <= self.max_samples:
                    in_collision = in_safe = False
                    sample = self.rng.uniform(self.workspace_min, self.workspace_max, 3)
                    nr_sampled += 1
                    in_collision = self._in_collision(sample)        # any obstacle with max(A x - b) < 1e-3
                    in_safe = self._in_safe(sample)                  # any known set with max(A x - b) < 1e-3
                if nr_sampled >= self.max_samples:
                    raise RuntimeError("(PosPath) Could not find collision-free sample")
                samples = [sample]
                nr_samples += 1
                if nr_samples > self.max_iters:
                    raise RuntimeError("(PosPath) Exceeded max iterations")
            for si, sample in enumerate(samples):
                j += 1
                optimize = not (nr_samples >= self.nr_optimized)
                # fixed_mid = (via_sample or (not sampled_first),) is a 1-tuple: always truthy (quirk Q3)
                if pre_answers is not None:
                    ans = pre_answers[si]                  # built in the sampling round
                    if isinstance(ans, Exception):
                        raise ans
                elif self.device_loop:
                    ans = yield ("set_point", np.asarray(sample, float), True, optimize, self)
                else:
                    ans = yield ("set_point", np.asarray(sample, float), True, optimize)
                _, _, q_ellipse, p_mid, a_set, b_set = ans[:6]
                sampled_first = True
                dvertex = ans[6] if len(ans) > 6 else self._min_node_distance(q_ellipse, p_mid)
                if dvertex > 0.01:
                    self.id_graph += 1
                    graph.add_node(self.id_graph, cset=[a_set, b_set], size=1 / float(_det(q_ellipse)),
                                   q_ellipse=q_ellipse, p_mid=p_mid, a_set=np.array(a_set), b_set=np.array(b_set))
                    self._nodes_add(a_set, b_set, q_ellipse, p_mid)
                    self.nr_sets += 1
                    conn = yield from self._add_edges(self.id_graph, graph, inter_graph, end, start)
                    connected = conn or connected
        self.graph, self.inter_graph = graph, inter_graph
        self.sets_via_prev = list(sets_via)                                                          # :556
        return dict(path=path, set_ids=seq_via, sets_via=sets_via, p_via=p_via, graph=graph, inter_graph=inter_graph)

    def plan_set_sequence(self, start, end, r0, r1, first_sample=None, replanning=False, p_horizon=(), new_obs=False):
        """Sequential driver: every request is answered at once by ``self.backend.execute``.
        Returns dict(path, set_ids, sets_via, p_via, graph, inter_graph).  replanning / p_horizon / new_obs as in
        plan_convex_set_path (:180-183): the start set then comes from the segment start .. horizon point that the
        previous plan's sets (``sets_via_prev``) still cover."""
        if self.backend is None:
            if self.polytopes:
                self.backend = GpuBackend(None, self.obs_size_increase, self.workspace_max, self.workspace_min,
                                          obs_sets=self.obs_sets, obs_points_sets=self.obs_points_sets)
            else:
                self.backend = GpuBackend(self._obstacles, self.obs_size_increase, self.workspace_max,
                                          self.workspace_min)
        gen = self.plan_gen(start, end, r0, r1, first_sample, replanning, p_horizon, new_obs)
        try:
            req = next(gen)
            while True:
                try:
                    res = self.backend.execute(req)
                except (RuntimeError, ValueError) as e:
                    req = gen.throw(e)
                    continue
                req = gen.send(res)
        except StopIteration as stop:
            return stop.value


# ---------------------------------------------------------------------------------------------
# Batched driver (BASELINE config C3): many independent queries, one scene each (or shared scenes), in lock step
# ---------------------------------------------------------------------------------------------
class BatchedGpuExecutor:
    """Answers the pending requests of many queries with one batched kernel call per primitive.

    Every query's known sets (rows of its graph nodes) and node ellipsoids live in fixed-size blocks of device
    tables, extended when a request shows that the query's planner has added nodes: the sampling rejection test
    (K11), the duplicate-set distance (K12) and the shortest path (K13) then run on the device in the same round as
    the set build they belong to (``device_loop``)."""

    device_loop = True
    MAX_NODES = 64           # graph nodes per query the tables hold (2 + 20 samples + via-point re-samples)
    NODE_ROWS = 24           # rows per reduced node set (the reference's sets have at most 20)

    def __init__(self, obstacles_list, obs_size_increase, workspace_max, workspace_min, polytope_scenes=None,
                 query_scene=None):
        """obstacles_list: one [N_k,6] box array per query; or polytope_scenes: one (obs_sets, obs_points_sets |
        None) pair per query (inflated polytopes, PolytopeSceneBatch), obstacles_list then unused.  query_scene [Q]:
        the queries share the scenes, query q plans in scene query_scene[q] (the lists then hold one entry per
        scene)."""
        from . import geometry as geo

        self.geo = geo
        if polytope_scenes is not None:
            self.scene = geo.PolytopeSceneBatch(polytope_scenes)
            self._n_queries = len(polytope_scenes)
        else:
            self.scene = geo.SceneBatch(obstacles_list, obs_size_increase)
            self._n_queries = len(obstacles_list)
        self._scene_of = None
        if query_scene is not None:
            self._scene_of = np.asarray(query_scene, np.int32).reshape(-1)
            self._n_queries = self._scene_of.shape[0]
        self.ws_min = np.asarray(workspace_min, float)
        self.ws_max = np.asarray(workspace_max, float)
        self.calls = 0
        self._tab = None

    # -- device tables of the queries' graph nodes -------------------------------------
    def _tables(self):
        import torch

        if self._tab is None:
            n = self._n_queries * self.MAX_NODES
            self._tab = dict(
                A=torch.zeros((n, self.NODE_ROWS, 3), dtype=torch.float64, device="cuda"),
                b=torch.full((n, self.NODE_ROWS), 10.0, dtype=torch.float64, device="cuda"),
                m=torch.zeros((n,), dtype=torch.int32, device="cuda"),
                q=torch.zeros((n, 9), dtype=torch.float64, device="cuda"),
                p=torch.zeros((n, 3), dtype=torch.float64, device="cuda"),
                count=torch.zeros((self._n_queries,), dtype=torch.int32, device="cuda"),
                begin=(torch.arange(self._n_queries, dtype=torch.int32, device="cuda") * self.MAX_NODES),
                count_host=np.zeros(self._n_queries, np.int64), owner=[None] * self._n_queries)
        return self._tab

    def _sync_tables(self, items):
        """items: [(qid, planner)].  Upload the nodes the planners have added since the last round (one H2D copy per
        table for the whole round).  Returns {qid: ValueError} for queries the tables cannot hold."""
        import torch

        tab = self._tables()
        slots, rows_a, rows_b, ms, qs, ps, bad = [], [], [], [], [], [], {}
        for q, pl in items:
            key = (pl, getattr(pl, "_plan_epoch", 0))
            if tab["owner"][q] is None or tab["owner"][q][0] is not pl or tab["owner"][q][1] != key[1]:
                tab["owner"][q] = key                     # a new planner (or a new plan of the same one) on this slot:
                tab["count_host"][q] = 0                  # its table starts empty
            have, n = int(tab["count_host"][q]), len(pl._row_start)
            if n > self.MAX_NODES:
                bad[q] = ValueError(f"more than {self.MAX_NODES} graph nodes in one query")
                continue
            starts = pl._row_start + [pl._rows_a.shape[0]]
            for k in range(have, n):
                r0, r1 = starts[k], starts[k + 1]
                if r1 - r0 > self.NODE_ROWS:
                    bad[q] = ValueError(f"graph node with more than {self.NODE_ROWS} rows")
                    break
                a = np.zeros((self.NODE_ROWS, 3))
                bb = np.full(self.NODE_ROWS, 10.0)
                a[: r1 - r0], bb[: r1 - r0] = pl._rows_a[r0:r1], pl._rows_b[r0:r1]
                slots.append(q * self.MAX_NODES + k)
                rows_a.append(a); rows_b.append(bb); ms.append(r1 - r0)
                qs.append(pl._node_q[k]); ps.append(pl._node_p[k])
            if q not in bad:
                tab["count_host"][q] = n
        if slots:
            idx = torch.as_tensor(np.asarray(slots, np.int64)).cuda()
            tab["A"].index_copy_(0, idx, torch.as_tensor(np.asarray(rows_a)).cuda())
            tab["b"].index_copy_(0, idx, torch.as_tensor(np.asarray(rows_b)).cuda())
            tab["m"].index_copy_(0, idx, torch.as_tensor(np.asarray(ms, np.int32)).cuda())
            tab["q"].index_copy_(0, idx, torch.as_tensor(np.asarray(qs)).cuda())
            tab["p"].index_copy_(0, idx, torch.as_tensor(np.asarray(ps)).cuda())
            tab["count"].copy_(torch.as_tensor(tab["count_host"].astype(np.int32)))
        return bad

    def _dvertex(self, batch, qi):
        """K12 against the queries' node tables: min ||Q - Q_v||_F + ||p - p_v|| (inf without nodes)."""
        tab = self._tables()
        return self.geo.dedupe_distance_tables(batch.q_ellipse, batch.p_mid, tab["q"], tab["p"],
                                               tab["begin"][qi], tab["count"][qi])[0]

    # -- helpers ----------------------------------------------------------------
    def _item_scene(self, qids):
        """The scene index of every query of qids (the query itself without a query -> scene map)."""
        qids = np.asarray(qids, np.int32)
        return qids if self._scene_of is None else self._scene_of[qids]

    def _reduced(self, batch):
        import torch

        Ar, br, mr, _, _ = self.geo.reduce_ineqs(batch.A, batch.b, batch.m)
        host = [t.cpu().numpy() for t in (batch.A, batch.b, batch.m, batch.q_ellipse, batch.p_mid, batch.status, Ar, br, mr)]
        torch.cuda.current_stream().synchronize()
        return host

    def _pack(self, sets):
        import torch

        m_max = max(max(s[0].shape[0] for s in sets), 1)
        A = np.zeros((len(sets), m_max, 3))
        b = np.full((len(sets), m_max), 10.0)
        m = np.zeros(len(sets), np.int32)
        for k, s in enumerate(sets):
            n = s[0].shape[0]
            A[k, :n], b[k, :n], m[k] = s[0], s[1], n
        return torch.as_tensor(A).cuda(), torch.as_tensor(b).cuda(), torch.as_tensor(m).cuda()

    @staticmethod
    def _row_limit_error(req):
        from ._lib import BP_MAX_ROWS

        kind = req[0]
        worst = 0
        if kind in ("edges", "intersect_many"):
            worst = max((s[0].shape[0] + req[2][0].shape[0] for s in req[1]), default=0)
        elif kind == "fit_many":
            worst = max((a.shape[0] for a, _, _ in req[1]), default=0)
        elif kind in ("project", "reduce"):
            worst = np.asarray(req[1]).shape[0]
        if worst > BP_MAX_ROWS:
            return ValueError(f"'{kind}' request with {worst} rows exceeds the kernels' {BP_MAX_ROWS}-row sets")
        return None

    # -- one round ----------------------------------------------------------------
    def execute(self, pending):
        """pending: {qid: request}.  Returns {qid: result | Exception}."""
        geo = self.geo
        out = {}
        by_kind = {}
        for qid, req in pending.items():
            # a request whose sets exceed the kernels' row capacity fails for ITS query only (the other queries of
            # the lock-step batch go on): pair / fit kernels take m_i + m_j <= BP_MAX_ROWS rows, the projection
            # one packed set of <= BP_MAX_ROWS rows
            err = self._row_limit_error(req)
            if err is not None:
                out[qid] = err
                continue
            by_kind.setdefault(req[0], []).append(qid)

        for (fixed_mid, optimize) in ((True, True), (True, False), (False, True), (False, False)):
            qids = [q for q in by_kind.get("set_point", []) if (pending[q][2], pending[q][3]) == (fixed_mid, optimize)]
            if not qids:
                continue
            self.calls += 1
            with_dv = [q for q in qids if len(pending[q]) > 4]          # requests that carry their planner
            bad = self._sync_tables([(q, pending[q][4]) for q in with_dv]) if with_dv else {}
            seeds = np.array([pending[q][1] for q in qids])
            batch = geo.build_sets_point(self.scene, seeds, self.ws_min, self.ws_max, fixed_mid=fixed_mid,
                                         optimize=optimize, row_cap=REFERENCE_MAX_ROWS,
                                         item_scene=self._item_scene(qids))
            dv = None
            if with_dv:
                import torch

                dv = self._dvertex(batch, torch.as_tensor(np.asarray(qids, np.int64)).cuda()).cpu().numpy()
            peak = batch.rows_peak.cpu().numpy()
            A, b, m, Q, P, st, Ar, br, mr = self._reduced(batch)
            for k, q in enumerate(qids):
                err = bad.get(q) or _set_errors(int(st[k]), int(peak[k]) if optimize else None)
                if err is not None:
                    out[q] = err
                    continue
                out[q] = (A[k, : m[k]].copy(), b[k, : m[k]].copy(), Q[k].copy(), P[k].copy(),
                          Ar[k, : mr[k]].copy(), br[k, : mr[k]].copy())
                if len(pending[q]) > 4:
                    out[q] = out[q] + (float(dv[k]),)

        # -- sampling round on the device: K11 (first accepted candidate) -> K5 at it -> K8 -> K12
        for optimize in (True, False):
            qids = [q for q in by_kind.get("sample_set", []) if bool(pending[q][2]) == optimize]
            if not qids:
                continue
            import torch

            self.calls += 1
            bad = self._sync_tables([(q, pending[q][3]) for q in qids])
            tab = self._tables()
            counts = [np.asarray(pending[q][1]).reshape(-1, 3).shape[0] for q in qids]
            C = max(counts)
            cand = np.empty((len(qids), C, 3))
            for k, q in enumerate(qids):
                c = np.asarray(pending[q][1], float).reshape(-1, 3)
                cand[k, : counts[k]] = c
                cand[k, counts[k]:] = c[0]               # padding: copies of the first candidate never win
            cand_d = torch.as_tensor(cand).cuda()
            qi = torch.as_tensor(np.asarray(qids, np.int64)).cuda()
            si = qi.to(torch.int32) if self._scene_of is None else torch.as_tensor(self._item_scene(qids)).cuda()
            first_d = geo.sample_filter_tables(self.scene, cand_d, tab["A"], tab["b"], tab["m"], tab["begin"][qi],
                                               tab["count"][qi], item_scene=si)
            pick = first_d.clamp(min=0).to(torch.int64)
            seeds_d = cand_d[torch.arange(len(qids), device="cuda"), pick]
            batch = geo.build_sets_point(self.scene, seeds_d, self.ws_min, self.ws_max, fixed_mid=True,
                                         optimize=optimize, row_cap=REFERENCE_MAX_ROWS, item_scene=si)
            dv = self._dvertex(batch, qi).cpu().numpy()
            first = first_d.cpu().numpy()
            peak = batch.rows_peak.cpu().numpy()
            A, b, m, Q, P, st, Ar, br, mr = self._reduced(batch)
            for k, q in enumerate(qids):
                if q in bad:
                    out[q] = bad[q]
                    continue
                f = int(first[k])
                if f < 0 or f >= counts[k]:
                    out[q] = (-1, None)
                    continue
                err = _set_errors(int(st[k]), int(peak[k]) if optimize else None)
                out[q] = (f, err if err is not None else
                          (A[k, : m[k]].copy(), b[k, : m[k]].copy(), Q[k].copy(), P[k].copy(),
                           Ar[k, : mr[k]].copy(), br[k, : mr[k]].copy(), float(dv[k])))

        # -- shortest paths through the intersection graphs (K13, one warp per graph)
        qids = by_kind.get("shortest_path", [])
        if qids:
            self.calls += 1
            node_off, edge_off, edge_dst, edge_w = [0], [], [], []
            for q in qids:
                g = pending[q][1]
                n = g.number_of_nodes()                 # intersection ids are 0 .. n-1 in insertion order
                adj = g._adj
                for v in range(n):
                    edge_off.append(len(edge_dst))
                    for u, d in adj[v].items():
                        edge_dst.append(u)
                        edge_w.append(d["weight"])
                node_off.append(node_off[-1] + n)
            edge_off.append(len(edge_dst))
            G = len(qids)
            path, plen, _ = geo.shortest_paths(np.asarray(node_off, np.int32), np.asarray(edge_off, np.int32),
                                               np.asarray(edge_dst, np.int32), np.asarray(edge_w, float),
                                               np.zeros(G, np.int32), np.ones(G, np.int32), max_len=64)
            path, plen = path.cpu().numpy(), plen.cpu().numpy()
            for k, q in enumerate(qids):
                if plen[k] <= 0:
                    out[q] = nx.NetworkXNoPath("No path between 0 and 1.")
                else:
                    out[q] = [int(v) for v in path[k, : plen[k]]]

        qids = by_kind.get("set_line", [])
        if qids:
            self.calls += 1
            p0 = np.array([pending[q][1] for q in qids])
            p1 = np.array([pending[q][2] for q in qids])
            batch = geo.build_sets_line(self.scene, p0, p1, self.ws_min, self.ws_max, compute_ellipsoid=True,
                                        item_scene=self._item_scene(qids))
            coll = batch.collision.cpu().numpy()
            A, b, m, Q, P, st, Ar, br, mr = self._reduced(batch)
            for k, q in enumerate(qids):
                err = _set_errors(int(st[k]), int(m[k]))
                out[q] = err if err is not None else (A[k, : m[k]].copy(), b[k, : m[k]].copy(), Q[k].copy(), P[k].copy(),
                                                      bool(coll[k]), Ar[k, : mr[k]].copy(), br[k, : mr[k]].copy())

        qids = by_kind.get("edges", [])
        if qids:
            groups = {}
            for q in qids:
                l_ee, om, on = pending[q][4]
                groups.setdefault((tuple(np.round(l_ee, 15)), tuple(np.round(om, 15)), round(float(on), 15),
                                   float(pending[q][3])), []).append(q)
            for gq in groups.values():
                self.calls += 1
                l_ee, om, on = pending[gq[0]][4]
                tol = pending[gq[0]][3]
                sets, pairs, spans = [], [], []
                for q in gq:
                    _, others, set_new, _, _ = pending[q]
                    base = len(sets)
                    sets.append(set_new)
                    sets.extend(others)
                    pairs.extend((base + 1 + k, base) for k in range(len(others)))  # rows of the old set first
                    spans.append(len(others))
                A, b, m = self._pack(sets)
                pairs = np.asarray(pairs, np.int32)
                ok, x = geo.pairs_feasible_list(A, b, m, pairs, tol)
                fits, omega = geo.check_fit(A, b, m, pairs, l_ee, om, on, x0=x, active=ok)   # x, ok stay on the device
                ok, x, fits, omega = ok.cpu().numpy(), x.cpu().numpy(), fits.cpu().numpy(), omega.cpu().numpy()
                o = 0
                for q, n in zip(gq, spans):
                    out[q] = [(x[o + k].copy() if ok[o + k] else None, bool(ok[o + k]), bool(fits[o + k]),
                               np.concatenate((x[o + k], [omega[o + k] if fits[o + k] else 0.0]))) for k in range(n)]
                    o += n

        qids = by_kind.get("intersect_many", [])
        if qids:
            self.calls += 1
            sets, pairs, spans = [], [], []
            tol = pending[qids[0]][3]
            for q in qids:
                _, others, set_new, _ = pending[q]
                base = len(sets)
                sets.append(set_new)
                sets.extend(others)
                pairs.extend((base + 1 + k, base) for k in range(len(others)))      # rows of the old set first
                spans.append(len(others))
            A, b, m = self._pack(sets)
            ok, x = geo.pairs_feasible_list(A, b, m, np.asarray(pairs, np.int32), tol)
            ok, x = ok.cpu().numpy(), x.cpu().numpy()
            o = 0
            for q, n in zip(qids, spans):
                out[q] = [(x[o + k].copy() if ok[o + k] else None, bool(ok[o + k])) for k in range(n)]
                o += n

        qids = by_kind.get("fit_many", [])
        if qids:
            groups = {}
            for q in qids:
                l_ee, om, on = pending[q][2]
                groups.setdefault((tuple(np.round(l_ee, 15)), tuple(np.round(om, 15)), round(float(on), 15)), []).append(q)
            for gq in groups.values():
                self.calls += 1
                l_ee, om, on = pending[gq[0]][2]
                sets, x0, spans = [], [], []
                for q in gq:
                    items = pending[q][1]
                    sets.extend([[a, b_] for a, b_, _ in items])
                    x0.extend(s for _, _, s in items)
                    spans.append(len(items))
                A, b, m = self._pack(sets)
                idx = np.arange(len(sets), dtype=np.int32)
                fits, omega = geo.check_fit(A, b, m, np.stack((idx, idx), axis=1), l_ee, om, on, x0=np.array(x0))
                fits, omega = fits.cpu().numpy(), omega.cpu().numpy()
                o = 0
                for q, n in zip(gq, spans):
                    items = pending[q][1]
                    out[q] = [(bool(fits[o + k]), np.concatenate((items[k][2], [omega[o + k] if fits[o + k] else 0.0])))
                              for k in range(n)]
                    o += n

        qids = by_kind.get("reduce", [])                   # reduce_ineqs of a given set (start-set fallback, :321-327)
        if qids:
            self.calls += 1
            A, b, m = self._pack([[pending[q][1], pending[q][2]] for q in qids])
            Ar, br, mr, _, _ = geo.reduce_ineqs(A, b, m)
            Ar, br, mr = Ar.cpu().numpy(), br.cpu().numpy(), mr.cpu().numpy()
            for k, q in enumerate(qids):
                out[q] = (Ar[k, : mr[k]].copy(), br[k, : mr[k]].copy())

        qids = by_kind.get("project", [])
        if qids:
            self.calls += 1
            A, b, m = self._pack([[pending[q][1], pending[q][2]] for q in qids])
            idx = np.arange(len(qids), dtype=np.int32)
            x, _ = geo.project_points(A, b, m, np.stack((idx, idx), axis=1), np.array([pending[q][3] for q in qids]))
            x = x.cpu().numpy()
            for k, q in enumerate(qids):
                out[q] = x[k].copy()
        return out


# the exits of plan_convex_set_path a query of a batch records (IndexError / AttributeError: the start-in-collision
# fallbacks of :296-324)
_QUERY_ERRORS = (RuntimeError, ValueError, IndexError, AttributeError)


def _planned(res, pl):
    """A planned query's result: the planner's dict plus what the next (re)planning call needs."""
    res["sets_via_prev"] = pl.sets_via_prev
    if pl.replanning:
        res["p_horizon_max"] = pl.p_horizon_max
    return res


def plan_batch(queries, obs_size_increase=0.01, workspace_max=(1.0, 1.0, 1.2), workspace_min=(-1.0, -1.0, 0.0),
               rng_seeds=None, executor=None, scenes=None):
    """Plan many independent queries in lock step.

    queries: list of dicts(obstacles [N,6], start, end, r0, r1[, first_sample]); or, for polytope obstacles,
    obs_sets (inflated [A (<= 15 x 3), b] per obstacle) [and obs_points_sets] instead of obstacles.  One kind per
    batch: a batch that mixes them raises ValueError.
    Replanning (an MPC loop calling the planner again, :231-276): a query may also carry ``replanning``,
    ``p_horizon`` [H,3], ``new_obs`` and ``sets_via_prev`` (the previous call's sets, [A, b] each; also used by the
    start-in-collision fallback of a first plan, :296-324).  A batch may mix replanning and first-plan queries.
    Returns (results, stats): results[i] is the planner's dict or the exception the sequential planner
    would have raised for that query.  A planned query's dict also holds ``sets_via_prev`` (what the planner keeps
    for its next call) and, when it replanned, ``p_horizon_max``.
    scenes: queries over shared scenes (planner_native.scene_map): a list of dicts with the obstacle keys above, each
    query carrying ``scene`` (its index) instead; every scene is stored on the device, and its host obstacle sets
    built, once."""
    from .planner_native import query_kind, scene_map

    query_scene = scene_map(queries, scenes)
    holders = queries if scenes is None else scenes
    polytopes = query_kind(holders, "query" if scenes is None else "scene") == "polytopes"
    if executor is None:
        if polytopes:
            executor = BatchedGpuExecutor(None, obs_size_increase, workspace_max, workspace_min,
                                          polytope_scenes=[(h["obs_sets"], h.get("obs_points_sets")) for h in holders],
                                          query_scene=query_scene)
        else:
            executor = BatchedGpuExecutor([h["obstacles"] for h in holders], obs_size_increase, workspace_max,
                                          workspace_min, query_scene=query_scene)
    # the obstacles of query i (its own, or its scene's) and, over shared scenes, the host obstacle sets of every
    # box scene, built once
    obs_of = (lambda i: queries[i]) if scenes is None else (lambda i: scenes[query_scene[i]])
    scene_sets = None
    if scenes is not None and not polytopes:
        scene_sets = [obstacle_sets(h["obstacles"], obs_size_increase) for h in scenes]
    import time

    t_start = time.perf_counter()
    planners, gens, pending, results = [], {}, {}, [None] * len(queries)
    finish = [0.0] * len(queries)              # seconds after the start of the batch at which query i was answered
    for i, q in enumerate(queries):
        ob = obs_of(i)
        pl = SetSequencePlanner(() if polytopes else ob["obstacles"], obs_size_increase, workspace_max, workspace_min,
                                rng=np.random.default_rng(rng_seeds[i] if rng_seeds is not None else None),
                                device_loop=bool(getattr(executor, "device_loop", False)),
                                obs_sets=ob["obs_sets"] if polytopes else
                                (scene_sets[query_scene[i]] if scene_sets is not None else None),
                                obs_points_sets=ob.get("obs_points_sets") if polytopes else None)
        pl.sets_via_prev = [[np.array(a, float), np.array(b, float)] for a, b in q.get("sets_via_prev", ())]
        planners.append(pl)
        gens[i] = pl.plan_gen(q["start"], q["end"], q["r0"], q["r1"], q.get("first_sample"),
                              bool(q.get("replanning", False)), q.get("p_horizon", ()), bool(q.get("new_obs", False)))
        try:
            pending[i] = next(gens[i])
        except StopIteration as stop:
            results[i] = _planned(stop.value, pl)
            finish[i] = time.perf_counter() - t_start
        except _QUERY_ERRORS as e:
            results[i] = e
            finish[i] = time.perf_counter() - t_start
    rounds = 0
    while pending:
        rounds += 1
        answers = executor.execute(pending)
        nxt = {}
        for i, ans in answers.items():
            try:
                nxt[i] = gens[i].throw(ans) if isinstance(ans, Exception) else gens[i].send(ans)
            except StopIteration as stop:
                results[i] = _planned(stop.value, planners[i])
                finish[i] = time.perf_counter() - t_start
            except _QUERY_ERRORS as e:
                results[i] = e
                finish[i] = time.perf_counter() - t_start
        pending = nxt
    return results, {"rounds": rounds, "kernel_batches": executor.calls, "finish_s": finish}
