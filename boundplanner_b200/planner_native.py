"""Native lock-step planner driver: ``plan_batch`` with the per-query loop in C++ (csrc/bp_planner.h) instead of
Python generators, and every round's requests answered by one batched kernel chain inside libbpgeo.so
(``bp_plan_batch``; BASELINE config C3).

Same loop, same results as ``planner.plan_batch`` -- BoundPlanner.plan_convex_set_path (:174-584) up to the planned
set sequence, add_edges (:789-896), compute_via_points (:586-743, no rotations) -- but no Python between the
rounds: the queries' graphs, generators (numpy's PCG64 stream, restated) and bookkeeping live on the host in C++,
their graph nodes in device tables.  What Python still does is the per-query set-up that involves rotations
(scipy's ``as_rotvec`` and the 20 Rodrigues samples of check_intersection, :745-772) and the result objects.
"""
from __future__ import annotations

import ctypes

import numpy as np

MAX_NODES, NODE_ROWS, SET_ROWS, MAX_PATH, FIT_SAMPLES = 64, 24, 48, 64, 20
OBS_ROWS = 15               # rows of a polytope obstacle (normalize_set_size)
MAX_POLY_OBSTACLES = 16384  # polytope obstacles per scene (the kernels of a planning round)
MAX_PREV_SETS = 64          # previous sets per query (sets_via_prev)
LENGTH_EE = 0.05            # BoundPlanner.__init__ (:54)

_dp = ctypes.POINTER(ctypes.c_double)
_ip = ctypes.POINTER(ctypes.c_int)
_up = ctypes.POINTER(ctypes.c_ulonglong)


class BpPlanIn(ctypes.Structure):
    _fields_ = [("Q", ctypes.c_int), ("boxes", _dp), ("box_off", _ip), ("inflate", ctypes.c_double), ("ws_min", _dp),
                ("ws_max", _dp), ("starts", _dp), ("ends", _dp), ("l_ee", _dp), ("l_ee_end", _dp), ("ee_samples", _dp),
                ("rng", _up), ("has_first", _ip), ("first_sample", _dp), ("sample_chunk", ctypes.c_int),
                ("max_rounds", ctypes.c_int), ("obs_rows", _dp), ("replanning", _ip), ("new_obs", _ip),
                ("horizon_off", _ip), ("p_horizon", _dp), ("prev_off", _ip), ("prev_row_off", _ip), ("prev_rows", _dp)]


class BpPlanOut(ctypes.Structure):
    _fields_ = [("err_kind", _ip), ("err_msg", ctypes.c_char_p), ("path", _ip), ("path_len", _ip), ("set_ids", _ip),
                ("n_ids", _ip), ("p_via", _dp), ("n_via", _ip), ("rng_out", _up), ("n_nodes", _ip), ("n_inter", _ip),
                ("n_edges", _ip), ("finish_round", _ip), ("finish_ms", _dp), ("node_A", _dp), ("node_b", _dp), ("node_m", _ip),
                ("stats", ctypes.POINTER(ctypes.c_longlong)), ("p_horizon_max", _dp)]

_ERRORS = {1: RuntimeError, 2: ValueError, 3: IndexError, 4: AttributeError}


def _ptr(a, t):
    return a.ctypes.data_as(t) if a is not None else None


def replan_arrays(queries):
    """The replanning inputs of bp_plan_in (ABI 4) from the queries' optional ``replanning``, ``new_obs``,
    ``p_horizon`` [H,3] and ``sets_via_prev`` ([A, b] per set): dict of host arrays, or None when no query carries
    any of them (the fields stay NULL).  ValueError for more than 64 previous sets in a query, or a set without rows
    or with more than 48 rows."""
    keys = ("replanning", "new_obs", "p_horizon", "sets_via_prev")
    if not any(k in q for q in queries for k in keys):
        return None
    Q = len(queries)
    rp = np.zeros(Q, np.int32)
    no = np.zeros(Q, np.int32)
    h_off = np.zeros(Q + 1, np.int32)
    p_off = np.zeros(Q + 1, np.int32)
    hz, rows, row_n = [], [], []
    for i, q in enumerate(queries):
        rp[i], no[i] = bool(q.get("replanning", False)), bool(q.get("new_obs", False))
        h = np.asarray(q.get("p_horizon", ()), float).reshape(-1, 3)
        hz.append(h)
        h_off[i + 1] = h_off[i] + h.shape[0]
        prev = q.get("sets_via_prev", ())
        if len(prev) > MAX_PREV_SETS:
            raise ValueError(f"query {i}: {len(prev)} previous sets (at most {MAX_PREV_SETS})")
        for a_set, b_set in prev:
            a_set = np.asarray(a_set, float).reshape(-1, 3)
            b_set = np.asarray(b_set, float).reshape(-1)
            if not 1 <= a_set.shape[0] <= SET_ROWS or b_set.shape[0] != a_set.shape[0]:
                raise ValueError(f"query {i}: a previous set has {a_set.shape[0]} rows (1 .. {SET_ROWS}, one b each)")
            rows.append(np.concatenate((a_set, b_set[:, None]), axis=1))
            row_n.append(a_set.shape[0])
        p_off[i + 1] = p_off[i] + len(prev)
    row_off = np.zeros(len(row_n) + 1, np.int32)
    row_off[1:] = np.cumsum(row_n)
    return dict(replanning=rp, new_obs=no, horizon_off=h_off,
                p_horizon=np.ascontiguousarray(np.concatenate(hz)) if Q else np.zeros((0, 3)), prev_off=p_off,
                prev_row_off=row_off, prev_rows=np.ascontiguousarray(np.concatenate(rows)) if rows else np.zeros((0, 4)))


def active_mask(active, Q):
    """The ``active`` argument of the batched drivers as int32 [Q] (None stays None); ValueError for another
    length."""
    if active is None:
        return None
    a = np.asarray(active).reshape(-1)
    if a.shape[0] != Q:
        raise ValueError(f"active has {a.shape[0]} entries for {Q} queries")
    return np.ascontiguousarray(a.astype(bool).astype(np.int32))


def pack_corridors(sets, query_scene):
    """Host packing of NativePlanner.corridor_hits: (buffer uint8, offsets of A [S,m_max,3] | b [S,m_max] | m [S] |
    set_scene [S] in it, S, m_max, per-query (first, count) or None).  Sets are padded with rows A = 0, b = 10.
    ValueError for a set without rows or with more than 48 rows, or rows and offsets of different counts."""
    spans, A_list, b_list, scene_of = [], [], [], []
    for i, qs in enumerate(sets):
        if qs is None:
            spans.append(None)
            continue
        spans.append((len(A_list), len(qs)))
        for a_set, b_set in qs:
            a_set = np.asarray(a_set, float).reshape(-1, 3)
            b_set = np.asarray(b_set, float).reshape(-1)
            if not 1 <= a_set.shape[0] <= SET_ROWS or b_set.shape[0] != a_set.shape[0]:
                raise ValueError(f"query {i}: a set has {a_set.shape[0]} rows (1 .. {SET_ROWS}, one b each)")
            A_list.append(a_set)
            b_list.append(b_set)
            scene_of.append(i if query_scene is None else int(query_scene[i]))
    S = len(A_list)
    m_max = max((a.shape[0] for a in A_list), default=1)
    sizes = (8 * S * m_max * 3, 8 * S * m_max, 4 * S, 4 * S)
    offs = np.concatenate(([0], np.cumsum([(n + 15) // 16 * 16 for n in sizes])))
    buf = np.zeros(int(offs[-1]), np.uint8)
    A = buf[offs[0]: offs[0] + sizes[0]].view(np.float64).reshape(S, m_max, 3)
    b = buf[offs[1]: offs[1] + sizes[1]].view(np.float64).reshape(S, m_max)
    b[:] = 10.0
    m = buf[offs[2]: offs[2] + sizes[2]].view(np.int32)
    sc = buf[offs[3]: offs[3] + sizes[3]].view(np.int32)
    for k, (a_set, b_set) in enumerate(zip(A_list, b_list)):
        A[k, : a_set.shape[0]] = a_set
        b[k, : b_set.shape[0]] = b_set
        m[k] = a_set.shape[0]
    sc[:] = scene_of
    return buf, [int(o) for o in offs[:4]], S, m_max, spans


def _rodrigues(omega, phi):
    k = np.array([[0.0, -omega[2], omega[1]], [omega[2], 0.0, -omega[0]], [-omega[1], omega[0], 0.0]])
    return np.eye(3) + np.sin(phi) * k + (1.0 - np.cos(phi)) * (k @ k)


def ee_setup(r0, r1, length_ee=LENGTH_EE):
    """plan_convex_set_path :207-219 for one (r0, r1): (l_ee, l_ee_end, the 20 rotated offsets of
    check_intersection)."""
    from scipy.spatial.transform import Rotation as R

    omega = R.from_matrix(r1 @ r0.T).as_rotvec()
    omega_norm = np.linalg.norm(omega)
    omega_normed = omega / omega_norm if omega_norm > 1e-6 else np.array([0, 0, 1.0])
    l_ee = r0 @ np.array([-length_ee, 0, 0])
    l_ee_end = r1 @ np.array([-length_ee, 0, 0])
    samples = np.ascontiguousarray([_rodrigues(omega_normed, omega_norm * k / (FIT_SAMPLES - 1)) @ l_ee
                                    for k in range(FIT_SAMPLES)])
    return l_ee, l_ee_end, samples


def query_kind(queries, what="query"):
    """'boxes' when every query carries ``obstacles`` ([N,6] lb | ub), 'polytopes' when every query carries
    ``obs_sets`` (inflated [A (<= 15 x 3), b] per obstacle, optionally ``obs_points_sets``).  One scene batch holds
    one kind: a batch that mixes them, or a query with both or neither, raises ValueError.  (Also the kind of a list
    of shared scenes, ``what="scene"``.)"""
    kinds = set()
    for i, q in enumerate(queries):
        has_boxes, has_sets = q.get("obstacles") is not None, q.get("obs_sets") is not None
        if has_boxes == has_sets:
            raise ValueError(f"{what} {i} must carry either 'obstacles' (boxes) or 'obs_sets' (polytopes)")
        kinds.add("polytopes" if has_sets else "boxes")
    if len(kinds) > 1:
        raise ValueError(f"a batch mixes box and polytope {'queries' if what == 'query' else what + 's'}: one scene "
                         "batch holds one obstacle kind")
    return kinds.pop() if kinds else "boxes"


_OBSTACLE_KEYS = ("obstacles", "obs_sets", "obs_points_sets")


def scene_map(queries, scenes=None):
    """The query -> scene map of a batch over shared scenes: None without ``scenes`` (every query carries its own
    obstacles), else int32 [Q] of the queries' ``scene`` indices.  ``scenes`` is a list of dicts with the obstacle keys
    a query carries otherwise (``obstacles``, or ``obs_sets`` [+ ``obs_points_sets``]), all of one kind; each query
    then carries ``scene`` (an int in [0, len(scenes))) and no obstacles.  ValueError (before anything touches the
    device) for a ``scene`` out of range or not an int, a query with both a scene and obstacles or neither, scenes of
    mixed kinds and ``scene`` keys without ``scenes``."""
    if scenes is None:
        for i, q in enumerate(queries):
            if "scene" in q:
                raise ValueError(f"query {i} carries 'scene' but no scenes were given")
        return None
    if len(scenes) == 0:
        raise ValueError("scenes is empty")
    query_kind(scenes, "scene")
    out = np.zeros(len(queries), np.int32)
    for i, q in enumerate(queries):
        has_obs = any(q.get(k) is not None for k in _OBSTACLE_KEYS)
        if "scene" not in q:
            raise ValueError(f"query {i} carries no 'scene'" + (" (it carries obstacles)" if has_obs else ""))
        if has_obs:
            raise ValueError(f"query {i} carries both 'scene' and obstacles")
        s = q["scene"]
        if isinstance(s, (bool, np.bool_)) or not isinstance(s, (int, np.integer)):
            raise ValueError(f"query {i}: scene {s!r} is not an int")
        if not 0 <= s < len(scenes):
            raise ValueError(f"query {i}: scene {s} out of range (0 .. {len(scenes) - 1})")
        out[i] = s
    return out


def pack_obstacles(holders, kind):
    """(box_off [n+1], boxes [sum N, 6] or None, obs_rows [sum N, 15, 4] or None) of a list of queries or scenes (the
    obstacle layout of bp_plan_in)."""
    n = len(holders)
    box_off = np.zeros(n + 1, np.int32)
    if kind == "polytopes":
        rows = [obs_rows_of(h["obs_sets"]) for h in holders]
        box_off[1:] = np.cumsum([r.shape[0] for r in rows])
        return box_off, None, np.ascontiguousarray(np.concatenate(rows)) if n else np.zeros((0, OBS_ROWS, 4))
    boxes = [np.asarray(h["obstacles"], float).reshape(-1, 6) for h in holders]
    box_off[1:] = np.cumsum([b.shape[0] for b in boxes])
    return box_off, np.ascontiguousarray(np.vstack(boxes)) if n else np.zeros((0, 6)), None


def obs_rows_of(obs_sets):
    """obs_sets -> [N, 15, 4] (a0, a1, a2, b) rows in the given order, padded with (0, 0, 0, 10) as
    normalize_set_size pads them."""
    rows = np.zeros((len(obs_sets), OBS_ROWS, 4))
    rows[:, :, 3] = 10.0
    for j, (a_set, b_set) in enumerate(obs_sets):
        a_set = np.asarray(a_set, float).reshape(-1, 3)
        b_set = np.asarray(b_set, float).reshape(-1)
        if a_set.shape[0] > OBS_ROWS or b_set.shape[0] != a_set.shape[0]:
            raise ValueError(f"obstacle {j}: at most {OBS_ROWS} rows (a, b) per polytope")
        rows[j, : a_set.shape[0], :3], rows[j, : a_set.shape[0], 3] = a_set, b_set
    return rows


def scene_batch(queries, obs_size_increase):
    """The device scene batch of a batch of queries (or of shared scenes): SceneBatch over the boxes, or
    PolytopeSceneBatch over the obs_sets (vertex lists from ``obs_points_sets``, enumerated on the device when
    missing)."""
    from . import geometry as geo

    if query_kind(queries) == "polytopes":
        return geo.PolytopeSceneBatch([(q["obs_sets"], q.get("obs_points_sets")) for q in queries])
    return geo.SceneBatch([q["obstacles"] for q in queries], obs_size_increase)


def rng_state_words(rng):
    """(state_hi, state_lo, inc_hi, inc_lo) of a numpy Generator over PCG64."""
    st = rng.bit_generator.state
    if st["bit_generator"] != "PCG64":
        raise ValueError("the native planner driver restates numpy's PCG64 stream only")
    s, inc = int(st["state"]["state"]), int(st["state"]["inc"])
    m = (1 << 64) - 1
    return [s >> 64, s & m, inc >> 64, inc & m]


class PackedQueries:
    """Host arrays of a batch in the layout of bp_plan_in / bp_plan_out (kept alive with the ctypes views).
    With ``scenes`` (see scene_map) the obstacles are the scenes', packed once (box_off of len(scenes) + 1), and
    ``query_scene`` is the batch's query -> scene map (else None).  ``scene_arrays``: the scenes already packed
    (pack_obstacles of the same scenes), for a planner that plans new queries over its resident scenes."""

    def __init__(self, queries, obs_size_increase, workspace_max, workspace_min, rng_seeds=None, sample_chunk=32,
                 want_nodes=True, scenes=None, scene_arrays=None):
        Q = len(queries)
        self.Q = Q
        self.query_scene = scene_map(queries, scenes)
        holders = queries if scenes is None else scenes
        self.kind = query_kind(holders, "query" if scenes is None else "scene")
        self.box_off, self.boxes, self.obs_rows = (scene_arrays if scene_arrays is not None else
                                                   pack_obstacles(holders, self.kind))
        self.ws_min = np.ascontiguousarray(np.asarray(workspace_min, float).reshape(3))
        self.ws_max = np.ascontiguousarray(np.asarray(workspace_max, float).reshape(3))
        self.starts = np.ascontiguousarray([np.asarray(q["start"], float) for q in queries]).reshape(Q, 3)
        self.ends = np.ascontiguousarray([np.asarray(q["end"], float) for q in queries]).reshape(Q, 3)
        self.l_ee = np.zeros((Q, 3))
        self.l_ee_end = np.zeros((Q, 3))
        self.ee_samples = np.zeros((Q, FIT_SAMPLES, 3))
        cache = {}
        for i, q in enumerate(queries):
            r0, r1 = np.asarray(q["r0"], float), np.asarray(q["r1"], float)
            key = (r0.tobytes(), r1.tobytes())
            if key not in cache:
                cache[key] = ee_setup(r0, r1)
            self.l_ee[i], self.l_ee_end[i], self.ee_samples[i] = cache[key]
        self.rng = np.zeros((Q, 4), np.uint64)
        for i in range(Q):
            g = np.random.default_rng(rng_seeds[i] if rng_seeds is not None else None)
            self.rng[i] = rng_state_words(g)
        self.has_first = np.zeros(Q, np.int32)
        self.first_sample = np.zeros((Q, 3))
        for i, q in enumerate(queries):
            if q.get("first_sample") is not None:
                self.has_first[i] = 1
                self.first_sample[i] = np.asarray(q["first_sample"], float)
        self.replan = replan_arrays(queries)
        rpa = self.replan or {}
        self.inp = BpPlanIn(Q, self.boxes.ctypes.data_as(_dp) if self.boxes is not None else None,
                            self.box_off.ctypes.data_as(_ip), float(obs_size_increase),
                            self.ws_min.ctypes.data_as(_dp), self.ws_max.ctypes.data_as(_dp),
                            self.starts.ctypes.data_as(_dp), self.ends.ctypes.data_as(_dp), self.l_ee.ctypes.data_as(_dp),
                            self.l_ee_end.ctypes.data_as(_dp), self.ee_samples.ctypes.data_as(_dp),
                            self.rng.ctypes.data_as(_up), self.has_first.ctypes.data_as(_ip),
                            self.first_sample.ctypes.data_as(_dp), int(sample_chunk), 0,
                            self.obs_rows.ctypes.data_as(_dp) if self.obs_rows is not None else None,
                            _ptr(rpa.get("replanning"), _ip), _ptr(rpa.get("new_obs"), _ip),
                            _ptr(rpa.get("horizon_off"), _ip), _ptr(rpa.get("p_horizon"), _dp),
                            _ptr(rpa.get("prev_off"), _ip), _ptr(rpa.get("prev_row_off"), _ip),
                            _ptr(rpa.get("prev_rows"), _dp))
        # outputs
        self.err_kind = np.zeros(Q, np.int32)
        self.err_msg = ctypes.create_string_buffer(160 * max(Q, 1))
        self.path = np.full((Q, MAX_PATH), -1, np.int32)
        self.path_len = np.zeros(Q, np.int32)
        self.set_ids = np.full((Q, MAX_PATH), -1, np.int32)
        self.n_ids = np.zeros(Q, np.int32)
        self.p_via = np.zeros((Q, MAX_PATH + 2, 3))
        self.n_via = np.zeros(Q, np.int32)
        self.rng_out = np.zeros((Q, 4), np.uint64)
        self.n_nodes = np.zeros(Q, np.int32)
        self.n_inter = np.zeros(Q, np.int32)
        self.n_edges = np.zeros(Q, np.int32)
        self.finish_round = np.full(Q, -1, np.int32)
        self.finish_ms = np.zeros(Q)
        self.node_A = np.zeros((Q, MAX_NODES, NODE_ROWS, 3)) if want_nodes else None
        self.node_b = np.zeros((Q, MAX_NODES, NODE_ROWS)) if want_nodes else None
        self.node_m = np.zeros((Q, MAX_NODES), np.int32) if want_nodes else None
        self.stats = np.zeros(8, np.int64)
        self.p_horizon_max = np.zeros((Q, 3))
        self.out = BpPlanOut(self.err_kind.ctypes.data_as(_ip), ctypes.cast(self.err_msg, ctypes.c_char_p),
                             self.path.ctypes.data_as(_ip), self.path_len.ctypes.data_as(_ip),
                             self.set_ids.ctypes.data_as(_ip), self.n_ids.ctypes.data_as(_ip),
                             self.p_via.ctypes.data_as(_dp), self.n_via.ctypes.data_as(_ip),
                             self.rng_out.ctypes.data_as(_up), self.n_nodes.ctypes.data_as(_ip),
                             self.n_inter.ctypes.data_as(_ip), self.n_edges.ctypes.data_as(_ip),
                             self.finish_round.ctypes.data_as(_ip), self.finish_ms.ctypes.data_as(_dp),
                             self.node_A.ctypes.data_as(_dp) if want_nodes else None,
                             self.node_b.ctypes.data_as(_dp) if want_nodes else None,
                             self.node_m.ctypes.data_as(_ip) if want_nodes else None,
                             self.stats.ctypes.data_as(ctypes.POINTER(ctypes.c_longlong)),
                             self.p_horizon_max.ctypes.data_as(_dp))

    def results(self, active=None):
        """Per query: dict(path, set_ids, sets_via, p_via, n_nodes, n_inter, n_edges) or the exception the Python
        planner raises for it (None for a query that ``active`` skipped).  With the node sets (want_nodes), a planned query also gets ``sets_via_prev``: what the
        planner keeps for its next call -- sets_via, or after the early exit of :361-375 (path [0]) the start set
        padded to 15 rows (:371-372).  A replanning query also gets ``p_horizon_max``."""
        from .utils import normalize_set_size

        out = []
        raw = self.err_msg.raw
        for q in range(self.Q):
            if active is not None and not active[q]:
                out.append(None)
                continue
            if self.err_kind[q]:
                msg = raw[160 * q: 160 * (q + 1)].split(b"\0", 1)[0].decode()
                out.append(_ERRORS[int(self.err_kind[q])](msg))
                continue
            ids = [int(v) for v in self.set_ids[q, : self.n_ids[q]]]
            res = dict(path=[int(v) for v in self.path[q, : self.path_len[q]]], set_ids=ids,
                       p_via=self.p_via[q, : self.n_via[q]].copy(), n_nodes=int(self.n_nodes[q]),
                       n_inter=int(self.n_inter[q]), n_edges=int(self.n_edges[q]))
            if self.node_A is not None:
                res["sets_via"] = [[self.node_A[q, s, : self.node_m[q, s]].copy(), self.node_b[q, s, : self.node_m[q, s]].copy()]
                                   for s in ids]
                prev = [[a.copy(), b.copy()] for a, b in res["sets_via"]]
                res["sets_via_prev"] = normalize_set_size(prev, 15) if res["path"] == [0] else prev
            if self.replan is not None and self.replan["replanning"][q]:
                res["p_horizon_max"] = self.p_horizon_max[q].copy()
            out.append(res)
        return out

    def stats_dict(self):
        return dict(rounds=int(self.stats[0]), set_requests=int(self.stats[1]), pair_tests=int(self.stats[2]),
                    projections=int(self.stats[3]), shortest_paths=int(self.stats[4]),
                    kernel_chains=int(self.stats[5]), device_wait_ms=self.stats[6] / 1e3, lanes=int(self.stats[7]),
                    finish_round=self.finish_round.copy(), finish_ms=self.finish_ms.copy())


class NativePlanner:
    """A batch of independent planning queries, one scene each, planned in lock step by libbpgeo's native driver.
    The queries carry boxes (``obstacles``) or polytopes (``obs_sets`` [, ``obs_points_sets``]), all of one kind.
    With ``scenes`` (a list of dicts with those obstacle keys), the queries share them instead: each query carries
    ``scene``, the index of the scene it plans in, and no obstacles (see scene_map).  Every scene is then packed,
    ingested and stored on the device once however many queries plan in it, and every query's results are the ones it
    gets with a copy of its scene of its own.
    The scene batch and the device tables are created once; ``run`` can be called again (same scenes), also with
    new per-query inputs (``queries=``: an MPC loop's replanning calls) over the same obstacles.  When the obstacles
    move, ``update_obstacles`` rewrites the resident scenes in place."""

    def __init__(self, queries, obs_size_increase=0.01, workspace_max=(1.0, 1.0, 1.2), workspace_min=(-1.0, -1.0, 0.0),
                 scenes=None):
        import torch

        from . import _lib

        # (a malformed or mixed batch fails before anything touches the device)
        self.query_scene = scene_map(queries, scenes)
        self.kind = query_kind(queries) if scenes is None else query_kind(scenes, "scene")
        if not torch.cuda.is_available():
            raise _lib.BpGeoError("boundplanner_b200 needs a CUDA device (no CPU fallback)")
        self._lib = _lib.load()
        self.queries = queries
        self.scenes = scenes
        self.infl, self.ws_max, self.ws_min = float(obs_size_increase), list(workspace_max), list(workspace_min)
        self.scene = scene_batch(queries if scenes is None else scenes, obs_size_increase)
        self._obstacles = None                   # (kind, offsets, rows) of the scenes, for run(queries=...)
        self._scene_pack = None                  # the shared scenes, packed (pack_obstacles)
        self._h = ctypes.c_void_p(0)
        self._packed = {}
        if scenes is None:
            _lib.check(self._lib.bp_plan_create(self.scene._h, len(queries), ctypes.byref(self._h)))
        else:
            _lib.check(self._lib.bp_plan_create_mapped(self.scene._h, len(queries),
                                                       self.query_scene.ctypes.data_as(_ip), ctypes.byref(self._h)))

    def update_obstacles(self, queries, scenes=None):
        """Move the obstacles: the scenes become those of ``queries`` (the constructor's format, as many queries, the
        same obstacle kind; ValueError before the device is touched otherwise), written into the resident scene batch
        in place (SceneBatch / PolytopeSceneBatch.update_scenes), and ``queries`` become the planner's queries.
        A planner over shared scenes takes the new ``scenes`` instead (as many as before, of the same kind), and
        ``queries`` must carry the planner's scene indices.
        ``run()`` and ``run(queries=...)`` then plan against the new obstacles.  A failed update leaves the planner
        as it was."""
        if len(queries) != len(self.queries):
            raise ValueError(f"{len(queries)} queries for a planner of {len(self.queries)} scenes")
        if (scenes is None) != (self.scenes is None):
            raise ValueError("a planner over shared scenes is updated with scenes=, a planner of one scene per query "
                             "without")
        holders = queries
        if scenes is not None:
            if len(scenes) != len(self.scenes):
                raise ValueError(f"{len(scenes)} scenes for a planner of {len(self.scenes)} scenes")
            m = scene_map(queries, scenes)
            if not np.array_equal(m, self.query_scene):
                raise ValueError("the queries' scene indices differ from the planner's")
            holders = scenes
        kind = query_kind(holders, "query" if scenes is None else "scene")
        if kind != self.kind:
            raise ValueError(f"the planner's scenes hold {self.kind}, the {'queries' if scenes is None else 'scenes'} "
                             f"{kind}")
        if kind == "polytopes":
            n_max = max(len(h["obs_sets"]) for h in holders)
            if n_max > MAX_POLY_OBSTACLES:
                raise ValueError(f"polytope scenes hold at most {MAX_POLY_OBSTACLES} obstacles (largest scene: {n_max})")
            self.scene.update_scenes([(h["obs_sets"], h.get("obs_points_sets")) for h in holders])
        else:
            self.scene.update_scenes([h["obstacles"] for h in holders])
        self.queries = queries
        if scenes is not None:
            self.scenes = scenes
        self._packed = {}
        self._obstacles = None
        self._scene_pack = None

    @staticmethod
    def _obstacles_of(pk):
        return pk.kind, pk.box_off, pk.boxes if pk.obs_rows is None else pk.obs_rows

    def _scene_arrays(self):
        """The shared scenes packed once (pack_obstacles), for run(queries=...)."""
        if self._scene_pack is None:
            self._scene_pack = pack_obstacles(self.scenes, self.kind)
        return self._scene_pack

    def corridor_hits(self, sets, tol=1e-3):
        """Check corridors against the resident scenes (after update_obstacles, say): ``sets`` has one entry per
        query, a list of [A, b] (e.g. a result's ``sets_via_prev``) or None.  Every set is tested against the
        obstacles of its query's scene (geometry.sets_obstacle_hits: the set and an obstacle, each shrunk by tol,
        share a point).  Returns per query None or np.int32 [n_sets]: the lowest index of an obstacle of the scene
        that hits the set, -1 where none does.  One host-to-device copy, one kernel chain and one device-to-host copy;
        ``corridor_events`` are CUDA events recorded around the library call.  ValueError, before the device is
        touched, for another number of entries than queries or a set without rows or with more than 48 rows."""
        import torch

        from . import _lib

        if len(sets) != len(self.queries):
            raise ValueError(f"{len(sets)} corridors for a planner of {len(self.queries)} queries")
        buf, offs, S, m_max, spans = pack_corridors(sets, self.query_scene)
        out = [None if sp is None else np.zeros(0, np.int32) for sp in spans]
        if S == 0:
            return out
        dev = torch.from_numpy(buf).to("cuda", non_blocking=False)
        base = dev.data_ptr()
        work = torch.empty((self._lib.bp_sets_obstacles_workspace_bytes(S),), dtype=torch.uint8, device="cuda")
        hit = torch.empty((S,), dtype=torch.int32, device="cuda")
        stream = torch.cuda.current_stream()
        self.corridor_events = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
        self.corridor_events[0].record(stream)
        _lib.check(self._lib.bp_sets_obstacles(self.scene._h, ctypes.c_void_p(base + offs[3]),
                                               ctypes.c_void_p(base + offs[0]), ctypes.c_void_p(base + offs[1]),
                                               ctypes.c_void_p(base + offs[2]), S, m_max, float(tol),
                                               ctypes.c_void_p(hit.data_ptr()), ctypes.c_void_p(work.data_ptr()),
                                               work.numel(), ctypes.c_void_p(stream.cuda_stream)))
        self.corridor_events[1].record(stream)
        h = hit.cpu().numpy()
        for i, sp in enumerate(spans):
            if sp is not None:
                out[i] = h[sp[0]: sp[0] + sp[1]].copy()
        return out

    def run(self, rng_seeds=None, sample_chunk=32, want_nodes=True, queries=None, active=None):
        """Plan the batch: (results, stats).  queries: new per-query inputs (start, end, r0, r1, first_sample and the
        replanning keys of planner.plan_batch) to plan against the scenes of this planner; their obstacles must be
        the ones it was created with, or last updated to (ValueError otherwise: the host push-out of `end` and the
        device scene must agree).  Over shared scenes, they carry the planner's scene indices instead (ValueError
        otherwise).  active: [Q] flags (or None: all): only the queries with a true flag are planned
        (bp_plan_run_active), each with the results it gets in a run of the whole batch; a skipped query's result is
        None and the stats count the active queries only."""
        active = active_mask(active, len(self.queries))
        if queries is not None:
            if len(queries) != len(self.queries):
                raise ValueError(f"{len(queries)} queries for a planner of {len(self.queries)} scenes")
            if self.scenes is not None:
                if not np.array_equal(scene_map(queries, self.scenes), self.query_scene):
                    raise ValueError("the queries' scene indices differ from the planner's")
                return self._run(PackedQueries(queries, self.infl, self.ws_max, self.ws_min, rng_seeds, sample_chunk,
                                               want_nodes, scenes=self.scenes, scene_arrays=self._scene_arrays()),
                                 active)
            pk = PackedQueries(queries, self.infl, self.ws_max, self.ws_min, rng_seeds, sample_chunk, want_nodes)
            if self._obstacles is None:
                self._obstacles = self._obstacles_of(
                    PackedQueries(self.queries, self.infl, self.ws_max, self.ws_min, None, sample_chunk, False))
            mine, theirs = self._obstacles, self._obstacles_of(pk)
            if mine[0] != theirs[0] or not np.array_equal(mine[1], theirs[1]) or not np.array_equal(mine[2], theirs[2]):
                raise ValueError("the queries' obstacles differ from the scenes this planner was created with")
            return self._run(pk, active)
        # the packed host arrays of the batch (inputs incl. every query's generator state, output buffers) are kept
        # per seed list: planning the same batch again only runs the driver
        key = (None if rng_seeds is None else tuple(int(v) for v in rng_seeds), int(sample_chunk), bool(want_nodes))
        pk = self._packed.get(key) if rng_seeds is not None else None
        if pk is None:
            pk = PackedQueries(self.queries, self.infl, self.ws_max, self.ws_min, rng_seeds, sample_chunk, want_nodes,
                               scenes=self.scenes,
                               scene_arrays=self._scene_arrays() if self.scenes is not None else None)
            if rng_seeds is not None:
                self._packed = {key: pk}
        return self._run(pk, active)

    def _run(self, pk, active=None):
        import torch

        from . import _lib

        stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
        if active is None:
            _lib.check(self._lib.bp_plan_run(self._h, ctypes.byref(pk.inp), ctypes.byref(pk.out), stream))
        else:
            _lib.check(self._lib.bp_plan_run_active(self._h, ctypes.byref(pk.inp), active.ctypes.data_as(_ip),
                                                    ctypes.byref(pk.out), stream))
        return pk.results(active), pk.stats_dict()

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._lib.bp_plan_destroy(self._h)
            self._h = ctypes.c_void_p(0)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def plan_batch_native(queries, obs_size_increase=0.01, workspace_max=(1.0, 1.0, 1.2), workspace_min=(-1.0, -1.0, 0.0),
                      rng_seeds=None, sample_chunk=32, scenes=None, active=None):
    """Drop-in for ``planner.plan_batch``: (results, stats).  Box or polytope queries, one kind per batch; with
    ``scenes``, queries over shared scenes (see NativePlanner); ``active``: plan only the flagged queries (see
    NativePlanner.run)."""
    active_mask(active, len(queries))
    pl = NativePlanner(queries, obs_size_increase, workspace_max, workspace_min, scenes=scenes)
    try:
        return pl.run(rng_seeds, sample_chunk, active=active)
    finally:
        pl.close()
