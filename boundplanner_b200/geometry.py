"""Batched device-side API over libbpgeo.so.

PyTorch is plumbing only (device memory, streams); every compute call goes
through the C ABI in include/bpgeo.h with raw device pointers.  All tensors are
float64 / int32 CUDA tensors.  Reference sites are cited per function.
"""
from __future__ import annotations

import ctypes
import time
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib
from ._lib import BP_MAX_ROWS, check

_dp = ctypes.POINTER(ctypes.c_double)


def _require_cuda():
    if not torch.cuda.is_available():
        raise _lib.BpGeoError("boundplanner_b200 needs a CUDA device (no CPU fallback)")


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _host3(v):
    a = np.ascontiguousarray(np.asarray(v, dtype=np.float64).reshape(3))
    return a, a.ctypes.data_as(_dp)


def _dev(x, dtype=torch.float64):
    """Host array / tensor -> contiguous CUDA tensor (H2D copy when needed)."""
    if isinstance(x, torch.Tensor):
        return x.to(device="cuda", dtype=dtype).contiguous()
    return torch.as_tensor(np.ascontiguousarray(x), dtype=dtype).cuda()


class Scene:
    """Obstacle boxes resident in HBM (SoA, inflated).

    Replaces BoundPlanner.make_box / add_obstacle_reps (BoundPlanner.py:126-152).
    ``boxes``: [N,6] rows (lb, ub) on the host; ``inflate`` = obs_size_increase."""

    def __init__(self, boxes, inflate=0.0):
        _require_cuda()
        self._lib = _lib.load()
        self._h = ctypes.c_void_p(0)
        boxes = np.ascontiguousarray(np.asarray(boxes, dtype=np.float64).reshape(-1, 6))
        torch.cuda.current_device()        # make sure a context exists on the current device
        check(self._lib.bp_scene_create(boxes.ctypes.data_as(_dp), boxes.shape[0], float(inflate),
                                        ctypes.byref(self._h)))
        self.n = boxes.shape[0]
        self.inflate = float(inflate)

    def update(self, boxes, inflate=None):
        boxes = np.ascontiguousarray(np.asarray(boxes, dtype=np.float64).reshape(-1, 6))
        if inflate is None:
            inflate = self.inflate
        check(self._lib.bp_scene_update(self._h, boxes.ctypes.data_as(_dp), boxes.shape[0], float(inflate), _stream()))
        self.n = boxes.shape[0]
        self.inflate = float(inflate)

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._lib.bp_scene_destroy(self._h)
            self._h = ctypes.c_void_p(0)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class PolytopeScene(Scene):
    """General convex polytope obstacles resident in HBM: what ConvexSetFinder is handed when the obstacles are not
    boxes -- obs_sets = [[A (<= 15 rows, zero-padded), b], ...] (already inflated) and obs_points_sets = [vertices
    (V x 3), ...] (the reference enumerates them with cddlib, util_functions.py:66-79).  At most 16384 obstacles
    (their closest points are cached in shared memory up to 3072; beyond that the winner of every pick is re-solved)."""

    MAX_ROWS = 15

    def __init__(self, obs_sets, obs_points_sets=None, _offsets=None):
        _require_cuda()
        self._lib = _lib.load()
        self._h = ctypes.c_void_p(0)
        n = len(obs_sets)
        if obs_points_sets is None and n > 0:
            # no vertex lists given: enumerate them on the device (compute_polytope_vertices, util_functions.py:66-79)
            from .utils import obstacle_points_sets

            obs_points_sets = obstacle_points_sets(obs_sets)
        if n == 0 or len(obs_points_sets) != n:
            raise ValueError("PolytopeScene needs one vertex array per obstacle set")
        rows = np.zeros((n, self.MAX_ROWS, 4))
        rows[:, :, 3] = 10.0
        nrows = np.zeros(n, np.int32)
        vmax = max(int(np.asarray(v).reshape(-1, 3).shape[0]) for v in obs_points_sets)
        verts = np.zeros((n, vmax, 3))
        nverts = np.zeros(n, np.int32)
        for j, ((a_set, b_set), v) in enumerate(zip(obs_sets, obs_points_sets)):
            a_set = np.asarray(a_set, float).reshape(-1, 3)
            b_set = np.asarray(b_set, float).reshape(-1)
            nz = np.linalg.norm(a_set, axis=1) > 0
            k = int(nz.sum())
            if k > self.MAX_ROWS:
                raise ValueError(f"obstacle {j} has more than {self.MAX_ROWS} rows")
            rows[j, :k, :3], rows[j, :k, 3] = a_set[nz], b_set[nz]
            nrows[j] = k
            v = np.asarray(v, float).reshape(-1, 3)
            verts[j, : v.shape[0]] = v
            nverts[j] = v.shape[0]
        ip = ctypes.POINTER(ctypes.c_int)
        torch.cuda.current_device()
        if _offsets is None:
            check(self._lib.bp_scene_create_polytopes(rows.ctypes.data_as(_dp), nrows.ctypes.data_as(ip),
                                                      verts.ctypes.data_as(_dp), nverts.ctypes.data_as(ip), n, vmax,
                                                      ctypes.byref(self._h)))
            self.n = n
        else:
            offs = np.ascontiguousarray(_offsets, dtype=np.int32)
            check(self._lib.bp_scene_create_polytopes_batch(rows.ctypes.data_as(_dp), nrows.ctypes.data_as(ip),
                                                            verts.ctypes.data_as(_dp), nverts.ctypes.data_as(ip),
                                                            offs.ctypes.data_as(ip), len(offs) - 1, vmax,
                                                            ctypes.byref(self._h)))
            self.n = int(np.diff(offs).max())
            self.n_scenes = len(offs) - 1
        self.inflate = 0.0

    def update(self, boxes, inflate=None):
        raise _lib.BpGeoError("PolytopeScene is immutable: create a new one")


def _concat_rows(arrays, width):
    """Per-obstacle arrays of rows ([R_j, width], or [R_j] for width 1) -> (all rows back to back [sum R_j, width] as
    float64, R_j [n]).  One concatenate when every array already has that shape, else a reshape per array."""
    n = len(arrays)
    if n == 0:
        return np.zeros((0, width)), np.zeros(0, np.int64)
    try:
        flat = np.concatenate(arrays).astype(np.float64, copy=False)
        if flat.ndim == (1 if width == 1 else 2) and (width == 1 or flat.shape[1] == width):
            return flat.reshape(-1, width), np.fromiter(map(len, arrays), np.int64, n)
    except ValueError:                                 # ragged ranks or widths
        pass
    arrays = [np.asarray(a, float).reshape(-1, width) for a in arrays]
    return np.concatenate(arrays), np.fromiter((a.shape[0] for a in arrays), np.int64, n)


def pack_polytope_rows(obs_sets, max_rows=PolytopeScene.MAX_ROWS):
    """obs_sets ([A, b] per obstacle) -> (rows [n, 15, 4] (a0, a1, a2, b), nrows [n] int32) as PolytopeScene packs
    them: the rows of nonzero norm in their order, then (0, 0, 0, 10).  Vectorised over all obstacles at once.
    ValueError for an obstacle with more than 15 such rows or with another number of b's than rows."""
    n = len(obs_sets)
    A, counts = _concat_rows([s[0] for s in obs_sets], 3)
    b, b_counts = _concat_rows([s[1] for s in obs_sets], 1)
    if not np.array_equal(counts, b_counts):
        raise ValueError("every obstacle needs one b per row of A")
    rows = np.zeros((n, max_rows, 4))
    rows[:, :, 3] = 10.0
    obs = np.repeat(np.arange(n), counts)
    nz = (A * A).sum(axis=1) > 0                       # (the sign of np.linalg.norm's sqrt(sum(a * a)))
    nrows = np.bincount(obs[nz], minlength=n)
    if (nrows > max_rows).any():
        raise ValueError(f"obstacle {int(np.argmax(nrows > max_rows))} has more than {max_rows} rows")
    o = obs[nz]
    start = np.cumsum(nrows) - nrows                   # first kept row of every obstacle among all kept rows
    rows.reshape(-1, 4)[o * max_rows + np.arange(o.shape[0]) - start[o]] = np.hstack((A[nz], b[nz]))
    return rows, nrows.astype(np.int32)


def pack_vertices(obs_points_sets):
    """Vertex lists ([V_j, 3] per obstacle) -> (verts [n, vmax, 3] zero-padded, nverts [n] int32, vmax = the largest
    V_j), as PolytopeScene packs them."""
    n = len(obs_points_sets)
    pts, nverts = _concat_rows(list(obs_points_sets), 3)
    vmax = int(nverts.max()) if n else 0
    verts = np.zeros((n, vmax, 3))
    obs = np.repeat(np.arange(n), nverts)
    verts.reshape(-1, 3)[obs * vmax + np.arange(obs.shape[0]) - (np.cumsum(nverts) - nverts)[obs]] = pts
    return verts, nverts.astype(np.int32), vmax


class PolytopeSceneBatch(PolytopeScene):
    """Several polytope scenes stored back to back in HBM (one per planning query): ``scenes`` is a list of
    (obs_sets, obs_points_sets | None) pairs.  Use with build_sets_point / build_sets_line / sample_filter and
    ``item_scene`` = scene index of every seed / segment.  ``update_scenes`` moves the obstacles in place."""

    def __init__(self, scenes_list):
        from .utils import obstacle_points_sets

        sets, pts, offs = [], [], [0]
        for obs_sets, obs_points in scenes_list:
            if obs_points is None:
                obs_points = obstacle_points_sets(obs_sets)
            sets.extend(obs_sets)
            pts.extend(obs_points)
            offs.append(len(sets))
        super().__init__(sets, pts, _offsets=offs)

    def update_scenes(self, scenes_list):
        """Replace every scene's obstacles (the constructor's format, as many scenes as the batch has) in place: one
        staging copy and a short kernel chain (bp_scene_update_polytopes_batch), the same device contents as a new
        PolytopeSceneBatch of scenes_list.  Scenes without vertex lists have them enumerated on the device when no
        scene carries any, else here like the constructor does.  On failure the batch is left as it was.
        ``pack_seconds``: the host time of the packing (everything before the library call); ``update_events``: CUDA
        events recorded on the current stream around the library call (staging copy, kernels, synchronisation)."""
        from .utils import obstacle_points_sets

        t0 = time.perf_counter()
        if len(scenes_list) != self.n_scenes:
            raise ValueError(f"{len(scenes_list)} scenes for a batch of {self.n_scenes}")
        sets, offs = [], np.zeros(len(scenes_list) + 1, np.int32)
        for k, (obs_sets, _) in enumerate(scenes_list):
            sets.extend(obs_sets)
            offs[k + 1] = len(sets)
        rows, nrows = pack_polytope_rows(sets)
        ip = ctypes.POINTER(ctypes.c_int)
        verts = nverts = None
        vmax = 0
        if any(pts is not None for _, pts in scenes_list):
            pts = []
            for obs_sets, obs_points in scenes_list:
                pts.extend(obs_points if obs_points is not None else obstacle_points_sets(obs_sets))
            if len(pts) != len(sets):
                raise ValueError("PolytopeScene needs one vertex array per obstacle set")
            verts, nverts, vmax = pack_vertices(pts)
        self.pack_seconds = time.perf_counter() - t0
        self.update_events = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
        self.update_events[0].record()
        check(self._lib.bp_scene_update_polytopes_batch(
            self._h, rows.ctypes.data_as(_dp), nrows.ctypes.data_as(ip),
            verts.ctypes.data_as(_dp) if verts is not None else None,
            nverts.ctypes.data_as(ip) if nverts is not None else None, offs.ctypes.data_as(ip), len(scenes_list),
            vmax, _stream()))
        self.update_events[1].record()
        self.n = int(np.diff(offs).max())


class SceneBatch(Scene):
    """Several scenes stored back to back in HBM (one per planning query, BASELINE config C3).
    ``boxes_list``: list of [N_k,6] arrays.  Use with build_sets_point / build_sets_line and
    ``item_scene`` = scene index of every seed / segment."""

    def __init__(self, boxes_list, inflate=0.0):
        _require_cuda()
        self._lib = _lib.load()
        self._h = ctypes.c_void_p(0)
        offs = np.zeros(len(boxes_list) + 1, dtype=np.int32)
        offs[1:] = np.cumsum([np.asarray(bx).reshape(-1, 6).shape[0] for bx in boxes_list])
        boxes = np.ascontiguousarray(np.vstack([np.asarray(bx, dtype=np.float64).reshape(-1, 6) for bx in boxes_list]))
        torch.cuda.current_device()
        check(self._lib.bp_scene_create_batch(boxes.ctypes.data_as(_dp), offs.ctypes.data_as(ctypes.POINTER(ctypes.c_int)),
                                              len(boxes_list), float(inflate), ctypes.byref(self._h)))
        self.n = int(np.diff(offs).max()) if len(boxes_list) else 0
        self.n_scenes = len(boxes_list)
        self.inflate = float(inflate)

    def update(self, boxes, inflate=None):
        raise _lib.BpGeoError("SceneBatch is immutable")

    def update_scenes(self, boxes_list):
        """Replace every scene's boxes (the constructor's format, as many scenes as the batch has; counts may change,
        down to 0) in place, with the batch's inflate: one staging copy and one kernel (bp_scene_update_batch), the
        same device contents as a new SceneBatch of boxes_list.  On failure the batch is left as it was.
        ``pack_seconds``: the host time of the packing (everything before the library call); ``update_events``: CUDA
        events recorded on the current stream around the library call (staging copy, kernels, synchronisation)."""
        t0 = time.perf_counter()
        if len(boxes_list) != self.n_scenes:
            raise ValueError(f"{len(boxes_list)} scenes for a batch of {self.n_scenes}")
        boxes_list = [np.asarray(bx, dtype=np.float64).reshape(-1, 6) for bx in boxes_list]
        offs = np.zeros(len(boxes_list) + 1, dtype=np.int32)
        offs[1:] = np.cumsum([bx.shape[0] for bx in boxes_list])
        boxes = np.ascontiguousarray(np.vstack(boxes_list))
        self.pack_seconds = time.perf_counter() - t0
        self.update_events = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
        self.update_events[0].record()
        check(self._lib.bp_scene_update_batch(self._h, boxes.ctypes.data_as(_dp),
                                              offs.ctypes.data_as(ctypes.POINTER(ctypes.c_int)), len(boxes_list),
                                              self.inflate, _stream()))
        self.update_events[1].record()
        self.n = int(np.diff(offs).max())


@dataclass
class SetBatch:
    """S convex sets {x : A[s,:m[s]] x <= b[s,:m[s]]} plus their ellipsoids."""

    A: torch.Tensor            # [S,m_max,3]
    b: torch.Tensor            # [S,m_max]
    m: torch.Tensor            # [S] int32
    q_ellipse: torch.Tensor    # [S,3,3]
    p_mid: torch.Tensor        # [S,3]
    status: torch.Tensor       # [S] int32
    iters: torch.Tensor | None = None      # [S] int32 (k of the IRIS loop)
    rows_peak: torch.Tensor | None = None  # [S] int32 largest row count of any pass (reference cap: 20)
    work: torch.Tensor | None = None       # loop workspace (kept with the batch so that it can be reused)
    collision: torch.Tensor | None = None  # [S] int32 (line sets)

    def to_sets(self):
        """Host list of [A (m,3), b (m,)] like the reference's set representation."""
        A, b, m = self.A.cpu().numpy(), self.b.cpu().numpy(), self.m.cpu().numpy()
        return [[A[s, : m[s]].copy(), b[s, : m[s]].copy()] for s in range(A.shape[0])]


def _alloc_sets(S, m_max):
    dev = "cuda"
    # padded rows follow normalize_set_size: A = 0, b = 10 (util_functions.py:121-122)
    A = torch.zeros((S, m_max, 3), dtype=torch.float64, device=dev)
    b = torch.full((S, m_max), 10.0, dtype=torch.float64, device=dev)
    m = torch.zeros((S,), dtype=torch.int32, device=dev)
    return A, b, m


def alloc_set_batch(S, m_max=BP_MAX_ROWS):
    """Device buffers of one SetBatch plus the loop workspace (reusable across calls via ``out=``)."""
    lib = _lib.load()
    A, b, m = _alloc_sets(S, m_max)
    batch = SetBatch(A, b, m, torch.zeros((S, 3, 3), dtype=torch.float64, device="cuda"),
                     torch.zeros((S, 3), dtype=torch.float64, device="cuda"),
                     torch.zeros((S,), dtype=torch.int32, device="cuda"),
                     iters=torch.zeros((S,), dtype=torch.int32, device="cuda"),
                     rows_peak=torch.zeros((S,), dtype=torch.int32, device="cuda"))
    batch.work = torch.empty((lib.bp_build_sets_workspace_bytes(S),), dtype=torch.uint8, device="cuda")
    return batch


def build_sets_point(scene, seeds, ws_min, ws_max, fixed_mid=False, optimize=True, max_iter=5, m_max=BP_MAX_ROWS,
                     row_cap=0, out=None, item_scene=None, aabb=None, peers=None, tail=None):
    """ConvexSetFinder.find_set_around_point (ConvexSetFinder.py:190-240) for S seeds.
    row_cap=20 reproduces the reference's failure on passes with more than 20 rows (status 5).
    out: a batch from alloc_set_batch to write into (no allocation, CUDA-graph capturable).
    aabb: [S,6] tensor that receives every set's exact bounding box from the kernel's epilogue.
    peers: dict(base=int64 tensor [world] of mapped base addresses, world, slot0, off_A, off_b, off_m, off_aabb):
    the sets are also stored into every rank's global tables (multi-GPU exchange by peer stores).
    tail: a BpTail from make_tail(): the finished CTAs also do the pair tests (see bp_build_sets_point_tail)."""
    lib = _lib.load()
    seeds = _dev(seeds).reshape(-1, 3)
    S = seeds.shape[0]
    if out is None:
        out = alloc_set_batch(S, m_max)
    A, b, m, q, p, status, iters, peak, work = (out.A, out.b, out.m, out.q_ellipse, out.p_mid, out.status, out.iters,
                                                out.rows_peak, out.work)
    m_max = A.shape[1]
    wbytes = work.numel()
    amin, pmin = _host3(ws_min)      # host arrays must outlive the call
    amax, pmax = _host3(ws_max)
    if item_scene is not None:
        item_scene = _dev(item_scene, torch.int32).reshape(S)
    pk = peers or {}
    check(lib.bp_build_sets_point_tail(scene._h, _ptr(item_scene), _ptr(seeds), S, pmin, pmax, int(bool(fixed_mid)),
                                       int(bool(optimize)), int(max_iter), int(m_max), _ptr(A), _ptr(b), _ptr(m),
                                       _ptr(q), _ptr(p), _ptr(status), _ptr(iters), _ptr(peak), int(row_cap),
                                       _ptr(aabb), _ptr(pk.get("base")), int(pk.get("world", 0)),
                                       int(pk.get("slot0", 0)), int(pk.get("off_A", 0)), int(pk.get("off_b", 0)),
                                       int(pk.get("off_m", 0)), int(pk.get("off_aabb", 0)),
                                       ctypes.byref(tail) if tail is not None else None, _ptr(work), wbytes, _stream()))
    del amin, amax
    return out


def build_sets_around_line(scene, p0, dp1, ws_min, ws_max, optimize=True, max_iter=5, m_max=BP_MAX_ROWS, row_cap=0):
    """ConvexSetFinder.find_set_around_line (ConvexSetFinder.py:242-307) for S segments p0 .. p0 + dp1."""
    lib = _lib.load()
    if getattr(scene, "n_scenes", 1) > 1:
        raise ValueError("build_sets_around_line works on a single scene")
    p0 = _dev(p0).reshape(-1, 3)
    dp1 = _dev(dp1).reshape(-1, 3)
    S = p0.shape[0]
    out = alloc_set_batch(S, m_max)
    amin, pmin = _host3(ws_min)      # host arrays must outlive the call
    amax, pmax = _host3(ws_max)
    check(lib.bp_build_sets_around_line(scene._h, _ptr(p0), _ptr(dp1), S, pmin, pmax, int(bool(optimize)),
                                        int(max_iter), int(m_max), _ptr(out.A), _ptr(out.b), _ptr(out.m),
                                        _ptr(out.q_ellipse), _ptr(out.p_mid), _ptr(out.status), _ptr(out.iters),
                                        _ptr(out.rows_peak), int(row_cap), _stream()))
    del amin, amax
    return out


def build_sets_line(scene, p0, p1, ws_min, ws_max, compute_ellipsoid=False, limit_space=False, e_max=0.3,
                    m_max=BP_MAX_ROWS, item_scene=None):
    """ConvexSetFinder.find_set_collision_avoidance (ConvexSetFinder.py:309-375) for S segments."""
    lib = _lib.load()
    p0 = _dev(p0).reshape(-1, 3)
    p1 = _dev(p1).reshape(-1, 3)
    S = p0.shape[0]
    A, b, m = _alloc_sets(S, m_max)
    q = torch.zeros((S, 3, 3), dtype=torch.float64, device="cuda")
    p = torch.zeros((S, 3), dtype=torch.float64, device="cuda")
    status = torch.zeros((S,), dtype=torch.int32, device="cuda")
    coll = torch.zeros((S,), dtype=torch.int32, device="cuda")
    wbytes = lib.bp_build_sets_workspace_bytes(S)
    work = torch.empty((wbytes,), dtype=torch.uint8, device="cuda")
    amin, pmin = _host3(ws_min)      # host arrays must outlive the call
    amax, pmax = _host3(ws_max)
    if item_scene is not None:
        item_scene = _dev(item_scene, torch.int32).reshape(S)
    check(lib.bp_build_sets_line_ms(scene._h, _ptr(item_scene), _ptr(p0), _ptr(p1), S, pmin, pmax,
                                    int(bool(limit_space)), float(e_max), int(bool(compute_ellipsoid)), int(m_max),
                                    _ptr(A), _ptr(b), _ptr(m), _ptr(q), _ptr(p), _ptr(coll), _ptr(status), _ptr(work),
                                    wbytes, _stream()))
    del amin, amax
    return SetBatch(A, b, m, q, p, status, collision=coll)


def closest_points(scene, seeds, q_inv):
    """ConvexSetFinder.compute_set_projs (:465-489) + dists (:429): y [S,N,3], dist [S,N]."""
    lib = _lib.load()
    seeds = _dev(seeds).reshape(-1, 3)
    q_inv = _dev(q_inv).reshape(-1, 3, 3)
    S = seeds.shape[0]
    y = torch.empty((S, scene.n, 3), dtype=torch.float64, device="cuda")
    dist = torch.empty((S, scene.n), dtype=torch.float64, device="cuda")
    check(lib.bp_closest_points(scene._h, _ptr(seeds), _ptr(q_inv), S, _ptr(y), _ptr(dist), _stream()))
    return y, dist


def closest_points_line(scene, p0, p1):
    """ConvexSetFinder.compute_set_projs_line (:491-510): x [S,N,3], phi [S,N]."""
    lib = _lib.load()
    p0 = _dev(p0).reshape(-1, 3)
    p1 = _dev(p1).reshape(-1, 3)
    S = p0.shape[0]
    x = torch.empty((S, scene.n, 3), dtype=torch.float64, device="cuda")
    phi = torch.empty((S, scene.n), dtype=torch.float64, device="cuda")
    check(lib.bp_closest_points_line(scene._h, _ptr(p0), _ptr(p1), S, _ptr(x), _ptr(phi), _stream()))
    return x, phi


def polyhedron(scene, seeds, q_inv, q_ellipse, init_rows, m_max=BP_MAX_ROWS):
    """ConvexSetFinder.compute_polyhedron (:423-463): one greedy pass for S seeds.
    init_rows: [S,6,4] (a | b)."""
    lib = _lib.load()
    seeds = _dev(seeds).reshape(-1, 3)
    S = seeds.shape[0]
    q_inv = _dev(q_inv).reshape(S, 3, 3)
    q_ellipse = _dev(q_ellipse).reshape(S, 3, 3)
    init_rows = _dev(init_rows).reshape(S, 6, 4)
    A, b, m = _alloc_sets(S, m_max)
    status = torch.zeros((S,), dtype=torch.int32, device="cuda")
    check(lib.bp_polyhedron(scene._h, _ptr(seeds), _ptr(q_inv), _ptr(q_ellipse), _ptr(init_rows), S, int(m_max),
                            _ptr(A), _ptr(b), _ptr(m), _ptr(status), _stream()))
    return A, b, m, status


def mvie(A, b, m, centre, free_centre):
    """mvie_socp (free_centre=True, :512-537) / mvie_socp_fixed_mid (:539-562) for S sets.
    Returns q_inv (= L L^T), q_ellipse (= q_inv^-1), centre, status, newton_iters."""
    lib = _lib.load()
    A = _dev(A)
    S, m_max = A.shape[0], A.shape[1]
    b = _dev(b).reshape(S, m_max)
    m = _dev(m, torch.int32).reshape(S)
    centre = _dev(centre).reshape(S, 3)
    q_inv = torch.empty((S, 3, 3), dtype=torch.float64, device="cuda")
    q_ell = torch.empty((S, 3, 3), dtype=torch.float64, device="cuda")
    c_out = torch.empty((S, 3), dtype=torch.float64, device="cuda")
    status = torch.zeros((S,), dtype=torch.int32, device="cuda")
    its = torch.zeros((S,), dtype=torch.int32, device="cuda")
    check(lib.bp_mvie(_ptr(A), _ptr(b), _ptr(m), S, m_max, int(bool(free_centre)), _ptr(centre), _ptr(q_inv),
                      _ptr(q_ell), _ptr(c_out), _ptr(status), _ptr(its), _stream()))
    return q_inv, q_ell, c_out, status, its


def mvie_fixed_r(A, b, m, centre, r_ellipse, a_lb):
    """mvie_socp_fixed_r (:564-588) for S sets.  Returns q_inv (= R diag(x^2) R^T), q_ellipse, eigs (= x), status,
    newton_iters."""
    lib = _lib.load()
    A = _dev(A)
    S, m_max = A.shape[0], A.shape[1]
    b = _dev(b).reshape(S, m_max)
    m = _dev(m, torch.int32).reshape(S)
    centre = _dev(centre).reshape(S, 3)
    r_ellipse = _dev(r_ellipse).reshape(S, 3, 3)
    a_lb = _dev(a_lb).reshape(S)
    q_inv = torch.empty((S, 3, 3), dtype=torch.float64, device="cuda")
    q_ell = torch.empty((S, 3, 3), dtype=torch.float64, device="cuda")
    eigs = torch.empty((S, 3), dtype=torch.float64, device="cuda")
    status = torch.zeros((S,), dtype=torch.int32, device="cuda")
    its = torch.zeros((S,), dtype=torch.int32, device="cuda")
    check(lib.bp_mvie_fixed_r(_ptr(A), _ptr(b), _ptr(m), S, m_max, _ptr(centre), _ptr(r_ellipse), _ptr(a_lb),
                              _ptr(q_inv), _ptr(q_ell), _ptr(eigs), _ptr(status), _ptr(its), _stream()))
    return q_inv, q_ell, eigs, status, its


def alloc_pair_buffers(S, rows=None):
    lib = _lib.load()
    rows = S if rows is None else rows
    bits = torch.empty((rows, (S + 31) // 32), dtype=torch.int32, device="cuda")
    work = torch.empty((lib.bp_pair_workspace_bytes(S, rows),), dtype=torch.uint8, device="cuda")
    return bits, work


def set_aabb(A, b, m, out=None):
    """Exact axis-aligned bounding boxes [S,6] (lo | hi) of S sets (pre-filter of pair_feasible)."""
    lib = _lib.load()
    S, m_max = A.shape[0], A.shape[1]
    if out is None:
        out = torch.empty((S, 6), dtype=torch.float64, device="cuda")
    check(lib.bp_set_aabb(_ptr(A), _ptr(b), _ptr(m), S, m_max, _ptr(out), _stream()))
    return out


def pair_feasible(A, b, m, tol=0.01, row_begin=0, row_end=None, want_points=False, out=None, aabb=None):
    """BoundPlanner.set_intersection (BoundPlanner.py:774-787, tol from :797) for all
    pairs (i, j>i), i in [row_begin,row_end).  Returns uint32-packed bits as an
    int32 tensor [rows, ceil(S/32)]; with want_points also x [rows,S,3], a point of
    each non-empty intersection (the reference's sol_lin.x)."""
    lib = _lib.load()
    S, m_max = A.shape[0], A.shape[1]
    if row_end is None:
        row_end = S
    words = (S + 31) // 32
    if out is None:
        out = alloc_pair_buffers(S, row_end - row_begin)
    bits, work = out
    wbytes = work.numel()
    assert bits.shape == (row_end - row_begin, words)
    x = torch.zeros((row_end - row_begin, S, 3), dtype=torch.float64, device="cuda") if want_points else None
    check(lib.bp_pair_feasible(_ptr(A), _ptr(b), _ptr(m), S, m_max, float(tol), int(row_begin), int(row_end),
                               _ptr(bits), _ptr(x), _ptr(aabb), _ptr(work), wbytes, _stream()))
    if want_points:
        return bits, x
    return bits


def pair_feasible_stages(A, b, m, tol=0.01, row_begin=0, row_end=None, out=None, aabb=None):
    """Diagnostics: pair_feasible with CUDA events between its kernels; synchronises and returns
    {"aabb": ms, "filter": ms, "lp": ms} (aabb = 0 when the boxes are given)."""
    lib = _lib.load()
    S, m_max = A.shape[0], A.shape[1]
    if row_end is None:
        row_end = S
    if out is None:
        out = alloc_pair_buffers(S, row_end - row_begin)
    bits, work = out
    ms = (ctypes.c_float * 3)()
    check(lib.bp_pair_feasible_stages(_ptr(A), _ptr(b), _ptr(m), S, m_max, float(tol), int(row_begin), int(row_end),
                                      _ptr(bits), _ptr(aabb), _ptr(work), work.numel(), _stream(), ms))
    return {"aabb": float(ms[0]), "filter": float(ms[1]), "lp": float(ms[2])}


def reduce_ineqs(A, b, m):
    """reduce_ineqs (util_functions.py:82-88) for S sets: returns (A_red, b_red, m_red, keep [S,m_max] bool)."""
    lib = _lib.load()
    A = _dev(A)
    S, m_max = A.shape[0], A.shape[1]
    b = _dev(b).reshape(S, m_max)
    m = _dev(m, torch.int32).reshape(S)
    Ao = torch.empty_like(A)
    bo = torch.empty_like(b)
    mo = torch.zeros_like(m)
    keep = torch.zeros((S, m_max), dtype=torch.uint8, device="cuda")
    status = torch.zeros((S,), dtype=torch.int32, device="cuda")
    check(lib.bp_reduce_ineqs(_ptr(A), _ptr(b), _ptr(m), S, m_max, _ptr(Ao), _ptr(bo), _ptr(mo), _ptr(keep),
                              _ptr(status), _stream()))
    return Ao, bo, mo, keep.bool(), status


def rodrigues_matrix(omega, phi):
    """R = I + sin(phi) K + (1 - cos(phi)) K^2 (optimization_functions.py:83-104)."""
    k = np.array([[0.0, -omega[2], omega[1]], [omega[2], 0.0, -omega[0]], [-omega[1], omega[0], 0.0]])
    return np.eye(3) + np.sin(phi) * k + (1.0 - np.cos(phi)) * (k @ k)


def check_fit(A, b, m, pairs, l_ee, omega_normed, omega_norm, x0=None, n_samples=20, margin=0.001, active=None):
    """BoundPlanner.check_intersection (BoundPlanner.py:745-772) for P intersection sets.
    pairs [P,2] int32: set indices (i, j); returns (fits [P] bool, omega_sample [P] float, -1 where none).
    active [P] (device bool/int, optional): pairs with 0 are skipped (fits False) -- add_edges only checks the
    pairs that intersect, and that answer is already on the device."""
    lib = _lib.load()
    S, m_max = A.shape[0], A.shape[1]
    pairs = _dev(pairs, torch.int32).reshape(-1, 2)
    P = pairs.shape[0]
    ls = np.ascontiguousarray([rodrigues_matrix(omega_normed, omega_norm * k / (n_samples - 1)) @ np.asarray(l_ee, float)
                               for k in range(n_samples)])
    fits = torch.zeros((P,), dtype=torch.int32, device="cuda")
    first = torch.full((P,), -1, dtype=torch.int32, device="cuda")
    x0 = _dev(x0).reshape(P, 3) if x0 is not None else None
    if active is not None:
        active = _dev(active, torch.int32).reshape(P)
    check(lib.bp_check_fit(_ptr(A), _ptr(b), _ptr(m), S, m_max, _ptr(pairs), P, _ptr(x0), _ptr(active),
                           ls.ctypes.data_as(_dp),
                           int(n_samples), float(margin), _ptr(fits), _ptr(first), _stream()))
    if bool((fits < 0).any().item()):
        raise _lib.BpGeoError("check_fit: an intersection set has more than 48 rows")
    omega = torch.where(first >= 0, first.double() / (n_samples - 1), torch.full_like(first, -1).double())
    return fits.bool(), omega


def project_points(A, b, m, pairs, xd):
    """Projection QP of add_edges (BoundPlanner.py:842-864) for P (intersection set, point) pairs -> x [P,3]."""
    lib = _lib.load()
    S, m_max = A.shape[0], A.shape[1]
    pairs = _dev(pairs, torch.int32).reshape(-1, 2)
    P = pairs.shape[0]
    xd = _dev(xd).reshape(P, 3)
    x = torch.empty((P, 3), dtype=torch.float64, device="cuda")
    status = torch.zeros((P,), dtype=torch.int32, device="cuda")
    check(lib.bp_project_points(_ptr(A), _ptr(b), _ptr(m), S, m_max, _ptr(pairs), P, _ptr(xd), _ptr(x), _ptr(status),
                                _stream()))
    return x, status


def pairs_feasible_list(A, b, m, pairs, tol=0.01):
    """set_intersection for an explicit list of set pairs [P,2] -> (ok [P] bool, x [P,3])."""
    lib = _lib.load()
    S, m_max = A.shape[0], A.shape[1]
    pairs = _dev(pairs, torch.int32).reshape(-1, 2)
    P = pairs.shape[0]
    res = torch.zeros((P,), dtype=torch.int32, device="cuda")
    x = torch.zeros((P, 3), dtype=torch.float64, device="cuda")
    work = torch.empty((max(S, 1) * 6,), dtype=torch.float64, device="cuda")
    check(lib.bp_pairs_feasible_list(_ptr(A), _ptr(b), _ptr(m), S, m_max, float(tol), _ptr(pairs), P, _ptr(res),
                                     _ptr(x), _ptr(work), work.numel() * 8, _stream()))
    return res.bool(), x


def sets_obstacle_hits(scene, A, b, m, set_scene=None, tol=1e-3):
    """Which obstacle of its scene does each of S sets meet (bp_sets_obstacles)?  A [S,m_max,3], b [S,m_max], m [S]
    (padded rows A = 0, b = 10 allowed), set_scene [S] (scene index of every set in a scene batch; None: scene 0).
    Returns first_hit, int32 [S] on the device: the lowest obstacle index (local to the set's scene) for which
    set_intersection([A_s, b_s], [A_o, b_o], tol) (BoundPlanner.py:774-787) succeeds, -1 where none does, -2 where
    set_scene lies outside the batch.  Box or polytope scenes, single scenes and batches."""
    lib = _lib.load()
    A = _dev(A)
    S, m_max = A.shape[0], A.shape[1]
    b = _dev(b).reshape(S, m_max)
    m = _dev(m, torch.int32).reshape(S)
    if set_scene is not None:
        set_scene = _dev(set_scene, torch.int32).reshape(S)
    out = torch.empty((S,), dtype=torch.int32, device="cuda")
    work = torch.empty((max(lib.bp_sets_obstacles_workspace_bytes(S), 1),), dtype=torch.uint8, device="cuda")
    check(lib.bp_sets_obstacles(scene._h, _ptr(set_scene), _ptr(A), _ptr(b), _ptr(m), S, m_max, float(tol), _ptr(out),
                                _ptr(work), work.numel(), _stream()))
    return out


def sample_filter(scene, cand, A=None, b=None, m=None, set_off=None, item_scene=None, want_flags=False):
    """Rejection loop of plan_convex_set_path (BoundPlanner.py:459-478) for Q queries: cand [Q,C,3] candidate
    points in draw order; known sets of query q are rows set_off[q]:set_off[q+1] of (A, b, m).
    Returns first_ok [Q] int32 (index of the first accepted candidate, -1: none) and, with want_flags, flags [Q,C]
    uint8 (bit 0: in an inflated obstacle, bit 1: in a known set)."""
    lib = _lib.load()
    cand = _dev(cand)
    Q, C = cand.shape[0], cand.shape[1]
    first = torch.empty((Q,), dtype=torch.int32, device="cuda")
    flags = torch.zeros((Q, C), dtype=torch.uint8, device="cuda") if want_flags else None
    if set_off is not None:
        A, b = _dev(A), _dev(b)
        m = _dev(m, torch.int32)
        set_off = _dev(set_off, torch.int32).reshape(Q + 1)
        m_max = A.shape[1]
    else:
        A = b = m = None
        m_max = 0
    if item_scene is not None:
        item_scene = _dev(item_scene, torch.int32).reshape(Q)
    check(lib.bp_sample_filter(scene._h, _ptr(item_scene), _ptr(cand), Q, C, _ptr(A), _ptr(b), _ptr(m), m_max,
                               _ptr(set_off), _ptr(first), _ptr(flags), _stream()))
    return (first, flags) if want_flags else first


def dedupe_distance(q_new, p_new, q_nodes, p_nodes, node_off):
    """Duplicate-set test of plan_convex_set_path (BoundPlanner.py:505-512): for P new sets, the smallest
    ||Q_new - Q_v||_F + ||p_new - p_v|| over nodes node_off[i]:node_off[i+1].  Returns (dmin [P], argmin [P])."""
    lib = _lib.load()
    q_new = _dev(q_new).reshape(-1, 9)
    P = q_new.shape[0]
    p_new = _dev(p_new).reshape(P, 3)
    q_nodes = _dev(q_nodes).reshape(-1, 9)
    p_nodes = _dev(p_nodes).reshape(-1, 3)
    node_off = _dev(node_off, torch.int32).reshape(P + 1)
    dmin = torch.empty((P,), dtype=torch.float64, device="cuda")
    arg = torch.empty((P,), dtype=torch.int32, device="cuda")
    check(lib.bp_dedupe_distance(_ptr(q_new), _ptr(p_new), P, _ptr(q_nodes), _ptr(p_nodes), _ptr(node_off), _ptr(dmin),
                                 _ptr(arg), _stream()))
    return dmin, arg


def shortest_paths(node_off, edge_off, edge_dst, edge_w, src, dst, max_len=64):
    """nx.shortest_path(inter_graph, src, dst, weight="weight") (BoundPlanner.py:434) for G graphs in CSR form
    (see include/bpgeo.h).  Returns (path [G,max_len] local ids, path_len [G], cost [G])."""
    lib = _lib.load()
    node_off = _dev(node_off, torch.int32)
    G = node_off.numel() - 1
    edge_off = _dev(edge_off, torch.int32)
    edge_dst = _dev(edge_dst, torch.int32)
    edge_w = _dev(edge_w)
    src = _dev(src, torch.int32).reshape(G)
    dst = _dev(dst, torch.int32).reshape(G)
    path = torch.full((G, max_len), -1, dtype=torch.int32, device="cuda")
    plen = torch.empty((G,), dtype=torch.int32, device="cuda")
    cost = torch.empty((G,), dtype=torch.float64, device="cuda")
    check(lib.bp_shortest_paths(_ptr(node_off), _ptr(edge_off), _ptr(edge_dst), _ptr(edge_w), _ptr(src), _ptr(dst), G,
                                int(max_len), _ptr(path), _ptr(plen), _ptr(cost), _stream()))
    return path, plen, cost


def unpack_adjacency(bits, S, row_begin=0):
    """int32 words [rows, words] -> bool [rows, S]."""
    shifts = torch.arange(32, device=bits.device, dtype=torch.int32)
    b = ((bits.unsqueeze(-1) >> shifts) & 1).to(torch.bool)
    return b.reshape(bits.shape[0], -1)[:, :S]


def fk_iiwa14(q, want_pose=False, want_jacobian=False):
    """RobotModel.fk_pos / fk_pos_col / hom_transform_endeffector / jacobian_fk
    (RobotModel.py:146-231) for B configurations.  Returns (p_ee [B,3],
    p_col [B,7,3], T_ee [B,4,4] | None, jac [B,6,7] | None)."""
    lib = _lib.load()
    q = _dev(q).reshape(-1, 7)
    B = q.shape[0]
    p_ee = torch.empty((B, 3), dtype=torch.float64, device="cuda")
    p_col = torch.empty((B, 7, 3), dtype=torch.float64, device="cuda")
    T = torch.empty((B, 4, 4), dtype=torch.float64, device="cuda") if want_pose else None
    J = torch.empty((B, 6, 7), dtype=torch.float64, device="cuda") if want_jacobian else None
    check(lib.bp_fk_iiwa14(_ptr(q), B, _ptr(p_ee), _ptr(p_col), _ptr(T), _ptr(J), _stream()))
    return p_ee, p_col, T, J


def fk_kinematics(q, dq=None):
    """RobotModel.forward_kinematics (RobotModel.py:70-77) for B (q, dq) pairs: returns (T_ee [B,4,4],
    jac [B,6,7], djac [B,6,7] | None) -- hom_transform_endeffector, jacobian_fk and djacobian_fk (:233-251)."""
    lib = _lib.load()
    q = _dev(q).reshape(-1, 7)
    B = q.shape[0]
    dq = None if dq is None else _dev(dq).reshape(-1, 7)
    if dq is not None and dq.shape[0] != B:
        raise ValueError("q and dq must hold the same number of configurations")
    T = torch.empty((B, 4, 4), dtype=torch.float64, device="cuda")
    J = torch.empty((B, 6, 7), dtype=torch.float64, device="cuda")
    dJ = torch.empty((B, 6, 7), dtype=torch.float64, device="cuda") if dq is not None else None
    check(lib.bp_fk_iiwa14_kin(_ptr(q), _ptr(dq), B, _ptr(T), _ptr(J), _ptr(dJ), _stream()))
    return T, J, dJ


def debug_counters(reset=False):
    """{"shell_fallbacks": polyhedron passes redone in the per-pick form because the closest-point shell overflowed}"""
    lib = _lib.load()
    buf = (ctypes.c_ulonglong * 4)()
    check(lib.bp_debug_counters(buf, 4, int(bool(reset))))
    return {"shell_fallbacks": int(buf[0])}


def polytope_vertices(A, b, m, vmax=64):
    """compute_polytope_vertices (util_functions.py:66-79) for S polytopes {A x <= b}: returns (V [S,vmax,3],
    nv [S], status [S]); status 6 = not a polytope (unbounded / empty), 2 = more than vmax vertices."""
    lib = _lib.load()
    A = _dev(A)
    S, m_max = A.shape[0], A.shape[1]
    b = _dev(b).reshape(S, m_max)
    m = _dev(m, torch.int32).reshape(S)
    V = torch.zeros((S, vmax, 3), dtype=torch.float64, device="cuda")
    nv = torch.zeros((S,), dtype=torch.int32, device="cuda")
    status = torch.zeros((S,), dtype=torch.int32, device="cuda")
    check(lib.bp_polytope_vertices(_ptr(A), _ptr(b), _ptr(m), S, m_max, int(vmax), _ptr(V), _ptr(nv), _ptr(status),
                                   _stream()))
    return V, nv, status


def sample_filter_tables(scene, cand, A, b, m, set_begin, set_count, item_scene=None):
    """K11 over device-resident per-query tables: the known sets of query q are rows set_begin[q] ..
    set_begin[q] + set_count[q] - 1 of (A, b, m).  Returns first_ok [Q] int32 (-1: no candidate accepted)."""
    lib = _lib.load()
    cand = _dev(cand)
    Q, C = cand.shape[0], cand.shape[1]
    first = torch.empty((Q,), dtype=torch.int32, device="cuda")
    set_begin = _dev(set_begin, torch.int32).reshape(Q)
    set_count = _dev(set_count, torch.int32).reshape(Q)
    if item_scene is not None:
        item_scene = _dev(item_scene, torch.int32).reshape(Q)
    check(lib.bp_sample_filter_tables(scene._h, _ptr(item_scene), _ptr(cand), Q, C, _ptr(A), _ptr(b), _ptr(m),
                                      int(A.shape[1]), _ptr(set_begin), _ptr(set_count), _ptr(first), _stream()))
    return first


def dedupe_distance_tables(q_new, p_new, q_nodes, p_nodes, node_begin, node_count):
    """K12 over device-resident node tables (see bp_dedupe_distance_tables): (dmin [P], argmin [P])."""
    lib = _lib.load()
    q_new = _dev(q_new).reshape(-1, 9)
    P = q_new.shape[0]
    p_new = _dev(p_new).reshape(P, 3)
    node_begin = _dev(node_begin, torch.int32).reshape(P)
    node_count = _dev(node_count, torch.int32).reshape(P)
    dmin = torch.empty((P,), dtype=torch.float64, device="cuda")
    arg = torch.empty((P,), dtype=torch.int32, device="cuda")
    check(lib.bp_dedupe_distance_tables(_ptr(q_new), _ptr(p_new), P, _ptr(q_nodes), _ptr(p_nodes), _ptr(node_begin),
                                        _ptr(node_count), _ptr(dmin), _ptr(arg), _stream()))
    return dmin, arg


def make_tail(A, b, m, aabb, count, log, bits, epoch, tol, off_count=0, off_log=0, off_bits=0):
    """bp_tail descriptor over device tensors: tables A [S,m_max,3], b, m, aabb [S,6]; arrival log: count (int32,
    one element) + log [S] int64; bits [S,words] or [2,S,words] int32; epoch: int32 tensor of one element.
    count, log, epoch must be 0 at allocation."""
    S = A.shape[0]
    t = _lib.BpTail()
    t.S_glob, t.words = int(S), int(bits.shape[-1])
    t.A, t.b, t.m, t.aabb = A.data_ptr(), b.data_ptr(), m.data_ptr(), aabb.data_ptr()
    t.count, t.log, t.bits, t.epoch = count.data_ptr(), log.data_ptr(), bits.data_ptr(), epoch.data_ptr()
    t.off_count, t.off_log, t.off_bits, t.tol = int(off_count), int(off_log), int(off_bits), float(tol)
    return t


def step_begin(tail, double_buffered):
    """Start a step of a tail pipeline: clear the adjacency buffer (of the next step when double-buffered) and
    bump the epoch."""
    check(_lib.load().bp_step_begin(ctypes.byref(tail), int(bool(double_buffered)), _stream()))
