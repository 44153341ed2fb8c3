"""Synthetic scenes for tests and bench.py (host-side NumPy, deterministic).

Definitions follow SURVEY.md section 8(d) / BASELINE.md section 3:

* ``example_scene``  -- C1, the 12 boxes of boundplanner_example.py:19-87 of the
  reference (scene constants restated, not imported).
* ``random_box_scene`` -- C2/C3 style clutter: boxes with uniform centres and
  uniform edge lengths in the planner's default workspace
  (BoundPlanner.py:32-33).
* ``shelf_scene`` -- C4: lattice of thin shelf plates (thickness 0.02 like the
  example's box walls) plus random clutter.
* ``config_c3_polytope_query`` -- C3 over general convex polytopes (``random_polytope_scene``).
* ``free_points`` -- rejection sampling that mirrors the planner's test
  "max(A x - b) < 1e-3 for any inflated obstacle => in collision"
  (BoundPlanner.py:467-471).
"""
from __future__ import annotations

import numpy as np

WORKSPACE_MIN = np.array([-1.0, -1.0, 0.0])
WORKSPACE_MAX = np.array([1.0, 1.0, 1.2])


def example_scene():
    """(obstacles [12,6] as lb|ub, workspace_min, workspace_max, obs_size_increase)."""
    size, s_box, w = 0.04, 0.12, 0.02
    px, py, pz, h = 0.45, -0.48, 0.05, 0.18
    obs = [
        [px + s_box - w, py - s_box, 0.0, px + s_box, py + s_box, pz + h],
        [px - s_box, py - s_box, 0.0, px - s_box + w, py + s_box, pz + h],
        [px - s_box, py - s_box - w, 0.0, px + s_box, py - s_box, pz + h],
        [px - s_box, py + s_box, 0.0, px + s_box, py + s_box + w, pz + h],
        [0.2, -1.0, -0.1, 1.0, 1.0, 0.0],
        [-0.3, -1.0, 0.53, 0.2, -0.35, 1.0],
        [-0.2, -1.0, 0.0, -0.14, 1.0, 1.0],
        [-1.0, 0.38, 0.0, 1.0, 0.5, 1.0],
        [0.4, -0.05, 0.0, 0.5, 0.05, 0.15],
        [0.1, -0.55, 0.0, 0.3, -0.35, 0.07],
        [0.5 - size, -0.2 - size, 0.03 - size, 0.5 + size, -0.2 + size, 0.03 + size],
        [0.4 - size, 0.3 - size, 0.03 - size, 0.4 + size, 0.3 + size, 0.03 + size],
    ]
    return (np.array(obs), np.array([-0.14, -1.0, 0.0]), np.array([1.0, 0.38, 1.0]), 0.08)


def random_box_scene(n_obs, rng, edge_lo=0.02, edge_hi=0.08,
                     ws_min=WORKSPACE_MIN, ws_max=WORKSPACE_MAX):
    centres = rng.uniform(ws_min, ws_max, (n_obs, 3))
    edges = rng.uniform(edge_lo, edge_hi, (n_obs, 3))
    return np.hstack((centres - 0.5 * edges, centres + 0.5 * edges))


def shelf_scene(n_obs, rng, ws_min=WORKSPACE_MIN, ws_max=WORKSPACE_MAX, thickness=0.02):
    """About one third shelf plates on a lattice, the rest clutter boxes U[0.01,0.05]."""
    plates = []
    nx, ny, nz = 12, 12, 8
    xs = np.linspace(ws_min[0], ws_max[0], nx + 1)
    ys = np.linspace(ws_min[1], ws_max[1], ny + 1)
    zs = np.linspace(ws_min[2], ws_max[2], nz + 1)
    n_plates = n_obs // 3
    k = 0
    # horizontal plates: one per (x cell, y cell, z level), shrunk so that cells connect
    for iz in range(1, nz):
        for ix in range(nx):
            for iy in range(ny):
                if k >= n_plates:
                    break
                if (ix + iy + iz) % 2 == 0:
                    continue
                lo = [xs[ix] + 0.03, ys[iy] + 0.03, zs[iz] - thickness / 2]
                hi = [xs[ix + 1] - 0.03, ys[iy + 1] - 0.03, zs[iz] + thickness / 2]
                plates.append(lo + hi)
                k += 1
    plates = np.array(plates).reshape(-1, 6)
    clutter = random_box_scene(n_obs - plates.shape[0], rng, 0.01, 0.05, ws_min, ws_max)
    return np.vstack((plates, clutter))


def in_collision(points, obstacles, inflate, margin=1e-3):
    """True where a point is inside (or within ``margin`` of) any inflated box."""
    lb = obstacles[:, :3] - inflate
    ub = obstacles[:, 3:] + inflate
    p = points[:, None, :]
    viol = np.maximum(p - ub[None], lb[None] - p).max(axis=2)     # max(A x - b)
    return (viol < margin).any(axis=1)


def free_points(n, obstacles, inflate, rng, ws_min=WORKSPACE_MIN, ws_max=WORKSPACE_MAX):
    out = np.empty((0, 3))
    while out.shape[0] < n:
        cand = rng.uniform(ws_min, ws_max, (2 * n, 3))
        cand = cand[~in_collision(cand, obstacles, inflate)]
        out = np.vstack((out, cand))
    return np.ascontiguousarray(out[:n])


def config_c2(n_obs=1000, n_seeds=256, seed=0):
    """C2 of BASELINE.json: 1k random boxes, 256 free seeds, default workspace."""
    rng = np.random.default_rng(seed)
    inflate = 0.01
    obstacles = random_box_scene(n_obs, rng)
    seeds = free_points(n_seeds, obstacles, inflate, rng)
    return obstacles, inflate, seeds, WORKSPACE_MIN.copy(), WORKSPACE_MAX.copy()


def config_c4(n_obs=10000, n_seeds=2048, seed=2):
    rng = np.random.default_rng(seed)
    inflate = 0.0
    obstacles = shelf_scene(n_obs, rng)
    seeds = free_points(n_seeds, obstacles, inflate, rng)
    return obstacles, inflate, seeds, WORKSPACE_MIN.copy(), WORKSPACE_MAX.copy()


def config_c3_query(i, n_obs=200):
    """Query i of C3: 200 boxes (edge U[0.05,0.2], inflate 0.01), free start/end at least 0.3 m apart."""
    rng = np.random.default_rng(1000 + i)
    inflate = 0.01
    obstacles = random_box_scene(n_obs, rng, 0.05, 0.2)
    while True:
        pts = free_points(2, obstacles, inflate + 0.06, rng, WORKSPACE_MIN + 0.1, WORKSPACE_MAX - 0.1)
        if np.linalg.norm(pts[0] - pts[1]) >= 0.3:
            break
    return obstacles, inflate, pts[0], pts[1], WORKSPACE_MIN.copy(), WORKSPACE_MAX.copy()


def config_c3_polytope_query(i, n_obs=200):
    """Query i of C3 over general convex polytopes: 200 obstacles of random_polytope_scene (boxes with edges
    U[0.05,0.2], as C3's, cut by up to 9 random planes; taken as already inflated), obs_size_increase 0.01, free
    start/end (max(A x - b) >= 0.06 for every obstacle) at least 0.3 m apart.
    Returns (obs_sets, obs_points_sets, inflate, start, end, workspace_min, workspace_max)."""
    rng = np.random.default_rng(2000 + i)
    inflate = 0.01
    obs_sets, obs_points = random_polytope_scene(n_obs, rng, 0.05, 0.2)
    while True:
        pts = polytope_free_points(2, obs_sets, 0.06, rng, WORKSPACE_MIN + 0.1, WORKSPACE_MAX - 0.1)
        if np.linalg.norm(pts[0] - pts[1]) >= 0.3:
            break
    return obs_sets, obs_points, inflate, pts[0], pts[1], WORKSPACE_MIN.copy(), WORKSPACE_MAX.copy()


def random_polytope_scene(n_obs, rng, size_lo=0.03, size_hi=0.12, max_rows=15, ws_min=WORKSPACE_MIN, ws_max=WORKSPACE_MAX):
    """n_obs random convex polytope obstacles in the layout ConvexSetFinder takes (what add_obstacle_reps would
    build for non-box obstacles): obs_sets = [[A (15x3, zero-padded), b (15, padded with 10)], ...] with unit
    normals, obs_points_sets = [vertices (V x 3), ...].  Each polytope is a random box cut by random planes."""
    from scipy.spatial import HalfspaceIntersection

    obs_sets, obs_points = [], []
    box = np.concatenate((np.eye(3), -np.eye(3)))
    while len(obs_sets) < n_obs:
        c = rng.uniform(ws_min, ws_max)
        half = 0.5 * rng.uniform(size_lo, size_hi, 3)
        n_cut = int(rng.integers(0, max_rows - 6 + 1))
        cuts = rng.normal(size=(n_cut, 3))
        cuts /= np.linalg.norm(cuts, axis=1)[:, None]
        A = np.vstack((box, cuts))
        b = np.concatenate((c + half, -(c - half), cuts @ c + rng.uniform(0.3, 0.9, n_cut) * (np.abs(cuts) @ half)))
        hs = HalfspaceIntersection(np.hstack((A, -b[:, None])), c)
        verts = hs.intersections
        # keep the rows that support a facet (>= 3 vertices on the plane), like the reference's reduced sets
        on = np.abs(verts @ A.T - b) < 1e-9
        keep = on.sum(axis=0) >= 3
        A, b = A[keep], b[keep]
        a_pad = np.zeros((max_rows, 3))
        b_pad = np.full(max_rows, 10.0)
        a_pad[: A.shape[0]], b_pad[: A.shape[0]] = A, b
        obs_sets.append([a_pad, b_pad])
        obs_points.append(np.ascontiguousarray(verts))
    return obs_sets, obs_points


def polytope_free_points(n, obs_sets, margin, rng, ws_min=WORKSPACE_MIN, ws_max=WORKSPACE_MAX):
    """Uniform points with max(A x - b) >= margin for every polytope."""
    A = np.stack([s[0] for s in obs_sets])
    b = np.stack([s[1] for s in obs_sets])
    out = np.empty((0, 3))
    while out.shape[0] < n:
        cand = rng.uniform(ws_min, ws_max, (2 * n, 3))
        viol = np.einsum("nrk,ck->cnr", A, cand) - b[None]
        viol[:, np.linalg.norm(A, axis=2) == 0] = -np.inf
        cand = cand[(viol.max(axis=2) >= margin).all(axis=1)]
        out = np.vstack((out, cand))
    return np.ascontiguousarray(out[:n])


def moved_obstacles(obstacles, rng, obs_points=None, move_frac=0.25, max_shift=0.05, n_add=4, n_remove=4):
    """One step of moving obstacles (an MPC loop's changing scene), seeded by ``rng``: a fraction ``move_frac`` of
    the obstacles is translated by U[-max_shift, max_shift]^3 each, ``n_remove`` are removed and ``n_add`` new ones
    (C3-sized: edges U[0.05, 0.2]) are appended.
    Boxes: ``obstacles`` [N,6] -> [N',6].  Polytopes: ``obstacles`` = obs_sets and ``obs_points`` = obs_points_sets
    (or None) -> (obs_sets', obs_points_sets' or None); a translation by t sets b += A t and vertices += t (padded rows,
    A = 0, keep b = 10)."""
    poly = not isinstance(obstacles, np.ndarray)
    n = len(obstacles)
    moved = rng.random(n) < move_frac
    shift = rng.uniform(-max_shift, max_shift, (n, 3))
    keep = np.sort(rng.permutation(n)[: max(n - n_remove, 0)])
    if not poly:
        out = obstacles + np.where(moved[:, None], np.hstack((shift, shift)), 0.0)
        return np.vstack((out[keep], random_box_scene(n_add, rng, 0.05, 0.2)))
    sets, pts = [], [] if obs_points is not None else None
    for j in keep:
        A, b = np.asarray(obstacles[j][0], float), np.asarray(obstacles[j][1], float)
        t = shift[j] if moved[j] else np.zeros(3)
        sets.append([A.copy(), b + A @ t])
        if pts is not None:
            pts.append(np.asarray(obs_points[j], float) + t)
    new_sets, new_pts = random_polytope_scene(n_add, rng, 0.05, 0.2)
    sets.extend(new_sets)
    if pts is not None:
        pts.extend(new_pts)
    return sets, pts
