"""The geometry BoundMPC evaluates every step, in one device-resident batch.

Replaces the block at bound_planner/BoundMPC/BoundMPC.py:480-496 of the reference:

    p_list   = [robot_model.fk_pos_col(q0, i) for i in range(6)]
    p_list_f = [robot_model.fk_pos_col(qf, i) for i in range(6)]
    for i, (pl, pf) in enumerate(zip(p_list, p_list_f)):
        a_c, b_c, _ = planner.set_finder.find_set_collision_avoidance(pl, pf, limit_space=True, e_max=0.7)
        set_joints.append([a_c, b_c - joint_sizes[i]])
    sets_normed = normalize_set_size(set_joints, 15)

i.e. 12 forward-kinematics evaluations and 6 line sets: here one FK launch for (q0, qf), one line-set
launch for the 6 segments (the FK output feeds it on the device) and one copy back.  Works for a
batch of T (q0, qf) pairs (horizon sweeps / many robots) as well.
"""
from __future__ import annotations

import numpy as np
import torch

from . import geometry as geo

COL_JOINT_SIZES = (0.09, 0.12, 0.09, 0.10, 0.07, 0.09, 0.075)      # RobotModel.py:37 (iiwa14)


def collision_sets(scene, q0, qf, ws_min, ws_max, e_max=0.7, n_points=6, max_set_size=15, robot_scene=None):
    """q0, qf: [7] or [T,7].  Returns (a_set_joints [T,6,15,3], b_set_joints [T,6,15], collision [T,6]) as
    NumPy arrays, padded like normalize_set_size(set_joints, 15) with b already reduced by the joint sizes.
    robot_scene [T]: ``scene`` is a scene batch (SceneBatch / PolytopeSceneBatch) and robot t's segments are built
    against its scene robot_scene[t] (a fleet of robots in a few shared cells); without it, ``scene`` is one scene."""
    q0 = np.asarray(q0, float).reshape(-1, 7)
    qf = np.asarray(qf, float).reshape(-1, 7)
    T = q0.shape[0]
    item_scene = None
    if robot_scene is not None:
        robot_scene = np.asarray(robot_scene).reshape(-1)
        if robot_scene.shape[0] != T:
            raise ValueError(f"robot_scene has {robot_scene.shape[0]} entries for {T} robots")
        item_scene = np.repeat(robot_scene.astype(np.int32), n_points)
    q = torch.as_tensor(np.concatenate((q0, qf))).cuda()
    _, p_col, _, _ = geo.fk_iiwa14(q)                                  # [2T,7,3]
    pl = p_col[:T, :n_points].reshape(-1, 3)                           # fk_pos_col(q0, i), i < 6
    pf = p_col[T:, :n_points].reshape(-1, 3)
    out = geo.build_sets_line(scene, pl, pf, ws_min, ws_max, compute_ellipsoid=False, limit_space=True, e_max=e_max,
                              m_max=max_set_size, item_scene=item_scene)
    sizes = torch.as_tensor(COL_JOINT_SIZES[:n_points], dtype=torch.float64, device="cuda").repeat(T)
    rows = torch.arange(max_set_size, device="cuda").unsqueeze(0) < out.m.unsqueeze(1)
    b = torch.where(rows, out.b - sizes.unsqueeze(1), out.b)           # b_c - joint_sizes[i]; padding stays 10
    status = out.status.cpu().numpy()
    if (status != 0).any():
        raise ValueError(f"a joint set needs more than {max_set_size} rows (the reference's normalize_set_size "
                         "would leave it ragged)")
    return (out.A.cpu().numpy().reshape(T, n_points, max_set_size, 3), b.cpu().numpy().reshape(T, n_points, max_set_size),
            out.collision.cpu().numpy().reshape(T, n_points).astype(bool))
