"""Optional TRUE-reference hook (SURVEY 8c, last row): when the reference's own dependencies import
(casadi + cvxpy/clarabel + pycddlib + pinocchio) and the reference tree is present, run the reference's
ConvexSetFinder / set_intersection / RobotModel themselves and compare the oracle with them.  In the build
container and on the GPU box none of them is installed and there is no network, so these tests SKIP with an
explicit "true reference unavailable" reason -- parity of the OSQP / qpOASES / Clarabel / cddlib rows stays
unpinned (oracle/__init__.py), the HiGHS and FK rows are pinned by other tests."""
import importlib
import os
import sys

import numpy as np
import pytest

REF = os.environ.get("BOUNDPLANNER_REFERENCE", "")     # a checkout of the reference, not part of this repository
NEEDED = ("casadi", "cvxpy", "cdd", "pinocchio")


def _reference():
    missing = []
    for name in NEEDED:
        try:
            importlib.import_module(name)
        except Exception:  # noqa: BLE001
            missing.append(name)
    if missing or not REF or not os.path.isdir(os.path.join(REF, "bound_planner")):
        pytest.skip("true reference unavailable: " + (", ".join(missing) + " not importable" if missing
                                                      else "set BOUNDPLANNER_REFERENCE to a checkout of it"))
    if REF not in sys.path:
        sys.path.insert(0, REF)
    os.chdir(REF)                       # CA_SAVE_PATH is relative (RobotModel.py:9)
    return importlib.import_module("bound_planner")


def test_reference_convex_set_finder_matches_oracle():
    _reference()
    from bound_planner.BoundPlanner.ConvexSetFinder import ConvexSetFinder as RefFinder

    from boundplanner_b200 import scenes
    from oracle.convex_set_finder import ConvexSetFinder as OracleFinder
    from oracle.obstacles import obstacle_reps

    boxes, ws_min, ws_max, inflate = scenes.example_scene()
    obs_sets, pts, _ = obstacle_reps(boxes, inflate)
    ref = RefFinder(obs_sets, pts, list(ws_max), list(ws_min))
    ora = OracleFinder(obs_sets, pts, list(ws_max), list(ws_min))
    for p in (np.array([0.3, 0.0, 0.7]), np.array([0.45, -0.5, 0.2])):
        A, b, Q, c = ref.find_set_around_point(p, fixed_mid=True)
        Ao, bo, Qo, co = ora.find_set_around_point(p, fixed_mid=True)
        assert np.asarray(A).shape == Ao.shape
        # bounded by the reference's solver tolerances (OSQP 1e-6, Clarabel ~1e-8)
        assert np.abs(np.asarray(A) - Ao).max() < 1e-4 and np.abs(np.asarray(b) - bo).max() < 1e-4
        assert np.abs(np.asarray(Q) - Qo).max() <= 1e-3 * np.abs(Qo).max()


def test_reference_robot_model_matches_oracle():
    _reference()
    from bound_planner.RobotModel import RobotModel as RefModel

    from oracle import fk_iiwa14 as ofk

    model = RefModel()
    rng = np.random.default_rng(3)
    for _ in range(8):
        q = rng.uniform(ofk.Q_LOWER, ofk.Q_UPPER)
        dq = rng.uniform(-1, 1, 7)
        assert np.abs(model.fk_pos(q) - ofk.fk_pos(q)).max() < 1e-9
        assert np.abs(model.hom_transform_endeffector(q) - ofk.hom_transform_endeffector(q)).max() < 1e-9
        assert np.abs(model.jacobian_fk(q) - ofk.jacobian_fk(q)).max() < 1e-9
        # records what Pinocchio's getFrameJacobianTimeVariation returns after the reference's call sequence
        # (RobotModel.py:233-251); the oracle is the time derivative of the Jacobian
        assert np.abs(model.djacobian_fk(q, dq) - ofk.djacobian_fk(q, dq)).max() < 1e-9


def test_reference_set_intersection_is_the_oracle_call():
    _reference()
    from bound_planner.BoundPlanner.BoundPlanner import BoundPlanner as RefPlanner

    from oracle.set_graph import set_intersection

    box = np.vstack((np.eye(3), -np.eye(3)))
    s1 = [box, np.array([1, 1, 1, 0, 0, 0.0])]
    s2 = [box, np.array([1.5, 1.5, 1.5, -0.5, -0.5, -0.5])]
    x, inter, ok = RefPlanner.set_intersection(None, s1, s2, tol=0.01)
    xo, intero, oko = set_intersection(s1, s2, tol=0.01)
    assert bool(ok) == bool(oko) and np.array_equal(inter[0], intero[0])
