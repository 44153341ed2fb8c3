"""Generates the committed golden fixtures under tests/golden/.

  python tests/golden/make_golden.py

fk_golden.npz       iiwa14 FK at fixed configurations.  Source: the ORACLE
                    (oracle/fk_iiwa14.py, chain constants of the reference's
                    iiwa.urdf).  The reference's own numeric FK needs pinocchio,
                    which is not installable here; the anchors of SURVEY.md 8c
                    are asserted separately in tests/test_oracle_graph_fk.py.
fk_reference_blobs.npz  The reference's OWN serialized CasADi functions (bound_planner/RobotModel/
                    fk_pos.ca, fk_pos_col_{0..5}.ca, hom_trans.ca, jacobian.ca -- what RobotModel.py:158,179,
                    209,229 load) evaluated at 64 configurations by oracle/casadi_blob.py (a CasADi-free
                    decoder + SX virtual machine); djacobian = the directional derivative of jacobian.ca
                    along dq (forward-mode AD through the same program).  Reference-generated golden vectors: they pin the FK oracle
                    and the FK kernel.  Needs a checkout of the reference named by
                    BOUNDPLANNER_REFERENCE.
c1_sets_golden.npz  The first two convex sets the reference's example plan builds
                    (boundplanner_example.py:89-92 -> BoundPlanner.py:278-294,
                    :381-389) as computed by the ORACLE; lets the GPU box check
                    the kernels without re-running the (slow) oracle and guards
                    the oracle itself against regressions.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from boundplanner_b200 import scenes  # noqa: E402
from oracle import fk_iiwa14 as ofk  # noqa: E402
from oracle.convex_set_finder import ConvexSetFinder  # noqa: E402
from oracle.obstacles import obstacle_reps  # noqa: E402


def main():
    rng = np.random.default_rng(1234)
    q = rng.uniform(ofk.Q_LOWER, ofk.Q_UPPER, (32, 7))
    q[0] = 0.0
    q[1] = [0, 0, 0, -np.pi / 2, 0, np.pi / 2, 0]
    q[2] = [0.1, -0.2, 0.3, -0.4, 0.5, -0.6, 0.7]
    np.savez(os.path.join(HERE, "fk_golden.npz"), q=q,
             p_ee=np.array([ofk.fk_pos(x) for x in q]),
             p_col=np.array([ofk.fk_pos_col_all(x) for x in q]),
             T_ee=np.array([ofk.hom_transform_endeffector(x) for x in q]),
             jac=np.array([ofk.jacobian_fk(x) for x in q]))

    ref_dir = os.path.join(os.environ.get("BOUNDPLANNER_REFERENCE", ""), "bound_planner", "RobotModel", "")
    if os.environ.get("BOUNDPLANNER_REFERENCE") and os.path.isdir(ref_dir):
        from oracle.casadi_blob import SXFunctionBlob

        qg = rng.uniform(ofk.Q_LOWER, ofk.Q_UPPER, (64, 7))
        qg[0] = 0.0
        qg[1] = [0, 0, 0, -np.pi / 2, 0, np.pi / 2, 0]
        f_pos = SXFunctionBlob(ref_dir + "fk_pos.ca")
        f_col = [SXFunctionBlob(ref_dir + f"fk_pos_col_{i}.ca") for i in range(6)]
        f_hom = SXFunctionBlob(ref_dir + "hom_trans.ca")
        f_jac = SXFunctionBlob(ref_dir + "jacobian.ca")
        # djacobian_fk (RobotModel.py:233-251): the reference ships no djacobian.ca; the golden value is the exact
        # directional derivative (forward-mode AD through the SX program) of its own jacobian.ca along dq
        dqg = np.random.default_rng(4321).uniform(-2.0, 2.0, (64, 7))
        dqg[0] = 0.0
        djac = np.array([f_jac.jvp([x], [v])[1] for x, v in zip(qg, dqg)])
        np.savez(os.path.join(HERE, "fk_reference_blobs.npz"), q=qg, dq=dqg, djacobian=djac,
                 fk_pos=np.array([f_pos(x).ravel() for x in qg]),
                 fk_pos_col=np.array([[f(x).ravel() for f in f_col] for x in qg]),
                 hom_trans=np.array([f_hom(x) for x in qg]),
                 jacobian=np.array([f_jac(x) for x in qg]))
        print("wrote fk_reference_blobs.npz from the reference's .ca files")

    boxes, ws_min, ws_max, inflate = scenes.example_scene()
    obs_sets, pts, _ = obstacle_reps(boxes, inflate)
    f = ConvexSetFinder(obs_sets, pts, ws_max, ws_min)
    p0 = np.array([0.3, 0.0, 0.7])
    p1 = np.array([0.45, -0.5, 0.2])
    l_ee = np.array([0.0, 0.0, 0.05])
    A0, b0, Q0, c0 = f.find_set_around_point(p0, fixed_mid=True)
    it0 = f.last_iters
    A1, b1, Q1, c1, coll = f.find_set_collision_avoidance(p1, p1 + l_ee, True)
    np.savez(os.path.join(HERE, "c1_sets_golden.npz"), p0=p0, p1=p1, l_ee=l_ee, A0=A0, b0=b0, Q0=Q0, c0=c0,
             iters0=it0, A1=A1, b1=b1, Q1=Q1, c1=c1, collision1=coll)
    print("wrote fk_golden.npz, c1_sets_golden.npz")


if __name__ == "__main__":
    main()
