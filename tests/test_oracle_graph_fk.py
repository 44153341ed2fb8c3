"""CPU: pin the set-graph oracle (the reference's own linprog call) and the FK oracle."""
import os

import numpy as np
import pytest

from oracle import fk_iiwa14 as ofk
from oracle.set_graph import adjacency, intersection_margin, set_intersection

BOX = np.vstack((np.eye(3), -np.eye(3)))
# the reference's RobotModel directory, in a checkout named by BOUNDPLANNER_REFERENCE (not part of this repository)
REF_MODEL = os.path.join(os.environ.get("BOUNDPLANNER_REFERENCE", ""), "bound_planner", "RobotModel")
NO_REF = "reference checkout not available (set BOUNDPLANNER_REFERENCE)"


def _box(lb, ub):
    return [BOX.copy(), np.concatenate((np.asarray(ub, float), -np.asarray(lb, float)))]


def test_boxes_intersect_iff_overlap_exceeds_two_tol():
    a = _box([0, 0, 0], [1, 1, 1])
    assert set_intersection(a, _box([0.97, 0, 0], [2, 1, 1]), tol=0.01)[2]
    assert not set_intersection(a, _box([0.99, 0, 0], [2, 1, 1]), tol=0.01)[2]
    assert set_intersection(a, _box([0.99, 0, 0], [2, 1, 1]), tol=0.0)[2]
    assert abs(intersection_margin(a, _box([0.97, 0, 0], [2, 1, 1]), 0.01) + 0.005) < 1e-9
    assert abs(intersection_margin(a, _box([1.5, 0, 0], [2, 1, 1]), 0.01) - 0.26) < 1e-9


def test_margin_sign_matches_highs_on_random_pairs():
    rng = np.random.default_rng(21)
    sets = []
    for _ in range(30):
        k = rng.integers(3, 14)
        c = rng.uniform(-0.6, 0.6, 3)
        An = rng.normal(size=(k, 3))
        An /= np.linalg.norm(An, axis=1)[:, None]
        sets.append([np.vstack((BOX, An)), np.concatenate((np.array([1, 1, 1.2, 1, 1, 0.0]),
                                                           An @ c + rng.uniform(0.05, 0.5, k)))])
    adj = adjacency(sets, 0.01)
    assert np.array_equal(adj, adj.T) and not adj.diagonal().any()
    for i in range(30):
        for j in range(i):
            mg = intersection_margin(sets[i], sets[j], 0.01)
            if abs(mg) > 1e-6:
                assert adj[i, j] == (mg <= 0)
    x, inter, ok = set_intersection(sets[0], sets[0], 0.01)
    assert ok and inter[0].shape[0] == 2 * sets[0][0].shape[0] and np.all(inter[0] @ x <= inter[1] - 0.01 + 1e-7)


def test_fk_anchors_from_urdf():
    """Anchors derived from iiwa.urdf (SURVEY.md 8c)."""
    assert np.abs(ofk.fk_pos(np.zeros(7)) - [0, 0, 1.4696]).max() < 1e-12
    assert np.abs(ofk.fk_pos_col_all(np.zeros(7))[:, 2] - [0.5925, 0.78, 0.9925, 1.18, 1.2596, 1.08, 1.3896]).max() < 1e-12
    assert np.abs(ofk.fk_pos(np.array([0, 0, 0, -np.pi / 2, 0, np.pi / 2, 0])) - [0.4, 0, 0.4904]).max() < 1e-12
    assert np.abs(ofk.fk_pos(np.array([0.1, -0.2, 0.3, -0.4, 0.5, -0.6, 0.7]))
                  - [-0.075099282696, -0.048154013641, 1.429984381972]).max() < 1e-11


def test_fk_jacobian_finite_differences():
    rng = np.random.default_rng(3)
    q = rng.uniform(ofk.Q_LOWER, ofk.Q_UPPER)
    J = ofk.jacobian_fk(q)
    for k in range(7):
        dq = np.zeros(7)
        dq[k] = 1e-6
        num = (ofk.fk_pos(q + dq) - ofk.fk_pos(q - dq)) / 2e-6
        assert np.abs(num - J[:3, k]).max() < 1e-8
    h = ofk.hom_transform_endeffector(q)
    assert np.abs(h[:3, :3] @ h[:3, :3].T - np.eye(3)).max() < 1e-12 and abs(np.linalg.det(h[:3, :3]) - 1) < 1e-12
    assert np.abs(ofk.fk(q)[:3] - h[:3, 3]).max() == 0


def test_fk_golden_fixture():
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "fk_golden.npz"))
    for i, q in enumerate(g["q"]):
        assert np.abs(ofk.fk_pos(q) - g["p_ee"][i]).max() < 1e-12
        assert np.abs(ofk.fk_pos_col_all(q) - g["p_col"][i]).max() < 1e-12
        assert np.abs(ofk.hom_transform_endeffector(q) - g["T_ee"][i]).max() < 1e-12


@pytest.mark.skipif(not os.environ.get("BOUNDPLANNER_REFERENCE") or
                    not os.path.exists(os.path.join(REF_MODEL, "iiwa.urdf")), reason=NO_REF)
def test_fk_constants_equal_the_reference_urdf():
    """Re-read the joint origins straight from the reference's URDF."""
    import xml.etree.ElementTree as ET

    root = ET.parse(os.path.join(REF_MODEL, "iiwa.urdf")).getroot()
    joints = {j.get("name"): j for j in root.findall("joint")}
    for k in range(7):
        o = joints[f"joint_{k + 1}"].find("origin")
        assert np.allclose([float(v) for v in o.get("xyz").split()], ofk.JOINT_ORIGINS[k][0], atol=0)
        assert np.allclose([float(v) for v in o.get("rpy").split()], ofk.JOINT_ORIGINS[k][1], atol=0)
        lim = joints[f"joint_{k + 1}"].find("limit")
        assert float(lim.get("upper")) == ofk.Q_UPPER[k] and float(lim.get("lower")) == ofk.Q_LOWER[k]
    for name, spec in (("joint_ee", ofk.EE), ("link4_col", ofk.LINK4_COL), ("end_effector_col", ofk.EE_COL)):
        o = joints[name].find("origin")
        assert [float(v) for v in o.get("xyz").split()] == list(spec[1])
        assert [float(v) for v in o.get("rpy").split()] == list(spec[2])
        assert joints[name].find("parent").get("link") == {4: "link_4", 7: "link_7"}[spec[0]]


def test_reduce_ineqs_oracle_known_answers():
    """oracle/reduce_ineqs.py (restating cddlib's redundancy removal, util_functions.py:82-88)."""
    from oracle.reduce_ineqs import reduce_ineqs, redundant_row_mask

    A = np.vstack((BOX, [[1, 1, 1], [1, 1, 1], [1, 0, 0], [1, 0, 0]]))
    b = np.concatenate((np.ones(6), [2.5, 3.0, 5.0, 1.0]))
    red = redundant_row_mask(A, b)
    # cut (2.5) kept; vertex-touching plane (3.0), far plane (5.0) and the LATER duplicate of the x face removed
    assert red.tolist() == [False] * 6 + [False, True, True, True]
    Ar, br = reduce_ineqs(A, b)
    assert np.array_equal(Ar, A[:7]) and np.array_equal(br, b[:7])
    # zero (padding) rows are redundant
    Ap = np.vstack((BOX, np.zeros((3, 3))))
    bp_ = np.concatenate((np.ones(6), 10 * np.ones(3)))
    assert redundant_row_mask(Ap, bp_).tolist() == [False] * 6 + [True] * 3


def test_fk_oracle_pinned_to_reference_casadi_blobs():
    """tests/golden/fk_reference_blobs.npz = the reference's serialized CasADi FK functions evaluated
    by oracle/casadi_blob.py (see tests/golden/make_golden.py)."""
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "fk_reference_blobs.npz"))
    for i, q in enumerate(g["q"]):
        assert np.abs(ofk.fk_pos(q) - g["fk_pos"][i]).max() < 1e-12
        assert np.abs(ofk.fk_pos_col_all(q)[:6] - g["fk_pos_col"][i]).max() < 1e-12     # no fk_pos_col_6.ca exists
        assert np.abs(ofk.hom_transform_endeffector(q) - g["hom_trans"][i]).max() < 1e-12
        assert np.abs(ofk.jacobian_fk(q) - g["jacobian"][i]).max() < 1e-12


@pytest.mark.skipif(not os.environ.get("BOUNDPLANNER_REFERENCE") or
                    not os.path.exists(os.path.join(REF_MODEL, "fk_pos.ca")), reason=NO_REF)
def test_casadi_blob_decoder_reproduces_committed_golden():
    from oracle.casadi_blob import SXFunctionBlob

    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "fk_reference_blobs.npz"))
    f_pos, f_c5, f_jac = (SXFunctionBlob(os.path.join(REF_MODEL, f)) for f in ("fk_pos.ca", "fk_pos_col_5.ca", "jacobian.ca"))
    assert f_pos.name_in == ["i0"] and f_pos.sp_in[0][:2] == (7, 1) and f_jac.sp_out[0][:2] == (6, 7)
    for i in (0, 1, 17, 63):
        q = g["q"][i]
        assert np.array_equal(f_pos(q).ravel(), g["fk_pos"][i])
        assert np.array_equal(f_c5(q).ravel(), g["fk_pos_col"][i][5])
        assert np.array_equal(f_jac(q), g["jacobian"][i])


def test_planner_loop_tests_oracle_known_answers():
    """oracle.planner_graph restatements of the planner's rejection / duplicate / shortest-path steps
    (BoundPlanner.py:459-478, :505-512, :434)."""
    from oracle.planner_graph import dedupe_distance, first_free_sample, sample_flags, shortest_path

    box = np.vstack((np.eye(3), -np.eye(3)))
    obs = [[np.vstack((box, np.zeros((9, 3)))), np.concatenate(([0.2, 0.2, 0.2, 0.2, 0.2, 0.2], 10 * np.ones(9)))]]
    node = [[box, np.array([1.0, 1.0, 1.0, -0.6, 1.0, 1.0])]]                    # 0.6 <= x <= 1
    assert sample_flags(obs, node, np.zeros(3)) == (True, False)
    assert sample_flags(obs, node, np.array([0.8, 0, 0])) == (False, True)
    assert sample_flags(obs, node, np.array([0.2005, 0, 0])) == (True, False)    # max(Ax - b) = 5e-4 < 1e-3: still "in"
    assert sample_flags(obs, node, np.array([0.202, 0, 0])) == (False, False)
    cands = np.array([[0, 0, 0], [0.8, 0, 0], [0.4, 0, 0], [0.5, 0, 0]])
    assert first_free_sample(obs, node, cands) == 2
    assert first_free_sample(obs, node, cands[:2]) == -1
    q, p = np.eye(3), np.zeros(3)
    assert dedupe_distance(q, p, []) == np.inf
    assert abs(dedupe_distance(q, p, [(2 * np.eye(3), np.ones(3)), (np.eye(3), np.array([0.003, 0.004, 0]))]) - 0.005) < 1e-15
    path, cost = shortest_path(3, [(0, 2, 0.4), (2, 1, 0.3), (0, 1, 0.9)], 0, 1)
    assert path == [0, 2, 1] and abs(cost - 0.7) < 1e-15
    assert shortest_path(2, [], 0, 1) == (None, np.inf)
