"""Set-intersection LP (K6) and fit-check LP (K9) at the tolerance boundary, against exact rational answers.

Every edge of the set graph comes from one decision: do two sets, each shrunk by tol, share a point?  The pairs
here are built so that the answer is decided exactly, in rational arithmetic on the fp64 values the kernels see
(the offsets c = fl(b - tol) included):

* face to face: row 0 of set 2 is the bitwise negation of row 0 of set 1 and every other row is slack on a wide
  patch of the contact plane, so the pair intersects iff c1 + c2 > 0;
* vertex to face: set 1 is a pyramid (or a cone, which is unbounded); its shrunk apex, by Cramer's rule from the
  three apex rows, must strictly satisfy the contact row of set 2, whose other rows are slack there;
* closed forms: containment (intersects), a set thinner than 2 tol (its shrunk set is empty), a slab of two rows.

Every case gets a random rotation (or a signed axis permutation) and translation, per-row scaling in [0.1, 10],
row permutations that put the deciding rows at indices >= 32 and >= 64 of the stacked pair, redundant far rows
that bring m1 + m2 into each of the three row forms of the warp LP (1, 2 or 3 rows per lane), and both pair
orders.  Margins (c units) of +-1e-3 ... +-1e-9 are asserted; +-1e-10 and 0 run, and there only a point that comes
with "intersects" is checked.  The CPU tests pin the thread-serial specification (bp_lp.cuh) and the reference
itself (against HiGHS); the GPU tests pin pair_feasible (k_pair_lp with the box filter and the margin pre-test),
pairs_feasible_list (k_pair_list), set_aabb (cta_set_aabb) and check_fit (k_fit_check + k_fit_finish).
"""
import ctypes
import itertools
from fractions import Fraction as Fr

import numpy as np
import pytest
from scipy.spatial.transform import Rotation

TOL = 0.01
ASSERTED = (1e-3, 1e-6, 1e-8, 1e-9)
RECORDED = (1e-10, 0.0)
MARGINS = [s * d for d in ASSERTED for s in (1.0, -1.0)] + [1e-10, -1e-10, 0.0]
FORMS = {1: (6, 32), 2: (33, 64), 3: (65, 96)}        # rows of the stacked LP per row form (rows per lane)
M_MAX = 48                                              # BP_MAX_ROWS
AABB_EPS = 1e-9                                         # BP_AABB_EPS of csrc/bpgeo.cu
P = ctypes.POINTER(ctypes.c_double)


def _form(rows):
    return next(f for f, (lo, hi) in FORMS.items() if rows <= hi)


def _asserted(delta):
    return abs(delta) >= min(ASSERTED)


# ---- exact reference -------------------------------------------------------------------------------------------
def _rotation(rng, aligned):
    if aligned:                                      # signed axis permutation: exact in fp64, boxes stay tight
        return np.eye(3)[rng.permutation(3)] * rng.choice([-1.0, 1.0], 3)[:, None]
    return Rotation.random(random_state=rng).as_matrix()


def _place(rows, R, t):
    """Local rows [(a, b)] -> world rows (a' = R a, b' = b + a'.t) in fp64."""
    A = np.array([r[0] for r in rows], float) @ R.T
    b = np.array([r[1] for r in rows], float) + A @ t
    return A, b


def _scales(rng, n, dominant):
    return 10.0 ** rng.uniform(-1.0, 0.0 if dominant else 1.0, n)


def _lateral(rng, k, h, radius, tilt):
    rows = []
    for j in range(k):
        th = 2 * np.pi * (j + rng.uniform(-0.2, 0.2)) / k
        w = rng.uniform(-tilt, tilt)
        rows.append(((np.cos(th), np.sin(th), w), radius + w * h))      # cos x + sin y <= radius on z = h
    return rows


def _fr(v):
    return v if isinstance(v, Fr) else Fr(float(v))


def _solve3(A3, c3):
    """Exact solution of the 3x3 system A3 x = c3 (fp64 or rational entries) by Cramer's rule; None if singular."""
    M = [[_fr(v) for v in row] for row in A3]
    c = [_fr(v) for v in c3]

    def det(X):
        return (X[0][0] * (X[1][1] * X[2][2] - X[1][2] * X[2][1]) - X[0][1] * (X[1][0] * X[2][2] - X[1][2] * X[2][0])
                + X[0][2] * (X[1][0] * X[2][1] - X[1][1] * X[2][0]))

    d = det(M)
    if d == 0:
        return None
    out = []
    for k in range(3):
        Mk = [row[:] for row in M]
        for r in range(3):
            Mk[r][k] = c[r]
        out.append(det(Mk) / d)
    return out


def _cramer(A3, c3):
    x = _solve3(A3, c3)
    assert x is not None
    return x


def _dot_exact(a, x):
    return sum(_fr(a[k]) * x[k] for k in range(3))


def _slack(a, b, x):
    """c - a.x with c = fl(b - tol), exactly."""
    return Fr(float(b) - TOL) - _dot_exact(a, x)


class Case:
    """One constructed pair: rows of set 1 and set 2 in the local 'base' order (deciding rows listed in dec1 and
    dec2), the exact margin (Fraction; > 0 <=> intersects) and the designed margin delta in c units."""

    def __init__(self, kind, delta, A1, b1, dec1, A2, b2, dec2, exact, centre, dominant, far_up=None):
        self.kind, self.delta = kind, delta
        self.A1, self.b1, self.dec1 = A1, b1, dec1
        self.A2, self.b2, self.dec2 = A2, b2, dec2
        self.exact, self.centre, self.dominant, self.far_up = exact, centre, dominant, far_up

    @property
    def truth(self):
        return self.exact > 0

    @property
    def asserted(self):
        return _asserted(self.delta)


def _face_to_face(rng, delta, aligned, dominant):
    R, t = _rotation(rng, aligned), rng.uniform(-0.4, 0.4, 3)
    h = rng.uniform(-0.2, 0.2)
    rows1 = [((0, 0, 1), h), ((0, 0, -1), -(h - 0.6))] + _lateral(rng, rng.integers(3, 7), h, 0.3, 0.3)
    rows2 = [((0, 0, -1), -h), ((0, 0, 1), h + 0.6)] + _lateral(rng, rng.integers(3, 7), h, 0.3, 0.3)
    A1, b1 = _place(rows1, R, t)
    A2, b2 = _place(rows2, R, t)
    s1, s2 = _scales(rng, len(rows1), dominant), _scales(rng, len(rows2), dominant)
    s1[0] = s2[0] = 10.0 if dominant else 10.0 ** rng.uniform(-1, 1)
    A1, b1, A2, b2 = A1 * s1[:, None], b1 * s1, A2 * s2[:, None], b2 * s2
    A2[0] = -A1[0]                                   # bitwise negation: the contact planes are exactly parallel
    c1 = b1[0] - TOL
    b2[0] = (delta - c1) + TOL
    if delta == 0.0:                                 # hit c1 + c2 == 0 exactly where an offset allows it
        for k in range(-8, 9):
            cand = b2[0] + k * np.spacing(b2[0])
            if cand - TOL == -c1:
                b2[0] = cand
                break
    exact = Fr(float(c1)) + Fr(float(b2[0] - TOL))
    return Case("face", delta, A1, b1, [0], A2, b2, [0], exact, t + R @ np.array([0, 0, h]), dominant)


def _vertex_to_face(rng, delta, aligned, dominant, cone=False):
    R, t = _rotation(rng, aligned), rng.uniform(-0.4, 0.4, 3)
    h = rng.uniform(-0.2, 0.2)
    apex = np.array([0.0, 0.0, h])
    rows1 = []
    for j in range(3):
        th = 2 * np.pi * (j + rng.uniform(-0.15, 0.15)) / 3
        n = np.array([np.cos(th), np.sin(th), rng.uniform(0.4, 1.0)])
        rows1.append((n, n @ apex))
    if not cone:
        rows1.append(((0, 0, -1), -(h - 0.5)))
    rows2 = [((0, 0, -1), -h), ((0, 0, 1), h + 0.6)] + _lateral(rng, rng.integers(3, 7), h, 0.4, 0.0)
    A1, b1 = _place(rows1, R, t)
    A2, b2 = _place(rows2, R, t)
    s1, s2 = _scales(rng, len(rows1), dominant), _scales(rng, len(rows2), dominant)
    if dominant:
        s1[:3] = 10.0
        s2[0] = 10.0
    A1, b1, A2, b2 = A1 * s1[:, None], b1 * s1, A2 * s2[:, None], b2 * s2
    xa = _cramer(A1[:3], b1[:3] - TOL)               # the shrunk apex, exactly
    ax = _dot_exact(A2[0], xa)
    b2[0] = float(Fr(delta) + ax) + TOL
    exact = Fr(float(b2[0] - TOL)) - ax
    up = R @ np.array([0.0, 0.0, 1.0]) if cone else None
    return Case("cone" if cone else "vertex", delta, A1, b1, [0, 1, 2], A2, b2, [0], exact, t + R @ apex, dominant,
                far_up=up)


def _containment(rng, dominant):
    R, t = _rotation(rng, False), rng.uniform(-0.4, 0.4, 3)
    rows1 = [((1, 0, 0), 0.5), ((-1, 0, 0), 0.5), ((0, 1, 0), 0.5), ((0, -1, 0), 0.5), ((0, 0, 1), 0.5),
             ((0, 0, -1), 0.5)]
    for _ in range(rng.integers(2, 6)):
        u = rng.normal(size=3)
        u /= np.linalg.norm(u)
        rows1.append((u, rng.uniform(0.3, 0.6)))
    rows2 = [((1, 0, 0), 0.1), ((-1, 0, 0), 0.1), ((0, 1, 0), 0.1), ((0, -1, 0), 0.1), ((0, 0, 1), 0.1),
             ((0, 0, -1), 0.1)]
    A1, b1 = _place(rows1, R, t)
    A2, b2 = _place(rows2, R, t)
    s1, s2 = _scales(rng, len(rows1), dominant), _scales(rng, len(rows2), dominant)
    A1, b1, A2, b2 = A1 * s1[:, None], b1 * s1, A2 * s2[:, None], b2 * s2
    # the centre t lies in both shrunk sets with slack >= 0.1 s - tol > 0: exact (fp rounding is ~1e-16)
    exact = min(Fr(float(b - TOL)) - _dot_exact(a, [Fr(float(v)) for v in t])
                for a, b in itertools.chain(zip(A1, b1), zip(A2, b2)))
    assert exact > Fr(1, 10 ** 4)
    return Case("contain", 1.0, A1, b1, [], A2, b2, [], exact, t, dominant)


def _thin(rng, dominant):
    """Set 1 is a slab thinner than 2 tol (bounded laterally): its shrunk set is empty; set 2 is a box around it."""
    R, t = _rotation(rng, False), rng.uniform(-0.4, 0.4, 3)
    w = 0.0015
    rows1 = [((0, 0, 1), w / 2), ((0, 0, -1), w / 2)] + _lateral(rng, 4, 0.0, 0.3, 0.0)
    rows2 = [((1, 0, 0), 0.5), ((-1, 0, 0), 0.5), ((0, 1, 0), 0.5), ((0, -1, 0), 0.5), ((0, 0, 1), 0.5),
             ((0, 0, -1), 0.5)]
    A1, b1 = _place(rows1, R, t)
    A2, b2 = _place(rows2, R, t)
    s1, s2 = _scales(rng, len(rows1), dominant), _scales(rng, len(rows2), dominant)
    s1[1] = s1[0]
    A1, b1, A2, b2 = A1 * s1[:, None], b1 * s1, A2 * s2[:, None], b2 * s2
    A1[1] = -A1[0]
    exact = Fr(float(b1[0] - TOL)) + Fr(float(b1[1] - TOL))        # < 0: the shrunk slab is empty
    assert exact < 0
    return Case("thin", -1.0, A1, b1, [0, 1], A2, b2, [], exact, t, dominant)


def _slab(rng, dominant):
    """Set 1 has two rows only (unbounded, no box) and contains the box set 2."""
    R, t = _rotation(rng, False), rng.uniform(-0.4, 0.4, 3)
    rows1 = [((0, 0, 1), 0.3), ((0, 0, -1), 0.3)]
    rows2 = [((1, 0, 0), 0.2), ((-1, 0, 0), 0.2), ((0, 1, 0), 0.2), ((0, -1, 0), 0.2), ((0, 0, 1), 0.2),
             ((0, 0, -1), 0.2)]
    A1, b1 = _place(rows1, R, t)
    A2, b2 = _place(rows2, R, t)
    s1, s2 = _scales(rng, 2, dominant), _scales(rng, 6, dominant)
    A1, b1, A2, b2 = A1 * s1[:, None], b1 * s1, A2 * s2[:, None], b2 * s2
    exact = min(Fr(float(b - TOL)) - _dot_exact(a, [Fr(float(v)) for v in t])
                for a, b in itertools.chain(zip(A1, b1), zip(A2, b2)))
    assert exact > 0
    # far rows with a positive component along the slab's x axis keep -x a recession direction: no box
    return Case("slab", 1.0, A1, b1, [], A2, b2, [], exact, t, dominant, far_up=R @ np.array([1.0, 0.0, 0.0]))


def _far_rows(rng, n, centre, dominant, up=None):
    """n redundant rows, each a real nonzero row, at least 1.6 from `centre` (>= 1 from every point of the sets).
    For a cone (`up` = its axis) the normals keep a positive component along the axis, so the cone stays
    unbounded."""
    A = np.zeros((n, 3))
    for k in range(n):
        u = rng.normal(size=3)
        if up is not None:
            u -= (u @ up) * up
            u = u / np.linalg.norm(u) + rng.uniform(0.3, 1.0) * up
        A[k] = u / np.linalg.norm(u)
    b = A @ centre + rng.uniform(1.6, 2.6, n)
    s = _scales(rng, n, dominant)
    return A * s[:, None], b * s


def _arrange(rng, A, b, dec, n_total, centre, dominant, last, up=None):
    """Pad one set with far rows to n_total rows and permute: deciding rows last (`last`) or anywhere."""
    Af, bf = _far_rows(rng, n_total - A.shape[0], centre, dominant, up)
    A, b = np.vstack((A, Af)), np.concatenate((b, bf))
    rest = [r for r in range(n_total) if r not in dec]
    order = list(rng.permutation(rest)) + list(dec) if last else list(rng.permutation(n_total))
    pos = [order.index(d) for d in dec]                  # where the deciding rows went
    return np.ascontiguousarray(A[order]), np.ascontiguousarray(b[order]), pos


def _certify(case, A1, b1, pos1, A2, b2, pos2):
    """Check, exactly, what makes case.truth the answer for these rows (far rows and permutation included):
    * face: the contact rows are bitwise +-a; for "intersects" every other row is slack at the middle of the
      slab -c2 <= a.x <= c1 (there both contact rows have slack margin / 2), else the slab alone is empty;
    * vertex / cone: the contact normal -a2 is a strictly positive combination of the three apex normals, so the
      shrunk apex minimises a2.x over the shrunk set 1 and "disjoint" follows from the contact row alone; for
      "intersects" every other row is slack at the shrunk apex;
    * contain / slab: every row is slack at the centre; thin: the two slab rows alone leave nothing."""
    others = [(a, b) for k, (a, b) in enumerate(zip(A1, b1)) if k not in pos1] + \
             [(a, b) for k, (a, b) in enumerate(zip(A2, b2)) if k not in pos2]
    if case.kind == "face":
        a = A1[pos1[0]]
        assert np.array_equal(A2[pos2[0]], -a)
        assert Fr(float(b1[pos1[0]]) - TOL) + Fr(float(b2[pos2[0]]) - TOL) == case.exact
        if not case.truth:
            return
        aa = _dot_exact(a, [_fr(v) for v in a])
        xc = [_fr(v) for v in case.centre]
        shift = (-_slack(a, b1[pos1[0]], xc) + case.exact / 2) / aa           # to a.x = c1 - margin / 2
        w = [xc[k] - shift * _fr(a[k]) for k in range(3)]
        assert _slack(a, b1[pos1[0]], w) == case.exact / 2 and _slack(-a, b2[pos2[0]], w) == case.exact / 2
    elif case.kind in ("vertex", "cone"):
        N, a2 = A1[pos1], A2[pos2[0]]
        lam = _cramer(N.T, -a2)
        assert all(v > 0 for v in lam), lam
        w = _cramer(N, [float(v) - TOL for v in b1[pos1]])
        assert _slack(a2, b2[pos2[0]], w) == case.exact
        if not case.truth:
            return
    elif case.kind == "thin":
        assert np.array_equal(A1[pos1[1]], -A1[pos1[0]])
        assert Fr(float(b1[pos1[0]]) - TOL) + Fr(float(b1[pos1[1]]) - TOL) < 0
        return
    else:
        w = [_fr(v) for v in case.centre]
    worst = min(_slack(a, b, w) for a, b in others)
    assert worst > 0, (case.kind, float(worst))


def _sized(rng, case, form, last):
    """(A1, b1, A2, b2) of `case` with m1 + m2 in the row range of `form`.  With `last` (forms 2 and 3) set 1 has
    at least 33 rows, so its deciding rows sit at set indices >= 32, and set 2's last row is stacked index
    m1 + m2 - 1 >= 32 (form 2) or >= 64 (form 3)."""
    n1, n2 = case.A1.shape[0], case.A2.shape[0]
    lo, hi = FORMS[form]
    if form == 1:
        T = int(rng.integers(max(lo, n1 + n2), hi + 1))
        # a cone or slab keeps its bare 3 or 2 rows here: a set of fewer than four rows
        m1 = n1 if case.far_up is not None else int(rng.integers(n1, T - n2 + 1))
    else:
        lo1 = 33 if last else n1
        T = int(rng.integers(max(lo, lo1 + n2), hi + 1))
        m1 = int(rng.integers(max(lo1, T - M_MAX), min(M_MAX, T - n2) + 1))
    A1, b1, pos1 = _arrange(rng, case.A1, case.b1, case.dec1, m1, case.centre, case.dominant, last, case.far_up)
    A2, b2, pos2 = _arrange(rng, case.A2, case.b2, case.dec2, T - m1, case.centre, case.dominant, last)
    _certify(case, A1, b1, pos1, A2, b2, pos2)
    return A1, b1, A2, b2


class Pair:
    def __init__(self, case, form, A1, b1, A2, b2):
        self.case, self.form = case, form
        self.A1, self.b1, self.A2, self.b2 = A1, b1, A2, b2

    def sets(self, swap=False):
        s1, s2 = [self.A1, self.b1], [self.A2, self.b2]
        return (s2, s1) if swap else (s1, s2)


def build_pairs(seed=2024):
    """The whole case set: every kind x margin x row form, in two variants (random rotation, mixed row scales and
    a random row order / signed axis permutation, the deciding rows carrying the largest row norm and placed
    last), plus the closed-form cases in every row form."""
    rng = np.random.default_rng(seed)
    pairs = []
    for form in FORMS:
        for delta in MARGINS:
            for variant in (0, 1):
                aligned = dominant = last = variant == 1
                for make in (_face_to_face, _vertex_to_face):
                    case = make(rng, delta, aligned, dominant)
                    pairs.append(Pair(case, form, *_sized(rng, case, form, last)))
            case = _vertex_to_face(rng, delta, aligned=bool(rng.integers(2)), dominant=False, cone=True)
            pairs.append(Pair(case, form, *_sized(rng, case, form, False)))
        for make in (_containment, _thin, _slab):
            for dominant in (False, True):
                case = make(rng, dominant)
                pairs.append(Pair(case, form, *_sized(rng, case, form, False)))
    return pairs


def inside_shrunk(A, b, x, tol=TOL):
    """x satisfies A x <= b - tol (up to the rounding of evaluating the rows, ~1e-16 relative)."""
    v = A @ x - (b - tol)
    return bool(np.all(v <= 1e-13 * (1.0 + np.abs(b) + np.abs(A) @ np.abs(x))))


class Tally:
    """Decisions per (kernel, row form): asserted cases by margin and answer, recorded outcomes at 1e-10 and 0."""

    def __init__(self):
        self.asserted, self.recorded = {}, {}

    def add(self, kernel, form, delta, truth, got):
        if _asserted(delta):
            key = (kernel, form, abs(delta), bool(truth))
            self.asserted[key] = self.asserted.get(key, 0) + 1
        else:
            key = (kernel, form, delta)
            self.recorded.setdefault(key, []).append(int(got))

    def report(self, kernels, capsys):
        lines = []
        for kernel in kernels:
            for form in FORMS:
                a = " ".join(f"{d:g}:{self.asserted.get((kernel, form, d, True), 0)}/"
                             f"{self.asserted.get((kernel, form, d, False), 0)}" for d in ASSERTED)
                r = " ".join(f"{d:+g}->{self.recorded.get((kernel, form, d), [])}" for d in (1e-10, -1e-10, 0.0))
                lines.append(f"{kernel:13s} {form} row(s)/lane  asserted |margin|:intersects/disjoint {a}  "
                             f"recorded {r}")
        with capsys.disabled():                         # shown under plain `pytest -q` as well
            print("\n" + "\n".join(lines))

    def check_both_answers(self, kernels, levels=ASSERTED):
        for kernel in kernels:
            for form in FORMS:
                for d in levels:
                    assert self.asserted.get((kernel, form, d, True), 0) > 0, (kernel, form, d, "intersects")
                    assert self.asserted.get((kernel, form, d, False), 0) > 0, (kernel, form, d, "disjoint")


@pytest.fixture(scope="module")
def pairs():
    return build_pairs()


# ---- CPU: the reference and the thread-serial specification ----------------------------------------------------
def test_case_set_covers_forms_and_margins(pairs):
    """Every row form, every margin, both answers; deciding rows at stacked indices >= 32 and >= 64."""
    seen = set()
    for p in pairs:
        m1, m2 = p.A1.shape[0], p.A2.shape[0]
        assert m1 <= M_MAX and m2 <= M_MAX and _form(m1 + m2) == p.form
        if p.case.kind in ("face", "vertex", "cone"):
            assert abs(float(p.case.exact) - p.case.delta) <= 1e-13 * (1 + np.abs(p.case.b1).max()), p.case.kind
        seen.add((p.form, p.case.delta, p.case.kind))
        # the deciding row of set 2 ends up last in the 'last' variant: stacked index m1 + m2 - 1
        if p.case.dominant and p.case.kind in ("face", "vertex") and p.form > 1:
            assert m1 >= 33 and np.array_equal(p.A2[-1], p.case.A2[0])
    for form in FORMS:
        for delta in MARGINS:
            for kind in ("face", "vertex", "cone"):
                assert (form, delta, kind) in seen
    assert sum(p.case.truth for p in pairs) > 80 and sum(not p.case.truth for p in pairs) > 80


def test_reference_agrees_with_highs(pairs):
    """The exact reference against HiGHS (oracle.set_graph.intersection_margin) wherever |margin| >= 1e-6."""
    from oracle.set_graph import intersection_margin

    n = 0
    for p in pairs:
        if abs(p.case.delta) < 1e-6:
            continue
        mg = intersection_margin(*p.sets(), TOL)
        assert (mg < 0) == p.case.truth and mg != 0, (p.case.kind, p.case.delta, mg)
        n += 1
    assert n >= 70


def test_spec_exact_at_the_boundary(pairs, host_harness, capsys):
    """hh_pair_lp and hh_pair_lp_t0(..., 8) (the spec of the warp LP) give the exact answer at every asserted
    margin, in both pair orders, and every 'intersects' comes with a point of both shrunk sets."""
    host_harness.hh_pair_lp_t0.restype = ctypes.c_int
    tally = Tally()
    for p in pairs:
        for swap in (False, True):
            (A1, b1), (A2, b2) = p.sets(swap)
            for name in ("hh_pair_lp", "hh_pair_lp_t0"):
                xo, it = np.zeros(3), ctypes.c_int()
                args = [A1.ctypes.data_as(P), b1.ctypes.data_as(P), A1.shape[0], A2.ctypes.data_as(P),
                        b2.ctypes.data_as(P), A2.shape[0], ctypes.c_double(TOL), xo.ctypes.data_as(P),
                        ctypes.byref(it)]
                if name == "hh_pair_lp_t0":
                    args.append(ctypes.c_double(8.0))
                r = bool(getattr(host_harness, name)(*args))
                tally.add(name, p.form, p.case.delta, p.case.truth, r)
                if p.case.asserted:
                    assert r == p.case.truth, (name, p.case.kind, p.form, p.case.delta, swap)
                if r:
                    assert inside_shrunk(A1, b1, xo) and inside_shrunk(A2, b2, xo), (name, p.case.kind, p.case.delta)
    tally.report(("hh_pair_lp", "hh_pair_lp_t0"), capsys)
    tally.check_both_answers(("hh_pair_lp", "hh_pair_lp_t0"))


# ---- GPU ---------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def geo():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from boundplanner_b200 import geometry

    return geometry


def _pack(sets):
    import torch

    S = len(sets)
    A = np.zeros((S, M_MAX, 3))
    b = np.full((S, M_MAX), 10.0)
    m = np.zeros(S, np.int32)
    for k, (As, bs) in enumerate(sets):
        A[k, : As.shape[0]] = As
        b[k, : As.shape[0]] = bs
        m[k] = As.shape[0]
    return torch.as_tensor(A).cuda(), torch.as_tensor(b).cuda(), torch.as_tensor(m).cuda()


def _batch(pairs):
    """Sets 4c .. 4c+3 of case c: (set 1, set 2, set 2, set 1), so (4c, 4c+1) and (4c+2, 4c+3) are the pair in both
    orders as (i, j > i) entries of pair_feasible."""
    sets = []
    for p in pairs:
        (s1, s2) = p.sets()
        sets += [s1, s2, s2, s1]
    return sets


@pytest.mark.gpu
def test_pair_feasible_exact_at_the_boundary(pairs, geo, capsys):
    import torch
    from oracle.set_graph import intersection_margin

    sets = _batch(pairs)
    S = len(sets)
    A, b, m = _pack(sets)
    bits, x = geo.pair_feasible(A, b, m, tol=TOL, want_points=True)
    adj = geo.unpack_adjacency(bits, S).cpu().numpy()
    x = x.cpu().numpy()
    # the same bits with given boxes, over row blocks, and through the staged diagnostics entry point
    aabb = geo.set_aabb(A, b, m)
    assert np.array_equal(geo.pair_feasible(A, b, m, tol=TOL, aabb=aabb).cpu().numpy(), bits.cpu().numpy())
    cuts = (0, 37, S // 2, S - 5, S)
    blocks = [geo.pair_feasible(A, b, m, tol=TOL, row_begin=r0, row_end=r1).cpu().numpy()
              for r0, r1 in zip(cuts[:-1], cuts[1:])]
    assert np.array_equal(np.vstack(blocks), bits.cpu().numpy())
    out = geo.alloc_pair_buffers(S)
    geo.pair_feasible_stages(A, b, m, tol=TOL, out=out)
    assert np.array_equal(out[0].cpu().numpy(), bits.cpu().numpy())
    torch.cuda.synchronize()

    tally = Tally()
    for c, p in enumerate(pairs):
        for i, j in ((4 * c, 4 * c + 1), (4 * c + 2, 4 * c + 3)):
            got = bool(adj[i, j])
            tally.add("k_pair_lp", p.form, p.case.delta, p.case.truth, got)
            if p.case.asserted:
                assert got == p.case.truth, (p.case.kind, p.form, p.case.delta, i, j)
    # every 1 bit, constructed or between cases, comes with a point of both shrunk sets
    ones = np.argwhere(adj)
    for i, j in ones:
        assert inside_shrunk(*sets[i], x[i, j]) and inside_shrunk(*sets[j], x[i, j]), (i, j)
    # pairs between cases: HiGHS on a sample
    rng = np.random.default_rng(5)
    n_checked = 0
    for _ in range(300):
        i, j = sorted(rng.choice(S, 2, replace=False))
        if j == i + 1 and i % 2 == 0:
            continue
        mg = intersection_margin(sets[i], sets[j], TOL)
        if abs(mg) >= 1e-6:
            assert bool(adj[i, j]) == (mg < 0), (i, j, mg)
            n_checked += 1
    assert n_checked > 150
    tally.report(("k_pair_lp",), capsys)
    tally.check_both_answers(("k_pair_lp",))


@pytest.mark.gpu
def test_pairs_feasible_list_exact_at_the_boundary(pairs, geo, capsys):
    from boundplanner_b200 import set_graph

    sets = _batch(pairs)
    A, b, m = _pack(sets)
    lst = np.array([(4 * c, 4 * c + 1) for c in range(len(pairs))] + [(4 * c + 1, 4 * c) for c in range(len(pairs))],
                   np.int32)
    ok, x = geo.pairs_feasible_list(A, b, m, lst, tol=TOL)
    ok, x = ok.cpu().numpy(), x.cpu().numpy()
    adj = geo.unpack_adjacency(geo.pair_feasible(A, b, m, tol=TOL), len(sets)).cpu().numpy()
    tally = Tally()
    n = len(pairs)
    for c, p in enumerate(pairs):
        for k, (i, j) in ((c, lst[c]), (n + c, lst[n + c])):
            tally.add("k_pair_list", p.form, p.case.delta, p.case.truth, ok[k])
            if p.case.asserted:
                assert ok[k] == p.case.truth, (p.case.kind, p.form, p.case.delta, i, j)
            if ok[k]:
                assert inside_shrunk(*sets[i], x[k]) and inside_shrunk(*sets[j], x[k]), (p.case.kind, p.case.delta)
        # same rows in the same order as pair_feasible's (4c, 4c+1) and (4c+2, 4c+3): the same LP, the same bit
        assert ok[c] == adj[4 * c, 4 * c + 1] and ok[n + c] == adj[4 * c + 2, 4 * c + 3], (p.case.kind, p.case.delta)
    tally.report(("k_pair_list",), capsys)
    tally.check_both_answers(("k_pair_list",))
    # the drop-in set_intersection on a few pairs of each form
    for p in pairs[::23]:
        for swap in (False, True):
            s1, s2 = p.sets(swap)
            pt, _, success = set_graph.set_intersection(s1, s2, TOL)
            if p.case.asserted:
                assert success == p.case.truth, (p.case.kind, p.case.delta)
            if success:
                assert inside_shrunk(*s1, pt) and inside_shrunk(*s2, pt)


@pytest.mark.gpu
def test_row_forms_same_decision(geo):
    """One geometric pair padded into the 1-, 2- and 3-row forms, in several row orders and both pair orders:
    the exact decision every time."""
    rng = np.random.default_rng(7)
    sets, meta = [], []
    for delta in (1e-3, -1e-3, 1e-6, -1e-6, 1e-9, -1e-9):
        for make, kw in ((_face_to_face, {}), (_vertex_to_face, {}), (_vertex_to_face, dict(cone=True))):
            for variant in (0, 1):
                case = make(rng, delta, aligned=variant == 1, dominant=variant == 1, **kw)
                for form in FORMS:
                    for last in (False, True, False):
                        A1, b1, A2, b2 = _sized(rng, case, form, last and form > 1 and case.kind != "cone")
                        for swap in (False, True):
                            sets += [[A2, b2], [A1, b1]] if swap else [[A1, b1], [A2, b2]]
                            meta.append((case, form))
    A, b, m = _pack(sets)
    lst = np.array([(2 * k, 2 * k + 1) for k in range(len(meta))], np.int32)
    ok = geo.pairs_feasible_list(A, b, m, lst, tol=TOL)[0].cpu().numpy()
    adj = geo.unpack_adjacency(geo.pair_feasible(A, b, m, tol=TOL), len(sets)).cpu().numpy()
    for k, (case, form) in enumerate(meta):
        assert ok[k] == case.truth, (case.kind, form, case.delta)
        assert adj[2 * k, 2 * k + 1] == case.truth, (case.kind, form, case.delta)


# ---- set_aabb -----------------------------------------------------------------------------------------------------
def _exact_box(A, b):
    """Exact box of the bounded set {A x <= b}, independent of the kernel's enumeration: for each of the six
    directions HiGHS finds an optimal vertex; every triple of the rows tight there (to 1e-7) is solved and checked
    for feasibility in rationals, and the extreme of those exact vertices is the box.  Returns the exact vertices
    found (as floats) and lo, hi."""
    from scipy.optimize import linprog

    Af = [[_fr(v) for v in row] for row in A]
    bf = [_fr(v) for v in b]
    cache = {}

    def vertex(tr):
        if tr not in cache:
            x = _solve3([Af[i] for i in tr], [bf[i] for i in tr])
            ok = x is not None and all(sum(Af[r][k] * x[k] for k in range(3)) <= bf[r] for r in range(len(bf)))
            cache[tr] = x if ok else None
        return cache[tr]

    lo, hi = np.zeros(3), np.zeros(3)
    for k in range(3):
        for sgn, out in ((1.0, lo), (-1.0, hi)):
            c = np.zeros(3)
            c[k] = sgn
            res = linprog(c, A_ub=A, b_ub=b, bounds=[(None, None)] * 3, method="highs-ds")
            assert res.status == 0, res.message
            x = res.x
            act = np.flatnonzero(b - A @ x <= 1e-7 * (1 + np.abs(b) + np.abs(A) @ np.abs(x))).tolist()
            vals = [v[k] for v in (vertex(tr) for tr in itertools.combinations(act, 3)) if v is not None]
            if not vals:        # x inside an optimal face: its vertices lie on every row tight at x
                tri = (tr for tr in itertools.combinations(range(len(bf)), 3) if set(tr) & set(act))
                vals = [v[k] for v in map(vertex, tri) if v is not None]
            assert vals, (k, sgn, act)
            out[k] = float(min(vals) if sgn > 0 else max(vals))
    V = np.array([[float(t) for t in v] for v in cache.values() if v is not None])
    return V, lo, hi


def _aabb_sets(rng):
    """(A, b, bounded) of the box test: random sets, boxes, a box whose corner is cut by its last row, pyramids
    with 12-20 faces through the apex, duplicate and near-parallel rows, the 48-row maximum; and sets without a
    box: cones, a semi-infinite prism, a slab, a half-space, an empty description, 0-2 rows."""
    out = []
    BOX = np.vstack((np.eye(3), -np.eye(3)))
    for k in range(12):                                        # random sets, up to the 48-row maximum
        n = (3, 10, 20, 42, 42, 42)[k % 6] if k < 6 else 42
        c = rng.uniform(-0.5, 0.5, 3)
        An = rng.normal(size=(n, 3))
        An /= np.linalg.norm(An, axis=1)[:, None]
        A = np.vstack((BOX, An)) * 10.0 ** rng.uniform(-1, 1, (n + 6, 1))
        R = _rotation(rng, False)
        A = A @ R.T
        b = A @ c + np.abs(A).sum(axis=1) * rng.uniform(0.05, 0.4, n + 6)
        out.append((A, b, True))
    for _ in range(3):                     # boxes, and boxes whose last row cuts a corner / moves a face inwards
        lo = rng.uniform(-1, 0, 3)
        hi = lo + rng.uniform(0.05, 1, 3)
        out.append((BOX.copy(), np.concatenate((hi, -lo)), True))
        u = np.array([1.0, 1.0, 1.0]) / np.sqrt(3)
        out.append((np.vstack((BOX, u)), np.concatenate((hi, -lo, [u @ hi - 0.02])), True))
        k = rng.integers(3)
        out.append((np.vstack((BOX, 2.0 * BOX[k])), np.concatenate((hi, -lo, [2.0 * (hi[k] - 0.01)])), True))
    for nf in (12, 16, 20):                                    # pyramids: nf faces through the apex, base last
        apex = rng.uniform(-0.3, 0.3, 3)
        th = np.sort(rng.uniform(0, 2 * np.pi, nf))
        N = np.stack((np.cos(th), np.sin(th), rng.uniform(0.3, 1.0, nf)), axis=1)
        R = _rotation(rng, nf == 16)
        A = np.vstack((N, [[0, 0, -1.0]])) @ R.T
        b = A @ apex + np.concatenate((np.zeros(nf), [0.5]))
        out.append((A, b, True))
    A, b, _ = out[2]                                           # duplicate rows and near-parallel rows
    out.append((np.vstack((A, A[:4])), np.concatenate((b, b[:4])), True))
    Ap = A[:6] + 1e-7 * rng.normal(size=(6, 3))
    out.append((np.vstack((A, Ap)), np.concatenate((b, b[:6] + 1e-8)), True))
    Ab, bb, _ = out[0]
    out.append((np.vstack((Ab, Ab[6:] * 2.0))[:48], np.concatenate((bb, bb[6:] * 2.0))[:48], True))
    # without a box
    for _ in range(3):                                         # cones: 3 or more rows through one apex
        c = _vertex_to_face(rng, 1e-3, aligned=False, dominant=False, cone=True)
        out.append((c.A1[:3], c.b1[:3], False))
    c = _vertex_to_face(rng, 1e-3, aligned=False, dominant=False, cone=True)
    Af, bf = _far_rows(rng, 8, c.centre, False, c.far_up)
    out.append((np.vstack((c.A1, Af)), np.concatenate((c.b1, bf)), False))
    th = np.array([0.1, 2.2, 4.2])                             # triangular prism closed at one end only
    Apr = np.vstack((np.stack((np.cos(th), np.sin(th), np.zeros(3)), axis=1), [[0, 0, 1.0]]))
    out.append((Apr, np.array([0.3, 0.3, 0.3, 0.2]), False))
    out.append((np.array([[0, 0, 1.0], [0, 0, -1.0]]), np.array([0.3, 0.3]), False))       # slab (2 rows)
    out.append((np.array([[0.3, 0.4, 1.0]]), np.array([0.1]), False))                      # half-space
    out.append((np.zeros((0, 3)), np.zeros(0), False))                                     # no rows
    out.append((BOX.copy(), np.array([0.5, 0.5, 0.5, -0.6, 0.5, 0.5]), False))              # empty: x >= 0.6 > 0.5
    return out


@pytest.mark.gpu
def test_set_aabb_against_exact_box(geo):
    rng = np.random.default_rng(11)
    cases = _aabb_sets(rng)
    A, b, m = _pack([(a, bb) for a, bb, _ in cases])
    box = geo.set_aabb(A, b, m).cpu().numpy()
    n_bounded = 0
    for k, (As, bs, bounded) in enumerate(cases):
        if not bounded:
            assert np.all(box[k, :3] == -np.inf) and np.all(box[k, 3:] == np.inf), (k, As.shape[0], box[k])
            continue
        V, lo, hi = _exact_box(As, bs)
        slack = AABB_EPS * (1 + np.abs(V))
        assert np.all(V >= box[k, :3] - slack) and np.all(V <= box[k, 3:] + slack), k     # contains every vertex
        assert np.abs(box[k, :3] - lo).max() <= 1e-9 and np.abs(box[k, 3:] - hi).max() <= 1e-9, (k, box[k], lo, hi)
        n_bounded += 1
    assert n_bounded >= 20


# ---- check_fit ------------------------------------------------------------------------------------------------------
def _fit_sets(rng, n_far_i, n_far_j, aligned=False):
    """Two rotated boxes whose intersection is [0.5 - w, 0.5] x [-0.2, 0.2]^2 in the local frame (w = 0.3), rows of
    unit norm; the rows along one axis are bitwise +-the same vector, so the shrunk intersection is exactly the
    parallelepiped |a_d.p - mid_d| <= W_d / 2 (W_d from c = fl(b - 0.001))."""
    R, t = _rotation(rng, aligned), rng.uniform(-0.4, 0.4, 3)
    ax = R.T.copy()                                           # ax[d] = R e_d in fp64
    def box(lo, hi):
        A = np.vstack((ax, -ax))
        return A, np.concatenate((hi + ax @ t, -(lo + ax @ t)))
    Ai, bi = box(np.array([0.0, -0.2, -0.2]), np.array([0.5, 0.2, 0.2]))
    Aj, bj = box(np.array([0.2, -0.25, -0.25]), np.array([1.0, 0.25, 0.25]))
    centre = t + R @ np.array([0.35, 0.0, 0.0])
    Fi, Fj = rng.normal(size=(n_far_i, 3)), rng.normal(size=(n_far_j, 3))
    Fi, Fj = Fi / np.linalg.norm(Fi, axis=1)[:, None], Fj / np.linalg.norm(Fj, axis=1)[:, None]
    fi, fj = Fi @ centre + rng.uniform(1.6, 2.6, n_far_i), Fj @ centre + rng.uniform(1.6, 2.6, n_far_j)
    pi, pj = rng.permutation(6 + n_far_i), rng.permutation(6 + n_far_j)
    Ai, bi = np.vstack((Ai, Fi))[pi], np.concatenate((bi, fi))[pi]
    Aj, bj = np.vstack((Aj, Fj))[pj], np.concatenate((bj, fj))[pj]
    return ax, Ai, bi, Aj, bj, centre


def _widths(ax, sets, margin=0.001):
    """W_d (exact) of the shrunk intersection of `sets` along the three axis vectors."""
    W = []
    for d in range(3):
        hi = min(Fr(float(b - margin)) for A, bb in sets for a, b in zip(A, bb) if np.array_equal(a, ax[d]))
        lo = min(Fr(float(b - margin)) for A, bb in sets for a, b in zip(A, bb) if np.array_equal(a, -ax[d]))
        W.append(hi + lo)
    return W


def _fit_margin(ax, W, l):
    """> 0 <=> p and p + l both fit: min_d (W_d - |a_d . l|), exactly."""
    lf = [Fr(float(v)) for v in l]
    return min(W[d] - abs(_dot_exact(ax[d], lf)) for d in range(3))


@pytest.mark.gpu
def test_check_fit_exact(geo, capsys):
    from boundplanner_b200._lib import BpGeoError
    from oracle.planner_graph import check_intersection

    rng = np.random.default_rng(13)
    sets, pairs, want, meta, l_list = [], [], [], [], []
    # (far rows of i, far rows of j): 2 (m_i + m_j) in the 1-, 2- and 3-row forms
    for n_far in ((0, 0), (2, 3), (5, 5), (10, 8), (20, 16), (30, 4)):
        for delta in MARGINS:
            ax, Ai, bi, Aj, bj, centre = _fit_sets(rng, *n_far, aligned=bool(rng.integers(2)))
            W = _widths(ax, [(Ai, bi), (Aj, bj)])
            # offset along the first axis: fits iff |l| < w - 2 margin, by delta
            l = ax[0] * (float(W[0]) - delta)
            mg = _fit_margin(ax, W, l)
            assert abs(float(mg) - delta) < 1e-14
            i = len(sets)
            sets += [[Ai, bi], [Aj, bj]]
            pairs.append((i, i + 1))
            want.append(mg)
            meta.append((2 * (Ai.shape[0] + Aj.shape[0]), delta, centre))
            l_list.append(l)
            # the single-set path (i, i): box i alone
            Wi = _widths(ax, [(Ai, bi)])
            l = ax[0] * (float(Wi[0]) - delta)
            pairs.append((i, i))
            want.append(_fit_margin(ax, Wi, l))
            meta.append((2 * Ai.shape[0], delta, centre))
            l_list.append(l)
    A, b, m = _pack(sets)
    tally = Tally()
    n_oracle = 0
    # one offset per call (check_fit takes one l_ee); batch the pairs that share nothing but the offset
    for k, ((i, j), mg, (rows, delta, centre), l) in enumerate(zip(pairs, want, meta, l_list)):
        fits, omega = geo.check_fit(A, b, m, np.array([[i, j]], np.int32), l, np.array([0.0, 1.0, 0.0]), 0.0,
                                    x0=centre[None] if k % 2 else None)
        got = bool(fits.cpu().numpy()[0])
        tally.add("k_fit_check", _form(rows), delta, mg > 0, got)
        if _asserted(delta):
            assert got == (mg > 0), (i, j, rows, delta)
            assert float(omega.cpu().numpy()[0]) == (0.0 if got else -1.0)
            if abs(delta) >= 1e-6 and k % 9 == 0:
                Ac = sets[i][0] if i == j else np.vstack((sets[i][0], sets[j][0]))
                bc = sets[i][1] if i == j else np.concatenate((sets[i][1], sets[j][1]))
                ok, _ = check_intersection(Ac, bc, l, centre, np.array([0.0, 1.0, 0.0]), 0.0)
                assert ok == got, (i, j, delta)
                n_oracle += 1
    assert n_oracle >= 5
    tally.report(("k_fit_check",), capsys)
    tally.check_both_answers(("k_fit_check",))

    # a rotating offset: omega is the first fitting sample, computed exactly; and the active mask
    ax, Ai, bi, Aj, bj, centre = _fit_sets(rng, 4, 4)
    sets2 = [[Ai, bi], [Aj, bj]]
    A2, b2, m2 = _pack(sets2)
    W = _widths(ax, sets2)
    omega_hat, omega_norm = ax[1], 1.2
    for L in (0.35, 0.33, 0.31, 0.25):
        l_ee = ax[0] * L
        ls = [geo.rodrigues_matrix(omega_hat, omega_norm * k / 19) @ l_ee for k in range(20)]
        mgs = [_fit_margin(ax, W, lk) for lk in ls]
        first = next((k for k, v in enumerate(mgs) if v > 0), -1)
        assert all(abs(v) > 1e-9 for v in mgs)
        pr = np.array([[0, 1], [0, 1], [1, 0], [0, 0]], np.int32)
        active = np.array([1, 0, 1, 1], np.int32)
        fits, omega = geo.check_fit(A2, b2, m2, pr, l_ee, omega_hat, omega_norm, active=active)
        fits, omega = fits.cpu().numpy(), omega.cpu().numpy()
        assert fits.tolist()[:3] == [first >= 0, False, first >= 0]
        assert omega[0] == omega[2] == (first / 19 if first >= 0 else -1.0) and omega[1] == -1.0
        Wi = _widths(ax, sets2[:1])
        first_i = next((k for k, lk in enumerate(ls) if _fit_margin(ax, Wi, lk) > 0), -1)
        assert bool(fits[3]) == (first_i >= 0) and omega[3] == (first_i / 19 if first_i >= 0 else -1.0)
        ok, p_inside = check_intersection(np.vstack((Ai, Aj)), np.concatenate((bi, bj)), l_ee, centre, omega_hat,
                                          omega_norm)
        assert ok == (first >= 0) and (not ok or p_inside[3] == first / 19)

    # more than 48 combined rows: a loud error
    Ab, bb = _fit_sets(rng, 20, 20)[1:3]
    big = [[Ab, bb], [np.vstack((Ab, Ab[:3])), np.concatenate((bb, bb[:3] + 1.0))]]
    A3, b3, m3 = _pack(big)
    with pytest.raises(BpGeoError):
        geo.check_fit(A3, b3, m3, np.array([[0, 1]], np.int32), ax[0] * 0.01, np.array([0.0, 1.0, 0.0]), 0.0)
