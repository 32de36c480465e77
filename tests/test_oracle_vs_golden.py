"""CPU: pins the oracle (oracle/toppra_oracle.c) to the reference's outputs.

Golden vectors come from the UNMODIFIED reference build (tests/golden/make_golden.py) and from the reference's
own test files (cited).  Everything is compared bit-for-bit unless a tolerance is written in the test."""
import numpy as np
import pytest

from conftest import BATCH_CASES
from oracle import oracle as orc


def _eq(a, b):
    return np.array_equal(np.asarray(a), np.asarray(b), equal_nan=True)


# ---- LP layer --------------------------------------------------------------------------------------------
# known-answer tests of tests/tests/lpsolvers/seidel/test_lp1d.py:6-13 (exact ==)
LP1D_KATS = [
    ([1.0, 2], [], [], -1.0, 1.0, 1, 3, 1, -2),
    ([-2.0, 2], [], [], -1.0, 1.0, 1, 4, -1, -1),
    ([1.0, 2], [4.0, -1.0], [-1.0, 0], -1.0, 1.0, 1, 2.25, 0.25, 0),
    ([1.0, 0], [1.0, -1.0, -1, 1, 0, 0], [-1.5, -.5, -1.5, -0.5, 0, 0], -10000.0, 10000.0, 1, 0.5, 0.5, 3),
]


@pytest.mark.parametrize("v,a,b,low,high,res,optval,optvar,active", LP1D_KATS)
def test_lp1d_kats(v, a, b, low, high, res, optval, optvar, active):
    out = orc.lp1d(v, np.array(a, dtype=float), np.array(b, dtype=float), low, high)
    assert out == (res, optval, optvar, active)


def test_lp1d_infeasible():
    # test_lp1d.py:41-48
    assert orc.lp1d([1.0, 2], [-1.0, 1.0], [0.0, 0.5], -1, 1.0)[0] == 0


_A10 = (1.36866544, 1.28199038, -0.19515422, 0.97578149, 0.64391477, -0.0811908, -0.70696349, -1.01804875,
        0.5742392, 0.02939029)
_B10 = (0.1969094, 1.13910161, 0.10109674, 1.71246466, -0.45206747, -0.51302219, -1.16558797, 0.19919171,
        -0.906885, 0.94722345)
_C10 = (-2.68926068, -1.59762444, -2.03337493, -2.04617298, -1.09241401, -1.67319798, -1.9483617, -1.57529407,
        -1.37795315, -3.47919232)
# tests/tests/lpsolvers/seidel/test_lp2d.py:7-34 (values allclose, active sets equal)
LP2D_KATS = [
    ([1, 2, 3.0], (), (), (), [-1, -1], [1, 1], [-1, 1], 1, 6, [1, 1], [-2, -4]),
    ([-2, 2, 2.0], (), (), (), [-1, -1], [1, 1], [-1, 1], 1, 6, [-1, 1], [-1, -4]),
    ([1, 2, 3], (1, -1), (1, 1), (-1, -0.5), [-1, -1], [1, 1], [-1, -1], 1, 4.75, [0.25, 0.75], [0, 1]),
    ([-1, 0.01, 0], (1, -1), (1, 1), (-1, -0.5), [-1, -1], [1, 1], [-1, -1], 1, 0.995, [-1, -0.5], [-1, 1]),
    ([1, 2, 0], _A10, _B10, _C10, [-100, -100], [100, 100], [0, 1], 1, 2.5547484757095305,
     [-1.18181729266432, 1.8682828841869252], [3, 7]),
    ([1, 2, 0], _A10, _B10, _C10, [-100, -100], [100, 100], [5, 9], 1, 2.5547484757095305,
     [-1.18181729266432, 1.8682828841869252], [3, 7]),
    ([1, 2, 0], [-0.01, 0.01], [-1, 1], [0, 0.5], [-1, -1], [1, 1], [0, 1], 0, None, None, None),
]


@pytest.mark.parametrize("v,a,b,c,low,high,active_c,res,optval,optvar,active", LP2D_KATS)
def test_lp2d_kats(v, a, b, c, low, high, active_c, res, optval, optvar, active):
    r, val, var, act = orc.lp2d(np.array(v, float), np.array(a, float), np.array(b, float), np.array(c, float),
                                np.array(low, float), np.array(high, float), active_c)
    assert r == res
    if res:
        np.testing.assert_allclose(val, optval)
        np.testing.assert_allclose(var, optvar)
        assert set(act.tolist()) == set(active)


def test_lp2d_random100(golden):
    """100 seeded random LPs of test_lp2d.py:74-95; expected values produced by the reference solve_lp2d."""
    g = golden("lp2d_random100")
    for i in range(100):
        r, val, var, act = orc.lp2d(g["v"][i], g["a"][i], g["b"][i], g["c"][i], g["low"], g["high"], g["active_in"][i])
        assert r == g["res"][i]
        if r:
            assert val == g["optval"][i] and _eq(var, g["optvar"][i]) and _eq(act, g["active_out"][i])


def test_lp2d_err_regressions():
    """test_lp2d.py:118-130 (test_err1) and :153-182 (test_err2): inputs that once broke the solver; both are
    feasible LPs with optimum x = high[1] resp. a finite x."""
    v = np.array([-1.e-09, 1.e+00, 0.e+00])
    a = np.array([-0.02020202, 0.02020202, 1.53515768, 4.3866269, -3.9954173, -1.53515768, -4.3866269, 3.9954173])
    b = np.array([-1., 1., -185.63664301, 156.27072783, -209.00954213, 185.63664301, -156.27072783, 209.00954213])
    c = np.array([0., -0.0062788, -1., -2., -4., -1., -1., -1.])
    r, val, var, act = orc.lp2d(v, a, b, c, np.array([-100., 0.]), np.array([1.0e+02, 6.26434609e-02]), [0, 5])
    assert r == 1
    assert np.all(a * var[0] + b * var[1] + c <= 1e-9)
    assert -100 <= var[0] <= 100 and 0 <= var[1] <= 6.26434609e-02 + 1e-12


# ---- spline fit / eval ------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [2, 3, 4, 5, 9, 20])
def test_spline_fit_vs_scipy(golden, n):
    """scipy CubicSpline coefficients (golden, scipy 1.18.1) for every supported boundary condition.
    Tolerance 1e-12 relative: LAPACK's banded solve may order operations differently; in practice bit-equal."""
    g = golden("spline_fits")
    x, y = g["x_%d" % n], g["y_%d" % n]
    cases = {"not-a-knot": "not-a-knot", "clamped": "clamped", "natural": "natural",
             "first": ((1, g["d0_%d" % n]), (1, g["d1_%d" % n])), "mixed": ((2, g["d0_%d" % n]), (1, g["d1_%d" % n]))}
    for key, bc in cases.items():
        c = orc.cubic_spline_fit(x, y, bc)
        ref = g["c_%d_%s" % (n, key)]
        np.testing.assert_allclose(c, ref, rtol=1e-12, atol=1e-12 * np.abs(ref).max())


# ---- whole path --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", BATCH_CASES)
def test_batch_cases_bit_exact(golden, case):
    g = golden(case)
    B = g["way"].shape[0]
    interp = bool(g["scheme"])
    for b in range(B):
        c = orc.cubic_spline_fit(g["ss"], g["way"][b])
        assert _eq(c, g["c"][b]), "spline fit differs from scipy"
        assert _eq(orc.ppoly_eval(c, g["ss"], g["grid"], 1), g["qs"][b])
        assert _eq(orc.ppoly_eval(c, g["ss"], g["grid"], 2), g["qss"][b])
        assert _eq(orc.velocity_xbound(g["qs"][b], g["vlim"][b]), g["xbound"][b])
        o = orc.solve_velacc(c, g["ss"], g["grid"], g["vlim"][b], g["alim"][b], interp, float(g["sd_start"]),
                             float(g["sd_end"]), want_rows=True)
        assert o["status"] == g["status"][b]
        assert _eq(o["K"], g["K"][b]) and _eq(o["sd"], g["sd"][b]) and _eq(o["u"], g["sdd"][b])
        # rows = F.a, F.b, F.c - g of the reference's (a, b, F, g): rows [a, -a, a+, -a+]
        dof = g["way"].shape[2]
        a_ref, b_ref = g["acc_a"][b], g["acc_b"][b]
        F = g["acc_F"][b]
        assert _eq(o["rows"][:, 0, :], a_ref.dot(F.T)) and _eq(o["rows"][:, 1, :], b_ref.dot(F.T))
        assert _eq(o["rows"][:, 2, :], np.zeros_like(o["rows"][:, 2, :]) - g["acc_g"][b])
        assert o["rows"].shape[2] == (4 if interp else 2) * dof


def test_cfg1_example(golden):
    """BASELINE config 1: examples/plot_kinematics.py, seed 9, 100 gridpoints."""
    g = golden("cfg1_seed9")
    c = orc.cubic_spline_fit(g["ss"], g["way"])
    assert _eq(c, g["c"])
    o = orc.solve_velacc(c, g["ss"], g["grid"], g["vlim"], g["alim"], True, 0, 0, want_rows=True)
    assert o["status"] == 0 and _eq(o["K"], g["K"]) and _eq(o["sd"], g["sd"]) and _eq(o["u"], g["sdd"])
    w = orc.Wrapper(g["grid"], o["rows"], o["xbound"])
    assert _eq(w.compute_feasible_sets(), g["X"])
    w = orc.Wrapper(g["grid"], o["rows"], o["xbound"])
    assert _eq(w.compute_controllable_sets(0.0, 0.5), g["K_0_05"])
    # the example's own automatic grid (290 points here)
    o = orc.solve_velacc(c, g["ss"], g["auto_grid"], g["vlim"], g["alim"], True, 0, 0)
    assert _eq(o["K"], g["auto_K"]) and _eq(o["sd"], g["auto_sd"])


# cpp/tests/test_algorithm.cpp:109-117,132-140,161-169 == tests/tests/cpp/test_toppra.py:29-36 (tolerance 1e-6 there)
CPP_K_MAX = [0.06666667, 0.07624309, 0.08631706, 0.09690258, 0.1005511, 0.09982804, 0.09979021, 0.1004364,
             0.10178673, 0.10184412, 0.09655088, 0.09173679, 0.08734254, 0.08331796, 0.07962037, 0.07621325,
             0.07306521, 0.07014913, 0.0674415, 0.06492188, 0.06257244, 0.06037764, 0.05832397, 0.05639984,
             0.05459563, 0.05290407, 0.05132158, 0.04985238, 0.04852317, 0.04745694, 0.04761905, 0.05457026,
             0.06044905, 0.06527948, 0.08479263, 0.10990991, 0.13252362, 0.15269631, 0.15777077, 0.12111776,
             0.09525987, 0.07641998, 0.06232537, 0.05154506, 0.04314353, 0.03257513, 0.02268898, 0.01495548,
             0.0088349, 0.00394283, 0.]
CPP_PARAM = [0., 0.00799999, 0.01559927, 0.02295854, 0.03021812, 0.0375065, 0.04494723, 0.05266502, 0.06079176,
             0.06947278, 0.07887417, 0.08890758, 0.08734253, 0.08331795, 0.07962036, 0.07621324, 0.0730652,
             0.07014912, 0.06744149, 0.06492187, 0.06257243, 0.06037763, 0.05832396, 0.05639983, 0.05459562,
             0.05290406, 0.05132157, 0.04985237, 0.04852316, 0.04745693, 0.04761904, 0.0285715, 0.05376003,
             0.04275653, 0.04126188, 0.04013804, 0.03912958, 0.03818766, 0.03729606, 0.0364472, 0.03563649,
             0.03486069, 0.03411724, 0.03340395, 0.03271895, 0.03206054, 0.02268897, 0.01495547, 0.00883489,
             0.00394282, 0.]
CPP_FEAS_MAX = [0.06666667, 0.07624309, 0.08631706, 0.09690258, 0.1005511, 0.09982804, 0.09979021, 0.1004364,
                0.10178673, 0.10388394, 0.10679654, 0.11062383, 0.11550389, 0.12162517, 0.12924407, 0.13871115,
                0.15051124, 0.16532619, 0.18413615, 0.20838854, 0.24029219, 0.27052997, 0.2601227, 0.2447933,
                0.22462845, 0.2, 0.17154989, 0.14013605, 0.10674847, 0.07241209, 0.04761905, 0.05457026, 0.06044905,
                0.06527948, 0.08479263, 0.10990991, 0.13252362, 0.15269631, 0.15777077, 0.12111776, 0.09525987,
                0.07641998, 0.06232537, 0.05154506, 0.04314353, 0.03648939, 0.0311448, 0.02679888, 0.02322632,
                0.02026086, 0.01777778]


def test_cpp_2dof_collocation_golden(golden):
    """The reference's 51-value golden vectors (x = sd^2, generated with Python + qpOASES, tolerance 1e-6)
    and the same case solved by the reference seidel build (bit-exact)."""
    g = golden("cpp_2dof_collocation")
    c = orc.cubic_spline_fit(g["ss"], g["way"])
    assert _eq(c, g["c"])
    o = orc.solve_velacc(c, g["ss"], g["grid"], g["vlim"], g["alim"], False, 0, 0, want_rows=True)
    assert o["status"] == 0
    assert _eq(o["K"], g["K"]) and _eq(o["sd"], g["sd"]) and _eq(o["u"], g["sdd"])
    np.testing.assert_allclose(o["K"][:, 1], CPP_K_MAX, atol=1e-6)
    np.testing.assert_allclose(o["sd"] ** 2, CPP_PARAM, atol=1e-6)
    X = orc.Wrapper(g["grid"], o["rows"], o["xbound"]).compute_feasible_sets()
    assert _eq(X, g["X"])
    np.testing.assert_allclose(X[:, 1], CPP_FEAS_MAX, atol=1e-6)


def test_stagewise_cases(golden):
    """solve_stagewise_optim at stages 3,10,30,40 (fixture of test_basic_can_linear.py:53-77), incl. the 1-D branch
    and NaN = absent bounds; warm-start state chained through the calls like the reference object."""
    g = golden("stagewise_6dof")
    c = orc.cubic_spline_fit(g["ss"], g["way"])
    o = orc.solve_velacc(c, g["ss"], g["grid"], g["vlim"], g["alim"], True, 0, 0, want_rows=True)
    w = orc.Wrapper(g["grid"], o["rows"], o["xbound"])
    for row in g["cases"]:
        i, gg, xb, xnb, ref = int(row[0]), row[1:3], row[3:5], row[5:7], row[7:9]
        res = w.solve_stagewise_optim(i, None, gg, xb[0], xb[1], xnb[0], xnb[1])
        assert _eq(res, ref), (row, res)


def test_robustness_suite(golden):
    """P4: tiny-motion paths of tests/tests/retime/robustness/problem_suite_1.yaml (clamped spline)."""
    g = golden("p4_robustness_suite")
    for name in g["names"]:
        ss, way, grid = g[name + "_ss"], g[name + "_way"], g[name + "_grid"]
        c = orc.cubic_spline_fit(ss, way, "clamped")
        ref_c = g[name + "_c"]
        np.testing.assert_allclose(c, ref_c, rtol=1e-12, atol=1e-15)
        o = orc.solve_velacc(ref_c, ss, grid, g[name + "_vlim"], g[name + "_alim"], True, 0, 0)
        assert o["status"] == int(g[name + "_status"]), name
        assert _eq(o["K"], g[name + "_K"]) and _eq(o["sd"], g[name + "_sd"]) and _eq(o["u"], g[name + "_sdd"]), name


def test_torque_second_order(golden):
    """cfg-3 shape: vel + acc + SecondOrder(torque) rows through the generic row interface."""
    from problems import inv_dyn_numpy
    g = golden("torque_dof6")
    for b in range(g["way"].shape[0]):
        c = orc.cubic_spline_fit(g["ss"], g["way"][b])
        base = orc.solve_velacc(c, g["ss"], g["grid"], g["vlim"][b], g["alim"][b], True, 0, 0, want_rows=True)
        a, bb, cc = g["tau_a"][b], g["tau_b"][b], g["tau_c"][b]  # interpolation-lifted [G, 12]
        tl = g["taulim"][b]
        gvec = np.r_[tl[:, 1], -tl[:, 0], tl[:, 1], -tl[:, 0]]
        F1 = np.vstack((np.eye(6), -np.eye(6)))
        F = np.zeros((24, 12)); F[:12, :6] = F1; F[12:, 6:] = F1
        rows = np.concatenate((base["rows"], np.stack((a.dot(F.T), bb.dot(F.T), cc.dot(F.T) - gvec), axis=1)), axis=2)
        o = orc.solve_rows(rows, base["xbound"], g["grid"], 0, 0)
        assert o["status"] == g["status"][b]
        assert _eq(o["K"], g["K"][b]) and _eq(o["sd"], g["sd"][b]) and _eq(o["u"], g["sdd"][b])


def test_joint_torque_constraint(golden):
    """JointTorqueConstraint (joint_torque.py:77-116, dry friction, identical F) for both discretisation schemes: the
    reference's (a, b, c, F, g) through the generic row interface reproduce its K / sd / sdd."""
    g = golden("joint_torque_dof6")
    for scheme in (0, 1):
        t = "s%d_" % scheme
        for b in range(g[t + "way"].shape[0]):
            a, bb, cc, F, gv = (g[t + k][b] for k in ("a", "b", "c", "F", "g"))
            assert F.shape == ((12, 6) if scheme == 0 else (24, 12)) and a.shape[1] == F.shape[1]
            rows = np.stack((a.dot(F.T), bb.dot(F.T), cc.dot(F.T) - gv), axis=1)
            o = orc.solve_rows(rows, g[t + "xbound"][b], g["grid"], 0, 0)
            assert o["status"] == g[t + "status"][b] == 0
            assert _eq(o["K"], g[t + "K"][b]) and _eq(o["sd"], g[t + "sd"][b]) and _eq(o["u"], g[t + "sdd"][b])


def test_forward_retry_rule(golden):
    """reachability_algorithm.py:315-343: x is lowered by max(x - 1e-8, 0.999 x) up to 10 times when the forward LP is
    infeasible.  (a) start velocities that are admissible only through the 1e-5 slack: an excess of 3e-8 is absorbed
    by retries (Ok), 5e-6 exhausts them (ErrUnknown); (b) row-level problems found by random search."""
    g = golden("retry_after_slack_start")
    n_ok = 0
    for b in range(g["way"].shape[0]):
        c = orc.cubic_spline_fit(g["ss"], g["way"][b])
        lin = orc.solve_velacc(c, g["ss"], g["grid"], g["vlim"][b], g["alim"][b], True, 0, 0, want_rows=True)
        w = orc.Wrapper(g["grid"], lin["rows"], lin["xbound"])
        o = w.compute_parameterization(float(g["sd_start"][b]), 0.0)
        assert o["status"] == g["status"][b] and o["retries"] > 0
        assert _eq(o["K"], g["K"][b]) and _eq(o["sd"], g["sd"][b]) and _eq(o["u"], g["sdd"][b])
        n_ok += o["status"] == 0
    assert 0 < n_ok < g["way"].shape[0]
    r = golden("retry_row_problems")
    for i in range(int(r["n"])):
        t = "c%d_" % i
        o = orc.solve_rows(r[t + "rows"], r[t + "xb"], r[t + "grid"], float(r[t + "sd_start"]), 0.0)
        assert o["status"] == int(r[t + "status"]), i
        assert _eq(o["K"], r[t + "K"]) and _eq(o["sd"], r[t + "sd"]) and _eq(o["u"], r[t + "sdd"]), i


@pytest.mark.parametrize("name", ["deg6", "deg20", "scaled14"])
def test_shortcut_stress_rows_vs_reference_golden(golden, name):
    """VERDICT r1 #4: the near-degenerate / badly scaled raw-row problems that stress the scan kernel's Seidel shortcuts.
    The golden holds the REFERENCE's own seidelWrapper results on them (tests/golden/make_golden.py shortcut_rows);
    the restatement must reproduce them bit for bit, so the GPU-vs-oracle tests on these inputs are pinned too."""
    from problems import SHORTCUT_SETS
    g = golden("shortcut_rows_" + name)
    gen, args = SHORTCUT_SETS[name]
    rows, xb = gen(*args)
    B, G = rows.shape[:2]
    grid = np.linspace(0, 1, G)
    nfail = 0
    for i in range(B):
        o = orc.solve_rows(rows[i], xb[i], grid, 0.0, 0.0)
        assert o["status"] == g[name + "_status"][i], i
        assert np.array_equal(o["K"], g[name + "_K"][i], equal_nan=True), i
        if o["status"] == 0:
            assert np.array_equal(o["sd"], g[name + "_sd"][i]) and np.array_equal(o["u"], g[name + "_sdd"][i]), i
        else:
            nfail += 1
    assert nfail == int((g[name + "_status"] != 0).sum())
