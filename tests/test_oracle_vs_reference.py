"""CPU: differential test of the oracle against the UNMODIFIED reference, on random problems beyond the other fixtures.
What the reference computed on these inputs (and its public API) is stored in tests/golden/oracle_vs_reference.npz,
written by `python tests/golden/make_golden.py oracle_vs_reference` from the reference build (oracle/_ref); the inputs
are regenerated here from the same seeds."""
import json

import numpy as np
import pytest

from oracle import oracle as orc
from problems import make_path


@pytest.fixture(scope="module")
def ref(golden):
    """{name: array} of the reference's results; a name absent for an `sd` means the reference returned None."""
    return golden("oracle_vs_reference")


@pytest.mark.parametrize("vel_active", [False, True])
def test_random_paths_bit_exact(ref, vel_active):
    ss = np.linspace(0, 1, 5)
    for seed in range(5000, 5040):
        key = "paths%d_%d_" % (vel_active, seed)
        G = 60 + (seed % 5) * 35
        grid = np.linspace(0, 1, G)
        way, vlim, alim = make_path(seed, vel_active=vel_active)
        sd0 = 0.0 if seed % 3 else 0.02
        K, sd, sdd = ref[key + "K"], ref.get(key + "sd"), ref.get(key + "sdd")
        c = orc.cubic_spline_fit(ss, way)
        assert np.array_equal(c, ref[key + "c"])
        o = orc.solve_velacc(c, ss, grid, vlim, alim, True, sd0, 0.0)
        assert np.array_equal(o["K"], K, equal_nan=True)
        if sd is None:
            assert o["status"] == 3
        else:
            assert np.array_equal(o["sd"], sd, equal_nan=True) and np.array_equal(o["u"], sdd, equal_nan=True)


def test_lp_shims_random(ref):
    """Random LPs with random warm-start pairs through the reference's solve_lp2d shim (pyx:65-87)."""
    rng = np.random.RandomState(0)
    for trial in range(300):
        n = rng.randint(1, 40)
        v = rng.randn(3)
        a, b = rng.randn(2, n)
        c = -rng.rand(n) if trial % 2 else rng.randn(n) * 0.3 - 0.5
        low, high = np.r_[-1.0, -2.0], np.r_[1.5, 0.7]
        act = rng.randint(-4, n + 2, size=2)
        r0, val0, var0, act0 = (ref["lp_" + k][trial] for k in ("ok", "val", "var", "act"))
        r1, val1, var1, act1 = orc.lp2d(v, a, b, c, low, high, act)
        assert r0 == r1
        if r0:
            assert val0 == val1 and np.array_equal(np.asarray(var0), var1) and np.array_equal(np.asarray(act0), act1)


def test_periodic_splines_random_vs_scipy():
    """bc_type='periodic': the restated condensed cyclic system against scipy on random closed curves (n = 2..40,
    non-uniform knots); the reference's SplineInterpolator is a thin wrapper over exactly this scipy call."""
    from scipy.interpolate import CubicSpline
    rng = np.random.RandomState(5)
    for trial in range(60):
        n = [2, 3, 4, 5][trial] if trial < 4 else rng.randint(4, 41)
        x = np.cumsum(0.05 + rng.rand(n))
        y = rng.randn(n, 1 + trial % 4)
        y[-1] = y[0]
        assert np.array_equal(orc.cubic_spline_fit(x, y, "periodic"), CubicSpline(x, y, bc_type="periodic").c), (trial, n)


def test_ubound_random_vs_reference(ref):
    """`ubound` of a constraint (seidelWrapper.__init__, pyx:512-515): random u-intervals and x-bounds through the reference's
    own TOPPRA (parameterisation, feasible and reachable sets) against the oracle's stateful wrapper with the same rows."""
    ss = np.linspace(0, 1, 5)
    rng = np.random.RandomState(17)
    for seed in range(6000, 6012):
        key = "ubound_%d_" % seed
        G = 40 + (seed % 4) * 25
        grid = np.linspace(0, 1, G)
        way, vlim, alim = make_path(seed)
        width = 0.05 + 1.5 * rng.rand()
        ub = np.stack((-width * (0.5 + rng.rand(G)), width * (0.5 + rng.rand(G))), axis=1)
        xb = np.stack((np.zeros(G), 20.0 + 80 * rng.rand(G)), axis=1)
        sdd, sd, K = ref.get(key + "sdd"), ref.get(key + "sd"), ref[key + "K"]
        X, L = ref[key + "X"], ref[key + "L"]
        # the same rows for the oracle: acceleration rows from its own K1 restatement, velocity bound intersected with xb
        c = orc.cubic_spline_fit(ss, way)
        lin = orc.solve_velacc(c, ss, grid, vlim, alim, True, 0, 0, want_rows=True)
        xbo = np.stack((np.maximum(lin["xbound"][:, 0], xb[:, 0]), np.minimum(lin["xbound"][:, 1], xb[:, 1])), axis=1)
        o = orc.solve_rows(lin["rows"], xbo, grid, 0.0, 0.0, ubound=ub)
        assert np.array_equal(o["K"], K, equal_nan=True), seed
        if sd is None:
            assert o["status"] == 3
        else:
            assert np.array_equal(o["sd"], sd, equal_nan=True) and np.array_equal(o["u"], sdd, equal_nan=True), seed
        w = orc.Wrapper(grid, lin["rows"], xbo, ub)
        assert np.array_equal(w.compute_feasible_sets(), X, equal_nan=True), seed
        # reachable sets: the reference runs the feasible-set pass first on the SAME wrapper object (stateful warm start)
        Lo = np.zeros((G, 2))
        Lo[0] = [0.0, 0.2 ** 2]
        deltas = np.diff(grid)
        for i in range(G - 1):
            dq = deltas[i - 1]
            obj = np.array([-2 * dq, -1.0])
            o1 = w.solve_stagewise_optim(i, None, obj, Lo[i, 0], Lo[i, 1], X[i + 1, 0], X[i + 1, 1])
            o0 = w.solve_stagewise_optim(i, None, -obj, Lo[i, 0], Lo[i, 1], X[i + 1, 0], X[i + 1, 1])
            Lo[i + 1] = [o0[1] + 2 * dq * o0[0], o1[1] + 2 * dq * o1[0]]
            if Lo[i + 1, 0] < 0:
                Lo[i + 1, 0] = 0
            if np.isnan(Lo[i + 1]).any():
                break
        assert np.array_equal(Lo, L, equal_nan=True), seed


def test_propose_gridpoints_and_spline_time_stamps_random_vs_reference(ref, monkeypatch):
    """The engine double's restatements (tests/cpu_engine.py) of propose_gridpoints and of ParametrizeSpline's time-stamp
    recurrence against the reference on random paths / velocity profiles with stalls and dropped knots."""
    import torch
    import cpu_engine
    ss = np.linspace(0, 1, 5)
    rng = np.random.RandomState(23)
    for seed in range(7000, 7008):
        way, _, _ = make_path(seed, dof=3 + seed % 4)
        kw = dict(max_err_threshold=10 ** rng.uniform(-4, -1.5), max_seg_length=rng.uniform(0.04, 0.4),
                  min_nb_points=int(rng.randint(5, 150)))
        want = ref["grid_%d_proposed" % seed]
        c = orc.cubic_spline_fit(ss, way)
        grid, glen, st = cpu_engine.propose_gridpoints(torch.from_numpy(c[None]), torch.from_numpy(ss), max_points=4096, **kw)
        assert int(st[0]) == 0 and int(glen[0]) == len(want) and np.array_equal(grid[0, :len(want)].numpy(), want), seed
        G = 80
        g = np.linspace(0, 1, G)
        vel = np.abs(rng.randn(G)) + 0.05
        vel[rng.randint(1, G - 1, size=3)] = 0.0              # stalled gridpoints: the 5 s rule
        vel[10:12] = 1e9                                      # increments below 1e-8: dropped knots
        knots = ref["grid_%d_time_stamps" % seed]             # ParametrizeSpline(path, g, vel).ss_waypoints
        t, s, nk = cpu_engine.spline_time_stamps(torch.from_numpy(vel[None]), torch.from_numpy(g))
        n = int(nk[0])
        assert n == len(knots) and np.array_equal(t[0, :n].numpy(), knots), seed


def test_toppra_sd_random_vs_reference(ref, monkeypatch):
    """TOPPRAsd (desired_duration_algorithm.py:42-191) through the package's host code on the engine double (two
    TOPPRAsd-rule scans + the duration bisection) against the reference class on random paths and desired durations
    (0.6, 1.3, 2.2 or 5 times the time-optimal duration)."""
    import cpu_engine
    ta = cpu_engine.install(monkeypatch)
    ss = np.linspace(0, 1, 5)
    for seed in range(8000, 8010):
        key = "sd_%d_" % seed
        G = 50 + (seed % 3) * 30
        grid = np.linspace(0, 1, G)
        way, vlim, alim = make_path(seed, vel_active=(seed % 4 == 0))
        want_t = float(ref[key + "duration"])
        sdd, sd, K = ref[key + "sdd"], ref[key + "sd"], ref[key + "K"]
        mine = ta.algorithm.TOPPRAsd([ta.constraint.JointVelocityConstraint(vlim), ta.constraint.JointAccelerationConstraint(alim)],
                                     ta.SplineInterpolator(ss, way), gridpoints=grid, solver_wrapper="seidel")
        mine.set_desired_duration(want_t)
        sdd2, sd2, _, K2 = mine.compute_parameterization(0, 0, return_data=True)
        assert np.array_equal(K2, K) and np.array_equal(sd2, sd) and np.array_equal(sdd2, sdd), seed


def test_univariate_spline_interpolator_vs_reference(ref, monkeypatch):
    """UnivariateSplineInterpolator (interpolator.py:508-581): the package's PPoly conversion of the FITPACK fits against
    the reference class — evaluations to rounding, the retimed solution to 1e-9 (the reference evaluates B-splines, this
    package local cubics, so the LP rows differ in the last bits)."""
    import cpu_engine
    ta = cpu_engine.install(monkeypatch)
    for seed in range(4):
        key = "univariate_%d_" % seed
        rng = np.random.RandomState(900 + seed)
        n = 25 + 10 * seed
        ss = np.sort(np.r_[0.0, rng.uniform(0.05, 2.95, n - 2), 3.0])
        way = np.stack([np.sin(ss), np.cos(1.7 * ss), 0.2 * ss ** 2 - ss, np.sin(0.5 * ss) * ss], axis=1)
        way += 0.03 * rng.randn(n, 4)
        mine = ta.UnivariateSplineInterpolator(ss, way)
        s = np.linspace(0, 3.0, 301)
        for order in (0, 1, 2):
            np.testing.assert_allclose(mine(s, order), ref[key + "eval%d" % order], rtol=1e-10, atol=1e-10)
        assert mine.dof == int(ref[key + "dof"]) == 4 and list(mine.path_interval) == list(ref[key + "path_interval"])
        vlim, alim = np.array([[-2.0, 2.0]] * 4), np.array([[-6.0, 5.0]] * 4)
        grid = np.linspace(0, 3.0, 151)
        inst = ta.algorithm.TOPPRA([ta.constraint.JointVelocityConstraint(vlim), ta.constraint.JointAccelerationConstraint(alim)],
                                   mine, gridpoints=grid, solver_wrapper="seidel")
        sdd2, sd2, _, K2 = inst.compute_parameterization(0, 0, return_data=True)
        sdd, sd, K = ref[key + "sdd"], ref[key + "sd"], ref[key + "K"]
        np.testing.assert_allclose(K2, K, rtol=1e-9, atol=1e-10)
        np.testing.assert_allclose(sd2, sd, rtol=1e-9, atol=1e-10)
        np.testing.assert_allclose(sdd2, sdd, rtol=1e-6, atol=1e-7)


FUZZ_SLICE_SEEDS = range(400000, 400120)


def test_randomly_shaped_problems_vs_reference(golden):
    """A slice of the campaign of scripts/fuzz_oracle_vs_reference.py (dof 1..14, 2..12 knots, 2..400 gridpoints, non-uniform
    knots and grids, every boundary condition, both discretisations, non-zero boundary velocities, tiny motions): spline
    coefficients, K, sd, u, status, feasible sets, propose_gridpoints, time stamps, TOPPRAsd, reachable sets, torque rows,
    both output parametrizers —
    bit for bit against the reference (31 000 + 10 000 problems in the full runs, profiles/r02_fuzz_oracle_vs_reference.txt)."""
    import importlib.util
    import os
    spec = importlib.util.spec_from_file_location(
        "fuzz_oracle_vs_reference", os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "scripts",
                                                 "fuzz_oracle_vs_reference.py"))
    fuzz = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(fuzz)
    fuzz.REPLAY = fuzz.unpack(golden("fuzz_slice"))   # the reference's results on these problems (make_golden.py)
    try:
        for seed in FUZZ_SLICE_SEEDS:
            rng = np.random.RandomState(seed)
            p = fuzz.random_problem(rng)
            fuzz.begin(seed)
            try:
                fuzz.check_all(p, rng)
            except AssertionError as e:
                raise AssertionError("seed %d: %s" % (seed, e))
            except Exception:
                pass            # the reference itself rejected the input (as in the campaign)
    finally:
        fuzz.release()          # the campaign installs the engine double process-wide
    assert fuzz.COUNTS.get("TOPPRAsd", 0) >= 10 and fuzz.COUNTS.get("propose_gridpoints", 0) >= 80


def test_public_classes_have_the_reference_methods_and_arguments(ref):
    """Introspection of the reference build against this package: every public class the two share has the reference's public
    methods / properties, and every shared callable takes the reference's argument names in the reference's order.  The
    reference's side (names, members, argument lists) is stored in the golden file as JSON."""
    import inspect
    import toppra_b200 as tb
    import toppra_b200.simplepath

    def params(f):
        try:
            return [p for p in inspect.signature(f).parameters if p not in ("args", "kwargs")]
        except (TypeError, ValueError):
            return None

    api = json.loads(str(ref["public_api_json"]))
    openrave_only = {"compute_rave_trajectory"}
    seen, problems = set(), []
    pairs = (("toppra", tb), ("toppra.algorithm", tb.algorithm), ("toppra.constraint", tb.constraint),
             ("toppra.parametrizer", tb.parametrizer), ("toppra.interpolator", tb.interpolator),
             ("toppra.simplepath", tb.simplepath), ("toppra.solverwrapper", tb.solverwrapper))
    for mod_r, mod_t in pairs:
        for name, entry in sorted(api[mod_r].items()):
            if name in seen or not hasattr(mod_t, name):
                continue
            mine = getattr(mod_t, name)
            seen.add(name)
            if entry["kind"] == "class":
                for member, pr in entry["members"].items():
                    if member in openrave_only:
                        continue
                    if not hasattr(mine, member):
                        problems.append("%s.%s missing" % (name, member))
                        continue
                    pt = params(getattr(mine, member)) if pr is not None else None
                    if pr is not None and pt is not None and [a for a in pr if a in pt] != pr:
                        problems.append("%s.%s(%s) vs (%s)" % (name, member, ", ".join(pr), ", ".join(pt)))
                    elif pr is not None and pt is not None and pt[:len(pr)] != pr and [a for a in pt if a in pr] != pr:
                        problems.append("%s.%s argument order" % (name, member))
            else:
                pr, pt = entry["params"], params(mine)
                if pr is not None and pt is not None and pt[:len(pr)] != pr:
                    problems.append("%s(%s) vs (%s)" % (name, ", ".join(pr), ", ".join(pt)))
    assert len(seen) >= 25, sorted(seen)
    assert not problems, problems
