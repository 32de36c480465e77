#!/usr/bin/env python
"""CPU campaign: the oracle (oracle/toppra_oracle.c, which the kernels are pinned to bit for bit on the GPU) against the
UNMODIFIED reference build (oracle/_ref) on randomly SHAPED problems — far more shapes than the committed tests: dof 1..14,
2..12 knots on non-uniform breakpoints, 2..400 gridpoints on non-uniform grids, all spline boundary conditions, collocation
and interpolation, active velocity bounds, non-zero boundary velocities (admissible or not), near-degenerate paths.
Any mismatch is printed with the seed that reproduces it.

usage: python scripts/fuzz_oracle_vs_reference.py [--minutes M] [--seed S]      (needs the reference build, oracle/_ref)

Every result of the reference goes through `theirs()`, so a slice of the campaign can be recorded once
(tests/golden/make_golden.py fuzz_slice) and replayed without the reference (tests/test_oracle_vs_reference.py)."""
import argparse
import os
import sys
import time
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
warnings.filterwarnings("ignore")

from oracle import oracle as orc  # noqa: E402

ta = algo = constraint = interp = ParametrizeSpline = None


def load():
    """Import the reference build (oracle/_ref) for live runs."""
    global ta, algo, constraint, interp, ParametrizeSpline
    from oracle.ref_loader import load_reference
    ta = load_reference()
    import toppra.algorithm as algo
    import toppra.constraint as constraint
    import toppra.interpolator as interp
    from toppra.parametrizer import ParametrizeSpline


REPLAY = None      # {key: array}: the reference's results as recorded into RECORD; None = call the reference
RECORD = None      # dict that collects the reference's results of a live run (stored with pack())
_PREFIX = [""]


class ReferenceRaised(Exception):
    """Replay of a reference call that raised."""


def begin(seed):
    """Key the reference's results of the next problem by its seed."""
    _PREFIX[0] = "%d/" % seed


def _encode(key, value, out, digest):
    if digest and not isinstance(value, (str, tuple, list)) and value is not None and np.size(value) > 1:
        d = Digest.of(value)
        out[key + "!shape"], out[key + "!sha256"] = np.array(d.shape, dtype=np.int64), np.array(d.sha)
    elif value is None:
        out[key + "!none"] = np.array(True)
    elif isinstance(value, str):
        out[key + "!str"] = np.array(value)
    elif isinstance(value, (tuple, list)):
        out[key + "!len"] = np.array(len(value))
        for i, v in enumerate(value):
            _encode("%s/%d" % (key, i), v, out, digest)
    else:
        out[key] = np.asarray(value)


def _decode(key, data):
    if not any(k in data for k in (key, key + "!raise", key + "!none", key + "!str", key + "!len", key + "!sha256")):
        raise AssertionError("no recorded reference result for " + key)
    if key + "!raise" in data:
        raise ReferenceRaised(str(data[key + "!raise"]))
    if key + "!none" in data:
        return None
    if key + "!sha256" in data:
        return Digest(data[key + "!shape"], data[key + "!sha256"])
    if key + "!str" in data:
        return str(data[key + "!str"])
    if key + "!len" in data:
        return tuple(_decode("%s/%d" % (key, i), data) for i in range(int(data[key + "!len"])))
    return data[key]


def pack(record):
    """RECORD as five arrays (keys, kinds, shapes, numbers, strings): one file entry per key would cost more than the data."""
    keys = sorted(record)
    kinds, shapes, nums, strs = [], [], [], []
    for k in keys:
        v = np.asarray(record[k])
        if v.dtype.kind == "U":
            kinds.append(1)
            strs.append(str(v))
        else:
            kinds.append(0)
            shapes += [v.ndim] + list(v.shape)
            nums.append(v.astype(np.float64).ravel())
    return {"keys": np.array(keys), "kinds": np.array(kinds, dtype=np.int8), "shapes": np.array(shapes, dtype=np.int64),
            "numbers": np.concatenate(nums) if nums else np.zeros(0), "strings": np.array(strs)}


def unpack(packed):
    """The inverse of pack()."""
    out, shapes, nums, strs = {}, iter(packed["shapes"].tolist()), packed["numbers"], iter(packed["strings"].tolist())
    pos = 0
    for k, kind in zip(packed["keys"].tolist(), packed["kinds"].tolist()):
        if kind == 1:
            out[k] = np.array(next(strs))
        else:
            shape = tuple(next(shapes) for _ in range(next(shapes)))
            n = int(np.prod(shape))
            out[k] = nums[pos:pos + n].reshape(shape)
            pos += n
    return out


def theirs(what, fn, digest=True):
    """The reference's result `fn()` (arrays, numbers, strings, None or tuples of them): live, recorded, or replayed.
    digest=True: its arrays are only compared with eq(), so a recording keeps their digests; digest=False for results
    that are computed with or compared to a tolerance."""
    key = _PREFIX[0] + what
    if REPLAY is not None:
        return _decode(key, REPLAY)
    try:
        value = fn()
    except Exception as e:
        if RECORD is not None:
            RECORD[key + "!raise"] = np.array(type(e).__name__)
        raise
    if RECORD is not None:
        _encode(key, value, RECORD, digest)
    return value


class Digest(object):
    """A recorded reference array that is only ever compared bit for bit (eq): its shape and a SHA-256 of its values with
    NaNs and signed zeros folded, so that two arrays have the same digest exactly when eq() holds for them."""

    def __init__(self, shape, sha):
        self.shape, self.sha = tuple(int(n) for n in shape), str(sha)

    @staticmethod
    def of(a):
        import hashlib
        a = np.asarray(a, dtype=float)
        a = np.where(np.isnan(a), np.nan, a) + 0.0
        return Digest(a.shape, hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest())

    def __len__(self):
        return self.shape[0]

    def __eq__(self, other):
        return isinstance(other, Digest) and (self.shape, self.sha) == (other.shape, other.sha)


def eq(a, b):
    if isinstance(a, Digest) or isinstance(b, Digest):
        return (a if isinstance(a, Digest) else Digest.of(a)) == (b if isinstance(b, Digest) else Digest.of(b))
    return np.array_equal(np.asarray(a, dtype=float), np.asarray(b, dtype=float), equal_nan=True)


from problems import random_shaped_problem as random_problem  # noqa: E402


def check_solve(p):
    def spline():
        path = ta.SplineInterpolator(p["ss"], p["way"], bc_type=p["bc"])
        return path.cspl.c if p["way"].shape[0] > 1 else None

    def solve():
        path = ta.SplineInterpolator(p["ss"], p["way"], bc_type=p["bc"])
        cons = [constraint.JointVelocityConstraint(p["vlim"]),
                constraint.JointAccelerationConstraint(p["alim"], discretization_scheme=p["interp"])]
        inst = algo.TOPPRA(cons, path, gridpoints=p["grid"], solver_wrapper="seidel")
        sdd, sd, _, K = inst.compute_parameterization(p["sd0"], p["sd1"], return_data=True)
        code = inst.problem_data.return_code
        assert algo.ParameterizationReturnCode.__members__[code.name] is code
        return sdd, sd, K, code.name

    def feasible_sets():
        path = ta.SplineInterpolator(p["ss"], p["way"], bc_type=p["bc"])
        cons = [constraint.JointVelocityConstraint(p["vlim"]),
                constraint.JointAccelerationConstraint(p["alim"], discretization_scheme=p["interp"])]
        return algo.TOPPRA(cons, path, gridpoints=p["grid"], solver_wrapper="seidel").compute_feasible_sets()

    c = orc.cubic_spline_fit(p["ss"], p["way"], p["bc"])
    ref_c = theirs("spline", spline, digest=False)
    if p["bc"] == "not-a-knot" and len(p["ss"]) != 3:
        assert eq(c, ref_c), "spline coefficients"
    else:
        # not pinned by scipy: clamped / natural go through LAPACK's banded solve, the 3-knot parabola through a DENSE solve
        # whose OpenBLAS kernels use FMA where the CPU has it (DESIGN.md section 2) -> agree to rounding, then continue
        # with the reference's coefficients so that everything downstream is compared bit for bit
        np.testing.assert_allclose(c, ref_c, rtol=1e-11, atol=1e-12 * max(1.0, np.abs(ref_c).max()))
        c = np.ascontiguousarray(ref_c)
    sdd, sd, K, code = theirs("solve", solve)
    o = orc.solve_velacc(c, p["ss"], p["grid"], p["vlim"], p["alim"], bool(p["interp"]), p["sd0"], p["sd1"])
    assert eq(o["K"], K), "K"
    want = {"Ok": 0, "ErrUnknown": 1, "ErrShortPath": 2, "FailUncontrollable": 3, "ErrForwardPassFail": 4}[code]
    assert o["status"] == want, ("status", o["status"], code)
    if sd is not None:
        assert eq(o["sd"], sd) and eq(o["u"], sdd), "sd / u"
    X = theirs("feasible_sets", feasible_sets)
    lin = orc.solve_velacc(c, p["ss"], p["grid"], p["vlim"], p["alim"], bool(p["interp"]), 0, 0, want_rows=True)
    w = orc.Wrapper(p["grid"], lin["rows"], lin["xbound"])
    assert eq(w.compute_feasible_sets(), X), "feasible sets"
    return want


def check_frows(p, rng):
    if p["way"].shape[0] < 2:
        return
    c = orc.cubic_spline_fit(p["ss"], p["way"])
    import torch
    import cpu_engine
    kw = dict(max_err_threshold=10 ** rng.uniform(-5, -1), max_seg_length=rng.uniform(0.02, 0.6) * p["ss"][-1],
              min_nb_points=int(rng.randint(2, 200)))
    def proposed():
        try:
            return np.asarray(interp.propose_gridpoints(ta.SplineInterpolator(p["ss"], p["way"]), **kw))
        except ValueError:
            return None

    want = theirs("propose_gridpoints", proposed)
    grid, glen, st = cpu_engine.propose_gridpoints(torch.from_numpy(c[None]), torch.from_numpy(p["ss"]), max_points=8192, **kw)
    if int(st[0]) < 0:
        pass                                    # more than max_points gridpoints needed: the cap of this harness, not a result
    elif want is None:
        assert int(st[0]) != 0, "propose_gridpoints: the reference raised"
    else:
        count("propose_gridpoints")
        assert int(st[0]) == 0 and int(glen[0]) == len(want) and eq(grid[0, :len(want)].numpy(), want), "propose_gridpoints"
    G = len(p["grid"])
    if G >= 3:
        vel = np.abs(rng.randn(G)) * 10 ** rng.uniform(-2, 1) + 1e-3
        if rng.rand() < 0.5:
            vel[rng.randint(0, G, size=2)] = 0.0
        if rng.rand() < 0.3:
            vel[G // 3:G // 3 + 2] = 1e10
        def knots():
            try:
                return ParametrizeSpline(ta.SplineInterpolator(p["ss"], p["way"]), p["grid"], vel).ss_waypoints
            except Exception:
                return None

        want = theirs("time_stamps", knots)
        if want is None:
            return
        t, s, nk = cpu_engine.spline_time_stamps(torch.from_numpy(vel[None]), torch.from_numpy(p["grid"]))
        k = int(nk[0])
        count("time stamps")
        assert k == len(want) and eq(t[0, :k].numpy(), want), "ParametrizeSpline time stamps"


_MINE = []
COUNTS = {}


def count(what):
    COUNTS[what] = COUNTS.get(what, 0) + 1


def mine():
    """toppra_b200 with its kernels replaced by the oracle-backed engine double (tests/cpu_engine.py)."""
    if not _MINE:
        import pytest
        import cpu_engine
        patch = pytest.MonkeyPatch()
        _MINE.extend([cpu_engine.install(patch), patch])
    return _MINE[0]


def release():
    """Undo the engine double (for callers that run inside another test process)."""
    if _MINE:
        _MINE[1].undo()
        del _MINE[:]


def check_sd_and_reachable(p, rng):
    """TOPPRAsd and compute_reachable_sets through the PACKAGE's host code on the engine double against the reference
    classes (the device forms of these two are pinned to the same restatements by the 16-path goldens on the GPU)."""
    if p["bc"] != "not-a-knot" or len(p["ss"]) == 3 or len(p["grid"]) < 3:
        return
    tb = mine()
    mk = lambda pkg, cons: [cons.JointVelocityConstraint(p["vlim"]),  # noqa: E731
                            cons.JointAccelerationConstraint(p["alim"], discretization_scheme=p["interp"])]
    ref_path = lambda: ta.SplineInterpolator(p["ss"], p["way"])  # noqa: E731
    ours = tb.SplineInterpolator(p["ss"], p["way"])
    sd_f = theirs("fast_sd", lambda: algo.TOPPRA(mk(algo, constraint), ref_path(), gridpoints=p["grid"],
                                                 solver_wrapper="seidel").compute_parameterization(0, 0)[1], digest=False)
    if sd_f is not None and np.all(sd_f[1:] + sd_f[:-1] > 0):
        t_fast = np.sum(2 * np.diff(p["grid"]) / (sd_f[1:] + sd_f[:-1]))
        want_t = t_fast * rng.choice([0.5, 1.0, 1.2, 2.0, 7.0, 1e3])

        def desired_duration():
            a = algo.TOPPRAsd(mk(algo, constraint), ref_path(), gridpoints=p["grid"], solver_wrapper="seidel")
            a.set_desired_duration(want_t)
            return a.compute_parameterization(0, 0, return_data=True) + (a.problem_data.return_code.name,)

        *ra, code_a = theirs("TOPPRAsd", desired_duration)
        b = tb.algorithm.TOPPRAsd(mk(tb.algorithm, tb.constraint), ours, gridpoints=p["grid"], solver_wrapper="seidel")
        b.set_desired_duration(want_t)
        rb = b.compute_parameterization(0, 0, return_data=True)
        count("TOPPRAsd")
        assert code_a == b.problem_data.return_code.name, "TOPPRAsd return code"
        for x, y, what in zip(ra, rb, ("sdd", "sd", "v", "K")):
            assert (x is None and y is None) or eq(x, y), "TOPPRAsd " + what
    sdmin = 0.0 if rng.rand() < 0.5 else 10 ** rng.uniform(-3, -0.5)
    sdmax = sdmin + (0.0 if rng.rand() < 0.3 else 10 ** rng.uniform(-3, 0))
    for v in ("sdmin", "sdmax"):
        val = locals()[v]
        while float(val) ** 2 != float(val) * float(val):
            val = float(np.nextafter(val, 10.0))
        if v == "sdmin":
            sdmin = val
        else:
            sdmax = val
    La = theirs("reachable_sets", lambda: algo.TOPPRA(mk(algo, constraint), ref_path(), gridpoints=p["grid"],
                                                      solver_wrapper="seidel").compute_reachable_sets(sdmin, sdmax))
    Lb = tb.algorithm.TOPPRA(mk(tb.algorithm, tb.constraint), ours, gridpoints=p["grid"],
                             solver_wrapper="seidel").compute_reachable_sets(sdmin, sdmax)
    count("reachable sets")
    assert eq(La, Lb), "reachable sets"


def check_parametrizers(p, rng):
    """ParametrizeConstAccel (time grid and accelerations bit for bit, evaluations to rounding) and ParametrizeSpline
    (knot times bit for bit, the clamped re-fit and its evaluations to rounding) on the solved velocity profile."""
    if p["bc"] != "not-a-knot" or len(p["ss"]) == 3 or len(p["grid"]) < 3:
        return
    tb = mine()
    ref_path = lambda: ta.SplineInterpolator(p["ss"], p["way"])  # noqa: E731
    ours = tb.SplineInterpolator(p["ss"], p["way"])

    def velocities():
        cons = [constraint.JointVelocityConstraint(p["vlim"]), constraint.JointAccelerationConstraint(p["alim"], p["interp"])]
        return algo.TOPPRA(cons, ref_path(), gridpoints=p["grid"], solver_wrapper="seidel").compute_parameterization(0, 0)[1]

    def const_accel():
        from toppra.parametrizer import ParametrizeConstAccel
        return ParametrizeConstAccel(ref_path(), p["grid"], sd)

    sd = theirs("parametrizer_sd", velocities, digest=False)
    if sd is None or not np.all(sd[1:] + sd[:-1] > 0):
        return
    a_ts, a_us, a_duration = theirs("ConstAccel", lambda: (lambda a: (a._ts, a._us, a.duration))(const_accel()))
    b = tb.ParametrizeConstAccel(ours, p["grid"], sd)
    count("ParametrizeConstAccel")
    assert eq(a_ts, b._ts) and eq(a_us, b._us) and a_duration == b.duration, "ConstAccel time grid"
    ts = np.r_[0.0, np.sort(rng.uniform(0, a_duration, 30)), a_duration]
    scale = max(1.0, np.abs(p["way"]).max())
    wants = theirs("ConstAccel_eval", lambda: (lambda a: [a(ts, order) for order in (0, 1, 2)])(const_accel()),
                   digest=False)
    for order, tol in ((0, 1e-11), (1, 1e-9), (2, 1e-7)):
        want = wants[order]
        np.testing.assert_allclose(b(ts, order), want, rtol=tol, atol=tol * max(scale, np.abs(want).max()),
                                   err_msg="ConstAccel order %d" % order)
    sa_knots, sa_duration = theirs("Spline", lambda: (lambda s: (s.ss_waypoints, s.duration))(
        ParametrizeSpline(ref_path(), p["grid"], sd)))
    sb = tb.ParametrizeSpline(ours, p["grid"], sd)
    count("ParametrizeSpline")
    assert eq(sa_knots, sb.ss_waypoints) and sa_duration == sb.duration, "ParametrizeSpline knots"
    ts = np.linspace(0, sa_duration, 25)
    want = theirs("Spline_eval", lambda: ParametrizeSpline(ref_path(), p["grid"], sd)(ts), digest=False)
    np.testing.assert_allclose(sb(ts), want, rtol=1e-9, atol=1e-9 * max(scale, np.abs(want).max()), err_msg="ParametrizeSpline q")


def _ub_class(cons):
    class UB(cons.LinearConstraint):
        """Acceleration rows + a u-interval and an x-interval per gridpoint (seidelWrapper.__init__, pyx:512-520)."""

        def __init__(self, acc, ub, xb):
            super(UB, self).__init__()
            self.acc, self.ub, self.xb = acc, ub, xb
            self.discretization_type = acc.discretization_type
            self.identical = True

        def get_dof(self):
            return self.acc.get_dof()

        def compute_constraint_params(self, path, gridpoints, *a):
            pa, pb, pc, F, g, _, _ = self.acc.compute_constraint_params(path, gridpoints)
            return pa, pb, pc, F, g, self.ub, self.xb

    return UB


def check_ubound(p, rng):
    """A user constraint that returns `ubound` / `xbound` next to its rows: parameterisation, feasible and reachable sets
    through the package's generic-constraint path (host 7-tuple -> rows_canlinear -> records with the u-bound pair)."""
    if p["bc"] != "not-a-knot" or len(p["ss"]) == 3 or len(p["grid"]) < 3 or p["way"].shape[1] > 7:
        return
    tb = mine()
    G = len(p["grid"])
    width = 10 ** rng.uniform(-1.5, 1.0) * max(1e-3, np.abs(p["alim"]).max())
    ub = np.stack((-width * (0.5 + rng.rand(G)), width * (0.5 + rng.rand(G))), axis=1)
    xb = np.stack((np.zeros(G), 10 ** rng.uniform(-2, 3) * (0.5 + rng.rand(G))), axis=1)
    def run(pkg, cons, path):
        mk = lambda: [cons.JointVelocityConstraint(p["vlim"]),  # noqa: E731
                      _ub_class(cons)(cons.JointAccelerationConstraint(p["alim"], p["interp"]), ub, xb)]
        inst = pkg.TOPPRA(mk(), path, gridpoints=p["grid"], solver_wrapper="seidel")
        res = inst.compute_parameterization(0, 0, return_data=True)
        X = pkg.TOPPRA(mk(), path, gridpoints=p["grid"], solver_wrapper="seidel").compute_feasible_sets()
        L = pkg.TOPPRA(mk(), path, gridpoints=p["grid"], solver_wrapper="seidel").compute_reachable_sets(0.0, 0.25)
        return (res[0], res[1], res[3], X, L)

    out = [theirs("ubound", lambda: run(algo, constraint, ta.SplineInterpolator(p["ss"], p["way"]))),
           run(tb.algorithm, tb.constraint, tb.SplineInterpolator(p["ss"], p["way"]))]
    count("ubound")
    for x, y, what in zip(out[0], out[1], ("sdd", "sd", "K", "feasible sets", "reachable sets")):
        assert (x is None and y is None) or (x is not None and y is not None and eq(x, y)), "ubound " + what


def check_other_constraints(p, rng):
    """JointVelocityConstraintVarying (limits as a function of s) and JointTorqueConstraint (dry friction, both schemes)."""
    dof = p["way"].shape[1]
    if p["bc"] != "not-a-knot" or len(p["ss"]) == 3 or len(p["grid"]) < 3 or len(p["grid"]) > 200:
        return
    from problems import inv_dyn_numpy
    tb = mine()
    k0, k1 = 0.05 + rng.rand(), rng.rand() / p["ss"][-1]
    vlim, span = p["vlim"], p["ss"][-1]
    def run(pkg, cons, path):
        var = cons.JointVelocityConstraintVarying(lambda s: vlim * (k0 + k1 * s))
        inst = pkg.TOPPRA([var, cons.JointAccelerationConstraint(p["alim"], p["interp"])], path, gridpoints=p["grid"],
                          solver_wrapper="seidel")
        res = inst.compute_parameterization(0, 0, return_data=True)
        item = [res[0], res[1], res[3], var.compute_constraint_params(path, p["grid"])[-1]]
        if 2 <= dof <= 7:
            taulim = np.stack((-(20 + 30 * np.arange(1, dof + 1) / dof), 25 + 30 * np.arange(1, dof + 1) / dof), axis=1)
            tau = cons.JointTorqueConstraint(inv_dyn_numpy, taulim, 0.3 * np.ones(dof), discretization_scheme=p["interp"])
            inst = pkg.TOPPRA([cons.JointVelocityConstraint(p["vlim"]), tau], path, gridpoints=p["grid"],
                              solver_wrapper="seidel")
            res = inst.compute_parameterization(0, 0, return_data=True)
            item += [res[0], res[1], res[3]]
        return item

    out = [theirs("other_constraints", lambda: run(algo, constraint, ta.SplineInterpolator(p["ss"], p["way"]))),
           run(tb.algorithm, tb.constraint, tb.SplineInterpolator(p["ss"], p["way"]))]
    count("varying velocity limits" + (" + JointTorqueConstraint" if len(out[0]) > 4 else ""))
    names = ("varying: sdd", "varying: sd", "varying: K", "varying: xbound", "joint torque: sdd", "joint torque: sd",
             "joint torque: K")
    for x, y, what in zip(out[0], out[1], names):
        assert (x is None and y is None) or (x is not None and y is not None and eq(x, y)), what


def check_batch(p, rng):
    """The batched entry points against per-path reference solves: B paths with per-path limits and start velocities on a
    common grid, and on the automatically proposed (ragged) grids — `BatchTOPPRA(gridpoints=None)` must equal
    `TOPPRA(constraints, path)` of the reference path by path."""
    dof, n = p["way"].shape[1], len(p["ss"])
    if n < 4 or dof > 7 or rng.rand() > 0.25:
        return
    tb = mine()
    B = int(rng.randint(2, 7))
    way = rng.randn(B, n, dof)
    vl, al = 1 + 20 * rng.rand(B, dof), 5 + 10 * rng.rand(B, dof)
    vlim, alim = np.stack((-vl, vl), axis=-1), np.stack((-al, al), axis=-1)
    sd0 = np.where(rng.rand(B) < 0.5, 0.0, 0.01)
    bpath = tb.BatchSplineInterpolator(p["ss"], way)
    cons_b = [tb.constraint.JointVelocityConstraint(vlim), tb.constraint.JointAccelerationConstraint(alim, p["interp"])]
    common = tb.BatchTOPPRA(cons_b, bpath, gridpoints=p["grid"]).compute_parameterization(sd0, 0.0).to_host()
    ragged_inst = tb.BatchTOPPRA(cons_b, bpath, gridpoints=None)
    ragged = ragged_inst.compute_parameterization(sd0, 0.0).to_host()
    glen = ragged_inst.glen.cpu().numpy()
    count("batch (common + ragged grids)")
    def solve(b, grid):
        path = ta.SplineInterpolator(p["ss"], way[b])
        cons = [constraint.JointVelocityConstraint(vlim[b]), constraint.JointAccelerationConstraint(alim[b], p["interp"])]
        inst = algo.TOPPRA(cons, path, gridpoints=grid, solver_wrapper="seidel")
        sdd, sd, _, K = inst.compute_parameterization(float(sd0[b]), 0.0, return_data=True)
        return sdd, sd, K, len(inst.gridpoints)

    for b in range(B):
        for grid, got, tag in ((p["grid"], common, "common grid"), (None, ragged, "proposed grid")):
            sdd, sd, K, G = theirs("batch/%d/%s" % (b, tag), lambda: solve(b, grid))
            G = int(G)
            if grid is None:
                assert glen[b] == G, "batch: proposed grid length"
            assert eq(got["K"][b, :G], K), "batch K (%s)" % tag
            if sd is not None:
                assert eq(got["sd"][b, :G], sd) and eq(got["sdd"][b, :G - 1], sdd), "batch sd / u (%s)" % tag
            else:
                assert got["status"][b] != 0, "batch status (%s)" % tag


def check_robust_params(p, rng):
    """RobustLinearConstraint (conic_constraint.py:47-124): the conic 6-tuple (a, b, c, P, ubound, xbound) of both packages.
    (The robust SOLVE has no reference here — ECOS is not installed — and stays pinned by tests/test_robust.py.)"""
    if p["bc"] != "not-a-knot" or len(p["ss"]) == 3 or len(p["grid"]) > 100:
        return
    tb = mine()
    ell = list(10 ** rng.uniform(-4, 0, 3))
    def run(cons, path):
        base = cons.JointAccelerationConstraint(p["alim"], p["interp"])
        return cons.RobustLinearConstraint(base, ell, p["interp"]).compute_constraint_params(path, p["grid"])

    out = [theirs("robust_params", lambda: run(constraint, ta.SplineInterpolator(p["ss"], p["way"]))),
           run(tb.constraint, tb.SplineInterpolator(p["ss"], p["way"]))]
    count("robust parameters")
    assert len(out[0]) == len(out[1]), "robust tuple length"
    for x, y, what in zip(out[0], out[1], ("a", "b", "c", "P", "ubound", "xbound")):
        assert (x is None and y is None) or (x is not None and y is not None and eq(x, y)), "robust " + what


def check_torque(p, rng):
    """vel + acc + SecondOrderConstraint.joint_torque_constraint with a numpy inverse dynamics (the reference-style callback
    route, bit-exact by construction: same user function, same call order) and JointTorqueConstraint with dry friction."""
    dof = p["way"].shape[1]
    if p["bc"] != "not-a-knot" or len(p["ss"]) == 3 or not 2 <= dof <= 7 or len(p["grid"]) > 200:
        return
    from problems import inv_dyn_numpy
    tb = mine()
    taulim = np.stack((-(20 + 30 * rng.rand(dof)), 20 + 30 * rng.rand(dof)), axis=1)
    fric = np.zeros(dof) if rng.rand() < 0.5 else 0.5 * rng.rand(dof)
    scheme = int(rng.rand() < 0.6)
    def run(pkg, cons, path):
        torque = cons.SecondOrderConstraint.joint_torque_constraint(inv_dyn_numpy, taulim, fric,
                                                                    discretization_scheme=scheme)
        inst = pkg.TOPPRA([cons.JointVelocityConstraint(p["vlim"]), cons.JointAccelerationConstraint(p["alim"]), torque],
                          path, gridpoints=p["grid"], solver_wrapper="seidel")
        return inst.compute_parameterization(p["sd0"], p["sd1"], return_data=True) + (inst.problem_data.return_code.name,)

    out = [theirs("torque", lambda: run(algo, constraint, ta.SplineInterpolator(p["ss"], p["way"]))),
           run(tb.algorithm, tb.constraint, tb.SplineInterpolator(p["ss"], p["way"]))]
    count("torque (%s)" % out[0][-1])
    for x, y, what in zip(out[0], out[1], ("sdd", "sd", "v", "K", "return code")):
        same = (x == y) if isinstance(x, str) else ((x is None and y is None) or (x is not None and y is not None and eq(x, y)))
        assert same, "torque " + what


def check_all(p, rng):
    """Every check on one problem; AssertionError on a mismatch, any other exception where the reference rejected the input.
    Returns the reference's status code."""
    st = check_solve(p)
    check_frows(p, rng)
    check_sd_and_reachable(p, rng)
    check_torque(p, rng)
    check_parametrizers(p, rng)
    check_ubound(p, rng)
    check_other_constraints(p, rng)
    check_batch(p, rng)
    check_robust_params(p, rng)
    return st


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--minutes", type=float, default=5.0)
    ap.add_argument("--seed", type=int, default=0)
    args = ap.parse_args()
    load()
    t_end = time.time() + 60 * args.minutes
    seed, bad, hist = args.seed, [], {}
    while time.time() < t_end:
        rng = np.random.RandomState(seed)
        p = random_problem(rng)
        try:
            st = check_all(p, rng)
            hist[st] = hist.get(st, 0) + 1
        except AssertionError as e:
            bad.append((seed, str(e)[:200]))
            print("MISMATCH seed %d: %s  (dof %d, n %d, G %d, bc %s, interp %d, sd %.3g -> %.3g)"
                  % (seed, str(e)[:200], p["way"].shape[1], len(p["ss"]), len(p["grid"]), p["bc"], p["interp"], p["sd0"],
                     p["sd1"]), flush=True)
        except Exception as e:                      # the reference itself raised (e.g. bad gridpoints): not a parity question
            hist["ref-raised:" + type(e).__name__] = hist.get("ref-raised:" + type(e).__name__, 0) + 1
        seed += 1
    print("problems: %d (seeds %d..%d), status histogram %s, checks run %s, mismatches: %d"
          % (seed - args.seed, args.seed, seed - 1, hist, COUNTS, len(bad)))
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
