"""Generates tests/golden/*.npz by running the UNMODIFIED reference (oracle/_ref, built by
oracle/build_ref.sh from /root/reference) and scipy.  Run where /root/reference exists:

    python tests/golden/make_golden.py

The fixtures pin the oracle (tests/test_oracle_vs_golden.py, CPU) and the CUDA path
(tests/test_gpu_*.py) to the reference's own outputs; /root/reference is not needed to RUN the tests.
Inputs follow SURVEY.md §8d (cfg 1/2, parity sets P1-P6) and the reference's own test fixtures
(cited per case)."""
import os
import sys
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
warnings.filterwarnings("ignore")

from oracle.ref_loader import load_reference  # noqa: E402
from problems import make_path  # noqa: E402

ta = load_reference()
import toppra.algorithm as algo  # noqa: E402
import toppra.constraint as constraint  # noqa: E402
import toppra.solverwrapper.cy_seidel_solverwrapper as seidel  # noqa: E402
from scipy.interpolate import CubicSpline  # noqa: E402

REF_TESTS = "/root/reference/tests/tests"


def solve_ref(ss, way, vlim, alim, grid, sd_start=0.0, sd_end=0.0, scheme=1, bc_type="not-a-knot"):
    """Reference TOPPRA(seidel) on one path -> dict of everything the tests compare."""
    path = ta.SplineInterpolator(ss, way, bc_type=bc_type)
    pc_vel = constraint.JointVelocityConstraint(vlim)
    pc_acc = constraint.JointAccelerationConstraint(alim, discretization_scheme=scheme)
    inst = algo.TOPPRA([pc_vel, pc_acc], path, gridpoints=grid, solver_wrapper="seidel")
    sdd, sd, _, K = inst.compute_parameterization(sd_start, sd_end, return_data=True)
    G = len(grid)
    code = inst.problem_data.return_code
    codes = list(algo.ParameterizationReturnCode)
    out = dict(c=path.cspl.c, K=K, status=codes.index(code),
               sd=np.full(G, np.nan) if sd is None else sd,
               sdd=np.full(G - 1, np.nan) if sdd is None else sdd,
               xbound=pc_vel.compute_constraint_params(path, grid)[-1])
    a, b, c, F, g, _, _ = pc_acc.compute_constraint_params(path, grid)
    out.update(acc_a=a, acc_b=b, acc_F=F, acc_g=g)
    out["qs"] = path(grid, 1)
    out["qss"] = path(grid, 2)
    return out, inst


def stack(dicts):
    return {k: np.stack([d[k] for d in dicts]) for k in dicts[0]}


def batch_case(name, seeds, G, vel_active=False, sd_start=0.0, sd_end=0.0, scheme=1, dof=7, grid=None):
    ss = np.linspace(0, 1, 5)
    grid = np.linspace(0, 1, G) if grid is None else grid
    rows, ways, vlims, alims = [], [], [], []
    for s in seeds:
        way, vlim, alim = make_path(s, dof=dof, vel_active=vel_active)
        out, _ = solve_ref(ss, way, vlim, alim, grid, sd_start, sd_end, scheme)
        rows.append(out)
        ways.append(way); vlims.append(vlim); alims.append(alim)
    data = stack(rows)
    data.update(ss=ss, way=np.stack(ways), vlim=np.stack(vlims), alim=np.stack(alims), grid=grid,
                sd_start=np.float64(sd_start), sd_end=np.float64(sd_end), scheme=np.int64(scheme),
                seeds=np.asarray(seeds))
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **data)
    print(name, "status histogram", np.bincount(data["status"], minlength=5))


def main():
    # ---- cfg 1: examples/plot_kinematics.py:22-40, np.random.seed(9), 100 gridpoints ---------------------
    np.random.seed(9)
    dof = 7
    way = np.random.randn(5, dof)
    ss = np.linspace(0, 1, 5)
    vl = 10 + np.random.rand(dof) * 20
    al = 10 + np.random.rand(dof) * 2
    vlim = np.vstack((-vl, vl)).T
    alim = np.vstack((-al, al)).T
    grid = np.linspace(0, 1, 100)
    out, inst = solve_ref(ss, way, vlim, alim, grid)
    out["X"] = inst.compute_feasible_sets()
    out["K_0_05"] = inst.compute_controllable_sets(0.0, 0.5)
    traj = algo.TOPPRA([constraint.JointVelocityConstraint(vlim), constraint.JointAccelerationConstraint(alim)],
                       ta.SplineInterpolator(ss, way), gridpoints=grid, solver_wrapper="seidel").compute_trajectory(0, 0)
    ts = np.linspace(0, traj.duration, 50)
    out.update(ss=ss, way=way, vlim=vlim, alim=alim, grid=grid, traj_duration=np.float64(traj.duration),
               traj_ts=ts, traj_q=traj(ts), traj_qd=traj(ts, 1), traj_qdd=traj(ts, 2))
    # constant-acceleration output (ParametrizeConstAccel, parametrizer.py:23-158)
    ca = algo.TOPPRA([constraint.JointVelocityConstraint(vlim), constraint.JointAccelerationConstraint(alim)],
                     ta.SplineInterpolator(ss, way), gridpoints=grid, solver_wrapper="seidel",
                     parametrizer="ParametrizeConstAccel").compute_trajectory(0, 0)
    ca_ts = np.linspace(0, ca.duration, 64)
    out.update(ca_duration=np.float64(ca.duration), ca_ts=ca_ts, ca_q=ca(ca_ts), ca_qd=ca(ca_ts, 1), ca_qdd=ca(ca_ts, 2),
               ca_tgrid=ca._ts, ca_us=ca._us)
    # TOPPRAsd (desired duration) and reachable sets on the same problem
    sd_inst = algo.TOPPRAsd([constraint.JointVelocityConstraint(vlim), constraint.JointAccelerationConstraint(alim)],
                            ta.SplineInterpolator(ss, way), gridpoints=grid, solver_wrapper="seidel")
    for tag, dur in (("sd5", 5.0), ("sd_fast", 1.0), ("sd_slow", 1e9)):
        sd_inst.set_desired_duration(dur)
        sdd_d, sd_d, _, _ = sd_inst.compute_parameterization(0, 0, return_data=True)
        out[tag + "_sd"], out[tag + "_sdd"] = sd_d, sdd_d
    out["L_0_05"] = inst.compute_reachable_sets(0.0, 0.5)
    # varying velocity limits (linear_joint_velocity.py:56-87): vlim(s) = vlim * (0.05 + 0.5 s) -> active bound
    vfun = lambda s: vlim * (0.05 + 0.5 * s)  # noqa: E731
    pc_var = constraint.JointVelocityConstraintVarying(vfun)
    out["var_xbound"] = pc_var.compute_constraint_params(ta.SplineInterpolator(ss, way), grid)[-1]
    var_inst = algo.TOPPRA([pc_var, constraint.JointAccelerationConstraint(alim)], ta.SplineInterpolator(ss, way),
                           gridpoints=grid, solver_wrapper="seidel")
    _, out["var_sd"], _, out["var_K"] = var_inst.compute_parameterization(0, 0, return_data=True)
    # the example's own automatic grid
    auto = algo.TOPPRA([constraint.JointVelocityConstraint(vlim), constraint.JointAccelerationConstraint(alim)],
                       ta.SplineInterpolator(ss, way), solver_wrapper="seidel")
    sdd, sd, _, K = auto.compute_parameterization(0, 0, return_data=True)
    out.update(auto_grid=auto.gridpoints, auto_sd=sd, auto_K=K)
    np.savez_compressed(os.path.join(HERE, "cfg1_seed9.npz"), **out)
    print("cfg1: duration", traj.duration, "auto gridpoints", len(auto.gridpoints))

    # ---- cfg 2 shape + parity-only sets (SURVEY.md §8d) --------------------------------------------------
    batch_case("cfg2_seeds1000", range(1000, 1016), 200)
    batch_case("p1_velocity_active", range(1000, 1016), 200, vel_active=True)
    batch_case("p2_boundary_speeds", range(1000, 1008), 100, sd_start=0.05, sd_end=0.03)
    batch_case("p3_inadmissible_start", range(1000, 1004), 50, sd_start=5.0)
    batch_case("p5_grid_on_breakpoints", range(1000, 1008), 201)
    batch_case("p6_collocation", range(1000, 1008), 100, scheme=0)
    batch_case("dof6_g500", range(2000, 2004), 500, dof=6)
    # non-uniform grid
    rng = np.random.RandomState(5)
    g = np.sort(np.r_[0.0, 1.0, rng.rand(148)])
    batch_case("nonuniform_grid", range(1000, 1008), 150, grid=g)

    # ---- forward-pass retry rule (reachability_algorithm.py:315-343; SURVEY §7 "cold but must exist") ----------
    # (a) start velocity admissible only through the 1e-5 slack: first forward LP infeasible, succeeds after a retry
    retry = dict(way=[], vlim=[], alim=[], sd_start=[], K=[], sd=[], sdd=[], status=[])
    ss5, grid200 = np.linspace(0, 1, 5), np.linspace(0, 1, 200)
    for seed in range(1000, 1006):
        way, vlim_, alim_ = make_path(seed)
        out0, _ = solve_ref(ss5, way, vlim_, alim_, grid200)
        s0 = float(np.sqrt(out0["K"][0, 1] + (3e-8 if seed % 2 else 5e-6)))
        out1, _ = solve_ref(ss5, way, vlim_, alim_, grid200, sd_start=s0)
        retry["way"].append(way); retry["vlim"].append(vlim_); retry["alim"].append(alim_); retry["sd_start"].append(s0)
        for k in ("K", "sd", "sdd", "status"):
            retry[k].append(out1[k])
    np.savez_compressed(os.path.join(HERE, "retry_after_slack_start.npz"), ss=ss5, grid=grid200,
                        **{k: np.asarray(v) for k, v in retry.items()})
    print("retry (slack start): statuses", retry["status"])

    # (b) random row-level problems whose forward pass exhausts the retry budget (found by random search with the
    #     oracle, seeds below), run through the REFERENCE via a pass-through CanonicalLinear constraint (F = I, g = 0)
    class RowConstraint(constraint.LinearConstraint):
        def __init__(self, rows, xb):
            super(RowConstraint, self).__init__()
            self.rows, self.xb, self.identical, self.dof = rows, xb, False, 1

        def compute_constraint_params(self, path, gridpoints):
            G_, _, R_ = self.rows.shape
            F = np.tile(np.eye(R_)[None], (G_, 1, 1))
            return self.rows[:, 0], self.rows[:, 1], self.rows[:, 2], F, np.zeros((G_, R_)), None, self.xb

    rng = np.random.RandomState(0)
    rc = {}
    n_found = 0
    for trial in range(200000):
        G_ = rng.randint(3, 8); R_ = rng.randint(2, 6)
        grid_ = np.sort(np.r_[0, 1, rng.rand(G_ - 2)])
        if np.any(np.diff(grid_) < 1e-3):
            continue
        rows_ = np.zeros((G_, 3, R_))
        rows_[:, 0, :] = rng.randn(G_, R_) * rng.choice([1, 0.1, 3])
        rows_[:, 1, :] = rng.randn(G_, R_)
        rows_[:, 2, :] = -rng.rand(G_, R_) * rng.choice([1, 0.2])
        xb_ = np.stack((np.zeros(G_), rng.rand(G_) * 2 + 0.05), axis=1)
        sd0_ = rng.rand() * 0.3
        if trial not in (4202, 27645, 52804, 67731, 100515, 160523, 11, 12, 13, 14):
            continue
        dummy = ta.SplineInterpolator([0.0, 1.0], [[0.0], [1.0]])
        inst_ = algo.TOPPRA([RowConstraint(rows_, xb_)], dummy, gridpoints=grid_, solver_wrapper="seidel")
        sdd_, sd_, _, K_ = inst_.compute_parameterization(sd0_, 0.0, return_data=True)
        codes = list(algo.ParameterizationReturnCode)
        tag = "c%d_" % n_found
        rc[tag + "grid"], rc[tag + "rows"], rc[tag + "xb"], rc[tag + "sd_start"] = grid_, rows_, xb_, np.float64(sd0_)
        rc[tag + "K"] = K_
        rc[tag + "sd"] = np.full(G_, np.nan) if sd_ is None else sd_
        rc[tag + "sdd"] = np.full(G_ - 1, np.nan) if sdd_ is None else sdd_
        rc[tag + "status"] = np.int64(codes.index(inst_.problem_data.return_code))
        n_found += 1
    rc["n"] = np.int64(n_found)
    np.savez_compressed(os.path.join(HERE, "retry_row_problems.npz"), **rc)
    print("retry (row problems):", n_found, "cases, statuses", [int(rc["c%d_status" % i]) for i in range(n_found)])

    # ---- P6: 2-DOF collocation golden of cpp/tests/test_algorithm.cpp:25-169 (generator script :25-57) ----
    path = ta.SplineInterpolator([0, 1, 2, 3], [[0, 0], [1, 3], [2, 4], [0, 0]])
    pc_vel = constraint.JointVelocityConstraint([1.0, 1.0])
    pc_acc = constraint.JointAccelerationConstraint([0.2, 0.2], discretization_scheme=0)
    grid = np.linspace(0, 3, 51)
    inst = algo.TOPPRA([pc_vel, pc_acc], path, gridpoints=grid, solver_wrapper="seidel")
    sdd, sd, _, K = inst.compute_parameterization(0, 0, return_data=True)
    X = inst.compute_feasible_sets()
    np.savez_compressed(os.path.join(HERE, "cpp_2dof_collocation.npz"), ss=np.array([0., 1, 2, 3]),
                        way=np.array([[0., 0], [1, 3], [2, 4], [0, 0]]), grid=grid, c=path.cspl.c, K=K, sd=sd, sdd=sdd,
                        X=X, vlim=np.array([[-1., 1], [-1, 1]]), alim=np.array([[-0.2, 0.2], [-0.2, 0.2]]))

    # ---- LP layer: 100 seeded random LPs of tests/tests/lpsolvers/seidel/test_lp2d.py:74-95 ----------------
    lp = dict(v=[], a=[], b=[], c=[], active_in=[], res=[], optval=[], optvar=[], active_out=[])
    for seed in range(100):
        d = 50
        np.random.seed(seed)
        seeds = np.random.randint(1000, size=7)
        np.random.seed(seeds[0])
        v = np.random.randn(3)
        np.random.seed(seeds[1])
        a, b = np.random.randn(2, d)
        np.random.seed(seeds[2])
        c = -np.random.rand(d) if seed % 2 == 0 else np.random.randn(d)
        low = np.r_[-0.5, -0.9]
        high = np.r_[0.5, 0.9]
        np.random.seed(seeds[3])
        active_c = np.random.choice(d, size=2)
        res, optval, optvar, act = seidel.solve_lp2d(v, a, b, c, low, high, active_c.astype(np.int64))
        lp["v"].append(v); lp["a"].append(a); lp["b"].append(b); lp["c"].append(c)
        lp["active_in"].append(active_c)
        lp["res"].append(res)
        lp["optval"].append(optval if res else np.nan)
        lp["optvar"].append(np.array(optvar) if res else np.full(2, np.nan))
        lp["active_out"].append(np.array(act) if res else np.zeros(2, dtype=int))
    lp = {k: np.asarray(val) for k, val in lp.items()}
    lp.update(low=np.r_[-0.5, -0.9], high=np.r_[0.5, 0.9])
    np.savez_compressed(os.path.join(HERE, "lp2d_random100.npz"), **lp)
    print("lp2d random: feasible", int(lp["res"].sum()), "/ 100")

    # ---- stage-level: tests/tests/solverwrapper/test_basic_can_linear.py:53-164 fixture (6-DOF, N=200, seed 1)
    np.random.seed(1)
    dof = 6
    way_pts = np.random.randn(4, dof) * 0.6
    path = ta.SplineInterpolator(np.linspace(0, 1, 4), way_pts)
    vlim_ = np.random.rand(dof) * 10 + 10
    vlim = np.vstack((-vlim_, vlim_)).T
    alim_ = np.random.rand(dof) * 10 + 100
    alim = np.vstack((-alim_, alim_)).T
    grid = np.linspace(0, path.duration, 201)
    cons = [constraint.JointVelocityConstraint(vlim), constraint.JointAccelerationConstraint(alim)]
    w = seidel.seidelWrapper(cons, path, grid, solve_lp1d=1)
    cases = []
    for i in (3, 10, 30, 40):
        for g in (np.array([0.2, -1.0]), np.array([0.5, 1.0]), np.array([2.0, 1.0])):
            for (x_ineq, xn_ineq) in ((( -1.0, 1.0), (0.0, 1.0)), ((0.2, 0.2), (0.0, 1.0)),
                                      ((np.nan, np.nan), (0.05, 0.5)), ((0.0, 0.05), (np.nan, np.nan))):
                res = np.array(w.solve_stagewise_optim(i, None, g, x_ineq[0], x_ineq[1], xn_ineq[0], xn_ineq[1]))
                cases.append(np.r_[i, g, x_ineq, xn_ineq, res])
    np.savez_compressed(os.path.join(HERE, "stagewise_6dof.npz"), ss=np.linspace(0, 1, 4), way=way_pts, vlim=vlim,
                        alim=alim, grid=grid, cases=np.asarray(cases))

    # ---- spline fits for the other boundary conditions (scipy) ------------------------------------------
    rng = np.random.RandomState(3)
    fits = {}
    for n in (2, 3, 4, 5, 9, 20):
        x = np.sort(rng.rand(n)) * 2.0
        x[0] = 0.0
        y = rng.randn(n, 3)
        fits["x_%d" % n] = x
        fits["y_%d" % n] = y
        for bc in ("not-a-knot", "clamped", "natural"):
            fits["c_%d_%s" % (n, bc)] = CubicSpline(x, y, bc_type=bc).c
        d0, d1 = rng.randn(3), rng.randn(3)
        fits["d0_%d" % n], fits["d1_%d" % n] = d0, d1
        fits["c_%d_first" % n] = CubicSpline(x, y, bc_type=((1, d0), (1, d1))).c
        fits["c_%d_mixed" % n] = CubicSpline(x, y, bc_type=((2, d0), (1, d1))).c
    np.savez_compressed(os.path.join(HERE, "spline_fits.npz"), **fits)

    # ---- P4: tiny-motion robustness suite tests/tests/retime/robustness/problem_suite_1.yaml (clamped BC) ----
    import yaml
    suite = yaml.safe_load(open(os.path.join(REF_TESTS, "retime/robustness/problem_suite_1.yaml")))
    rob = {}
    names = []
    for key, prob in suite.items():
        wp = np.array(prob["waypoints"], dtype=float)
        ssw = np.linspace(prob["ss_waypoints"][0], prob["ss_waypoints"][1], len(wp))
        vl = np.r_[prob["vlim"]].astype(float)
        al = np.r_[prob["alim"]].astype(float)
        for G in prob["nb_gridpoints"]:
            grid = np.linspace(ssw[0], ssw[-1], G)
            out, _ = solve_ref(ssw, wp, np.vstack((-vl, vl)).T, np.vstack((-al, al)).T, grid, bc_type="clamped")
            tag = "%s_%d" % (key, G)
            names.append(tag)
            rob[tag + "_ss"], rob[tag + "_way"], rob[tag + "_grid"] = ssw, wp, grid
            rob[tag + "_vlim"], rob[tag + "_alim"] = np.vstack((-vl, vl)).T, np.vstack((-al, al)).T
            for k in ("c", "K", "sd", "sdd", "status"):
                rob[tag + "_" + k] = out[k]
    rob["names"] = np.array(names)
    np.savez_compressed(os.path.join(HERE, "p4_robustness_suite.npz"), **rob)
    print("robustness suite:", len(names), "cases, statuses", [int(rob[n + "_status"]) for n in names])

    # ---- SecondOrder (cfg-3 shape, small): synthetic closed-form torque model, SURVEY.md §8d cfg 3 -------------
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from problems import make_torque_problem, inv_dyn_numpy
    outs = []
    for seed in range(2000, 2004):
        way, vlim, alim, taulim = make_torque_problem(seed)
        ssw = np.linspace(0, 1, 5)
        grid = np.linspace(0, 1, 100)
        path = ta.SplineInterpolator(ssw, way)
        pc_vel = constraint.JointVelocityConstraint(vlim)
        pc_acc = constraint.JointAccelerationConstraint(alim)
        pc_tau = constraint.SecondOrderConstraint.joint_torque_constraint(inv_dyn_numpy, taulim, np.zeros(6))
        inst = algo.TOPPRA([pc_vel, pc_acc, pc_tau], path, gridpoints=grid, solver_wrapper="seidel")
        sdd, sd, _, K = inst.compute_parameterization(0, 0, return_data=True)
        a, b, c, F, g, _, _ = pc_tau.compute_constraint_params(path, grid)
        codes = list(algo.ParameterizationReturnCode)
        outs.append(dict(way=way, vlim=vlim, alim=alim, taulim=taulim, K=K, sd=sd, sdd=sdd, tau_a=a, tau_b=b, tau_c=c,
                         status=codes.index(inst.problem_data.return_code)))
    data = stack(outs)
    data.update(ss=np.linspace(0, 1, 5), grid=np.linspace(0, 1, 100))
    np.savez_compressed(os.path.join(HERE, "torque_dof6.npz"), **data)
    print("torque: statuses", data["status"])


def torque_g500_case():
    """BASELINE cfg 3 at its stated shape (6-DOF, 500 gridpoints, vel + acc + SecondOrder torque rows -> nC = 50),
    4 paths with seeds 2000+b solved by the reference with the numpy inv_dyn of tests/problems.py."""
    from problems import make_torque_problem, inv_dyn_numpy
    codes = list(algo.ParameterizationReturnCode)
    outs = []
    for seed in range(2000, 2004):
        way, vlim, alim, taulim = make_torque_problem(seed)
        ssw = np.linspace(0, 1, 5)
        grid = np.linspace(0, 1, 500)
        path = ta.SplineInterpolator(ssw, way)
        pc_tau = constraint.SecondOrderConstraint.joint_torque_constraint(inv_dyn_numpy, taulim, np.zeros(6))
        inst = algo.TOPPRA([constraint.JointVelocityConstraint(vlim), constraint.JointAccelerationConstraint(alim), pc_tau],
                           path, gridpoints=grid, solver_wrapper="seidel")
        sdd, sd, _, K = inst.compute_parameterization(0, 0, return_data=True)
        outs.append(dict(way=way, vlim=vlim, alim=alim, taulim=taulim, K=K, sd=sd, sdd=sdd,
                         status=codes.index(inst.problem_data.return_code)))
    data = stack(outs)
    data.update(ss=np.linspace(0, 1, 5), grid=np.linspace(0, 1, 500))
    np.savez_compressed(os.path.join(HERE, "torque_dof6_g500.npz"), **data)
    print("torque g500: statuses", data["status"])


def shortcut_rows_case():
    """VERDICT r1 #4: the degenerate-row and badly-scaled problems that stress the scan kernel's Seidel shortcuts, solved
    by the REFERENCE's seidelWrapper.  The raw rows reach it through a LinearConstraint whose F is the identity and
    g = 0 (rows = F.a, F.b, F.c - g = a, b, c exactly, cy_seidel_solverwrapper.pyx:483-510), xbound as given.
    Only the outputs are stored (float64 K, sd, sdd + status); the inputs are regenerated from the seeds in
    tests/problems.py:SHORTCUT_SETS."""
    from problems import SHORTCUT_SETS

    class RowsConstraint(constraint.LinearConstraint):
        def __init__(self, rows, xbound):
            super(RowsConstraint, self).__init__()
            self.rows, self.xb = rows, xbound
            self.identical = True
            self.dof = 1

        def compute_constraint_params(self, path, gridpoints, *args, **kwargs):
            R = self.rows.shape[2]
            return (self.rows[:, 0].copy(), self.rows[:, 1].copy(), self.rows[:, 2].copy(), np.eye(R), np.zeros(R), None,
                    self.xb.copy())

    codes = list(algo.ParameterizationReturnCode)
    for name, (gen, args) in SHORTCUT_SETS.items():
        rows, xb = gen(*args)
        B, G = rows.shape[:2]
        grid = np.linspace(0, 1, G)
        path = ta.SplineInterpolator([0, 1], [[0.0], [1.0]])
        K = np.empty((B, G, 2)); sd = np.full((B, G), np.nan); sdd = np.full((B, G - 1), np.nan)
        status = np.empty(B, dtype=np.int64)
        for i in range(B):
            inst = algo.TOPPRA([RowsConstraint(rows[i], xb[i])], path, gridpoints=grid, solver_wrapper="seidel")
            u_, s_, _, K[i] = inst.compute_parameterization(0, 0, return_data=True)
            status[i] = codes.index(inst.problem_data.return_code)
            if s_ is not None:
                sd[i], sdd[i] = s_, u_
        data = {name + "_K": K, name + "_sd": sd, name + "_sdd": sdd, name + "_status": status}
        print("shortcut rows", name, "status histogram", np.bincount(status, minlength=5))
        # one file per set keeps every fixture under 1 MB
        np.savez_compressed(os.path.join(HERE, "shortcut_rows_%s.npz" % name), **data)


def joint_torque_case():
    """JointTorqueConstraint (toppra/constraint/joint_torque.py:7-116, SURVEY §8 f4): vel + torque with dry friction,
    both discretisation schemes, synthetic closed-form inverse dynamics of tests/problems.py."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from problems import make_torque_problem, inv_dyn_numpy
    codes = list(algo.ParameterizationReturnCode)
    data = {}
    ssw, grid = np.linspace(0, 1, 5), np.linspace(0, 1, 60)
    for scheme in (0, 1):
        outs = []
        for seed in range(2100, 2103):
            way, vlim, alim, taulim = make_torque_problem(seed)
            fric = 0.5 + 0.25 * np.arange(6)
            path = ta.SplineInterpolator(ssw, way)
            pc_vel = constraint.JointVelocityConstraint(vlim)
            pc_tau = constraint.JointTorqueConstraint(inv_dyn_numpy, taulim, fric, discretization_scheme=scheme)
            inst = algo.TOPPRA([pc_vel, pc_tau], path, gridpoints=grid, solver_wrapper="seidel")
            sdd, sd, _, K = inst.compute_parameterization(0, 0, return_data=True)
            a, b, c, F, g, _, _ = pc_tau.compute_constraint_params(path, grid)
            xb = pc_vel.compute_constraint_params(path, grid)[-1]
            outs.append(dict(way=way, vlim=vlim, taulim=taulim, fric=fric, K=K, sd=sd, sdd=sdd, a=a, b=b, c=c, F=F, g=g,
                             xbound=xb, status=codes.index(inst.problem_data.return_code)))
        for k, v in stack(outs).items():
            data["s%d_%s" % (scheme, k)] = v
    data.update(ss=ssw, grid=grid)
    np.savez_compressed(os.path.join(HERE, "joint_torque_dof6.npz"), **data)
    print("joint torque: statuses", data["s0_status"], data["s1_status"])


def other_paths_case():
    """SimplePath (toppra/simplepath.py, cubic Hermite via scipy BPoly) and PolynomialPath (interpolator.py:584-686):
    evaluations at sample positions and the vel+acc parameterisation along them (SURVEY §8 f4 'other path types')."""
    codes = list(algo.ParameterizationReturnCode)
    rng = np.random.RandomState(77)
    data = {}
    x = np.array([0.0, 0.3, 0.9, 1.4, 2.0, 2.5])
    y = rng.randn(6, 3)
    yd = rng.randn(6, 3) * 0.5
    vlim = np.vstack((-np.ones(3) * 3, np.ones(3) * 3)).T
    alim = np.vstack((-np.ones(3) * 8, np.ones(3) * 8)).T
    s = np.linspace(0, 2.5, 41)
    grid = np.linspace(0, 2.5, 80)
    for tag, path in (("sp_auto", ta.SimplePath(x, y)), ("sp_yd", ta.SimplePath(x, y, yd)),
                      ("poly", ta.PolynomialPath([[1, 2, 3], [-2, 3, 4, 5], [0.5, -1.0]], s_start=0.0, s_end=2.5))):
        for order in (0, 1, 2):
            data["%s_q%d" % (tag, order)] = np.asarray(path(s, order), dtype=float)
        inst = algo.TOPPRA([constraint.JointVelocityConstraint(vlim), constraint.JointAccelerationConstraint(alim)], path,
                           gridpoints=grid, solver_wrapper="seidel")
        sdd, sd, _, K = inst.compute_parameterization(0, 0, return_data=True)
        data[tag + "_K"], data[tag + "_sd"], data[tag + "_sdd"] = K, sd, sdd
        data[tag + "_status"] = codes.index(inst.problem_data.return_code)
    data.update(x=x, y=y, yd=yd, vlim=vlim, alim=alim, s=s, grid=grid)
    np.savez_compressed(os.path.join(HERE, "other_paths.npz"), **data)
    print("other paths: statuses", [int(data[t + "_status"]) for t in ("sp_auto", "sp_yd", "poly")])


def periodic_case():
    """scipy CubicSpline(bc_type='periodic') (reference SplineInterpolator passes bc_type through, interpolator.py:419):
    closed curves, y[0] == y[-1]; n = 2, 3 (special cases), 4, 5, 9, 20 (the workspace path of the fit kernel)."""
    rng = np.random.RandomState(11)
    fits = {}
    for n in (2, 3, 4, 5, 9, 20):
        x = np.sort(rng.rand(n)) * 3.0
        x[0] = 0.0
        y = rng.randn(n, 3)
        y[-1] = y[0]
        cs = CubicSpline(x, y, bc_type="periodic")
        se = np.linspace(x[0], x[-1], 41)
        csd = cs.derivative()          # the reference evaluates derivatives like this (interpolator.py:419-430)
        fits.update({"x_%d" % n: x, "y_%d" % n: y, "c_%d" % n: cs.c, "s_%d" % n: se, "q_%d" % n: cs(se),
                     "qd_%d" % n: csd(se), "qdd_%d" % n: csd.derivative()(se)})
    # a closed 7-DOF path through the reference's TOPPRA (the solver evaluates q', q'' at the gridpoints through scipy's
    # periodic extrapolation: the last gridpoint wraps to the first)
    way = rng.randn(6, 7)
    way[-1] = way[0]
    ssp = np.linspace(0, 1, 6)
    vl, al = 10 + rng.rand(7) * 20, 10 + rng.rand(7) * 2
    vlim, alim = np.vstack((-vl, vl)).T, np.vstack((-al, al)).T
    grid = np.linspace(0, 1, 100)
    o, _ = solve_ref(ssp, way, vlim, alim, grid, bc_type="periodic")
    fits.update(solve_ss=ssp, solve_way=way, solve_vlim=vlim, solve_alim=alim, solve_grid=grid, solve_K=o["K"],
                solve_sd=o["sd"], solve_sdd=o["sdd"], solve_status=np.int32(o["status"]))
    np.savez_compressed(os.path.join(HERE, "spline_periodic.npz"), **fits)
    print("spline_periodic: written")


def frows_batch_case():
    """Rows f1-f3 + ubound for BATCHES (VERDICT r1 "next" #8, #9): 16 paths each through the reference's own
    propose_gridpoints (ragged grids), compute_reachable_sets, TOPPRAsd, ParametrizeSpline, and a user-defined
    LinearConstraint that returns a ubound (seidelWrapper.__init__, cy_seidel_solverwrapper.pyx:512-515)."""
    import toppra.interpolator as interp
    from toppra.parametrizer import ParametrizeSpline
    B, dof = 16, 7
    ss = np.linspace(0, 1, 5)
    probs = [make_path(5000 + b, dof=dof) for b in range(B)]       # (way, vlim, alim)
    way = np.stack([p[0] for p in probs])
    vlim = np.stack([p[1] for p in probs])
    alim = np.stack([p[2] for p in probs])
    vlim[:4] *= 0.04                                              # some velocity-limited paths
    data = dict(ss=ss, way=way, vlim=vlim, alim=alim)

    # ---- propose_gridpoints (interpolator.py:49-122): two parameter sets, ragged results, padded with NaN
    for tag, kw in (("pg_default", {}), ("pg_toppra", dict(max_err_threshold=1e-3, min_nb_points=100)),
                    ("pg_coarse", dict(max_err_threshold=5e-2, max_seg_length=0.3, min_nb_points=20))):
        grids = [np.asarray(interp.propose_gridpoints(ta.SplineInterpolator(ss, way[b]), **kw)) for b in range(B)]
        glen = np.array([len(g) for g in grids], dtype=np.int32)
        pad = np.full((B, glen.max()), np.nan)
        for b, g in enumerate(grids):
            pad[b, :len(g)] = g
        data[tag + "_grid"], data[tag + "_len"] = pad, glen
    # solve on the ragged pg_toppra grids (what TOPPRA(gridpoints=None) does)
    Gmax = data["pg_toppra_grid"].shape[1]
    rK, rsd, rsdd, rst = (np.full((B, Gmax, 2), np.nan), np.full((B, Gmax), np.nan), np.full((B, Gmax - 1), np.nan),
                          np.zeros(B, dtype=np.int32))
    for b in range(B):
        n = data["pg_toppra_len"][b]
        o, _ = solve_ref(ss, way[b], vlim[b], alim[b], data["pg_toppra_grid"][b, :n])
        rK[b, :n], rsd[b, :n], rsdd[b, :n - 1], rst[b] = o["K"], o["sd"], o["sdd"], o["status"]
    data.update(ragged_K=rK, ragged_sd=rsd, ragged_sdd=rsdd, ragged_status=rst)

    # ---- reachable sets, TOPPRAsd, ParametrizeSpline on a shared 120-point grid
    grid = np.linspace(0, 1, 120)
    data["grid"] = grid
    sdmin = np.where(np.arange(B) % 3 == 0, 0.0, 0.2)
    sdmax = np.where(np.arange(B) % 2 == 0, sdmin, sdmin + 0.5)   # equal pairs take the 1-variable branch at stage 0
    L = np.zeros((B, 120, 2))
    X = np.zeros((B, 120, 2))
    sd_out, sdd_out, sd_status = np.zeros((B, 120)), np.zeros((B, 119)), np.zeros(B, dtype=np.int32)
    desired = np.zeros(B)
    ps_t, ps_n = np.full((B, 120), np.nan), np.zeros(B, dtype=np.int32)
    ts_eval = np.linspace(0, 1, 33)
    ps_q, ps_qd, ps_qdd = (np.zeros((B, 33, dof)) for _ in range(3))
    ps_dur = np.zeros(B)
    for b in range(B):
        cons = lambda: [constraint.JointVelocityConstraint(vlim[b]), constraint.JointAccelerationConstraint(alim[b])]  # noqa: E731
        path = ta.SplineInterpolator(ss, way[b])
        inst = algo.TOPPRA(cons(), path, gridpoints=grid, solver_wrapper="seidel")
        X[b] = inst.compute_feasible_sets()
        inst = algo.TOPPRA(cons(), path, gridpoints=grid, solver_wrapper="seidel")
        L[b] = inst.compute_reachable_sets(sdmin[b], sdmax[b])
        # fastest duration first, then a desired duration below / inside / above the achievable range
        o, _ = solve_ref(ss, way[b], vlim[b], alim[b], grid)
        fastest = np.sum(2 * np.diff(grid) / (o["sd"][1:] + o["sd"][:-1]))
        desired[b] = fastest * (0.5, 1.7, 3.0, 1e6)[b % 4]
        sdi = algo.TOPPRAsd(cons(), path, gridpoints=grid, solver_wrapper="seidel")
        sdi.set_desired_duration(desired[b])
        sdd_d, sd_d, _, _ = sdi.compute_parameterization(0, 0, return_data=True)
        sd_out[b], sdd_out[b] = sd_d, sdd_d
        sd_status[b] = list(algo.ParameterizationReturnCode).index(sdi.problem_data.return_code)
        # ParametrizeSpline on the time-optimal velocities; path 5 gets two stationary gridpoints (5 s rule), path 6 a
        # huge speed (increment below 1e-8 -> dropped knot)
        vel = o["sd"].copy()
        if b == 5:
            vel[40:42] = 0.0
        if b == 6:
            vel[60:62] = 1e9
        traj = ParametrizeSpline(path, grid, vel)
        n = len(traj.ss_waypoints)
        ps_t[b, :n], ps_n[b] = traj.ss_waypoints, n
        ps_dur[b] = traj.duration
        te = ts_eval * traj.duration
        ps_q[b], ps_qd[b], ps_qdd[b] = traj(te), traj(te, 1), traj(te, 2)
        data.setdefault("ps_vel", np.zeros((B, 120)))[b] = vel
    data.update(X=X, L=L, sdmin=sdmin, sdmax=sdmax, sd_desired=desired, sd_sd=sd_out, sd_sdd=sdd_out, sd_status=sd_status,
                ps_t=ps_t, ps_n=ps_n, ps_dur=ps_dur, ps_ts=ts_eval, ps_q=ps_q, ps_qd=ps_qd, ps_qdd=ps_qdd)

    # ---- ubound from a constraint: acceleration rows + a u-interval that tightens with s (and an x-bound), 8 paths
    class UBoundConstraint(constraint.LinearConstraint):
        def __init__(self, acc, ulim):
            super(UBoundConstraint, self).__init__()
            self.acc, self.ulim = acc, ulim
            self.discretization_type = acc.discretization_type
            self.identical = True

        def get_dof(self):
            return self.acc.get_dof()

        def compute_constraint_params(self, path, gridpoints, *a):
            pa, pb, pc, F, g, _, _ = self.acc.compute_constraint_params(path, gridpoints)
            n = len(gridpoints)
            ub = np.stack((-self.ulim * (1.0 + gridpoints), self.ulim * (2.0 - gridpoints)), axis=1)
            xb = np.stack((np.zeros(n), 40.0 + 30 * gridpoints), axis=1)
            return pa, pb, pc, F, g, ub, xb

    ub_K, ub_sd, ub_sdd, ub_status, ub_X, ub_L = ([] for _ in range(6))
    ulims = np.array([0.3, 0.1, 0.12, 0.08, 0.6, 0.4, 0.5, 0.2])
    for b in range(8):
        path = ta.SplineInterpolator(ss, way[b])
        mk = lambda: [constraint.JointVelocityConstraint(vlim[b]),  # noqa: E731
                      UBoundConstraint(constraint.JointAccelerationConstraint(alim[b]), ulims[b])]
        inst = algo.TOPPRA(mk(), path, gridpoints=grid, solver_wrapper="seidel")
        sdd, sd, _, K = inst.compute_parameterization(0, 0, return_data=True)
        ub_K.append(K)
        ub_status.append(list(algo.ParameterizationReturnCode).index(inst.problem_data.return_code))
        ub_sd.append(np.full(120, np.nan) if sd is None else sd)
        ub_sdd.append(np.full(119, np.nan) if sdd is None else sdd)
        ub_X.append(algo.TOPPRA(mk(), path, gridpoints=grid, solver_wrapper="seidel").compute_feasible_sets())
        ub_L.append(algo.TOPPRA(mk(), path, gridpoints=grid, solver_wrapper="seidel").compute_reachable_sets(0.0, 0.3))
    data.update(ub_ulim=ulims, ub_K=np.stack(ub_K), ub_sd=np.stack(ub_sd), ub_sdd=np.stack(ub_sdd),
                ub_status=np.array(ub_status, dtype=np.int32), ub_X=np.stack(ub_X), ub_L=np.stack(ub_L))
    np.savez_compressed(os.path.join(HERE, "frows_batch.npz"), **data)
    print("frows_batch: grid lengths", data["pg_toppra_len"], "| sd status", sd_status, "| kept knots", ps_n,
          "| ubound status", ub_status)


def oracle_vs_reference_case():
    """The reference's outputs on the random problems of tests/test_oracle_vs_reference.py (same seeds, same inputs),
    and the reference's public API (classes, members, argument names) for the introspection test there."""
    import json
    import inspect
    import toppra.interpolator as interp
    import toppra.parametrizer
    import toppra.simplepath
    import toppra.solverwrapper
    from toppra.parametrizer import ParametrizeSpline
    data = {}
    ss = np.linspace(0, 1, 5)
    # test_random_paths_bit_exact
    for vel_active in (0, 1):
        for seed in range(5000, 5040):
            key = "paths%d_%d_" % (vel_active, seed)
            grid = np.linspace(0, 1, 60 + (seed % 5) * 35)
            way, vlim, alim = make_path(seed, vel_active=bool(vel_active))
            path = ta.SplineInterpolator(ss, way)
            inst = algo.TOPPRA([constraint.JointVelocityConstraint(vlim), constraint.JointAccelerationConstraint(alim)],
                               path, gridpoints=grid, solver_wrapper="seidel")
            sdd, sd, _, K = inst.compute_parameterization(0.0 if seed % 3 else 0.02, 0.0, return_data=True)
            data.update({key + "c": path.cspl.c, key + "K": K})
            if sd is not None:
                data.update({key + "sd": sd, key + "sdd": sdd})
    # test_lp_shims_random
    rng = np.random.RandomState(0)
    lp = {"ok": [], "val": [], "var": [], "act": []}
    for trial in range(300):
        n = rng.randint(1, 40)
        v = rng.randn(3)
        a, b = rng.randn(2, n)
        c = -rng.rand(n) if trial % 2 else rng.randn(n) * 0.3 - 0.5
        act = rng.randint(-4, n + 2, size=2)
        r, val, var, act_out = seidel.solve_lp2d(v, a, b, c, np.r_[-1.0, -2.0], np.r_[1.5, 0.7], act.astype(np.int64))
        lp["ok"].append(bool(r))
        lp["val"].append(val if r else np.nan)
        lp["var"].append(np.asarray(var, dtype=float) if r else np.full(2, np.nan))
        lp["act"].append(np.asarray(act_out, dtype=np.int64) if r else np.full(2, -99, dtype=np.int64))
    data.update({"lp_" + k: np.array(v) for k, v in lp.items()})
    # test_ubound_random_vs_reference
    rng = np.random.RandomState(17)

    class UB(constraint.LinearConstraint):
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

    for seed in range(6000, 6012):
        key = "ubound_%d_" % seed
        G = 40 + (seed % 4) * 25
        grid = np.linspace(0, 1, G)
        way, vlim, alim = make_path(seed)
        width = 0.05 + 1.5 * rng.rand()
        ub = np.stack((-width * (0.5 + rng.rand(G)), width * (0.5 + rng.rand(G))), axis=1)
        xb = np.stack((np.zeros(G), 20.0 + 80 * rng.rand(G)), axis=1)
        path = ta.SplineInterpolator(ss, way)
        mk = lambda: [constraint.JointVelocityConstraint(vlim),  # noqa: E731
                      UB(constraint.JointAccelerationConstraint(alim), ub, xb)]
        sdd, sd, _, K = algo.TOPPRA(mk(), path, gridpoints=grid, solver_wrapper="seidel").compute_parameterization(
            0, 0, return_data=True)
        data[key + "K"] = K
        if sd is not None:
            data.update({key + "sd": sd, key + "sdd": sdd})
        data[key + "X"] = algo.TOPPRA(mk(), path, gridpoints=grid, solver_wrapper="seidel").compute_feasible_sets()
        data[key + "L"] = algo.TOPPRA(mk(), path, gridpoints=grid, solver_wrapper="seidel").compute_reachable_sets(0.0, 0.2)
    # test_propose_gridpoints_and_spline_time_stamps_random_vs_reference
    rng = np.random.RandomState(23)
    for seed in range(7000, 7008):
        key = "grid_%d_" % seed
        way, _, _ = make_path(seed, dof=3 + seed % 4)
        path = ta.SplineInterpolator(ss, way)
        kw = dict(max_err_threshold=10 ** rng.uniform(-4, -1.5), max_seg_length=rng.uniform(0.04, 0.4),
                  min_nb_points=int(rng.randint(5, 150)))
        data[key + "proposed"] = np.asarray(interp.propose_gridpoints(path, **kw))
        G = 80
        vel = np.abs(rng.randn(G)) + 0.05
        vel[rng.randint(1, G - 1, size=3)] = 0.0
        vel[10:12] = 1e9
        data[key + "time_stamps"] = np.asarray(ParametrizeSpline(path, np.linspace(0, 1, G), vel).ss_waypoints)
    # test_toppra_sd_random_vs_reference
    rng = np.random.RandomState(31)
    for seed in range(8000, 8010):
        key = "sd_%d_" % seed
        grid = np.linspace(0, 1, 50 + (seed % 3) * 30)
        way, vlim, alim = make_path(seed, vel_active=(seed % 4 == 0))
        mk = lambda: [constraint.JointVelocityConstraint(vlim), constraint.JointAccelerationConstraint(alim)]  # noqa: E731
        inst = algo.TOPPRAsd(mk(), ta.SplineInterpolator(ss, way), gridpoints=grid, solver_wrapper="seidel")
        fast = algo.TOPPRA(mk(), ta.SplineInterpolator(ss, way), gridpoints=grid, solver_wrapper="seidel")
        _, sd_f, _ = fast.compute_parameterization(0, 0)
        want_t = np.sum(2 * np.diff(grid) / (sd_f[1:] + sd_f[:-1])) * rng.choice([0.6, 1.3, 2.2, 5.0])
        inst.set_desired_duration(want_t)
        sdd, sd, _, K = inst.compute_parameterization(0, 0, return_data=True)
        data.update({key + "duration": np.float64(want_t), key + "K": K, key + "sd": sd, key + "sdd": sdd})
    # test_univariate_spline_interpolator_vs_reference
    for seed in range(4):
        key = "univariate_%d_" % seed
        rng = np.random.RandomState(900 + seed)
        n = 25 + 10 * seed
        s_w = np.sort(np.r_[0.0, rng.uniform(0.05, 2.95, n - 2), 3.0])
        way = np.stack([np.sin(s_w), np.cos(1.7 * s_w), 0.2 * s_w ** 2 - s_w, np.sin(0.5 * s_w) * s_w], axis=1)
        way += 0.03 * rng.randn(n, 4)
        path = ta.UnivariateSplineInterpolator(s_w, way)
        s = np.linspace(0, 3.0, 301)
        for order in (0, 1, 2):
            data[key + "eval%d" % order] = path(s, order)
        data[key + "dof"] = np.int64(path.dof)
        data[key + "path_interval"] = np.asarray(path.path_interval, dtype=float)
        vlim, alim = np.array([[-2.0, 2.0]] * 4), np.array([[-6.0, 5.0]] * 4)
        inst = algo.TOPPRA([constraint.JointVelocityConstraint(vlim), constraint.JointAccelerationConstraint(alim)], path,
                           gridpoints=np.linspace(0, 3.0, 151), solver_wrapper="seidel")
        sdd, sd, _, K = inst.compute_parameterization(0, 0, return_data=True)
        data.update({key + "K": K, key + "sd": sd, key + "sdd": sdd})
    # test_public_classes_have_the_reference_methods_and_arguments: {module: {name: {member: [argument names] or None}}}
    def params(f):
        try:
            return [p for p in inspect.signature(f).parameters if p not in ("args", "kwargs")]
        except (TypeError, ValueError):
            return None

    api = {}
    for mod in (ta, algo, constraint, toppra.parametrizer, interp, toppra.simplepath, toppra.solverwrapper):
        entries = api.setdefault(mod.__name__, {})
        for name in dir(mod):
            obj = getattr(mod, name)
            if name.startswith("_") or not (getattr(obj, "__module__", None) or "").startswith("toppra"):
                continue
            if inspect.isclass(obj):
                members = {}
                for member in ["__init__"] + [m for m in dir(obj) if not m.startswith("_")]:
                    fr = getattr(obj, member)
                    members[member] = params(fr) if callable(fr) and not isinstance(fr, type) else None
                entries[name] = {"kind": "class", "members": members}
            elif inspect.isfunction(obj):
                entries[name] = {"kind": "function", "params": params(obj)}
    data["public_api_json"] = np.array(json.dumps(api, sort_keys=True))
    np.savez_compressed(os.path.join(HERE, "oracle_vs_reference.npz"), **data)
    print("oracle_vs_reference:", len(data), "arrays")


def fuzz_slice_case():
    """The reference's results on the randomly shaped problems of test_randomly_shaped_problems_vs_reference, recorded
    through the campaign's own checks (scripts/fuzz_oracle_vs_reference.py, `theirs`) while they run live."""
    import importlib.util
    from test_oracle_vs_reference import FUZZ_SLICE_SEEDS
    spec = importlib.util.spec_from_file_location("fuzz_oracle_vs_reference",
                                                  os.path.join(ROOT, "scripts", "fuzz_oracle_vs_reference.py"))
    fuzz = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(fuzz)
    fuzz.load()
    fuzz.RECORD = {}
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
                pass
    finally:
        fuzz.release()
    np.savez_compressed(os.path.join(HERE, "fuzz_slice.npz"), **fuzz.pack(fuzz.RECORD))
    print("fuzz slice:", len(fuzz.RECORD), "arrays; checks", fuzz.COUNTS)


PLUGIN_SINGLE_CASES = [(1000, 200, False, 0.0, 0.0, 1), (1003, 100, True, 0.0, 0.0, 1), (1005, 150, False, 0.1, 0.1, 1),
                       (1007, 64, False, 0.0, 0.0, 0), (1002, 100, False, 30.0, 0.0, 1)]


def plugin_batch_case():
    """The reference solved path by path on the batch of tests/test_reference_plugin.py (make_batch(24, 1000), 120
    gridpoints, vel + acc)."""
    from problems import make_batch
    ss, way, vlim, alim = make_batch(24, 1000)
    grid = np.linspace(0, 1, 120)
    outs = [solve_ref(ss, way[b], vlim[b], alim[b], grid)[0] for b in range(way.shape[0])]
    data = {k: np.stack([o[k] for o in outs]) for k in ("K", "sd", "sdd", "status")}
    # single paths with boundary velocities, the collocation scheme and an inadmissible start (status 3)
    for seed, G, vel_active, s0, s1, scheme in PLUGIN_SINGLE_CASES:
        way1, vlim1, alim1 = make_path(seed, vel_active=vel_active)
        o, _ = solve_ref(ss, way1, vlim1, alim1, np.linspace(0, 1, G), s0, s1, scheme)
        data.update({"single%d_%s" % (seed, k): o[k] for k in ("K", "sd", "sdd", "status")})
    np.savez_compressed(os.path.join(HERE, "plugin_batch.npz"), **data)
    print("plugin batch: statuses", data["status"])


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "shortcut_rows":
        shortcut_rows_case()
    elif len(sys.argv) > 1 and sys.argv[1] == "oracle_vs_reference":
        oracle_vs_reference_case()
    elif len(sys.argv) > 1 and sys.argv[1] == "fuzz_slice":
        fuzz_slice_case()
    elif len(sys.argv) > 1 and sys.argv[1] == "plugin_batch":
        plugin_batch_case()
    elif len(sys.argv) > 1 and sys.argv[1] == "torque_g500":
        torque_g500_case()
    elif len(sys.argv) > 1 and sys.argv[1] == "joint_torque":
        joint_torque_case()
    elif len(sys.argv) > 1 and sys.argv[1] == "other_paths":
        other_paths_case()
    elif len(sys.argv) > 1 and sys.argv[1] == "frows_batch":
        frows_batch_case()
    elif len(sys.argv) > 1 and sys.argv[1] == "periodic":
        periodic_case()
    else:
        main()
        joint_torque_case()
        other_paths_case()
        frows_batch_case()
        periodic_case()
