#!/usr/bin/env python
"""bench.py — paths/sec of batched TOPP-RA (7-DOF, 200 gridpoints, vel+accel) on N B200s vs the reference CPU
seidel path.  Contract: see the task statement; one JSON line on stdout (rank 0).

  python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo (CUDA kernels)
  python bench.py --impl reference [--gpus N] [--steps K] ...    # the reference's own CPU path on the host cores
  python bench.py --dump-outputs DIR ...                         # also write the last timed step's results to DIR

A "step" = one pass of the hot path over one batch of `--batch` synthetic paths per GPU (BASELINE.json configs[1]:
4096 random 7-DOF spline paths, 200 gridpoints, vel+acc): K0 spline fit -> K1 coefficient records -> K2
backward+forward scan.  `value` times it with the inputs resident in HBM; `e2e` goes through the public API
(BatchSplineInterpolator / BatchTOPPRA) with pinned HOST buffers, H2D and D2H inside the timed region."""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True   # the benchmark leaves the tree it runs from untouched (it may be read-only)
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "paths/sec (7-DOF, 200 gridpoints, vel+accel)"
UNIT = "paths/s"


def workload_text(B, dof, G):
    """One string for both arms (the driver compares the arms' `config.workload`)."""
    return ("configs[1]: batch %d random %d-DOF cubic-spline paths (5 waypoints), %d gridpoints, "
            "JointVelocity+JointAcceleration(interp), per GPU" % (B, dof, G))


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=4096, help="paths per GPU per step (BASELINE configs[1]: 4096)")
    ap.add_argument("--gridpoints", type=int, default=200)
    ap.add_argument("--dof", type=int, default=7)
    ap.add_argument("--cpu-sample", type=int, default=0, help="paths in the cpu_baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--configs", default="1,3,4,5", help="BASELINE configs reported in the `configs` block besides the "
                    "headline cfg 2 (comma list out of 1,3,4,5; 'none' to skip)")
    ap.add_argument("--cfg3-batch", type=int, default=65536)
    ap.add_argument("--cfg5-batch", type=int, default=1 << 20)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write K, sd, u, status, fail_stage of the last timed step of "
                    "the headline path as DIR/<name>.npy (float64; rank 0's shard), for comparing two builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out, directory):
    """Writes the arrays the headline path returns as float64 .npy files.  The inputs are seeded, so two builds run with
    the same arguments can be compared file by file.  If the batch exceeds DUMP_LIMIT_BYTES, a fixed seeded sample of
    paths is written; path_index.npy always lists the paths (rows) written."""
    host = {k: v.cpu().numpy().astype(np.float64) for k, v in out.items() if v is not None}
    B = host["K"].shape[0]
    per_path = sum(a[0].nbytes for a in host.values()) + 8
    idx = np.arange(B)
    if per_path * B > DUMP_LIMIT_BYTES:
        idx = np.sort(np.random.RandomState(0).choice(B, DUMP_LIMIT_BYTES // per_path, replace=False))
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, "path_index.npy"), idx.astype(np.float64))
    for name, a in host.items():
        np.save(os.path.join(directory, name + ".npy"), np.ascontiguousarray(a[idx]))


# ----------------------------------------------------------------------------------------------------------
# CPU arms: the reference's own implementation (oracle/_ref) or, if that build is absent, the C port.
# ----------------------------------------------------------------------------------------------------------
_REF = {}


def _ref_worker_init():
    import warnings
    warnings.filterwarnings("ignore")
    try:  # one BLAS thread per worker process: the reference's a_j.dot(F_j.T) must not oversubscribe the cores
        from threadpoolctl import threadpool_limits
        _REF["blas_limit"] = threadpool_limits(1)
    except Exception:
        pass
    from oracle.ref_loader import load_reference
    ta = load_reference()
    import toppra.algorithm as algo
    import toppra.constraint as constraint
    _REF.update(ta=ta, algo=algo, constraint=constraint)


def _ref_solve_chunk(args):
    """Reference hot path for a chunk of paths: SplineInterpolator + TOPPRA(seidel).compute_parameterization."""
    ss, way, vlim, alim, grid = args
    ta, algo, constraint = _REF["ta"], _REF["algo"], _REF["constraint"]
    n_ok = 0
    for b in range(way.shape[0]):
        path = ta.SplineInterpolator(ss, way[b])
        inst = algo.TOPPRA([constraint.JointVelocityConstraint(vlim[b]), constraint.JointAccelerationConstraint(alim[b])],
                           path, gridpoints=grid, solver_wrapper="seidel")
        inst.compute_parameterization(0, 0)
        n_ok += inst.problem_data.return_code == algo.ParameterizationReturnCode.Ok
    return n_ok


def _cgroup_cpu_limit():
    """CPU quota of this container (cgroup v2 cpu.max / v1 cfs quota), or None."""
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            return max(1, int(float(q) / float(p) + 0.5))
    except Exception:
        pass
    try:
        q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
        p = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        if q > 0:
            return max(1, int(q / p + 0.5))
    except Exception:
        pass
    return None


class CpuArm(object):
    """Times the reference CPU path on the host cores (multiprocessing, one chunk of paths per task).

    The number of worker processes is calibrated (a few candidates up to the visible CPU count, best throughput on
    a small sample wins): on shared hosts the visible CPUs exceed what the container may actually use, and an
    oversubscribed pool would understate the reference."""

    def __init__(self, dof, G, calibrate=None):
        from oracle.ref_loader import reference_available
        self.kind = "reference" if reference_available() else "port"
        self.visible = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
        quota = _cgroup_cpu_limit()
        self.cores = min(self.visible, quota) if quota else self.visible
        self.G, self.dof = G, dof
        self.pool = None
        self.note = "visible cpus %d%s" % (self.visible, (", cgroup quota %d" % quota) if quota else "")
        if self.kind == "reference":
            if calibrate is not None:
                self._calibrate(*calibrate)
            self._make_pool(self.cores)
        else:
            from oracle import oracle as orc
            self.orc = orc

    def _make_pool(self, n):
        import multiprocessing as mp
        if self.pool is not None:
            self.pool.close()
            self.pool.join()
        self.pool = mp.get_context("fork").Pool(n, initializer=_ref_worker_init)
        self.nproc = n

    def _calibrate(self, ss, way, vlim, alim, grid):
        """Pool size = min(visible CPUs, cgroup quota), or half of it when that is measurably faster (SMT siblings):
        two candidates, each timed on >= 2 s of work so that the choice and the reported value are stable run to run."""
        cands = sorted({max(1, self.cores // 2), self.cores})
        best, best_rate, log = cands[-1], 0.0, []
        for n in cands:
            self._make_pool(n)
            self.run(ss, way[:min(way.shape[0], 4 * n)], vlim[:4 * n], alim[:4 * n], grid)  # import warm-up
            S = min(way.shape[0], max(64, 300 * n))  # ~150 paths/s per core -> ~2 s
            rate = S / self.run(ss, way[:S], vlim[:S], alim[:S], grid)
            log.append("%d:%.0f" % (n, rate))
            if rate > best_rate * 1.03:   # prefer the smaller pool unless the larger one is clearly faster
                best, best_rate = n, rate
        self.cores = best
        self.note += "; pool-size calibration (procs:paths/s) " + " ".join(log)

    def run(self, ss, way, vlim, alim, grid):
        """Solve all given paths; returns seconds."""
        B = way.shape[0]
        t0 = time.perf_counter()
        if self.kind == "reference":
            nchunk = min(B, self.nproc * 4)
            idx = np.array_split(np.arange(B), nchunk)
            tasks = [(ss, way[i], vlim[i], alim[i], grid) for i in idx if len(i)]
            self.pool.map(_ref_solve_chunk, tasks, chunksize=1)
        else:
            c = np.stack([self.orc.cubic_spline_fit(ss, way[b]) for b in range(B)])
            self.orc.solve_velacc_batch(c, np.tile(ss, (B, 1)), grid, vlim, alim, True, nthreads=self.cores)
        return time.perf_counter() - t0

    def close(self):
        if self.pool is not None:
            self.pool.close()
            self.pool.join()


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from problems import make_batch_fast
    G, dof = args.gridpoints, args.dof
    grid = np.linspace(0, 1, G)
    ss, way, vlim, alim = make_batch_fast(args.batch, seed=1234, dof=dof)
    arm = CpuArm(dof, G, calibrate=(ss, way, vlim, alim, grid))
    # bounded sample of the workload per step: ~2 s of wall time per step on this box
    per_core = 150.0 if arm.kind == "reference" else 4000.0
    S = args.cpu_sample or int(min(args.batch, max(arm.cores * 8, per_core * arm.cores * 2.0)))
    way, vlim, alim = way[:S], vlim[:S], alim[:S]
    for _ in range(max(args.warmup, 1)):
        arm.run(ss, way, vlim, alim, grid)
    secs = [arm.run(ss, way, vlim, alim, grid) for _ in range(args.steps)]
    arm.close()
    total = float(np.sum(secs))
    value = S * args.steps / total
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_text(args.batch, dof, G),
                   "sample_paths_per_step": S, "solver": "reference seidelWrapper (Cython, -O1) via TOPPRA(..., 'seidel')"
                   if arm.kind == "reference" else "oracle C port (reference build absent)"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": arm.cores, "kind": arm.kind,
                         "sample": "%d paths/step x %d steps, spline fit + wrapper construction + compute_parameterization, "
                                   "multiprocessing over %d processes (%s)" % (S, args.steps, arm.cores, arm.note)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.02)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}



# ----------------------------------------------------------------------------------------------------------
# `configs` block: the other BASELINE.json configurations on the same box, after the headline measurement
# ----------------------------------------------------------------------------------------------------------
def extra_configs(args, torch, dist, ta, dev, world, rank, peak):
    """cfg 1 (B = 1 latency), cfg 3 (6-DOF, 500 gridpoints, vel + acc + torque rows, 65536 paths per GPU), cfg 4 (robust,
    4096 paths per GPU) and cfg 5 (2^20 paths STRONG-scaled over the ranks, chunked all-gather of the results inside the
    timed region) through the public API with device-resident inputs; CUDA events, max over ranks.  Each entry: paths/s,
    ms split (fit / records / scan), status histogram over all ranks, and the scan kernel's roofline against the
    materialised-record algorithmic bytes of SURVEY.md section 8d."""
    from problems import make_batch_fast
    want = [] if args.configs == "none" else [int(c) for c in args.configs.split(",") if c]
    out = {}
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731

    def allmax(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def allminmax(x):
        t = torch.tensor([x, -x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [-float(t[1].item()), float(t[0].item())]

    def timed(fn, steps, warmup):
        """ms per step = MEDIAN of per-step CUDA-event times (an allocator hiccup in one step does not skew the figure);
        ranks enter the timed steps together."""
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()
        pairs = []
        for _ in range(steps):
            s, e = ev(), ev()
            s.record()
            r = fn()
            e.record()
            pairs.append((s, e))
        torch.cuda.synchronize()
        return float(np.median([a.elapsed_time(b) for a, b in pairs])), r

    def hist(status):
        h = torch.bincount(status.to(torch.int64), minlength=5)[:5].clone()
        if world > 1:
            dist.all_reduce(h)
        return dict(zip(("Ok", "ErrUnknown", "ErrShortPath", "FailUncontrollable", "ErrForwardPassFail"), h.cpu().tolist()))

    def roof(R, G, B, ms):
        by = (2 * G * (3 * R + 2) * 8 + G * 16 + G * 8 + (G - 1) * 8 + 8) * B
        return {"bound": "hbm", "achieved": by / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                "frac": by / (ms * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_launch": by, "ms_per_launch": ms}

    def staged(cons, d_ss, d_way, d_grid, steps=3):
        """fit / records (or xbound) / scan, timed separately on a fresh instance (single-chunk problems only)."""
        fit, path = timed(lambda: ta.BatchSplineInterpolator(d_ss, d_way, validate=False), steps, 2)
        inst = ta.BatchTOPPRA(cons, path, d_grid, validate=False)
        if inst.chunk_size() < inst.B:
            return {"fit_ms": allmax(fit), "chunk_paths": inst.chunk_size()}, None
        rec, _ = timed(inst.setup, steps, 2)
        scan, _ = timed(lambda: inst.compute_parameterization(0.0, 0.0), steps, 2)
        return {"fit_ms": allmax(fit), "records_ms": allmax(rec), "scan_ms": allmax(scan),
                "scan_ms_ranks_min_max": allminmax(scan)}, scan

    if 1 in want:
        # cfg 1: one 7-DOF path, 100 gridpoints (examples/plot_kinematics.py, seed 9): latency of the single-path drop-in
        # API (host in, host out, every sync included) and of the B = 1 batched call
        np.random.seed(9)
        way1 = np.random.randn(5, 7)
        vl, al = 10 + np.random.rand(7) * 20, 10 + np.random.rand(7) * 2
        ss1, grid1 = np.linspace(0, 1, 5), np.linspace(0, 1, 100)

        def one_api():
            path = ta.SplineInterpolator(ss1, way1)
            inst = ta.algorithm.TOPPRA([ta.constraint.JointVelocityConstraint(vl), ta.constraint.JointAccelerationConstraint(al)],
                                       path, gridpoints=grid1, solver_wrapper="seidel")
            return inst.compute_parameterization(0, 0)

        def one_batch():
            path = ta.BatchSplineInterpolator(ss1, way1[None], device=dev)
            inst = ta.BatchTOPPRA([ta.constraint.JointVelocityConstraint(vl), ta.constraint.JointAccelerationConstraint(al)],
                                  path, grid1)
            return inst.compute_parameterization(0.0, 0.0).to_host()

        lat = {}
        for name, fn in (("TOPPRA.compute_parameterization", one_api), ("BatchTOPPRA_B1_to_host", one_batch)):
            for _ in range(5):
                fn()
            ts = []
            for _ in range(30):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                fn()
                torch.cuda.synchronize()
                ts.append(time.perf_counter() - t0)
            lat[name] = {"median_ms": 1e3 * float(np.median(ts)), "min_ms": 1e3 * float(np.min(ts))}
        d_w1 = torch.as_tensor(way1[None]).to(dev)
        d_s1, d_g1 = torch.as_tensor(ss1).to(dev), torch.as_tensor(grid1).to(dev)
        c1 = [ta.constraint.JointVelocityConstraint(vl), ta.constraint.JointAccelerationConstraint(al)]
        for c in c1:
            c.device_limits(dev)
        k_ms, _ = timed(lambda: ta.BatchTOPPRA(c1, ta.BatchSplineInterpolator(d_s1, d_w1, validate=False), d_g1,
                                               validate=False).compute_parameterization(0.0, 0.0), 20, 5)
        out["cfg1"] = {"workload": "configs[0]: one 7-DOF path, 100 gridpoints, vel+acc (seed 9), wall clock on the host "
                                   "incl. H2D/D2H and every synchronisation", "latency": lat,
                       "device_resident_step_ms": k_ms, "n_gpus_used": 1}

    if 3 in want:
        B, G, dof = args.cfg3_batch, 500, 6
        ss, way, vlim, alim = make_batch_fast(B, seed=2000 + rank, dof=dof)
        tl = 40 + np.random.RandomState(7 + rank).rand(B, dof) * 10
        taulim = np.stack((-tl, tl), axis=-1)
        cons = [ta.constraint.JointVelocityConstraint(vlim), ta.constraint.JointAccelerationConstraint(alim),
                ta.constraint.SecondOrderConstraint.joint_torque_constraint(
                    None, taulim, np.zeros(dof), device_model=("coupled_cosine", [2.0, 0.3, 0.1, 4.9]))]
        for c in cons[:2]:
            c.device_limits(dev)
        d_way, d_ss = torch.as_tensor(way).to(dev), torch.as_tensor(ss).to(dev)
        d_grid = torch.as_tensor(np.linspace(0, 1, G)).to(dev)

        def step3():
            path = ta.BatchSplineInterpolator(d_ss, d_way, validate=False)
            return ta.BatchTOPPRA(cons, path, d_grid, validate=False).compute_parameterization(0.0, 0.0)

        ms, res = timed(step3, 3, 2)
        ms = allmax(ms)
        h = hist(res.status)
        del res
        # stage split on a sub-batch that fits one record buffer (the full batch runs chunked)
        nsub = min(B, 16384)
        sub = [ta.constraint.JointVelocityConstraint(vlim[:nsub]), ta.constraint.JointAccelerationConstraint(alim[:nsub]),
               ta.constraint.SecondOrderConstraint.joint_torque_constraint(
                   None, taulim[:nsub], np.zeros(dof), device_model=("coupled_cosine", [2.0, 0.3, 0.1, 4.9]))]
        split, scan_ms = staged(sub, d_ss, d_way[:nsub].contiguous(), d_grid)
        split["split_measured_on_paths"] = nsub
        out["cfg3"] = {"workload": "configs[2]: %d 6-DOF paths per GPU, 500 gridpoints, JointVelocity + JointAcceleration + "
                                   "SecondOrder torque rows (R = 48, nC = 50), inverse dynamics by the library's device "
                                   "model 'coupled_cosine' inside tb_coeff_second_order" % B,
                       "paths_per_s": B * world / (ms * 1e-3), "ms_per_step": ms, "scaling": "weak", "status": h,
                       "split": split, "roofline": roof(48, G, nsub, scan_ms) if scan_ms else None}
        del d_way, cons, sub
        torch.cuda.empty_cache()

    if 4 in want:
        B, G, dof = args.batch, 200, 7
        ss, way, vlim, alim = make_batch_fast(B, seed=3000 + rank, dof=dof)
        cons = [ta.constraint.JointVelocityConstraint(vlim),
                ta.constraint.RobustLinearConstraint(ta.constraint.JointAccelerationConstraint(alim), [1e-3, 5e-2, 9e-3], 1)]
        cons[0].device_limits(dev)
        d_way, d_ss = torch.as_tensor(way).to(dev), torch.as_tensor(ss).to(dev)
        d_grid = torch.as_tensor(np.linspace(0, 1, G)).to(dev)

        def step4():
            path = ta.BatchSplineInterpolator(d_ss, d_way, validate=False)
            return ta.BatchTOPPRA(cons, path, d_grid, validate=False).compute_parameterization(0.0, 0.0)

        ms, res = timed(step4, 5, 3)
        ms = allmax(ms)
        split, scan_ms = staged(cons, d_ss, d_way, d_grid)
        out["cfg4"] = {"workload": "configs[3]: robust TOPP-RA, %d 7-DOF paths per GPU, 200 gridpoints, JointVelocity + "
                                   "RobustLinearConstraint(JointAcceleration, ellipsoid [1e-3, 5e-2, 9e-3], interpolation): "
                                   "3 two-variable SOCPs per stage (tb_scan_robust)" % B,
                       "paths_per_s": B * world / (ms * 1e-3), "ms_per_step": ms, "scaling": "weak", "status": hist(res.status),
                       "split": split, "roofline": roof(28, G, B, scan_ms) if scan_ms else None,
                       "parity": "unpinned (no ECOS): optimality certificate + SLSQP cross-check in tests/test_robust.py"}
        del d_way, res
        torch.cuda.empty_cache()

    if 5 in want:
        from toppra_b200.distributed import ShardedSolver
        Btot, G, dof = args.cfg5_batch, 200, 7
        Btot -= Btot % world
        shard = Btot // world
        ss, way, vlim, alim = make_batch_fast(shard, seed=1000 + rank, dof=dof)
        d_way, d_ss = torch.as_tensor(way).to(dev), torch.as_tensor(ss).to(dev)
        d_vlim, d_alim = torch.as_tensor(vlim).to(dev), torch.as_tensor(alim).to(dev)
        d_grid = torch.as_tensor(np.linspace(0, 1, G)).to(dev)
        # chunks of >= 32768 paths where the shard allows it (the scan's large-batch forward pass starts at 24576 paths)
        solver = ShardedSolver(Btot, G, dev, nchunks=max(2, min(8, shard // 32768)), gather=True)

        ms, full = timed(lambda: solver.solve(d_ss, d_way, d_grid, d_vlim, d_alim), 3, 2)
        ms = allmax(ms)
        solver.kernel_events = []
        solver.solve(d_ss, d_way, d_grid, d_vlim, d_alim, record_events=True)
        torch.cuda.synchronize()
        k_ms = sum(a.elapsed_time(b) for a, b in solver.kernel_events)   # this rank's K0 + xbound + scan, all chunks
        lo = rank * shard if solver.gather else 0
        h = hist(full["status"][lo:lo + shard])
        out["cfg5"] = {"workload": "configs[4]: %d 7-DOF paths, 200 gridpoints, vel+acc, sharded contiguously over %d GPU(s) "
                                   "(%d per GPU, %d chunks per shard); NCCL all-gather of K, sd, sdd, status per chunk on a "
                                   "side stream INSIDE the timed region, results in global order on every rank"
                                   % (Btot, world, shard, solver.nchunks),
                       "paths_per_s": Btot / (ms * 1e-3), "ms_per_step": ms, "scaling": "strong", "status": h,
                       "kernels_ms_ranks_min_max": allminmax(k_ms), "gather_exposed_ms": ms - allmax(k_ms),
                       "gathered_bytes_per_rank": int(sum(v.numel() * v.element_size() for v in full.values())) if world > 1 else 0,
                       "roofline": roof(28, G, shard, k_ms)}
        del solver, full, d_way
        torch.cuda.empty_cache()
    return out

def run_b200(args):
    import torch
    import torch.distributed as dist
    import toppra_b200 as ta
    from toppra_b200 import engine
    from problems import make_batch_fast

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    B, G, dof, nway = args.batch, args.gridpoints, args.dof, 5
    R = 4 * dof
    ss, way, vlim, alim = make_batch_fast(B, seed=1234 + rank, dof=dof, nway=nway)  # every rank: its own shard
    grid = np.linspace(0, 1, G)

    # CPU baseline first: the worker pool is forked before this process touches CUDA
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        try:
            arm = CpuArm(dof, G, calibrate=(ss, way, vlim, alim, grid))
            S = args.cpu_sample or min(B, 4096)  # the whole cfg-2 batch: ~20 s of CPU work for the reference
            arm.run(ss, way[:min(S, 256)], vlim[:min(S, 256)], alim[:min(S, 256)], grid)  # warm-up (imports, pool)
            secs = arm.run(ss, way[:S], vlim[:S], alim[:S], grid)
            arm.close()
            cpu = {"value": S / secs, "unit": UNIT, "cores": arm.cores, "kind": arm.kind,
                   "sample": "%d paths of the same batch (spline fit + wrapper construction + compute_parameterization), "
                             "%s, %d processes (%s)" % (S, "reference TOPPRA(seidel)" if arm.kind == "reference" else "C port", arm.cores, arm.note)}
        except Exception as exc:  # never lose the GPU line
            cpu = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": "failed: %r" % (exc,)}

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # NCCL's copy kernels share the SMs with the scan (whose resident one-warp CTAs hold the whole register file); the
        # high-priority NCCL stream is the cheap half of the remedy (measured at N = 8: no change on its own, DESIGN.md 7)
        opts = None
        try:
            opts = dist.ProcessGroupNCCL.Options(is_high_priority_stream=True)
        except Exception:
            pass
        if opts is not None:
            dist.init_process_group("nccl", device_id=dev, pg_options=opts)
        else:
            dist.init_process_group("nccl", device_id=dev)
    # pinned host buffers (e2e) and device-resident inputs (value)
    h_way = torch.as_tensor(way).pin_memory()
    h_vlim = torch.as_tensor(vlim).pin_memory()
    h_alim = torch.as_tensor(alim).pin_memory()
    h_ss = torch.as_tensor(ss).pin_memory()
    h_grid = torch.as_tensor(grid).pin_memory()
    d_way, d_vlim, d_alim, d_ss, d_grid = (t.to(dev) for t in (h_way, h_vlim, h_alim, h_ss, h_grid))
    def pinned_set():
        return {"K": torch.empty((B, G, 2), dtype=torch.float64).pin_memory(),
                "sd": torch.empty((B, G), dtype=torch.float64).pin_memory(),
                "sdd": torch.empty((B, G - 1), dtype=torch.float64).pin_memory(),
                "status": torch.empty((B,), dtype=torch.int32).pin_memory(),
                "fail_stage": torch.empty((B,), dtype=torch.int32).pin_memory()}

    h_sets = [pinned_set(), pinned_set()]   # a pipelined caller alternates between two result buffers
    h_out = h_sets[0]
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)  # 256 MB > 126 MB L2
    W = engine.record_doubles(R)
    records = torch.empty((B, G, W), dtype=torch.float64, device=dev)
    gathered = torch.empty((world * B, G), dtype=torch.float64, device=dev) if world > 1 else None

    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    k_events = []  # (k0_start, k1_start, k2_start, k2_end) per timed step

    scan_mode = {"fast_lower": False}
    last_out = {}   # results of the latest timed headline step (for --dump-outputs)

    xbound = torch.empty((B, G, 2), dtype=torch.float64, device=dev)

    def step_device(record_kernels=False):
        """Hot path with inputs resident in HBM: 3 kernel launches: K0 spline fit, K1 velocity bound (xbound only),
        K2 scan with the acceleration rows built inside the kernel (tb_scan_velacc: K1's record stream fused away)."""
        e = [ev() for _ in range(4)] if record_kernels else None
        if e: e[0].record()
        ppoly = engine.spline_fit(d_ss, d_way)
        if e: e[1].record()
        engine.xbound_constant(ppoly, d_ss, d_grid, d_vlim, xbound, 0, 1)
        if e: e[2].record()
        out = engine.scan_velacc(ppoly, d_ss, d_grid, d_alim, True, xbound, fast_lower=scan_mode["fast_lower"])
        if e:
            e[3].record()
            k_events.append(e)
            if args.dump_outputs and len(k_events) == args.steps:   # keep nothing alive between timed steps
                last_out["out"] = out
        return out

    rec_events = []

    def step_records():
        """The same problem through materialised stage records (K0 -> K1 records -> K2 record scan): what generic
        constraint lists use; timed for the K1 / K2 rooflines of that path, not part of `value`."""
        e = [ev() for _ in range(4)]
        e[0].record()
        ppoly = engine.spline_fit(d_ss, d_way)
        e[1].record()
        engine.coeff_velacc(ppoly, d_ss, d_grid, d_vlim, d_alim, True, records, R, 0, 1)
        e[2].record()
        out = engine.scan(records, R, d_grid)
        e[3].record()
        rec_events.append(e)
        return out

    # the e2e step builds constraint objects from host limit arrays each step (their H2D copy is part of the step)
    e2e_mode = {"sync": False, "k": 0, "ready": {}}
    from toppra_b200.batch import copy_stream
    d2h_stream = copy_stream(dev)
    nccl_side = torch.cuda.Stream(dev) if world > 1 else None

    def step_e2e_full():
        # the public API with HOST inputs (pinned tensors): the H2D copies happen inside the constructors; inputs are
        # validated on the host (no device synchronisation)
        path = ta.BatchSplineInterpolator(h_ss, h_way, device=dev)
        pc_vel = ta.constraint.JointVelocityConstraint(vlim)
        pc_acc = ta.constraint.JointAccelerationConstraint(alim)
        pc_vel._d_cache[str(dev)] = h_vlim.to(dev, non_blocking=True)
        pc_acc._d_cache[str(dev)] = h_alim.to(dev, non_blocking=True)
        inst = ta.BatchTOPPRA([pc_vel, pc_acc], path, h_grid)
        # K leaves on a copy stream while the forward pass runs; sync=False: pipelined caller, the pinned buffers are
        # valid at inst.host_ready (all copies are still inside the timed region); sync=True: host waits every step
        e2e_mode["k"] += 1
        k = e2e_mode["k"]
        if not e2e_mode["sync"]:
            # double buffering as a real pipelined caller does it: result buffer k & 1 is reused only after the solve that
            # filled it last (step k - 2) has landed on the host — at most two steps are in flight
            prev = e2e_mode["ready"].get(k & 1)
            if prev is not None:
                prev.synchronize()
        inst.solve_to_host(0.0, 0.0, pinned=h_sets[k & 1], sync=e2e_mode["sync"])
        if not e2e_mode["sync"]:
            e2e_mode["ready"][k & 1] = inst.host_ready
        if world > 1:
            # NCCL: gather the result velocities; on a side stream, so the next step's kernels overlap the collective
            sd = inst.last_result.sd
            done = torch.cuda.Event()
            done.record()
            with torch.cuda.stream(nccl_side):
                nccl_side.wait_event(done)
                dist.all_gather_into_tensor(gathered, sd)
            sd.record_stream(nccl_side)
        return inst

    def timed_pipelined(fn, steps, warmup):
        """e2e throughput of a pipelined caller: ONE event pair around the K steps; every H2D copy, kernel, D2H copy and
        the NCCL gather of all K steps completes inside it (the caller's stream waits for the copy / NCCL side streams
        before the closing event).  The L2 flush between iterations is inside the timed region here."""
        main = torch.cuda.current_stream(dev)
        for _ in range(warmup):
            fn()
            flush.zero_()
        main.wait_stream(d2h_stream)
        if nccl_side is not None:
            main.wait_stream(nccl_side)
        barrier()
        s, e = ev(), ev()
        s.record()
        for _ in range(steps):
            flush.zero_()
            fn()
        main.wait_stream(d2h_stream)
        if nccl_side is not None:
            main.wait_stream(nccl_side)
        e.record()
        barrier()
        t = torch.tensor([s.elapsed_time(e)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, steps, warmup, record_kernels=False):
        for _ in range(warmup):
            fn()
            flush.zero_()
        barrier()
        pairs = []
        for _ in range(steps):
            flush.zero_()  # L2 flush between timed iterations (outside the event pair)
            s, e = ev(), ev()
            s.record()
            fn(True) if record_kernels else fn()
            e.record()
            pairs.append((s, e))
        barrier()
        ms = sum(s.elapsed_time(e) for s, e in pairs)
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def measure():
        sampler = ClockSampler(local_rank)
        sampler.start()
        del k_events[:]
        a = timed(step_device, args.steps, max(args.warmup, 3), record_kernels=True)
        e2e_mode["sync"] = False
        b = timed_pipelined(step_e2e_full, args.steps, max(args.warmup, 3))
        e2e_mode["sync"] = True
        c = timed(step_e2e_full, args.steps, max(args.warmup, 3))
        torch.cuda.synchronize()
        sampler.stop_flag = True
        sampler.join(timeout=1.0)
        return a, b, c, sampler.summary()

    ms_dev, ms_e2e, ms_e2e_sync, clocks = measure()
    bad = {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    if bad & set(clocks.get("reasons", [])):  # throttled: take the measurement again, once
        clocks_first = clocks
        ms_dev, ms_e2e, ms_e2e_sync, clocks = measure()
        clocks["remeasured_after"] = clocks_first
    if args.dump_outputs and rank == 0:
        dump_outputs(last_out["out"], args.dump_outputs)

    # opt-in mode (BatchTOPPRA(exact=False), TB_SCAN_FAST_LOWER): reported beside the headline, never instead of it
    scan_mode["fast_lower"] = True
    ms_fast = timed(step_device, args.steps, max(args.warmup, 3))
    scan_mode["fast_lower"] = False
    ms_rec = timed(step_records, args.steps, max(args.warmup, 3))

    status = h_out["status"].numpy()
    n_ok = int((status == 0).sum())
    total_paths = B * world
    value = total_paths * args.steps / (ms_dev * 1e-3)
    e2e_value = total_paths * args.steps / (ms_e2e * 1e-3)
    k0 = float(np.mean([e[0].elapsed_time(e[1]) for e in k_events]))
    k1 = float(np.mean([e[1].elapsed_time(e[2]) for e in k_events]))
    k2 = float(np.mean([e[2].elapsed_time(e[3]) for e in k_events]))

    peaks0 = {}
    try:
        peaks0 = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    # per-rank K2 time (SCALE: explains the max-over-ranks step time)
    k2_ranks = torch.tensor([k2, -k2], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(k2_ranks, op=dist.ReduceOp.MAX)
    k2_min, k2_max = -float(k2_ranks[1].item()), float(k2_ranks[0].item())
    try:
        configs = extra_configs(args, torch, dist, ta, dev, world, rank, float(peaks0.get("hbm_gbs", 6650.0)))
    except Exception as exc:  # never lose the headline line
        configs = {"error": repr(exc)}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # roofline of the dominant kernel: the fused scan (tb_scan_velacc).  SURVEY.md section 8d's contract: report against the
    # MATERIALISED-record algorithmic bytes (rows read twice + outputs) and note what the fused form really moves.
    peak = float(peaks0.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks0 else "fallback 6.65 TB/s"
    bytes_k1 = (4 * (nway - 1) * dof * 8 + G * (3 * R + 2) * 8) * B
    bytes_k2 = (2 * G * (3 * R + 2) * 8 + G * 16 + G * 8 + (G - 1) * 8 + 8) * B
    bytes_fused = (4 * (nway - 1) * dof * 8 + G * 16 + G * 16 + G * 8 + (G - 1) * 8 + 8) * B
    bytes_xb = (4 * (nway - 1) * dof * 8 + G * 16) * B
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        pass
    roof = {"kernel": "scan_kernel<FUSED> (tb_scan_velacc: K1 rows built inside K2)", "bound": "hbm",
            "achieved": bytes_k2 / (k2 * 1e-3) / 1e9, "peak": peak,
            "unit": "GB/s", "frac": bytes_k2 / (k2 * 1e-3) / 1e9 / peak,
            "traffic": (traffic or {}).get("scan_velacc_bytes_per_launch"), "peak_source": peak_src,
            "algorithmic_bytes_per_launch": bytes_k2, "ms_per_launch": k2,
            "fused_bytes_per_launch": bytes_fused,
            "note": "algorithmic bytes = the materialised-record figure of SURVEY 8d (281,600 B/path); the fused kernel "
                    "itself reads spline + velocity bound and writes K, sd, u (fused_bytes_per_launch): the scan is a "
                    "latency/issue-bound chain of 597 dependent LPs per path, see lp_solves_per_s and profiles/"}
    roof_k1 = {"kernel": "xbound_velocity_kernel (K1 of the fused path: velocity bound only)", "bound": "hbm",
               "achieved": bytes_xb / (k1 * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
               "frac": bytes_xb / (k1 * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_launch": bytes_xb, "ms_per_launch": k1}
    timed_rec = rec_events[-args.steps:]        # the warm-up steps (first launch = module load) are not part of the figure
    rk0 = float(np.mean([e[0].elapsed_time(e[1]) for e in timed_rec]))
    rk1 = float(np.mean([e[1].elapsed_time(e[2]) for e in timed_rec]))
    rk2 = float(np.mean([e[2].elapsed_time(e[3]) for e in timed_rec]))
    records_path = {
        "what": "the same batch through materialised stage records (generic constraint lists: K0 -> K1 coeff_velacc -> "
                "K2 record scan); not part of `value`",
        "ms_per_step": ms_rec / args.steps, "kernels_ms": {"K0": rk0, "K1_coeff_velacc": rk1, "K2_scan_records": rk2},
        "roofline_k1": {"bound": "hbm", "achieved": bytes_k1 / (rk1 * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                        "frac": bytes_k1 / (rk1 * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_launch": bytes_k1,
                        "traffic": (traffic or {}).get("coeff_velacc_kernel_bytes_per_launch")},
        "roofline_k2": {"bound": "hbm", "achieved": bytes_k2 / (rk2 * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                        "frac": bytes_k2 / (rk2 * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_launch": bytes_k2,
                        "traffic": (traffic or {}).get("scan_kernel_bytes_per_launch")}}

    h2d = int(h_way.numel() + h_vlim.numel() + h_alim.numel() + h_ss.numel() + h_grid.numel()) * 8
    d2h = int(h_out["K"].numel() + h_out["sd"].numel() + h_out["sdd"].numel()) * 8 + int(h_out["status"].numel()) * 8
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_text(B, dof, G),
                   "global_batch": total_paths, "parallelism": "paths sharded over %d GPU(s), no data-path collective" % world,
                   "l2": "256 MB buffer written between timed iterations (L2 flush)", "ok_paths_last_step": n_ok},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": ms_e2e / args.steps,
                "host_sync_every_step": {"value": total_paths * args.steps / (ms_e2e_sync * 1e-3), "unit": UNIT,
                                         "ms_per_step": ms_e2e_sync / args.steps},
                "api": "BatchSplineInterpolator + BatchTOPPRA.solve_to_host(sync=False) with pinned HOST inputs and "
                       "outputs: a pipelined caller with two result buffers (at most two steps in flight: a buffer is "
                       "reused once its previous solve has landed); all D2H copies run on the package's copy "
                       "stream and overlap the next step's kernels; ONE event pair around the K steps, every copy of "
                       "every step (and the L2 flushes) inside it; host_sync_every_step = the same call with sync=True "
                       "(host waits for each step's results; per-step event pairs)"
                       + (", NCCL all_gather of sd" if world > 1 else "")},
        "gpu_launches": 3 * args.steps,
        "kernels_ms": {"K0_spline_fit": k0, "K1_xbound": k1, "K2_scan_velacc": k2, "K2_ranks_min_max": [k2_min, k2_max]},
        "configs": configs,
        "roofline": roof, "roofline_k1": roof_k1, "records_path": records_path,
        "lp_solves_per_s": 597.0 / 199 * (G - 1) * B / (k2 * 1e-3),
        "opt_in_fast_lower_bound": {
            "value": total_paths * args.steps / (ms_fast * 1e-3), "unit": UNIT, "ms_per_step": ms_fast / args.steps,
            "note": "BatchTOPPRA(exact=False): the min-x LP of each backward stage returns xbound_lo when some u is "
                    "feasible there (the exact LP optimum) instead of replaying the reference's Seidel re-solves; "
                    "deviates from the reference by its rounding noise (<= ~1e-15 on K, sd; tests: 1e-12). "
                    "NOT the default; value/e2e above are the bit-identical default."},
        "clocks": clocks,
        "cpu_baseline": cpu,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
