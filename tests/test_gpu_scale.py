"""GPU (-m gpu): BASELINE.json sizes.  cfg 2 (B=4096, 7-DOF, 200 gridpoints) is checked bit-for-bit against the
oracle (the C restatement solves 4096 paths in about a second on a few threads); the larger batch is checked
through size-independent properties of a correct parameterisation."""
import os

import numpy as np
import pytest

from problems import make_batch, make_batch_fast

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ta():
    import toppra_b200
    return toppra_b200


def _solve(ta, ss, way, vlim, alim, grid, counters=False):
    path = ta.BatchSplineInterpolator(ss, way)
    inst = ta.BatchTOPPRA([ta.constraint.JointVelocityConstraint(vlim), ta.constraint.JointAccelerationConstraint(alim)],
                          path, grid)
    res = inst.compute_parameterization(0.0, 0.0, counters=counters)
    return path, inst, res


def test_cfg2_full_batch_vs_oracle(ta):
    from oracle import oracle as orc
    B, G = 4096, 200
    ss, way, vlim, alim = make_batch(B, 1000)          # path b uses RandomState(1000 + b), SURVEY §8d cfg 2
    grid = np.linspace(0, 1, G)
    path, inst, res = _solve(ta, ss, way, vlim, alim, grid, counters=True)
    h = res.to_host()
    c = path.d_ppoly.cpu().numpy()
    o = orc.solve_velacc_batch(c, np.tile(ss, (B, 1)), grid, vlim, alim, True, nthreads=min(16, os.cpu_count() or 1))
    assert np.array_equal(h["status"], o["status"]) and not h["status"].any()
    assert np.array_equal(h["K"], o["K"]) and np.array_equal(h["sd"], o["sd"]) and np.array_equal(h["sdd"], o["u"])
    cnt = res.counters.cpu().numpy()
    assert (cnt[:, 0] == 2 * (G - 1)).all() and (cnt[:, 1] == G - 1).all()   # 398 2-D + 199 1-D LPs per path


def test_velocity_active_batch_vs_oracle(ta):
    from oracle import oracle as orc
    B, G = 512, 200
    ss, way, vlim, alim = make_batch(B, 1000, vel_active=True)
    grid = np.linspace(0, 1, G)
    path, inst, res = _solve(ta, ss, way, vlim, alim, grid)
    h = res.to_host()
    o = orc.solve_velacc_batch(path.d_ppoly.cpu().numpy(), np.tile(ss, (B, 1)), grid, vlim, alim, True, nthreads=8)
    assert np.array_equal(h["status"], o["status"])
    assert np.array_equal(h["K"], o["K"]) and np.array_equal(h["sd"], o["sd"]) and np.array_equal(h["sdd"], o["u"])


def test_large_batch_properties(ta):
    """65536 paths (cfg-5 shard size order): properties that hold for every correct parameterisation."""
    import torch
    B, G = 65536, 200
    ss, way, vlim, alim = make_batch_fast(B, seed=77)
    grid = np.linspace(0, 1, G)
    path, inst, res = _solve(ta, ss, way, vlim, alim, grid)
    assert int((res.status != 0).sum()) == 0
    K, sd, u = res.K, res.sd, res.sdd
    x = sd * sd
    assert bool((sd[:, 0] == 0).all()) and bool((sd[:, -1] == 0).all())
    assert bool((K[:, :, 0] <= K[:, :, 1]).all()) and bool((K[:, :, 0] >= 0).all())
    assert bool((x <= K[:, :, 1] * (1 + 1e-12) + 1e-15).all()) and bool((x >= K[:, :, 0] - 1e-15).all())
    d_grid = inst.d_grid
    qs = path.eval_device(d_grid, 1)
    qss = path.eval_device(d_grid, 2)
    # joint accelerations q' u + q'' x within limits at every stage (u constant on the stage)
    acc = qs[:, :-1] * u[:, :, None] + qss[:, :-1] * x[:, :-1, None]
    amax = torch.as_tensor(alim[:, None, :, 1], device=acc.device)
    assert float((acc.abs() - amax).max()) < 1e-6
    vel = qs * sd[:, :, None]
    vmax = torch.as_tensor(vlim[:, None, :, 1], device=vel.device)
    assert float((vel.abs() - vmax).max()) < 1e-6
    # dynamics consistency: x_{i+1} <= x_i + 2 ds u_i (equality before the safety shrink 1e-8 / 0.9999)
    ds = d_grid[1:] - d_grid[:-1]
    xn = x[:, :-1] + 2 * ds * u
    assert float((x[:, 1:] - xn).max()) <= 1e-12
    assert float((xn - x[:, 1:]).max()) <= 1e-4 * float(xn.max()) + 2e-8
    # determinism + independence of batch composition: first 256 paths alone give identical bits
    _, _, res2 = _solve(ta, ss, way[:256], vlim[:256], alim[:256], grid)
    assert torch.equal(res2.sd, sd[:256]) and torch.equal(res2.K, K[:256])


def test_chunked_solve_equals_single_launch(ta):
    """Batches whose records exceed the budget run chunk by chunk through one record buffer (fused=False: materialised
    stage records): identical bits to the single fused launch (rows built inside the scan)."""
    import torch
    B, G = 1000, 120
    ss, way, vlim, alim = make_batch_fast(B, seed=5)
    grid = np.linspace(0, 1, G)
    path = ta.BatchSplineInterpolator(ss, way)
    cons = [ta.constraint.JointVelocityConstraint(vlim), ta.constraint.JointAccelerationConstraint(alim)]
    full = ta.BatchTOPPRA(cons, path, grid).compute_parameterization(0.0, 0.0)
    per_path = 8 * 86 * G
    inst = ta.BatchTOPPRA(cons, path, grid, max_record_bytes=per_path * 96 + 7, fused=False)   # 96 paths per chunk, ragged tail
    assert inst.chunk_size() == 96
    part = inst.compute_parameterization(0.0, 0.0)
    for key in ("K", "sd", "sdd", "status"):
        assert torch.equal(getattr(full, key), getattr(part, key)), key
    # per-path boundary speeds are sliced with the chunks
    s0 = np.where(np.arange(B) % 2 == 0, 0.0, 0.05)
    a = ta.BatchTOPPRA(cons, path, grid).compute_parameterization(s0, 0.0)
    b = ta.BatchTOPPRA(cons, path, grid, max_record_bytes=per_path * 96, fused=False).compute_parameterization(s0, 0.0)
    assert torch.equal(a.sd, b.sd) and torch.equal(a.status, b.status)
    assert float(a.sd[1, 0]) == 0.05 and float(a.sd[0, 0]) == 0.0


def test_cfg5_shard_size_chunked(ta):
    """cfg-5 style: 2^17 paths (one GPU's shard of the 1M-path batch) through the chunked path."""
    B, G = 1 << 17, 200
    ss, way, vlim, alim = make_batch_fast(B, seed=11)
    grid = np.linspace(0, 1, G)
    path = ta.BatchSplineInterpolator(ss, way)
    cons = [ta.constraint.JointVelocityConstraint(vlim), ta.constraint.JointAccelerationConstraint(alim)]
    inst = ta.BatchTOPPRA(cons, path, grid, max_record_bytes=4 << 30, fused=False)
    assert inst.chunk_size() < B
    res = inst.compute_parameterization(0.0, 0.0)
    assert int((res.status != 0).sum()) == 0
    import torch
    one = ta.BatchTOPPRA(cons, path, grid)   # fused scan: the whole shard in ONE launch, no record buffer
    assert one.fused and one.chunk_size() == B
    res1 = one.compute_parameterization(0.0, 0.0)
    for key in ("K", "sd", "sdd", "status"):
        assert torch.equal(getattr(res, key), getattr(res1, key)), key
    assert bool((res.sd[:, 0] == 0).all()) and bool((res.sd[:, -1] == 0).all()) and bool((res.sd[:, 1:-1] > 0).all())
    x = res.sd * res.sd
    assert bool((x <= res.K[:, :, 1] * (1 + 1e-12) + 1e-15).all())


@pytest.mark.parametrize("dof,G,B", [(1, 2, 1), (2, 3, 5), (12, 37, 5), (20, 64, 3), (31, 50, 2), (7, 1000, 2)])
def test_shapes_rows_per_lane_and_tiny_grids(ta, dof, G, B):
    """1..4 LP rows per lane (R = 4*dof up to 124), one-stage grids, batches that do not fill a CTA: vs the oracle."""
    from oracle import oracle as orc
    ss, way, vlim, alim = make_batch(B, 4000 + dof, dof=dof)
    grid = np.linspace(0, 1, G)
    path, inst, res = _solve(ta, ss, way, vlim, alim, grid)
    h = res.to_host()
    c = path.d_ppoly.cpu().numpy()
    for b in range(B):
        assert np.array_equal(c[b], orc.cubic_spline_fit(ss, way[b]))
        o = orc.solve_velacc(c[b], ss, grid, vlim[b], alim[b], True, 0, 0)
        assert h["status"][b] == o["status"]
        assert np.array_equal(h["K"][b], o["K"], equal_nan=True) and np.array_equal(h["sd"][b], o["sd"], equal_nan=True)
        assert np.array_equal(h["sdd"][b], o["u"], equal_nan=True)


def test_split_backward_forward_and_host_copy(ta):
    """BatchTOPPRA.solve_to_host: backward-only + forward-only launches (K copied out in between) == single launch."""
    import torch
    B, G = 777, 150
    ss, way, vlim, alim = make_batch_fast(B, seed=21)
    vlim[:50] *= 0.03  # some velocity-active paths
    grid = np.linspace(0, 1, G)
    path = ta.BatchSplineInterpolator(ss, way)
    cons = [ta.constraint.JointVelocityConstraint(vlim), ta.constraint.JointAccelerationConstraint(alim)]
    inst = ta.BatchTOPPRA(cons, path, grid)
    s0 = np.where(np.arange(B) % 7 == 0, 30.0, 0.0)   # every 7th path starts inadmissibly fast -> FailUncontrollable
    one = inst.compute_parameterization(s0, 0.0).to_host()
    host = inst.solve_to_host(s0, 0.0)
    torch.cuda.synchronize()
    assert (one["status"][::7] == 3).all() and (one["status"][1::7] == 0).all()
    for key in ("K", "sd", "sdd", "status"):
        assert np.array_equal(one[key], host[key].numpy(), equal_nan=True), key
    # pipelined caller (sync=False): several solves in flight on two result buffers; every device-to-host copy runs on the
    # package's copy stream; each buffer is valid when its own host_ready event has completed — no device-wide sync
    sets = [inst._pinned_outputs(None), inst._pinned_outputs(None)]
    starts = [s0, np.zeros(B), 0.5 * s0, s0]
    refs = [inst.compute_parameterization(v, 0.0).to_host() for v in starts]
    pending = []
    for k, v in enumerate(starts):
        if k >= 2:   # the buffer about to be reused: its previous solve must have landed and been checked
            kk, evt, buf = pending.pop(0)
            evt.synchronize()
            for key in ("K", "sd", "sdd", "status"):
                assert np.array_equal(refs[kk][key], buf[key].numpy(), equal_nan=True), (kk, key)
        buf = inst.solve_to_host(v, 0.0, pinned=sets[k & 1], sync=False)
        pending.append((k, inst.host_ready, buf))
    for kk, evt, buf in pending:
        evt.synchronize()
        for key in ("K", "sd", "sdd", "status"):
            assert np.array_equal(refs[kk][key], buf[key].numpy(), equal_nan=True), (kk, key)


def test_fast_lower_bound_mode(ta):
    """exact=False (TB_SCAN_FAST_LOWER): same LP optima, not the reference's rounding noise: deviations <= 1e-12
    (measured ~1e-16), statuses equal; exact=True stays bit-identical (all the other tests)."""
    B, G = 2048, 200
    ss, way, vlim, alim = make_batch_fast(B, seed=99)
    vlim[:256] *= 0.03
    grid = np.linspace(0, 1, G)
    path = ta.BatchSplineInterpolator(ss, way)
    cons = [ta.constraint.JointVelocityConstraint(vlim), ta.constraint.JointAccelerationConstraint(alim)]
    exact = ta.BatchTOPPRA(cons, path, grid).compute_parameterization(0.0, 0.0, counters=True)
    fast = ta.BatchTOPPRA(cons, path, grid, exact=False).compute_parameterization(0.0, 0.0, counters=True)
    he, hf = exact.to_host(), fast.to_host()
    assert np.array_equal(he["status"], hf["status"]) and not he["status"].any()
    assert np.abs(he["K"] - hf["K"]).max() <= 1e-12 and np.abs(he["sd"] - hf["sd"]).max() <= 1e-12
    assert np.abs(he["sdd"] - hf["sdd"]).max() <= 1e-9 * max(1.0, np.abs(he["sdd"]).max())
    ce, cf = exact.counters.cpu().numpy(), fast.counters.cpu().numpy()
    assert cf[:, 2].sum() < 0.7 * ce[:, 2].sum()      # far fewer projected re-solves


def test_skip_ahead_is_bit_identical_on_many_paths(ta):
    """The Seidel skip-ahead of the min-x LP (csrc/tb_scan.cu) must not change a single bit: 16384 fresh random
    paths + 2048 velocity-limited ones + mixed start/end speeds against the sequential oracle."""
    from oracle import oracle as orc
    G = 200
    grid = np.linspace(0, 1, G)
    for B, seed, scale in ((16384, 4242, 1.0), (2048, 777, 0.03)):
        ss, way, vlim, alim = make_batch_fast(B, seed=seed)
        vlim = vlim * scale
        path, inst, res = _solve(ta, ss, way, vlim, alim, grid, counters=True)
        h = res.to_host()
        o = orc.solve_velacc_batch(path.d_ppoly.cpu().numpy(), np.tile(ss, (B, 1)), grid, vlim, alim, True,
                                   nthreads=min(16, os.cpu_count() or 1))
        assert np.array_equal(h["status"], o["status"])
        assert np.array_equal(h["K"], o["K"], equal_nan=True) and np.array_equal(h["sd"], o["sd"], equal_nan=True)
        assert np.array_equal(h["sdd"], o["u"], equal_nan=True)
    # fewer projected re-solves than LPs x 3 shows the skip-ahead is actually taken
    cnt = res.counters.cpu().numpy()
    assert cnt[:, 2].mean() < 2.5 * (G - 1)


@pytest.mark.parametrize("interp", [True, False])
def test_large_batch_forward_threads_bit_identical(ta, interp):
    """Batches of >= 24576 paths run the forward pass with one thread per path (csrc/tb_scan_fwd.cu) after a backward-only
    launch of the warp kernel: same bits as the sequential oracle.  An odd batch size, velocity-limited paths (the retry
    rule), inadmissible and non-zero boundary speeds, both discretisation schemes; the split launch of solve_to_host too."""
    from oracle import oracle as orc
    B, G = 24576 + 37, 48
    ss, way, vlim, alim = make_batch_fast(B, seed=9090)
    vlim[:3000] *= 0.03
    s0 = np.where(np.arange(B) % 13 == 0, 30.0, np.where(np.arange(B) % 5 == 0, 0.05, 0.0))
    s1 = np.where(np.arange(B) % 7 == 0, 0.04, 0.0)
    grid = np.linspace(0, 1, G)
    path = ta.BatchSplineInterpolator(ss, way)
    inst = ta.BatchTOPPRA([ta.constraint.JointVelocityConstraint(vlim),
                           ta.constraint.JointAccelerationConstraint(alim, discretization_scheme=1 if interp else 0)], path, grid)
    assert inst.fused
    h = inst.compute_parameterization(s0, s1).to_host()
    o = orc.solve_velacc_batch(path.d_ppoly.cpu().numpy(), np.tile(ss, (B, 1)), grid, vlim, alim, interp, sd_start=s0,
                               sd_end=s1, nthreads=min(16, os.cpu_count() or 1))
    assert np.array_equal(h["status"], o["status"]) and (h["status"] == 3).sum() >= B // 13 and (h["status"] == 0).sum() > B // 2
    assert np.array_equal(h["K"], o["K"], equal_nan=True) and np.array_equal(h["sd"], o["sd"], equal_nan=True)
    assert np.array_equal(h["sdd"], o["u"], equal_nan=True)
    host = inst.solve_to_host(s0, s1)                 # backward-only launch, then the forward pass alone
    for key, ref in (("K", o["K"]), ("sd", o["sd"]), ("sdd", o["u"]), ("status", o["status"])):
        assert np.array_equal(host[key].numpy(), ref, equal_nan=True), key


@pytest.mark.parametrize("name", ["deg6", "deg20", "scaled14"])
def test_seidel_shortcuts_on_stress_rows_vs_reference_golden(ta, golden, name):
    """The K2 shortcuts (csrc/tb_scan.cu, A: jump to the last visited row, B: skip the first warm-start re-solve) must
    fall back to the ordinary walk whenever a decision is close to the TINY threshold.  Raw rows with near-duplicate,
    scaled, parallel and slightly rotated copies (perturbations 1e-14 .. 1e-6) and badly scaled rows (coefficients down
    to 1e-8, optima up to the 1e10 sentinel): 4200 problems, one and two rows per lane, bit for bit against the
    REFERENCE's own seidelWrapper results (tests/golden/shortcut_rows_<set>.npz, generated by make_golden.py shortcut_rows
    from the unmodified reference).  The kernel's per-path re-solve counters must also equal those of the scalar
    shortcut model (oracle/shortcut_model.c), which ties the model campaigns to the kernel's decisions."""
    import torch
    from oracle import oracle as orc
    from problems import SHORTCUT_SETS
    g = golden("shortcut_rows_" + name)
    gen, args = SHORTCUT_SETS[name]
    rows, xb = gen(*args)
    B, G, _, R = rows.shape
    grid = np.linspace(0, 1, G)
    dev = torch.device("cuda:0")
    rec, W = ta.engine.alloc_records(B, G, R, dev)
    host = np.zeros((B, G, W))
    host[:, :, 0:R] = rows[:, :, 0]
    host[:, :, R:2 * R] = rows[:, :, 1]
    host[:, :, 2 * R:3 * R] = rows[:, :, 2]
    # the xbound slots hold the bound intersected with the solver box, as every record producer writes them
    # (seidelWrapper low/high init, pyx:477-478,517-520; scaled14 has xbound_hi up to 1e9)
    host[:, :, 3 * R] = np.maximum(xb[:, :, 0], -1e8)
    host[:, :, 3 * R + 1] = np.minimum(xb[:, :, 1], 1e8)
    rec.copy_(torch.from_numpy(host))
    z = torch.zeros(B, dtype=torch.float64, device=dev)
    out = ta.engine.scan(rec, R, torch.from_numpy(grid).to(dev), z, z, z, counters=True)
    K, sd, u, st, cnt = (out[k].cpu().numpy() for k in ("K", "sd", "u", "status", "counters"))
    assert np.array_equal(st, g[name + "_status"])
    assert np.array_equal(K, g[name + "_K"], equal_nan=True)
    ok = st == 0
    assert ok.sum() > B // 2
    assert np.array_equal(sd, g[name + "_sd"], equal_nan=True) and np.array_equal(u, g[name + "_sdd"], equal_nan=True)
    # re-solve counters: kernel == scalar model of the shortcut rules, path by path
    for i in range(0, B, 7):
        with orc.shortcut_model() as sm:
            orc.solve_rows(rows[i], xb[i], grid, 0.0, 0.0)
            stt = sm.stats()
        assert stt["mismatches"] == 0
        assert cnt[i, 2] == stt["resolves_model"], (i, cnt[i], stt)
