"""Stage rows of the torque constraint (tb_coeff_second_order) and of generic CanonicalLinear constraints
(tb_rows_canlinear), checked record by record.

  * The torque rows are compared with an independent restatement: q, q', q'' from oracle.ppoly_eval (bit-identical to the
    device evaluator), the model of include/toppra_b200.h evaluated in mpmath at 40 digits (cos(q_i - q_j) as written, not
    the kernel's expanded form), F = [I; -I], g = [tau_max; -tau_min], dry friction sign(q') * f, the Interpolation lift
    a+ = a_{i+1} + 2 delta_i b_{i+1}.  Each entry must lie within 16 eps S of it, S being the sum of the magnitudes of the
    terms that make up the entry (see `_scales`); the pendulum model's a and b entries are single products and must equal
    the same float64 operations exactly.  The reference is anchored on the rows that reproduce the upstream golden.
    Worst |got - ref| / (eps S) measured on an NVIDIA B200 (1000 W power limit): 1.82 for coupled_cosine, 1.13 for
    pendulums; a float64 numpy model of the kernel's arithmetic reaches the same.  The tests print it per model.
  * Shapes and edges: both models and schemes, dof 1..16, G from 1 to one gridpoint past three 32-point tiles, shared and
    per-path breaks / grids / limits, asymmetric limits, friction with q' of both signs and q' = 0 on a frozen joint, rows
    at row 0 and inside a larger odd R.  Every slot the call does not own must keep a sentinel bit pattern.
  * End to end: BatchTOPPRA with a device model, the records it built fed to oracle.solve_rows reproduce the GPU scan bit for
    bit, and a solve in several chunks equals the one-launch solve bit for bit.
  * tb_rows_canlinear records, every F mode, against a numpy restatement of its summation order, bit for bit.
  * A CPU test corrupts correct records in the ways these kernels could go wrong and checks that the comparison notices.

Every test with the `ta` fixture runs on the GPU (-m gpu) and on the CPU engine double (tests/cpu_engine.py)."""
import ctypes
import functools

import mpmath
import numpy as np
import pytest

import cpu_engine
from oracle import oracle as orc

EPS = np.finfo(np.float64).eps
TOL = 16.0                                  # |got - ref| <= TOL * eps * S
SENTINEL = np.int64(0x7FF4DEADBEEFCAFE)     # a signalling-NaN bit pattern no kernel writes
MODELS = ("coupled_cosine", "pendulums")
DOFS = (1, 2, 6, 7, 16)                     # 16 = SO_MAX_DOF of csrc/tb_coeff.cu
GS = (1, 2, 31, 32, 33, 64, 65, 97)         # around the 32-gridpoint tile of second_order_rows_tiled_kernel
WORST = {}                                  # (engine, model) -> largest |got - ref| / (eps S) seen


@pytest.fixture(params=[pytest.param("gpu", marks=pytest.mark.gpu), "cpu_double"])
def ta(request, monkeypatch):
    if request.param == "cpu_double":
        return cpu_engine.install(monkeypatch)
    import toppra_b200
    return toppra_b200


@pytest.fixture(scope="module", autouse=True)
def _report_worst():
    yield
    for key in sorted(WORST):
        print("torque rows, %s %s: worst |got - ref| / (eps S) = %.3f (bound %g)" % (key + (WORST[key], TOL)))


def _note(engine, model, ratio):
    WORST[(engine, model)] = max(WORST.get((engine, model), 0.0), ratio)


def _engine_name(ta):
    return "gpu" if ta.engine.default_device().type == "cuda" else "cpu_double"


# ---- the independent reference ---------------------------------------------------------------------------------------
def _dd(x):
    """mpf -> (hi, lo) with hi + lo = x to about 2^-106 relative."""
    hi = float(x)
    return hi, float(x - hi)


def _model_terms_mp(model, params, q, qd, qdd, friction):
    """a = tau(q, 0, q') - tau(q, 0, 0), b = tau(q, q', q'') - tau(q, 0, 0), c = tau(q, 0, 0) + sign(q') f at every
    gridpoint, straight from the model definition, in 40-digit arithmetic.  Returns (A, B, C) as mpf lists [G][dof]."""
    G, dof = q.shape
    mpf = mpmath.mpf
    A, B, C = [], [], []
    with mpmath.workdps(40):
        P = [mpf(float(x)) for x in params]
        for i in range(G):
            Q, QD, QDD = ([mpf(float(x)) for x in v[i]] for v in (q, qd, qdd))
            S = [mpmath.sin(x) for x in Q]
            if model == "coupled_cosine":
                cosm = [[mpf(1)] * dof for _ in range(dof)]
                for k in range(dof):
                    for j in range(k + 1, dof):
                        cosm[k][j] = cosm[j][k] = mpmath.cos(Q[k] - Q[j])
                v2 = mpmath.fdot(QD, QD)
                A.append([P[0] * QD[k] + P[1] * mpmath.fdot(cosm[k], QD) for k in range(dof)])
                B.append([P[0] * QDD[k] + P[1] * mpmath.fdot(cosm[k], QDD) + P[2] * S[k] * v2 for k in range(dof)])
                C.append([P[3] * S[k] for k in range(dof)])
            else:
                A.append([P[2 * k] * QD[k] for k in range(dof)])
                B.append([P[2 * k] * QDD[k] for k in range(dof)])
                C.append([P[2 * k + 1] * S[k] for k in range(dof)])
            if friction is not None:
                C[-1] = [C[-1][k] + int(np.sign(qd[i, k])) * mpf(float(friction[k])) for k in range(dof)]
    return A, B, C


def _scales(model, params, qd, qdd, friction):
    """Per-entry magnitude S of a, b, c (float64 [G, dof]):
    S(b) = |p0 q''_k| + 2 |p1| sum_j |q''_j| + |p2| sum_j q'_j^2, S(a) the same with q' for q'' (no p2 term), S(c) = |p3| + |f|
    (pendulums: |p_2k q''_k|, |p_2k q'_k|, |p_2k+1| + |f|)."""
    p = np.abs(np.asarray(params, dtype=np.float64))
    f = np.zeros(qd.shape[1]) if friction is None else np.abs(friction)
    if model == "coupled_cosine":
        sa = p[0] * np.abs(qd) + 2 * p[1] * np.abs(qd).sum(1, keepdims=True)
        sb = p[0] * np.abs(qdd) + 2 * p[1] * np.abs(qdd).sum(1, keepdims=True) + p[2] * (qd * qd).sum(1, keepdims=True)
        sc = p[3] + f + 0 * qd
    else:
        sa, sb, sc = p[0::2] * np.abs(qd), p[0::2] * np.abs(qdd), p[1::2] + f + 0 * qd
    return sa, sb, sc


def _assemble(a, b, cmax, cmin, aplus, interp, neg=np.negative):
    """Rows [G, 3, nrows] of F = [I; -I]: blocks (+, -) at s_i, then (+, -) lifted from s_{i+1} (interp).  cmax = c - tau_max,
    cmin = c - tau_min; the negated copy's c row is -c + tau_min = -cmin.  The last gridpoint duplicates itself."""
    G = a.shape[0]
    src = np.minimum(np.arange(G) + 1, G - 1)
    blocks = [(a, b, cmax), (neg(a), neg(b), neg(cmin))]
    if interp:
        blocks += [(aplus, b[src], cmax[src]), (neg(aplus), neg(b[src]), neg(cmin[src]))]
    return np.stack([np.concatenate([blk[part] for blk in blocks], axis=1) for part in range(3)], axis=1)


def torque_rows_reference(model, params, q, qd, qdd, grid, taulim, friction, interp):
    """Reference rows of one path: dict(hi, lo, S [G, 3, nrows], exact [G, 3, nrows] (float64 restatement where the
    kernel's arithmetic is a single product, NaN elsewhere))."""
    G, dof = q.shape
    A, B, C = _model_terms_mp(model, params, q, qd, qdd, friction)
    tmin, tmax = taulim[:, 0], taulim[:, 1]
    hi = {n: np.empty((G, dof)) for n in ("a", "b", "cmax", "cmin", "aplus")}
    lo = {n: np.empty((G, dof)) for n in hi}
    with mpmath.workdps(40):
        for i in range(G):
            j = min(i + 1, G - 1)
            two_delta = 2 * (mpmath.mpf(float(grid[j])) - mpmath.mpf(float(grid[i])))
            for k in range(dof):
                vals = dict(a=A[i][k], b=B[i][k], cmax=C[i][k] - float(tmax[k]), cmin=C[i][k] - float(tmin[k]),
                            aplus=A[j][k] + two_delta * B[j][k])
                for n, v in vals.items():
                    hi[n][i, k], lo[n][i, k] = _dd(v)
    sa, sb, sc = _scales(model, params, qd, qdd, friction)
    src = np.minimum(np.arange(G) + 1, G - 1)
    s_aplus = sa[src] + 2 * np.abs(grid[src] - grid)[:, None] * sb[src]
    out = dict(hi=_assemble(*(hi[n] for n in ("a", "b", "cmax", "cmin", "aplus")), interp),
               lo=_assemble(*(lo[n] for n in ("a", "b", "cmax", "cmin", "aplus")), interp),
               S=_assemble(sa, sb, sc + np.abs(tmax), sc + np.abs(tmin), s_aplus, interp, neg=lambda x: x))
    exact = np.full_like(out["hi"], np.nan)
    if model == "pendulums":
        pk = np.asarray(params, dtype=np.float64)[0::2]
        ea, eb = pk * qd, pk * qdd
        ap = ea[src] + (2 * (grid[src] - grid))[:, None] * eb[src]
        ap[G - 1] = ea[G - 1]
        nan = np.full_like(ea, np.nan)
        exact = _assemble(ea, eb, nan, nan, ap, interp)
    out["exact"] = exact
    return out


def compare_rows(got, ref):
    """got [G, 3, nrows] against a reference.  Returns (number of entries outside the bound or not exactly equal where
    required, worst |got - ref| / (eps S))."""
    S = ref["S"]
    with np.errstate(divide="ignore", invalid="ignore"):           # a sentinel (NaN) where a row belongs is a mismatch
        err = np.abs((got - ref["hi"]) - ref["lo"])
        ratio = np.where(S > 0, err / (EPS * S), np.where(err == 0, 0.0, np.inf))
    bad = ~(err <= TOL * EPS * S)                                  # NaN counts as bad
    ex = ~np.isnan(ref["exact"])
    bad |= ex & (got != ref["exact"])
    return int(bad.sum()), float(np.nanmax(ratio)) if ratio.size else 0.0


def check_records(rec, refs, R_total, row0, nrows):
    """rec [B, G, W] (float64) of one launch: problems found (list of str) and the worst error ratio.  The rows of every
    path must match `refs[b]`; every other slot (other rows, x bound, padding) must still hold the sentinel."""
    problems, worst = [], 0.0
    B, G, W = rec.shape
    own = np.zeros(W, dtype=bool)
    for part in range(3):
        own[part * R_total + row0:part * R_total + row0 + nrows] = True
    touched = rec.view(np.int64)[:, :, ~own] != SENTINEL
    if touched.any():
        problems.append("%d slots outside the rows were written" % int(touched.sum()))
    for b in range(B):
        got = np.stack([rec[b, :, part * R_total + row0:part * R_total + row0 + nrows] for part in range(3)], axis=1)
        nbad, ratio = compare_rows(got, refs[b])
        worst = max(worst, ratio)
        if nbad:
            problems.append("path %d: %d row entries off (worst %.3g eps S)" % (b, nbad, ratio))
    return problems, worst


# ---- problem set for tb_coeff_second_order ----------------------------------------------------------------------------
CASES = [(model, interp, dof) for model in MODELS for interp in (1, 0) for dof in DOFS]


def _launches(case):
    """Three launches per (model, scheme, dof); over the five dofs of one (model, scheme) every G of GS appears and every
    sharing / placement flag takes both values."""
    model, interp, dof = case
    off = 4 * (1 - interp) + 2 * MODELS.index(model)
    out = []
    for t in range(3):
        n = 3 * DOFS.index(dof) + t
        out.append(dict(G=GS[(n + off) % len(GS)], breaks_shared=n % 2 == 0, grid_shared=n % 3 != 1,
                        lim_shared=(n // 2) % 2 == 0, friction=n % 4 != 3, inner=n % 5 in (1, 2, 4),
                        seed=1000 * MODELS.index(model) + 100 * interp + 10 * DOFS.index(dof) + t))
    return out


def _model_params(model, dof, rng, standard=False):
    if model == "coupled_cosine":
        return np.array([2.0, 0.3, 0.1, 4.9]) if standard else np.array([1.3, -0.7, 0.45, -6.2])
    return np.stack((0.5 + 2.5 * rng.rand(dof), 1.0 + 9.0 * rng.rand(dof)), axis=1).reshape(-1)


def _asym_limits(rng, dof):
    """tau_min != -tau_max on every joint."""
    return np.stack((-(5.0 + 40.0 * rng.rand(dof)), 20.0 + 30.0 * rng.rand(dof)), axis=1)


def _grid(rng, x0, x1, G):
    if G == 1:
        return np.array([x0 + (0.2 + 0.6 * rng.rand()) * (x1 - x0)])
    return np.r_[x0, np.sort(rng.uniform(x0, x1, G - 2)), x1]


def make_problem(model, interp, dof, G, breaks_shared, grid_shared, lim_shared, friction, inner, seed, B=3):
    """B = 3 paths on non-uniform knots over [0.5, 2]: path 0 ordinary, path 1 with |q| up to ~100 (range reduction of
    sin / cos), path 2 with joint 0 frozen (constant waypoints: q' = q'' = 0 exactly)."""
    rng = np.random.RandomState(seed)
    nway, x0, x1 = 6, 0.5, 2.0
    breaks = np.empty((B, nway))
    ppoly = np.empty((B, 4, nway - 1, dof))
    for b in range(B):
        if b == 0 or not breaks_shared:
            d = np.cumsum(np.r_[0.0, 0.2 + rng.rand(nway - 1)])
            x = x0 + (x1 - x0) * d / d[-1]
            x[-1] = x1
        breaks[b] = x
        way = 1.5 * rng.randn(nway, dof)
        if b == 1:
            way = 25.0 * way + 60.0
        if b == 2:
            way[:, 0] = way[0, 0]
        ppoly[b] = orc.cubic_spline_fit(x, way)
    grid = _grid(rng, x0, x1, G) if grid_shared else np.stack([_grid(rng, x0, x1, G) for _ in range(B)])
    taulim = _asym_limits(rng, dof) if lim_shared else np.stack([_asym_limits(rng, dof) for _ in range(B)])
    nrows = (4 if interp else 2) * dof
    row0, R_total = (3, nrows + 5) if inner else (0, nrows)          # inner: odd R, one padding slot
    return dict(model=model, params=_model_params(model, dof, rng), interp=interp, ppoly=ppoly,
                breaks=breaks[0] if breaks_shared else breaks, grid=grid, taulim=taulim,
                friction=(0.3 + 2.0 * rng.rand(dof)) if friction else None, row0=row0, R_total=R_total, nrows=nrows)


def _per(arr, b, ndim):
    return arr if arr.ndim == ndim else arr[b]


def path_inputs(pr, b):
    """(q, q', q'', grid, taulim) of path b, the derivatives from the oracle's PPoly evaluation."""
    grid = _per(pr["grid"], b, 1)
    qs = [orc.ppoly_eval(pr["ppoly"][b], _per(pr["breaks"], b, 1), grid, o) for o in (0, 1, 2)]
    return qs + [grid, _per(pr["taulim"], b, 2)]


def problem_reference(pr):
    refs = []
    for b in range(pr["ppoly"].shape[0]):
        q, qd, qdd, grid, tl = path_inputs(pr, b)
        refs.append(torque_rows_reference(pr["model"], pr["params"], q, qd, qdd, grid, tl, pr["friction"], pr["interp"]))
    return refs


@functools.lru_cache(maxsize=None)
def case_data(case):
    """[(problem, reference rows per path)] of the three launches of `case` (computed once, shared by every engine)."""
    out = []
    for ln in _launches(case):
        pr = make_problem(case[0], case[1], case[2], **ln)
        out.append((pr, problem_reference(pr)))
    return out


def sentinel_records(B, G, W):
    return np.full((B, G, W), SENTINEL, dtype=np.int64).view(np.float64)


def sentinel_tensor(shape, dev):
    import torch
    return torch.full(shape, int(SENTINEL), dtype=torch.int64, device=dev).view(torch.float64)


def _tensor(x, dev):
    import torch
    return None if x is None else torch.as_tensor(np.ascontiguousarray(x), dtype=torch.float64, device=dev)


def launch_second_order(ta, pr, on_device=False):
    """engine.coeff_second_order on problem `pr` into sentinel-filled records; returns the records (numpy, or the device
    tensor with on_device=True)."""
    dev = ta.engine.default_device()
    B, G = pr["ppoly"].shape[0], pr["grid"].shape[-1]
    rec = sentinel_tensor((B, G, ta.engine.record_doubles(pr["R_total"])), dev)
    n = ta.engine.coeff_second_order(pr["model"], pr["params"], *(_tensor(pr[key], dev) for key in ("ppoly", "breaks", "grid")),
                                     _tensor(pr["taulim"], dev), _tensor(pr["friction"], dev), pr["interp"], rec,
                                     pr["R_total"], pr["row0"])
    assert n == pr["nrows"]
    return rec if on_device else rec.cpu().numpy()


def test_problem_set_has_the_edges_it_claims():
    """Every (model, scheme) meets every G and dof, both values of every flag; q' takes both signs and is exactly 0 on the
    frozen joint."""
    for model in MODELS:
        for interp in (1, 0):
            lns = [ln for dof in DOFS for ln in _launches((model, interp, dof))]
            assert sorted(set(ln["G"] for ln in lns)) == sorted(GS)
            for flag in ("breaks_shared", "grid_shared", "lim_shared", "friction", "inner"):
                assert set(ln[flag] for ln in lns) == {True, False}, (model, interp, flag)
    pr = make_problem("coupled_cosine", 1, 6, 33, False, False, False, True, True, 7)
    q, qd, qdd, _, _ = path_inputs(pr, 2)
    assert np.all(qd[:, 0] == 0) and np.all(qdd[:, 0] == 0)
    assert (qd[:, 1:] > 0).any() and (qd[:, 1:] < 0).any()
    assert np.abs(path_inputs(pr, 1)[0]).max() > 50
    assert np.all(pr["taulim"][..., 0] != -pr["taulim"][..., 1])


# ---- 1. the reference, anchored on the rows that reproduce the upstream golden ----------------------------------------
def numpy_callback_torque_rows(ss, way, taulim, grid):
    """Torque rows as the reference builds them from a numpy inv_dyn (3 calls per gridpoint, canlinear_colloc_to_interpolate,
    F = [I; -I], g = [tau_max; -tau_min]); with the oracle's vel + acc rows they reproduce tests/golden/torque_dof6_g500
    bit for bit (checked below)."""
    from problems import inv_dyn_numpy
    from toppra_b200.constraint.linear_constraint import canlinear_colloc_to_interpolate
    c = orc.cubic_spline_fit(ss, way)
    q, qd, qdd = (orc.ppoly_eval(c, ss, grid, o) for o in (0, 1, 2))
    zero = np.zeros(q.shape[1])
    cv = np.array([inv_dyn_numpy(p, zero, zero) for p in q])
    av = np.array([inv_dyn_numpy(p, zero, ps) for p, ps in zip(q, qd)]) - cv
    bv = np.array([inv_dyn_numpy(p, ps, pss) for p, ps, pss in zip(q, qd, qdd)]) - cv
    dof = q.shape[1]
    F = np.vstack((np.eye(dof), -np.eye(dof)))
    g = np.concatenate((taulim[:, 1], -taulim[:, 0]))
    a2, b2, c2, F2, g2, _, _ = canlinear_colloc_to_interpolate(av, bv, cv, F, g, None, None, grid, identical=True)
    return np.stack((a2.dot(F2.T), b2.dot(F2.T), c2.dot(F2.T) - g2), axis=1), c, (q, qd, qdd)


def test_reference_anchored_on_upstream_golden_rows(golden):
    g = golden("torque_dof6_g500")
    params = _model_params("coupled_cosine", 6, None, standard=True)
    worst = 0.0
    for b in range(2):
        rows, c, (q, qd, qdd) = numpy_callback_torque_rows(g["ss"], g["way"][b], g["taulim"][b], g["grid"])
        lin = orc.solve_velacc(c, g["ss"], g["grid"], g["vlim"][b], g["alim"][b], True, 0, 0, want_rows=True)
        o = orc.solve_rows(np.concatenate((lin["rows"], rows), axis=2), lin["xbound"], g["grid"], 0.0, 0.0)
        assert o["status"] == g["status"][b] == 0
        assert np.array_equal(o["K"], g["K"][b]) and np.array_equal(o["sd"], g["sd"][b])
        ref = torque_rows_reference("coupled_cosine", params, q, qd, qdd, g["grid"], g["taulim"][b], None, 1)
        nbad, ratio = compare_rows(rows, ref)
        assert nbad == 0, (b, ratio)
        worst = max(worst, ratio)
    print("numpy-callback rows of the upstream golden vs the mpmath reference: worst %.3f eps S" % worst)


# ---- 2. tb_coeff_second_order: shapes, edges, untouched slots ---------------------------------------------------------
@pytest.mark.parametrize("case", CASES, ids=["%s-%s-dof%d" % (m, "interp" if i else "colloc", d) for m, i, d in CASES])
def test_second_order_rows_match_mpmath_reference(ta, case):
    worst = 0.0
    for pr, refs in case_data(case):
        rec = launch_second_order(ta, pr)
        problems, ratio = check_records(rec, refs, pr["R_total"], pr["row0"], pr["nrows"])
        assert not problems, (pr["grid"].shape, pr["row0"], pr["R_total"], problems)
        worst = max(worst, ratio)
    _note(_engine_name(ta), case[0], worst)


@pytest.mark.gpu
def test_second_order_rows_beyond_65535_ctas():
    """B = 4096 paths x 16 tiles of G = 500: 65 536 CTAs in one launch (cfg 3 shape: coupled_cosine, 6 DOF, Interpolation).
    Sampled paths (the first, the middle, the last CTA's) match the reference and equal a launch of that path alone."""
    import torch
    import toppra_b200 as ta
    B, G, dof = 4096, 500, 6
    rng = np.random.RandomState(42)
    ss = np.r_[0.0, np.cumsum(0.2 + rng.rand(4))]
    ss /= ss[-1]
    way = rng.randn(B, 5, dof)
    pr = dict(model="coupled_cosine", params=_model_params("coupled_cosine", dof, rng, standard=True), interp=1,
              ppoly=np.stack([orc.cubic_spline_fit(ss, w) for w in way]), breaks=ss, grid=_grid(rng, 0.0, 1.0, G),
              taulim=np.stack([_asym_limits(rng, dof) for _ in range(B)]), friction=0.3 + 2.0 * rng.rand(dof),
              row0=0, R_total=4 * dof, nrows=4 * dof)
    big = launch_second_order(ta, pr, on_device=True)
    R = pr["R_total"]
    assert bool((big[:, :, 3 * R:].view(torch.int64) == int(SENTINEL)).all())     # x bound slots untouched
    for p in (0, 1, B // 2, B - 2, B - 1):
        rec = big[p:p + 1].cpu().numpy()
        one = dict(pr, ppoly=pr["ppoly"][p:p + 1], taulim=pr["taulim"][p:p + 1])
        alone = launch_second_order(ta, one)
        assert np.array_equal(alone.view(np.int64), rec.view(np.int64)), p
        problems, ratio = check_records(rec, problem_reference(one), R, 0, pr["nrows"])
        assert not problems, (p, problems)
        _note("gpu", "coupled_cosine", ratio)


TB_ERR_ARG, TB_ERR_UNSUPPORTED = -1, -2


@pytest.mark.parametrize("where", [pytest.param("gpu", marks=pytest.mark.gpu), "host"])
def test_second_order_rejects_bad_arguments(where):
    """tb_coeff_second_order validates on the host and returns before any launch: dof above SO_MAX_DOF, a parameter count
    that does not match the model, an unknown model, rows that do not fit R_total or W.  On the GPU the record buffer is
    checked to be untouched and the same arguments with the bad one corrected do run."""
    from toppra_b200 import _lib
    import torch
    if where == "host" and torch.cuda.is_available():
        pytest.skip("host addresses stand in for device arrays: run without a GPU")
    lib = _lib.load()
    n = 1 << 12
    # params, ppoly, breaks [0, 1, 2], grid [0, 0.5], taulim, friction: large enough for every call below
    host = [np.zeros(n), np.zeros(n), np.arange(n, dtype=np.float64), 0.5 * np.arange(n), np.zeros(n), np.zeros(n),
            sentinel_records(1, 1, n).reshape(-1)]
    if where == "gpu":
        keep = [torch.from_numpy(a).cuda() for a in host]
        ptrs = [_lib.ptr(t) for t in keep]
        rec = keep[-1]
    else:
        keep = host
        ptrs = [ctypes.c_void_p(a.ctypes.data) for a in keep]
    prm, pp, br, gr, tl, fr, rc_ = ptrs

    def call(model=1, nparams=32, dof=16, interp=1, W=3 * 64 + 2, R_total=64, row0=0):
        rc = lib.tb_coeff_second_order(model, prm, nparams, pp, br, 1, 1, 2, dof, gr, 1, 2, tl, 1, fr, interp, rc_, W,
                                       R_total, row0, None)
        return rc, (lib.tb_last_error() or b"").decode()

    rc, msg = call(dof=17, nparams=34, W=3 * 68 + 2, R_total=68)
    assert rc == TB_ERR_UNSUPPORTED and "dof=17" in msg
    for model, nparams in ((1, 31), (1, 33), (1, 4), (0, 3), (0, 5), (0, 32)):
        rc, msg = call(model=model, nparams=nparams)
        assert rc == TB_ERR_ARG and "parameters" in msg, (model, nparams)
    for model in (2, -1):
        rc, msg = call(model=model)
        assert rc == TB_ERR_UNSUPPORTED and "unknown device model" in msg
    for kw in (dict(R_total=63, W=3 * 63 + 2), dict(row0=1), dict(row0=-1, R_total=65, W=3 * 65 + 3), dict(W=3 * 64 + 1),
               dict(interp=0, R_total=31, W=3 * 31 + 3)):
        rc, msg = call(**kw)
        assert rc == TB_ERR_ARG and "do not fit" in msg, kw
    if where == "gpu":
        torch.cuda.synchronize()
        assert bool((rec.view(torch.int64) == int(SENTINEL)).all())
        assert call()[0] == 0 and call(model=0, nparams=4, dof=1, R_total=4, W=14)[0] == 0
        torch.cuda.synchronize()
        assert not bool((rec.view(torch.int64) == int(SENTINEL)).all())


# ---- 3. end to end through BatchTOPPRA, no tolerance ---------------------------------------------------------------------
def _same(a, b):
    """array_equal with NaN == NaN."""
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and bool(np.all((a == b) | (np.isnan(a) & np.isnan(b))))


@pytest.mark.parametrize("torque_first", [True, False], ids=["torque-rows-first", "torque-rows-last"])
def test_device_model_records_reproduce_scan_and_chunks(ta, torque_first):
    """[torque, vel, acc] (vel + acc rows at row0 = 24) and [vel, acc, torque] with a device model, asymmetric per-path
    torque limits and friction, record scan.  The records' torque rows match the reference; oracle.solve_rows on the
    records reproduces K, sd, u and status of the scan bit for bit; 11 paths in chunks of 4, 4, 3 (each chunk slices the
    per-path limits) equal the single launch bit for bit."""
    B, G, dof = 11, 101, 6
    rng = np.random.RandomState(31 if torque_first else 32)
    ss = np.r_[0.0, np.cumsum(0.2 + rng.rand(4))]
    ss /= ss[-1]
    way = rng.randn(B, 5, dof)
    way[3, :, 2] = way[3, 0, 2]                                           # one frozen joint
    vlim = np.stack((-(10 + 20 * rng.rand(B, dof)), 10 + 20 * rng.rand(B, dof)), axis=-1)
    alim = np.stack((-(10 + 2 * rng.rand(B, dof)), 10 + 2 * rng.rand(B, dof)), axis=-1)
    taulim = np.stack((-(18 + 15 * rng.rand(B, dof)), 22 + 15 * rng.rand(B, dof)), axis=-1)
    fric = 0.5 + 1.5 * rng.rand(dof)
    params = _model_params("coupled_cosine", dof, rng, standard=True)
    grid = _grid(rng, 0.0, 1.0, G) if torque_first else np.stack([_grid(rng, 0.0, 1.0, G) for _ in range(B)])
    path = ta.BatchSplineInterpolator(ss, way)

    def cons(torque=True):
        c = [ta.constraint.JointVelocityConstraint(vlim), ta.constraint.JointAccelerationConstraint(alim)]
        if torque:
            tq = ta.constraint.SecondOrderConstraint.joint_torque_constraint(None, taulim, fric,
                                                                             device_model=("coupled_cosine", params))
            c = [tq] + c if torque_first else c + [tq]
        return c

    inst = ta.BatchTOPPRA(cons(), path, grid, fused=False)
    assert inst.R == 48 and not inst.fused and inst.chunk_size() == B
    h = inst.compute_parameterization(0.0, 0.0).to_host()
    rec = inst.records.cpu().numpy()
    W, R = rec.shape[-1], inst.R
    t0 = 0 if torque_first else 4 * dof
    ppoly = path.d_ppoly.cpu().numpy()
    for b in range(B):
        g_b = grid if grid.ndim == 1 else grid[b]
        q, qd, qdd = (orc.ppoly_eval(ppoly[b], ss, g_b, o) for o in (0, 1, 2))
        ref = torque_rows_reference("coupled_cosine", params, q, qd, qdd, g_b, taulim[b], fric, 1)
        got = np.stack([rec[b, :, p * R + t0:p * R + t0 + 4 * dof] for p in range(3)], axis=1)
        nbad, ratio = compare_rows(got, ref)
        assert nbad == 0, (b, ratio)
        _note(_engine_name(ta), "coupled_cosine", ratio)
        rows = np.stack([rec[b, :, p * R:(p + 1) * R] for p in range(3)], axis=1)
        o = orc.solve_rows(rows, rec[b, :, 3 * R:3 * R + 2], g_b, 0.0, 0.0)
        assert h["status"][b] == o["status"], b
        assert _same(h["K"][b], o["K"]), b
        if o["status"] != 3:
            assert _same(h["sd"][b], o["sd"]) and _same(h["sdd"][b], o["u"]), b
    assert (h["status"] == 0).sum() >= B - 2
    # the torque rows are active: without them most paths get another parameterisation
    plain = ta.BatchTOPPRA(cons(torque=False), path, grid).compute_parameterization(0.0, 0.0).to_host()
    assert sum(not _same(plain["sd"][b], h["sd"][b]) for b in range(B)) >= B - 2
    # chunks 4 + 4 + 3: every chunk slices the per-path torque limits (and per-path grid) of its own paths
    per_path = 8 * W * G
    chunked = ta.BatchTOPPRA(cons(), path, grid, fused=False, max_record_bytes=4 * per_path)
    assert chunked.chunk_size() == 4
    hc = chunked.compute_parameterization(0.0, 0.0).to_host()
    for key in ("K", "sd", "sdd", "status", "fail_stage"):
        assert _same(hc[key], h[key]), key


# ---- 4. tb_rows_canlinear records, bit for bit ------------------------------------------------------------------------
def canlinear_rows_numpy(a, b, c, F, g, F_mode, grid, interp):
    """Rows [B, G, 3, nrows] of the generic row assembly: acc = acc + F[j, q] * a[q] for q = 0..m-1 (left to right), the
    lifted block reading a, b, c, F, g at s_{i+1} with a + 2 delta_i b; the last gridpoint duplicates itself."""
    B, G, m = a.shape
    k = 2 * m if F_mode >= 2 else (F.shape[0] if F_mode == 0 else F.shape[2])
    grid = np.broadcast_to(grid, (B, G))
    idx = np.arange(G)
    src = np.minimum(idx + 1, G - 1)
    two_delta = 2 * (grid[:, src] - grid)
    out = []
    for second in ((0, 1) if interp else (0,)):
        s = src if second else idx
        lift = (idx < G - 1) if second else np.zeros(G, dtype=bool)
        av = np.where(lift[None, :, None], a[:, s] + two_delta[:, :, None] * b[:, s], a[:, s])
        bv, cv = b[:, s], c[:, s]
        if F_mode >= 2:
            sgn = np.r_[np.ones(m), -np.ones(m)]
            col = np.r_[np.arange(m), np.arange(m)]
            ta_, tb_, tc_ = sgn * av[..., col], sgn * bv[..., col], sgn * cv[..., col]
            gv = np.broadcast_to(g if F_mode == 2 else g[:, None, :], (B, G, k))
        else:
            Fr = np.broadcast_to(F, (B, G, k, m)) if F_mode == 0 else F[:, s]
            ta_ = tb_ = tc_ = np.zeros((B, G, k))
            for q in range(m):
                ta_ = ta_ + Fr[..., q] * av[:, :, None, q]
                tb_ = tb_ + Fr[..., q] * bv[:, :, None, q]
                tc_ = tc_ + Fr[..., q] * cv[:, :, None, q]
            gv = np.broadcast_to(g, (B, G, k)) if F_mode == 0 else g[:, s]
        out.append(np.stack((ta_, tb_, tc_ - gv), axis=2))
    return np.concatenate(out, axis=3)


@pytest.mark.parametrize("F_mode", [0, 1, 2, 3])
def test_rows_canlinear_records_bit_exact(ta, F_mode):
    dev = ta.engine.default_device()
    B, m = 3, 3
    k = 2 * m if F_mode >= 2 else 5
    rng = np.random.RandomState(70 + F_mode)
    d = lambda x: _tensor(x, dev)  # noqa: E731
    n = 0
    for interp in (1, 0):
        for G in (1, 2, 33):
            n += 1
            a, b, c = (rng.randn(B, G, m) * 10 ** rng.uniform(-2, 2) for _ in range(3))
            F = {0: rng.randn(k, m), 1: rng.randn(B, G, k, m)}.get(F_mode)
            gsh = {0: (k,), 1: (B, G, k), 2: (k,), 3: (B, k)}[F_mode]
            g = 5 + 20 * rng.rand(*gsh)                                    # asymmetric: tau_max-like | -tau_min-like
            grid = _grid(rng, 0.0, 1.0, G) if n % 2 else np.stack([_grid(rng, 0.0, 1.0, G) for _ in range(B)])
            nrows = (2 if interp else 1) * k
            row0, R_total = (2, nrows + 3) if n % 3 else (0, nrows)
            W = ta.engine.record_doubles(R_total)
            rec = sentinel_tensor((B, G, W), dev)
            assert ta.engine.rows_canlinear(d(a), d(b), d(c), d(F), d(g), F_mode, d(grid), interp, rec, R_total, row0) == nrows
            got = rec.cpu().numpy()
            want = canlinear_rows_numpy(a, b, c, F, g, F_mode, grid, interp)
            for part in range(3):
                blk = got[:, :, part * R_total + row0:part * R_total + row0 + nrows]
                assert np.array_equal(blk.view(np.int64), np.ascontiguousarray(want[:, :, part]).view(np.int64)), \
                    (interp, G, part)
            own = np.zeros(W, dtype=bool)
            for part in range(3):
                own[part * R_total + row0:part * R_total + row0 + nrows] = True
            assert np.all(got.view(np.int64)[:, :, ~own] == SENTINEL), (interp, G)


# ---- 5. the comparison notices the bugs it is there for ---------------------------------------------------------------
def kernel_model_records(pr, bug=None):
    """float64 numpy model of second_order_rows_tiled_kernel (its summation order, the expanded cos(q_i - q_j)) writing
    records [B, G, W] with a sentinel elsewhere; `bug` injects one mistake."""
    B, G = pr["ppoly"].shape[0], pr["grid"].shape[-1]
    R, row0, nrows = pr["R_total"], pr["row0"], pr["nrows"]
    W = cpu_engine.record_doubles(R)
    rec = sentinel_records(B, G, W)
    for p in range(B):
        q, qd, qdd, grid, tl = path_inputs(pr, p)
        sq, cq = np.sin(q), np.cos(q)
        prm = pr["params"]
        if pr["model"] == "coupled_cosine":
            m0, m1, h, gr = prm
            cs1 = ss1 = cs2 = ss2 = v2 = np.zeros((G, 1))
            for j in range(q.shape[1]):
                cs1, ss1 = cs1 + cq[:, j:j + 1] * qd[:, j:j + 1], ss1 + sq[:, j:j + 1] * qd[:, j:j + 1]
                cs2, ss2 = cs2 + cq[:, j:j + 1] * qdd[:, j:j + 1], ss2 + sq[:, j:j + 1] * qdd[:, j:j + 1]
                v2 = v2 + qd[:, j:j + 1] * qd[:, j:j + 1]
            cv = gr * sq
            if bug == "coupling_dropped":
                av, bv = m0 * qd, m0 * qdd + h * sq * v2
            else:
                av = m0 * qd + m1 * (cq * cs1 + sq * ss1)
                bv = m0 * qdd + m1 * (cq * cs2 + sq * ss2) + h * sq * v2
        else:
            cv, av, bv = prm[1::2] * sq, prm[0::2] * qd, prm[0::2] * qdd
        if pr["friction"] is not None:
            sg = np.sign(qd) * (-1.0 if bug == "friction_sign" else 1.0)
            cv = cv + sg * pr["friction"]
        tmin, tmax = (tl[:, 1], tl[:, 0]) if bug == "tau_swapped" else (tl[:, 0], tl[:, 1])
        src = np.minimum(np.arange(G) + 1, G - 1)
        lift_src = np.arange(G) if bug == "lift_reads_i" else src
        aplus = av[lift_src] + (2 * (grid[src] - grid))[:, None] * bv[lift_src]
        aplus[G - 1] = av[G - 1]
        rows = _assemble(av, bv, cv - tmax, cv - tmin, aplus, pr["interp"])
        r0 = row0 + 1 if bug == "row0_off_by_one" else row0
        for part in range(3):
            rec[p, :, part * R + r0:part * R + r0 + nrows] = rows[:, part]
        if bug == "tile_edge_record" and G > 31:
            rec[p, 31] = rec[p, 30]
    return rec


BUGS = ("lift_reads_i", "tau_swapped", "friction_sign", "coupling_dropped", "row0_off_by_one", "tile_edge_record")


def _bug_applies(bug, pr):
    G = pr["grid"].shape[-1]
    return {"lift_reads_i": pr["interp"] and G >= 2, "friction_sign": pr["friction"] is not None,
            "coupling_dropped": pr["model"] == "coupled_cosine", "tile_edge_record": G > 31}.get(bug, True)


def test_float64_kernel_model_within_bound():
    """The kernel's own float64 arithmetic (numpy, its summation order) passes the comparison on every launch of the
    problem set: the bound is not tighter than what correct fp64 code can meet."""
    for case in CASES:
        for pr, refs in case_data(case):
            problems, ratio = check_records(kernel_model_records(pr), refs, pr["R_total"], pr["row0"], pr["nrows"])
            assert not problems, (case, problems)
            _note("numpy float64 model", case[0], ratio)


@pytest.mark.parametrize("bug", BUGS)
def test_comparison_detects_corrupted_records(bug):
    applicable = 0
    for case in CASES:
        for pr, refs in case_data(case):
            if not _bug_applies(bug, pr):
                continue
            applicable += 1
            problems, _ = check_records(kernel_model_records(pr, bug), refs, pr["R_total"], pr["row0"], pr["nrows"])
            assert problems, (bug, case, pr["grid"].shape)
    assert applicable >= 10
