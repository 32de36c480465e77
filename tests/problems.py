"""Seeded synthetic TOPP-RA problems shared by tests, bench.py and smoke() (SURVEY.md §8d).

Generation order per path follows the reference example examples/plot_kinematics.py:22-33:
way_pts = randn(n, dof); vlims = 10 + rand(dof)*20; alims = 10 + rand(dof)*2; ss = linspace(0,1,n)."""
import numpy as np


def make_path(seed, dof=7, nway=5, vel_active=False):
    rng = np.random.RandomState(seed)
    way = rng.randn(nway, dof)
    vl = (0.5 + rng.rand(dof)) if vel_active else (10 + rng.rand(dof) * 20)
    al = 10 + rng.rand(dof) * 2
    vlim = np.vstack((-vl, vl)).T
    alim = np.vstack((-al, al)).T
    return way, vlim, alim


def make_batch(B, seed0=1000, dof=7, nway=5, vel_active=False):
    """B paths with seeds seed0+b.  Returns ss [n], way [B,n,dof], vlim [B,dof,2], alim [B,dof,2]."""
    way = np.empty((B, nway, dof))
    vlim = np.empty((B, dof, 2))
    alim = np.empty((B, dof, 2))
    for b in range(B):
        way[b], vlim[b], alim[b] = make_path(seed0 + b, dof, nway, vel_active)
    return np.linspace(0, 1, nway), way, vlim, alim


def make_batch_fast(B, seed=1234, dof=7, nway=5):
    """Large batches for the bench: one RandomState for the whole batch (same distributions)."""
    rng = np.random.RandomState(seed)
    way = rng.randn(B, nway, dof)
    vl = 10 + rng.rand(B, dof) * 20
    al = 10 + rng.rand(B, dof) * 2
    vlim = np.stack((-vl, vl), axis=-1)
    alim = np.stack((-al, al), axis=-1)
    return np.linspace(0, 1, nway), way, vlim, alim


# ---- cfg 3: synthetic closed-form torque model (SURVEY.md §8d):
#      tau = M(q) qdd + h(q) |qd|^2 + g(q),  M = 2 I + 0.3 cos(q_i - q_j),  h = 0.1 sin q,  g = 4.9 sin q
def inv_dyn_numpy(q, qd, qdd):
    q, qd, qdd = np.asarray(q), np.asarray(qd), np.asarray(qdd)
    M = 2.0 * np.eye(len(q)) + 0.3 * np.cos(q[:, None] - q[None, :])
    return M.dot(qdd) + 0.1 * np.sin(q) * np.dot(qd, qd) + 4.9 * np.sin(q)


def inv_dyn_torch(q, qd, qdd):
    """Batched form on tensors [M, dof] (same formula).  M(q) qdd is evaluated without materialising the [M, dof, dof]
    matrices: sum_j cos(q_i - q_j) qdd_j = cos q_i * sum_j cos q_j qdd_j + sin q_i * sum_j sin q_j qdd_j."""
    import torch
    cq, sq = torch.cos(q), torch.sin(q)
    mq = 2.0 * qdd + 0.3 * (cq * (cq * qdd).sum(-1, keepdim=True) + sq * (sq * qdd).sum(-1, keepdim=True))
    return mq + 0.1 * sq * (qd * qd).sum(-1, keepdim=True) + 4.9 * sq


def make_torque_problem(seed, dof=6, nway=5):
    rng = np.random.RandomState(seed)
    way = rng.randn(nway, dof)
    vl = 10 + rng.rand(dof) * 20
    al = 10 + rng.rand(dof) * 2
    tl = 40 + rng.rand(dof) * 10
    return way, np.vstack((-vl, vl)).T, np.vstack((-al, al)).T, np.vstack((-tl, tl)).T


# ---- raw stage rows that stress the Seidel shortcuts of the scan kernel (VERDICT r1 #4): near-duplicate, scaled,
#      parallel and slightly rotated copies of random rows (perturbations 1e-14 .. 1e-6), and badly scaled rows
def degenerate_rows_batch(R0, G, B, seed):
    """B problems of 2*R0 rows, G gridpoints: rows [B, G, 3, 2*R0], xbound [B, G, 2]."""
    rng = np.random.RandomState(seed)
    R = 2 * R0
    rows = np.empty((B, G, 3, R))
    xb = np.empty((B, G, 2))
    for i in range(B):
        a = rng.randn(G, R0)
        b = rng.randn(G, R0)
        c = -rng.rand(G, R0) * 10 ** rng.uniform(-1, 1)
        eps = 10 ** rng.uniform(-14, -6)
        kind = i % 4
        if kind == 0:
            a2, b2, c2 = a * (1 + eps * rng.randn(G, R0)), b * (1 + eps * rng.randn(G, R0)), c * (1 + eps * rng.randn(G, R0))
        elif kind == 1:
            sc = 10 ** rng.uniform(-3, 3, size=(G, R0))
            a2, b2, c2 = a * sc, b * sc, c * sc + eps * rng.randn(G, R0)
        elif kind == 2:
            a2, b2, c2 = a.copy(), b.copy(), c + eps * rng.randn(G, R0)
        else:
            a2, b2, c2 = a + eps * rng.randn(G, R0), b.copy(), c.copy()
        perm = rng.permutation(R)
        rows[i, :, 0] = np.concatenate((a, a2), 1)[:, perm]
        rows[i, :, 1] = np.concatenate((b, b2), 1)[:, perm]
        rows[i, :, 2] = np.concatenate((c, c2), 1)[:, perm]
        xb[i, :, 0] = 0.0
        xb[i, :, 1] = 10 ** rng.uniform(-2, 3)
    return rows, xb


def badly_scaled_rows_batch(R, G, B, seed):
    """Coefficients down to 1e-8 (rows look 'parallel' to the 1e-10 test of pyx:339-345), optima up to the +-1e10
    sentinel of the 1-D LP (pyx:376-383); a third of the problems vary smoothly along the path (warm starts stay valid)."""
    rng = np.random.RandomState(seed)
    rows = np.empty((B, G, 3, R))
    xb = np.empty((B, G, 2))
    for it in range(B):
        sa, sb, sc = 10 ** rng.uniform(-8, 1), 10 ** rng.uniform(-8, 1), 10 ** rng.uniform(-3, 5)
        if it % 3 == 0:
            a = np.cumsum(rng.randn(G, R) * 0.05, 0) * sa + rng.randn(1, R) * sa
            b = np.cumsum(rng.randn(G, R) * 0.05, 0) * sb + rng.randn(1, R) * sb
        else:
            a, b = rng.randn(G, R) * sa, rng.randn(G, R) * sb
        rows[it, :, 0], rows[it, :, 1], rows[it, :, 2] = a, b, -rng.rand(G, R) * sc
        xb[it, :, 0] = 0.0
        xb[it, :, 1] = 1e8 if it % 2 else 10 ** rng.uniform(-2, 9)
    return rows, xb


SHORTCUT_SETS = {  # name -> (generator, args): the problems of tests/golden/shortcut_rows_<name>.npz
    "deg6": (degenerate_rows_batch, (6, 24, 1500, 105)),
    "deg20": (degenerate_rows_batch, (20, 16, 1500, 119)),
    "scaled14": (badly_scaled_rows_batch, (14, 20, 1200, 6)),
}


def random_shaped_problem(rng):
    """One randomly SHAPED vel+acc problem (used by scripts/fuzz_oracle_vs_reference.py and the GPU shape campaign): dof
    1..14, 2..12 knots on uniform or non-uniform breakpoints, 2..400 gridpoints (uniform, random, some on breakpoints), any
    boundary condition, both discretisations, symmetric or asymmetric limits, active velocity bounds, tiny motions, a
    motionless joint now and then, zero / small / inadmissible boundary velocities."""
    dof = int(rng.choice([1, 2, 3, 6, 7, 7, 7, 10, 14]))
    n = int(rng.randint(2, 13))
    ss = np.r_[0.0, np.cumsum(0.05 + rng.rand(n - 1))]
    if rng.rand() < 0.5:
        ss = np.linspace(0, ss[-1], n)
    scale = 10 ** rng.uniform(-3, 1) if rng.rand() < 0.25 else 1.0          # tiny motions now and then
    way = rng.randn(n, dof) * scale
    if rng.rand() < 0.1:
        way[:, rng.randint(dof)] = way[0, 0]                                 # a joint that does not move
    vl = (0.5 + rng.rand(dof)) * scale if rng.rand() < 0.4 else 10 + 20 * rng.rand(dof)
    al = (10 + 2 * rng.rand(dof)) * (scale if rng.rand() < 0.5 else 1.0)
    if rng.rand() < 0.3:                                                     # asymmetric limits
        vlim = np.stack((-vl * (0.3 + rng.rand(dof)), vl), axis=1)
        alim = np.stack((-al, al * (0.3 + rng.rand(dof))), axis=1)
    else:
        vlim, alim = np.stack((-vl, vl), axis=1), np.stack((-al, al), axis=1)
    G = int(rng.choice([2, 3, 5, 17, 50, 100, 200, 400]))
    grid = np.linspace(0, ss[-1], G)
    if G > 3 and rng.rand() < 0.4:
        grid = np.r_[0.0, np.sort(rng.uniform(0, ss[-1], G - 2)), ss[-1]]
        if np.any(np.diff(grid) <= 0):
            grid = np.linspace(0, ss[-1], G)
    if G > n and rng.rand() < 0.2:                                           # gridpoints exactly on breakpoints
        k = rng.randint(1, G - 1, size=min(n - 2, 3)) if n > 2 else []
        for j, idx in enumerate(np.unique(k)):
            cand = ss[1 + j % max(n - 2, 1)]
            if grid[idx - 1] < cand < grid[idx + 1]:
                grid[idx] = cand
    bc = rng.choice(["not-a-knot", "clamped", "natural"]) if n > 2 else "not-a-knot"
    interp_scheme = int(rng.rand() < 0.7)
    r = rng.rand()
    sd0 = 0.0 if r < 0.6 else (10 ** rng.uniform(-3, 0) if r < 0.9 else 50.0)
    sd1 = 0.0 if rng.rand() < 0.6 else 10 ** rng.uniform(-3, 0)
    # the reference squares the boundary velocities with libm pow(x, 2.0), which is not always correctly rounded
    # (DESIGN.md section 2); keep to velocities where it is, so that everything else is compared bit for bit
    while float(sd0) ** 2 != float(sd0) * float(sd0):
        sd0 = float(np.nextafter(sd0, 1.0))
    while float(sd1) ** 2 != float(sd1) * float(sd1):
        sd1 = float(np.nextafter(sd1, 1.0))
    return dict(ss=ss, way=way, vlim=vlim, alim=alim, grid=grid, bc=str(bc), interp=interp_scheme, sd0=sd0, sd1=sd1)
