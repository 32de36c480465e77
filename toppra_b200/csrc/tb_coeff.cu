// tb_coeff.cu — K1: constraint coefficients -> stage records, one coalesced pass over batch x gridpoint.
//
// Replaces (reference):
//   path(gridpoints, 1), path(gridpoints, 2)                       toppra/interpolator.py:423-430 (scipy PPoly)
//   JointVelocityConstraint.compute_constraint_params             toppra/constraint/linear_joint_velocity.py:43-53
//   _create_velocity_constraint (fp32 accumulators!)              toppra/_CythonUtils.pyx:16-59
//   JointAccelerationConstraint.compute_constraint_params         toppra/constraint/linear_joint_acceleration.py:63-104
//   canlinear_colloc_to_interpolate                               toppra/constraint/linear_constraint.py:84-192
//   seidelWrapper.__init__ row assembly (F.a, F.b, F.c - g)        toppra/solverwrapper/cy_seidel_solverwrapper.pyx:474-520
//
// Bound: HBM write bandwidth (3R+2 doubles per path and gridpoint; the PPoly input is 4*nseg*dof doubles
// per path).  One CTA per (path, chunk of CH gridpoints): q', q'' of the chunk (+1 gridpoint for the
// interpolation lift) are evaluated once into shared memory, then every thread writes consecutive doubles of
// the record stream, so the stores are fully coalesced.
#include "tb_common.cuh"

namespace tb {
namespace {

#ifndef TB_COEFF_THREADS
#define TB_COEFF_THREADS 128
#endif
#ifndef TB_COEFF_CH
#define TB_COEFF_CH 32
#endif
constexpr int COEFF_THREADS = TB_COEFF_THREADS;
constexpr int COEFF_CH_SMALL = 32, COEFF_CH_LARGE = TB_COEFF_CH;  // gridpoints per CTA

__device__ __forceinline__ int R_total_or1(int R_total) { return R_total > 0 ? R_total : 1; }

// Shared-memory plan of one CTA (dof = d, VS = 6d + 3 doubles per gridpoint, CH gridpoints per CTA):
//   dco  [nseg][d][5]   derivative coefficients of the path's PPoly: q' = (3c0, 2c1, c2), q'' = (6c0, 2c1)
//   raw  [(CH+1)][2d]   q'(s_i), q''(s_i) of the chunk (+1 gridpoint for the lift)
//   cand [CH][2d]       velocity-bound candidates vlim/q' per joint (upper, lower)
//   vec  [CH][VS]       per gridpoint: q' | a+ | q'' | b+ | -amax | +amin | xlo | xhi | 0
//   tab  [W]            per record column: offset into vec (bit 15 = negate, 0x7fff = column not owned)
// Phase 2: every thread owns one 16-byte column pair and walks down the gridpoints:
//   rec[ci][col] = +-vec[ci][tab[col]]  -> two shared loads + one coalesced 16-byte store per iteration.
template <int CH>
__global__ void __launch_bounds__(COEFF_THREADS)
coeff_velacc_kernel(const double *__restrict__ ppoly, const double *__restrict__ breaks, const int breaks_shared,
                    const int nseg, const int dof, const double *__restrict__ grid, const int grid_shared, const int G,
                    const double *__restrict__ vlim, const double *__restrict__ alim, const int lim_shared,
                    const int interp, double *__restrict__ records, const int W, const int R_total, const int row0,
                    const int write_xbound, const int nchunks, const int pp_in_smem) {
  extern __shared__ double sm[];
  const int VS = 6 * dof + 3;
  double *raw = sm;                                  // [(CH+1)][2*dof]
  double *cand = raw + (CH + 1) * 2 * dof;           // [CH][2*dof]
  double *vec = cand + CH * 2 * dof;                 // [CH][VS]
  double *sgrid = vec + CH * VS;                     // [CH+1]
  // long splines (many waypoints): breakpoints and coefficients stay in global memory (L1/L2)
  double *sx_s = sgrid + CH + 1;                     // [nseg+1] breakpoints
  double *dco = sx_s + (pp_in_smem ? nseg + 1 : 0);  // [nseg][dof][5]
  unsigned short *tab = reinterpret_cast<unsigned short *>(dco + (pp_in_smem ? nseg * dof * 5 : 0));  // [W]
  const long path = blockIdx.x / nchunks;
  const int chunk = blockIdx.x % nchunks;
  const int i0 = chunk * CH;
  const int N = G - 1;
  const int npts = min(CH, G - i0);          // gridpoints written by this CTA
  const int nev = min(CH + 1, G - i0);       // gridpoints evaluated (one extra for the lift)
  const double *c = ppoly + path * 4 * nseg * dof;
  const double *x = breaks + (breaks_shared ? 0 : path * (nseg + 1));
  const double *gp = grid + (grid_shared ? 0 : path * G);
  const double *al = alim ? alim + (lim_shared ? 0 : path * dof * 2) : nullptr;
  const double *vl = vlim ? vlim + (lim_shared ? 0 : path * dof * 2) : nullptr;
  const int tid = threadIdx.x;
  const int Racc = al ? (interp ? 4 : 2) * dof : 0;

  // ---- phase 0: gridpoints, breakpoints, derivative coefficients, column table ----
  for (int ci = tid; ci < nev; ci += COEFF_THREADS) sgrid[ci] = gp[i0 + ci];
  const double *sx = pp_in_smem ? sx_s : x;
  for (int q = tid; pp_in_smem && q <= nseg; q += COEFF_THREADS) sx_s[q] = x[q];
  for (int q = tid; pp_in_smem && q < nseg * dof; q += COEFF_THREADS) {
    // scipy PPoly.derivative: c'[j] = c[j] * (k - j); cspldd = cspld.derivative() (interpolator.py:419-421)
    const double c0 = c[q], c1 = c[nseg * dof + q], c2 = c[2 * nseg * dof + q];
    const double d0 = c0 * 3.0, d1 = c1 * 2.0, d2 = c2 * 1.0;
    double *o = dco + q * 5;
    o[0] = d0; o[1] = d1; o[2] = d2; o[3] = d0 * 2.0; o[4] = d1 * 1.0;
  }
  for (int w = tid; w < W; w += COEFF_THREADS) {
    unsigned short code = 0x7fff;  // not owned by this call: leave untouched
    const int kind = w / R_total_or1(R_total), r = w - kind * R_total - row0;
    if (kind < 3 && R_total > 0 && r >= 0 && r < Racc) {
      const int blk = r / dof, k = r - blk * dof;
      const int neg = blk & 1, second = blk >> 1;
      if (kind == 0) code = (unsigned short)((second ? dof + k : k) | (neg << 15));
      else if (kind == 1) code = (unsigned short)((second ? 3 * dof + k : 2 * dof + k) | (neg << 15));
      else code = (unsigned short)(neg ? 5 * dof + k : 4 * dof + k);
    } else if (w >= 3 * R_total) {
      // xlo | xhi | padding zeros; records with a u-bound pair (W >= 3R+4, TB_SCAN_UBOUND) keep those two slots
      const bool ub_slot = (W >= 3 * R_total + 4) && (w == 3 * R_total + 2 || w == 3 * R_total + 3);
      if (write_xbound && !ub_slot)
        code = (unsigned short)(w == 3 * R_total ? 6 * dof : (w == 3 * R_total + 1 ? 6 * dof + 1 : 6 * dof + 2));
    }
    tab[w] = code;
  }
  __syncthreads();

  // ---- phase 1: q', q'' at the chunk's gridpoints (+ per-joint velocity-bound candidates) ----
  const double inf_d = __longlong_as_double(0x7ff0000000000000LL);
  for (int idx = tid; idx < nev * dof; idx += COEFF_THREADS) {
    const int ci = idx / dof, k = idx - ci * dof;
    const double s = sgrid[ci];
    const int seg = find_interval(sx, nseg, s);
    double v1, v2;
    if (seg < 0) {
      v1 = v2 = __longlong_as_double(0x7ff8000000000000LL);
    } else {
      // scipy evaluate_poly1: res = 0; z = 1; for each power: res += c * z; z *= ds
      const double ds = s - sx[seg];
      double oloc[5];
      const double *o = dco + (seg * dof + k) * 5;
      if (!pp_in_smem) {
        const int q = seg * dof + k;
        const double c0 = c[q], c1 = c[nseg * dof + q], c2 = c[2 * nseg * dof + q];
        oloc[0] = c0 * 3.0; oloc[1] = c1 * 2.0; oloc[2] = c2 * 1.0; oloc[3] = oloc[0] * 2.0; oloc[4] = oloc[1] * 1.0;
        o = oloc;
      }
      double z = ds;
      v1 = 0.0 + o[2];
      v1 = v1 + o[1] * z;
      z = z * ds;
      v1 = v1 + o[0] * z;
      v2 = 0.0 + o[4];
      v2 = v2 + o[3] * ds;
    }
    raw[ci * 2 * dof + k] = v1;
    raw[ci * 2 * dof + dof + k] = v2;
    if (vl && write_xbound && ci < npts) {
      // _CythonUtils.pyx:44-50: q' > 0: (vmax/q', vmin/q'); q' < 0: (vmin/q', vmax/q'); q' == 0 (or NaN): no update
      const bool posq = v1 > 0, negq = v1 < 0;
      const double qd = (posq || negq) ? v1 : 1.0;
      const double r1 = vl[k * 2 + 1] / qd, r0 = vl[k * 2 + 0] / qd;
      cand[ci * 2 * dof + k] = posq ? r1 : (negq ? r0 : inf_d);          // candidate for sdmax
      cand[ci * 2 * dof + dof + k] = posq ? r0 : (negq ? r1 : -inf_d);   // candidate for sdmin
    }
  }
  __syncthreads();

  // ---- phase 1b: per-gridpoint value vectors ----
  double *rec0 = records + (path * G + i0) * (long)W;
  for (int idx = tid; idx < npts * dof; idx += COEFF_THREADS) {
    const int ci = idx / dof, k = idx - ci * dof;
    const int gi = i0 + ci;
    double *v = vec + ci * VS;
    const double a = raw[ci * 2 * dof + k], b = raw[ci * 2 * dof + dof + k];
    double ap = a, bp = b;  // last gridpoint duplicates itself, linear_constraint.py:171,175
    if (gi < N) {
      const double delta = sgrid[ci + 1] - sgrid[ci];
      ap = raw[(ci + 1) * 2 * dof + k] + (2 * delta) * raw[(ci + 1) * 2 * dof + dof + k];  // linear_constraint.py:170
      bp = raw[(ci + 1) * 2 * dof + dof + k];
    }
    v[k] = a; v[dof + k] = ap; v[2 * dof + k] = b; v[3 * dof + k] = bp;
    if (al) {
      v[4 * dof + k] = 0.0 - al[k * 2 + 1];       // F.c - g with c = 0, g = [amax; -amin]
      v[5 * dof + k] = 0.0 - (-al[k * 2 + 0]);
    }
    if (k == 0 && write_xbound) {
      // velocity bound of this gridpoint: fp32 running min/max over the joints exactly like _CythonUtils.pyx:41-58
      double xlo = VAR_MIN, xhi = VAR_MAX;  // seidelWrapper low_arr/high_arr init, pyx:477-478
      if (vl) {
        // The reference keeps the running min/max in C floats: s <- (float)min(cand_k, (double)s), k = 0..dof-1,
        // s_0 = 1e8f (_CythonUtils.pyx:41-50).  Round-to-nearest is monotone and idempotent, so that chain equals
        // (float)min(1e8, min_k cand_k) (likewise for the max): reduce in fp64, round once.
        double mhi = JVEL_MAXSD, mlo = -JVEL_MAXSD;
        for (int kk = 0; kk < dof; ++kk) {
          const double hi = cand[ci * 2 * dof + kk], lo = cand[ci * 2 * dof + dof + kk];
          mhi = (hi <= mhi) ? hi : mhi;
          mlo = (lo >= mlo) ? lo : mlo;
        }
        const float sdmax = __double2float_rn(mhi), sdmin = __double2float_rn(mlo);
        const float up = __fmul_rn(sdmax, sdmax);                          // powf(sdmax, 2) in fp32
        const double lo_d = ((double)sdmin >= 0.0) ? (double)sdmin : 0.0;  // float64_max(sdmin, 0.)
        xlo = lo_d * lo_d;
        xhi = (double)up;
        if (write_xbound != 2) {
          // pyx:517-520: low = max(VAR_MIN, xbound_lo), high = min(VAR_MAX, xbound_hi)
          xlo = fmax(VAR_MIN, xlo);
          xhi = fmin(VAR_MAX, xhi);
        }
      }
      if (write_xbound == 3) {  // intersect with what the record already holds
        const double *rec = rec0 + (long)ci * W;
        xlo = fmax(rec[3 * R_total], xlo);
        xhi = fmin(rec[3 * R_total + 1], xhi);
      }
      v[6 * dof] = xlo; v[6 * dof + 1] = xhi; v[6 * dof + 2] = 0.0;
    }
  }
  __syncthreads();

  // ---- phase 2: stream the records out; thread -> fixed 16-byte column pair, loop over gridpoints ----
  const int Wh = W >> 1;
  const int ngrp = COEFF_THREADS / Wh;  // gridpoints written per sweep (threads beyond ngrp * Wh idle)
  const int g = tid / Wh, j = tid - g * Wh;
  if (ngrp > 0 && g < ngrp) {
    const unsigned short c0 = tab[2 * j], c1 = tab[2 * j + 1];
    const int o0 = c0 & 0x7fff, o1 = c1 & 0x7fff;
    const bool n0 = (c0 & 0x8000) != 0, n1 = (c1 & 0x8000) != 0;
    const bool own0 = c0 != 0x7fff, own1 = c1 != 0x7fff;
    double *dst = rec0 + (long)g * W + 2 * j;
    const double *v = vec + g * VS;
    if (own0 && own1) {
      for (int ci = g; ci < npts; ci += ngrp, dst += (long)ngrp * W, v += ngrp * VS) {
        double2 o;
        o.x = n0 ? -v[o0] : v[o0];
        o.y = n1 ? -v[o1] : v[o1];
        __stcs(reinterpret_cast<double2 *>(dst), o);  // streaming store: written once, read later by K2
      }
    } else if (own0 || own1) {
      for (int ci = g; ci < npts; ci += ngrp, dst += (long)ngrp * W, v += ngrp * VS) {
        if (own0) dst[0] = n0 ? -v[o0] : v[o0];
        if (own1) dst[1] = n1 ? -v[o1] : v[o1];
      }
    }
  } else if (ngrp == 0) {  // records wider than 2 * COEFF_THREADS columns: column loop per gridpoint
    for (int ci = 0; ci < npts; ++ci)
      for (int w = tid; w < W; w += COEFF_THREADS) {
        const unsigned short cw = tab[w];
        if (cw != 0x7fff) {
          const double t = vec[ci * VS + (cw & 0x7fff)];
          rec0[(long)ci * W + w] = (cw & 0x8000) ? -t : t;
        }
      }
  }
}

// Generic CanonicalLinear row assembly (seidelWrapper.__init__ pyx:483-510 +
// canlinear_colloc_to_interpolate linear_constraint.py:134-192).  One thread per (path, gridpoint, out row).
__global__ void rows_canlinear_kernel(const double *__restrict__ a, const double *__restrict__ b,
                                      const double *__restrict__ c, const double *__restrict__ F,
                                      const double *__restrict__ g, const int F_mode, const long B, const int G,
                                      const int m, const int k, const double *__restrict__ grid,
                                      const int grid_shared, const int interp, double *__restrict__ records,
                                      const int W, const int R_total, const int row0) {
  const int nrows = interp ? 2 * k : k;
  const long total = B * G * nrows;
  const int N = G - 1;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    const int r = (int)(idx % nrows);
    const long pg = idx / nrows;
    const int gi = (int)(pg % G);
    const long p = pg / G;
    const int second = r >= k;           // second block: constraint at s_{i+1} in stage-i variables
    const int j = second ? r - k : r;    // row of F
    const int src = (second && gi < N) ? gi + 1 : gi;  // last stage duplicates itself
    const double *ap = a + (p * G + src) * m, *bp = b + (p * G + src) * m, *cp = c + (p * G + src) * m;
    double two_delta = 0.0;
    const bool lift = second && gi < N;
    if (lift) {
      const double *gp = grid + (grid_shared ? 0 : p * G);
      two_delta = 2 * (gp[gi + 1] - gp[gi]);
    }
    double ta = 0.0, tb_ = 0.0, tc = 0.0, gv;
    if (F_mode >= 2) {  // F = [I; -I]
      const int col = (j < m) ? j : j - m;
      const double sgn = (j < m) ? 1.0 : -1.0;
      const double av = lift ? ap[col] + two_delta * bp[col] : ap[col];
      ta = sgn * av;
      tb_ = sgn * bp[col];
      tc = sgn * cp[col];
      gv = (F_mode == 3) ? g[p * k + j] : g[j];
    } else {
      const double *Fr = (F_mode == 0) ? F + (long)j * m : F + ((p * G + src) * k + j) * (long)m;
      for (int q = 0; q < m; ++q) {
        const double av = lift ? ap[q] + two_delta * bp[q] : ap[q];
        ta = ta + Fr[q] * av;
        tb_ = tb_ + Fr[q] * bp[q];
        tc = tc + Fr[q] * cp[q];
      }
      gv = (F_mode == 0) ? g[j] : g[(p * G + src) * k + j];
    }
    double *rec = records + (p * G + gi) * (long)W;
    rec[row0 + r] = ta;
    rec[R_total + row0 + r] = tb_;
    rec[2 * R_total + row0 + r] = tc - gv;
  }
}

// JointVelocityConstraintVarying (linear_joint_velocity.py:56-87, _CythonUtils.pyx:61-101): velocity limits that
// vary along the path, vlim_grid [G][dof][2] (shared) or [B][G][dof][2].  One thread per (path, gridpoint).
__global__ void xbound_varying_kernel(const double *__restrict__ ppoly, const double *__restrict__ breaks,
                                      const int breaks_shared, const long B, const int nseg, const int dof,
                                      const double *__restrict__ grid, const int grid_shared, const int G,
                                      const double *__restrict__ vlim_grid, const int vlim_shared, const int per_grid,
                                      double *__restrict__ records, const int W, const int R_total, const int mode) {
  const long total = B * G;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    const int gi = (int)(idx % G);
    const long p = idx / G;
    const double *x = breaks + (breaks_shared ? 0 : p * (nseg + 1));
    const double *c = ppoly + p * 4 * nseg * dof;
    const double s = grid[(grid_shared ? 0 : p * G) + gi];
    // per_grid: limits per gridpoint (JointVelocityConstraintVarying); else one (dof, 2) array per path / batch
    const double *vl = per_grid ? vlim_grid + ((vlim_shared ? 0 : p * G) + gi) * (long)dof * 2
                                : vlim_grid + (vlim_shared ? 0 : p) * (long)dof * 2;
    const int seg = find_interval(x, nseg, s);
    float sdmin = -(float)JVEL_MAXSD, sdmax = (float)JVEL_MAXSD;
    for (int k = 0; k < dof && seg >= 0; ++k) {
      const double q = ppoly_eval1(c, nseg, dof, seg, k, s - x[seg], 1);
      if (q > 0) {
        const double hi = vl[k * 2 + 1] / q, lo = vl[k * 2 + 0] / q;
        sdmax = __double2float_rn(hi <= (double)sdmax ? hi : (double)sdmax);
        sdmin = __double2float_rn(lo >= (double)sdmin ? lo : (double)sdmin);
      } else if (q < 0) {
        const double hi = vl[k * 2 + 0] / q, lo = vl[k * 2 + 1] / q;
        sdmax = __double2float_rn(hi <= (double)sdmax ? hi : (double)sdmax);
        sdmin = __double2float_rn(lo >= (double)sdmin ? lo : (double)sdmin);
      }
    }
    const float up = __fmul_rn(sdmax, sdmax);
    const double lo_d = ((double)sdmin >= 0.0) ? (double)sdmin : 0.0;
    double xlo = lo_d * lo_d, xhi = (double)up;
    double *rec = records + idx * W;
    if (mode != 2) { xlo = fmax(VAR_MIN, xlo); xhi = fmin(VAR_MAX, xhi); }
    if (mode == 3) { xlo = fmax(rec[3 * R_total], xlo); xhi = fmin(rec[3 * R_total + 1], xhi); }
    rec[3 * R_total] = xlo;
    rec[3 * R_total + 1] = xhi;
  }
}

// ---- SecondOrderConstraint on device (BASELINE cfg 3) -------------------------------------------------------------
// SecondOrderConstraint.compute_constraint_params (toppra/constraint/linear_second_order.py:142-173):
//     c = tau(q, 0, 0);  a = tau(q, 0, q') - c;  b = tau(q, q', q'') - c;  c += sign(q') * friction  (:138)
// for the joint-torque factory (:114-140): F = [I; -I], g = [tau_max; -tau_min], Interpolation lift
// (linear_constraint.py:134-163).  The reference calls a user Python inv_dyn 3 (N+1) times per path; here the inverse
// dynamics is a DEVICE MODEL picked from a small registry (TB_INVDYN_*), evaluated straight from the spline: no
// [B*G, dof] intermediates, no host round trip.  The lifted block of record i (a+ = a_{i+1} + 2 delta_i b_{i+1}) reads the
// values of gridpoint i+1 from shared memory; the last gridpoint duplicates itself (linear_constraint.py:141-153).
//   TB_INVDYN_COUPLED_COSINE: tau_i = p0 qdd_i + p1 sum_j cos(q_i - q_j) qdd_j + p2 sin(q_i) |qd|^2 + p3 sin(q_i)
//                             (SURVEY.md section 8d cfg 3: p = (2, 0.3, 0.1, 4.9));  cos(q_i - q_j) is expanded
//                             into cos q_i cos q_j + sin q_i sin q_j: dof sincos instead of dof^2 cosines
//   TB_INVDYN_PENDULUMS:      tau_i = p[2i] qdd_i + p[2i+1] sin(q_i)   (independent joints; params [dof][2])
constexpr int SO_MAX_DOF = 16;

// second_order_rows_tiled_kernel: one CTA per (path, 32 gridpoints).
//   phase 1  thread per (gridpoint, joint): q, q', q'' from the spline and sincos(q) — the expensive part, spread over
//            all threads instead of one thread per gridpoint;
//   phase 2  thread per (gridpoint, joint): the model's coupling sums over the joints (same summation order as
//            the first version of this kernel) -> a, b, c in shared memory (33 gridpoints: one more than the tile for the lifted block);
//   phase 3  the CTA streams the 3 x (2 | 4) dof row entries of its 32 records out in record order: consecutive
//            threads write consecutive doubles (runs of (2 | 4) dof doubles) instead of one thread striding through 72
//            scattered 8-byte stores per gridpoint.
constexpr int SO_TILE = 32;
constexpr int SO_THREADS = 128;

template <int MODEL>
__global__ void __launch_bounds__(SO_THREADS)
second_order_rows_tiled_kernel(const double *__restrict__ ppoly, const double *__restrict__ breaks,
                               const int breaks_shared, const int nseg, const int dof, const double *__restrict__ grid,
                               const int grid_shared, const int G, const double *__restrict__ prm,
                               const double *__restrict__ taulim, const int lim_shared,
                               const double *__restrict__ friction, const int interp, double *__restrict__ records,
                               const int W, const int R_total, const int row0) {
  extern __shared__ double so_sm[];
  const int tiles = (G + SO_TILE - 1) / SO_TILE;
  const long p = blockIdx.x / tiles;
  const int gi0 = (int)(blockIdx.x % tiles) * SO_TILE;
  const int npts = min(SO_TILE, G - gi0);                  // records of this tile
  const int nev = min(npts + 1, G - gi0);                  // gridpoints evaluated (one more for the lift)
  const int tid = threadIdx.x, N = G - 1;
  const double *x = breaks + (breaks_shared ? 0 : p * (nseg + 1));
  const double *cpp = ppoly + p * 4 * nseg * dof;
  const double *gp = grid + (grid_shared ? 0 : p * G);
  const double *tl = taulim + (lim_shared ? 0 : p * dof * 2);
  // shared: per evaluated gridpoint and joint: qd, qdd, sin q, cos q, then a, b, c; the gridpoints; the row decode table
  const int ne = (SO_TILE + 1) * dof;
  double *s_qd = so_sm, *s_qdd = so_sm + ne, *s_sq = so_sm + 2 * ne, *s_cq = so_sm + 3 * ne;
  double *s_a = so_sm + 4 * ne, *s_b = so_sm + 5 * ne, *s_c = so_sm + 6 * ne, *s_g = so_sm + 7 * ne;
  const int nrows = (interp ? 4 : 2) * dof;
  const int per_rec = 3 * nrows;
  unsigned *s_tab = reinterpret_cast<unsigned *>(s_g + SO_TILE + 2);
  const double nan_d = __longlong_as_double(0x7ff8000000000000LL);
  // row decode table, once per CTA (the only integer divisions of the kernel): entry r of a record's 3 * nrows values ->
  // part (a | b | c), row j, joint k, negated copy, lifted block
  for (int r = tid; r < per_rec; r += SO_THREADS) {
    const int part = r / nrows, j = r - part * nrows;
    const int blk = j / dof, k = j - blk * dof;
    s_tab[r] = (unsigned)part | ((unsigned)k << 2) | ((unsigned)(blk & 1) << 8) | ((unsigned)(blk >> 1) << 9) | ((unsigned)j << 10);
  }
  for (int t = tid; t < nev; t += SO_THREADS) s_g[t] = gp[gi0 + t];
  // e -> (gridpoint t, joint k) without a division: t = floor(e / dof) by a multiply-high with ceil(2^32 / dof) (exact
  // for e < 2^16).  For dof = 1 that multiplier is 2^32, which does not fit 32 bits: t = e there.
  const unsigned inv_dof = dof > 1 ? (unsigned)((0x100000000ULL + (unsigned)dof - 1u) / (unsigned)dof) : 0u;
  for (int e = tid; e < nev * dof; e += SO_THREADS) {
    const int t = dof > 1 ? (int)__umulhi((unsigned)e, inv_dof) : e, k = e - t * dof;
    const double s = gp[gi0 + t];
    const int seg = find_interval(x, nseg, s);
    const double q = seg < 0 ? nan_d : ppoly_eval1(cpp, nseg, dof, seg, k, s - x[seg], 0);
    s_qd[e] = seg < 0 ? nan_d : ppoly_eval1(cpp, nseg, dof, seg, k, s - x[seg], 1);
    s_qdd[e] = seg < 0 ? nan_d : ppoly_eval1(cpp, nseg, dof, seg, k, s - x[seg], 2);
    double sv, cv;
    sincos(q, &sv, &cv);
    s_sq[e] = sv;
    s_cq[e] = cv;
  }
  __syncthreads();
  for (int e = tid; e < nev * dof; e += SO_THREADS) {
    const int t = dof > 1 ? (int)__umulhi((unsigned)e, inv_dof) : e, k = e - t * dof;
    const double *qd = s_qd + t * dof, *qdd = s_qdd + t * dof, *sq = s_sq + t * dof, *cq = s_cq + t * dof;
    double av, bv, cv;
    if (MODEL == TB_INVDYN_COUPLED_COSINE) {
      const double m0 = prm[0], m1 = prm[1], h = prm[2], gr = prm[3];
      double cs1 = 0.0, ss1 = 0.0, cs2 = 0.0, ss2 = 0.0, v2 = 0.0;
      for (int j = 0; j < dof; ++j) {
        cs1 += cq[j] * qd[j]; ss1 += sq[j] * qd[j];
        cs2 += cq[j] * qdd[j]; ss2 += sq[j] * qdd[j];
        v2 += qd[j] * qd[j];
      }
      cv = gr * sq[k];
      av = m0 * qd[k] + m1 * (cq[k] * cs1 + sq[k] * ss1);
      bv = m0 * qdd[k] + m1 * (cq[k] * cs2 + sq[k] * ss2) + h * sq[k] * v2;
    } else {
      cv = prm[2 * k + 1] * sq[k];
      av = prm[2 * k] * qd[k];
      bv = prm[2 * k] * qdd[k];
    }
    if (friction) {  // np.sign(q') * joint_friction, linear_second_order.py:138
      const double sg = (qd[k] > 0) ? 1.0 : ((qd[k] < 0) ? -1.0 : 0.0);
      cv = cv + sg * friction[k];
    }
    s_a[e] = av; s_b[e] = bv; s_c[e] = cv;
  }
  __syncthreads();
  // phase 3: a warp takes one record at a time, its lanes the record's 3 * nrows values in record order (runs of nrows
  // consecutive doubles per part).  Row j of the constraint: bit 0 of blk = negated copy, bit 1 = the block evaluated at
  // s_{i+1} and lifted.
  double *rec0 = records + (p * G + gi0) * (long)W;
  const int warp = tid >> 5, lane = tid & 31;
  for (int gl = warp; gl < npts; gl += SO_THREADS / 32) {
    const bool last = (gi0 + gl) >= N;                  // the last gridpoint duplicates itself (linear_constraint.py:141-153)
    const double two_delta = last ? 0.0 : 2 * (s_g[gl + 1] - s_g[gl]);
    double *rec = rec0 + (long)gl * W;
    for (int r = lane; r < per_rec; r += 32) {
      const unsigned code = s_tab[r];
      const int part = code & 3, k = (code >> 2) & 63, j = code >> 10;
      const bool neg = (code >> 8) & 1, second = (code >> 9) & 1;
      const bool lift = second && !last;
      const int src = (lift ? gl + 1 : gl) * dof + k;
      double v;
      if (part == 0) {
        v = lift ? s_a[src] + two_delta * s_b[src] : s_a[src];
        v = neg ? -v : v;
      } else if (part == 1) {
        v = neg ? -s_b[src] : s_b[src];
      } else {
        v = neg ? (-s_c[src] - (-tl[k * 2 + 0])) : (s_c[src] - tl[k * 2 + 1]);   // F c - g, g = [tau_max; -tau_min]
      }
      rec[part * R_total + row0 + j] = v;
    }
  }
}

// Fill the xbound slots (and padding) with the defaults +-1e8 when no constraint supplies them.
__global__ void init_bounds_kernel(double *__restrict__ records, const long BG, const int W, const int R_total) {
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < BG; idx += (long)gridDim.x * blockDim.x) {
    double *rec = records + idx * W;
    rec[3 * R_total] = VAR_MIN;
    rec[3 * R_total + 1] = VAR_MAX;
    int j = 3 * R_total + 2;
    if (W >= 3 * R_total + 4) {  // records with a u-bound pair (TB_SCAN_UBOUND): u in [-1e8, 1e8] by default
      rec[j] = VAR_MIN;
      rec[j + 1] = VAR_MAX;
      j += 2;
    }
    for (; j < W; ++j) rec[j] = 0.0;
  }
}

}  // namespace
}  // namespace tb

extern "C" int tb_record_doubles(int R) {
  if (R < 0) return TB_ERR_ARG;
  const int w = 3 * R + 2;
  return (w + 1) & ~1;
}

extern "C" int tb_coeff_velacc(const double *ppoly, const double *breaks, int breaks_shared, int B, int nseg, int dof,
                               const double *grid, int grid_shared, int G, const double *vlim, const double *alim,
                               int lim_shared, int interp, double *records, int W, int R_total, int row0,
                               int write_xbound, void *stream) {
  using namespace tb;
  if (!ppoly || !breaks || !grid || (!alim && !vlim) || !records || B <= 0 || nseg <= 0 || dof <= 0 || G <= 0) {
    set_error("tb_coeff_velacc: bad argument");
    return TB_ERR_ARG;
  }
  const int Racc = alim ? (interp ? 4 : 2) * dof : 0;
  if (row0 < 0 || row0 + Racc > R_total || W < 3 * R_total + 2) {
    set_error("tb_coeff_velacc: rows [%d,%d) do not fit R_total=%d / W=%d", row0, row0 + Racc, R_total, W);
    return TB_ERR_ARG;
  }
  if (R_total > MAX_ROWS) { set_error("tb_coeff_velacc: R=%d > %d", R_total, MAX_ROWS); return TB_ERR_UNSUPPORTED; }
  if (6 * dof + 3 >= 0x7fff) { set_error("tb_coeff_velacc: dof=%d too large", dof); return TB_ERR_UNSUPPORTED; }
  const int CH = (G > 96) ? COEFF_CH_LARGE : COEFF_CH_SMALL;
  const int nchunks = (G + CH - 1) / CH;
  const long blocks = (long)B * nchunks;
  if (blocks > 0x7fffffffL) { set_error("tb_coeff_velacc: batch too large for one launch"); return TB_ERR_UNSUPPORTED; }
  const size_t pp_doubles = (size_t)nseg + 1 + (size_t)nseg * dof * 5;
  const int pp_in_smem = pp_doubles * sizeof(double) <= 32 * 1024;
  const size_t smem = (size_t)((CH + 1) * dof * 2 + CH * dof * 2 + CH * (6 * dof + 3) + CH + 1 +
                               (pp_in_smem ? pp_doubles : 0)) * sizeof(double) + (size_t)W * sizeof(unsigned short) + 16;
  auto kern = (CH == COEFF_CH_LARGE) ? coeff_velacc_kernel<COEFF_CH_LARGE> : coeff_velacc_kernel<COEFF_CH_SMALL>;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) { set_error("tb_coeff_velacc: dof=%d too large for shared memory", dof); return TB_ERR_UNSUPPORTED; }
  }
  kern<<<(unsigned)blocks, COEFF_THREADS, smem, (cudaStream_t)stream>>>(
      ppoly, breaks, breaks_shared, nseg, dof, grid, grid_shared, G, vlim, alim, lim_shared, interp, records, W,
      R_total, row0, write_xbound, nchunks, pp_in_smem);
  return check_launch("tb_coeff_velacc");
}

extern "C" int tb_rows_canlinear(const double *a, const double *b, const double *c, const double *F, const double *g,
                                 int F_mode, int B, int G, int m, int k, const double *grid, int grid_shared,
                                 int interp, double *records, int W, int R_total, int row0, void *stream) {
  using namespace tb;
  if (!a || !b || !c || !g || !records || !grid || B <= 0 || G <= 0 || m <= 0 || k <= 0 || F_mode < 0 || F_mode > 3) {
    set_error("tb_rows_canlinear: bad argument");
    return TB_ERR_ARG;
  }
  if (F_mode < 2 && !F) { set_error("tb_rows_canlinear: F is null"); return TB_ERR_ARG; }
  if (F_mode >= 2 && k != 2 * m) { set_error("tb_rows_canlinear: F=[I;-I] needs k == 2m"); return TB_ERR_ARG; }
  const int nrows = interp ? 2 * k : k;
  if (row0 < 0 || row0 + nrows > R_total || W < 3 * R_total + 2) {
    set_error("tb_rows_canlinear: rows [%d,%d) do not fit R_total=%d / W=%d", row0, row0 + nrows, R_total, W);
    return TB_ERR_ARG;
  }
  const long total = (long)B * G * nrows;
  const int threads = 256;
  long blocks = (total + threads - 1) / threads;
  if (blocks > 148L * 32) blocks = 148L * 32;
  rows_canlinear_kernel<<<(unsigned)blocks, threads, 0, (cudaStream_t)stream>>>(a, b, c, F, g, F_mode, B, G, m, k, grid,
                                                                               grid_shared, interp, records, W,
                                                                               R_total, row0);
  return check_launch("tb_rows_canlinear");
}

extern "C" int tb_init_bounds(double *records, int B, int G, int W, int R_total, void *stream) {
  using namespace tb;
  if (!records || B <= 0 || G <= 0 || W < 3 * R_total + 2) { set_error("tb_init_bounds: bad argument"); return TB_ERR_ARG; }
  const long BG = (long)B * G;
  const int threads = 256;
  long blocks = (BG + threads - 1) / threads;
  if (blocks > 148L * 32) blocks = 148L * 32;
  init_bounds_kernel<<<(unsigned)blocks, threads, 0, (cudaStream_t)stream>>>(records, BG, W, R_total);
  return check_launch("tb_init_bounds");
}

extern "C" int tb_xbound_varying(const double *ppoly, const double *breaks, int breaks_shared, int B, int nseg, int dof,
                                 const double *grid, int grid_shared, int G, const double *vlim_grid, int vlim_shared,
                                 double *records, int W, int R_total, int write_xbound, void *stream) {
  using namespace tb;
  if (!ppoly || !breaks || !grid || !vlim_grid || !records || B <= 0 || nseg <= 0 || dof <= 0 || G <= 0 ||
      write_xbound < 1 || write_xbound > 3 || W < 3 * R_total + 2) {
    set_error("tb_xbound_varying: bad argument");
    return TB_ERR_ARG;
  }
  const long total = (long)B * G;
  const int threads = 128;
  long blocks = (total + threads - 1) / threads;
  if (blocks > 148L * 64) blocks = 148L * 64;
  xbound_varying_kernel<<<(unsigned)blocks, threads, 0, (cudaStream_t)stream>>>(
      ppoly, breaks, breaks_shared, B, nseg, dof, grid, grid_shared, G, vlim_grid, vlim_shared, 1, records, W, R_total,
      write_xbound);
  return check_launch("tb_xbound_varying");
}

extern "C" int tb_coeff_second_order(int model, const double *params, int nparams, const double *ppoly, const double *breaks,
                                     int breaks_shared, int B, int nseg, int dof, const double *grid, int grid_shared,
                                     int G, const double *taulim, int lim_shared, const double *friction, int interp,
                                     double *records, int W, int R_total, int row0, void *stream) {
  using namespace tb;
  if (!params || !ppoly || !breaks || !grid || !taulim || !records || B <= 0 || nseg <= 0 || dof <= 0 || G <= 0) {
    set_error("tb_coeff_second_order: bad argument");
    return TB_ERR_ARG;
  }
  if (dof > SO_MAX_DOF) { set_error("tb_coeff_second_order: dof=%d > %d", dof, SO_MAX_DOF); return TB_ERR_UNSUPPORTED; }
  const int need = (model == TB_INVDYN_COUPLED_COSINE) ? 4 : ((model == TB_INVDYN_PENDULUMS) ? 2 * dof : -1);
  if (need < 0) { set_error("tb_coeff_second_order: unknown device model %d", model); return TB_ERR_UNSUPPORTED; }
  if (nparams != need) { set_error("tb_coeff_second_order: model %d takes %d parameters, got %d", model, need, nparams); return TB_ERR_ARG; }
  const int nrows = (interp ? 4 : 2) * dof;
  if (row0 < 0 || row0 + nrows > R_total || W < 3 * R_total + 2) {
    set_error("tb_coeff_second_order: rows [%d,%d) do not fit R_total=%d / W=%d", row0, row0 + nrows, R_total, W);
    return TB_ERR_ARG;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const int tiles = (G + SO_TILE - 1) / SO_TILE;
  const long blocks = (long)B * tiles;
  if (blocks > 0x7fffffffL) { set_error("tb_coeff_second_order: B * ceil(G / 32) = %ld CTAs exceed the grid limit", blocks); return TB_ERR_UNSUPPORTED; }
  const size_t smem = (size_t)(7 * (SO_TILE + 1) * dof + SO_TILE + 2) * sizeof(double) + (size_t)3 * nrows * sizeof(unsigned);
  if (model == TB_INVDYN_COUPLED_COSINE)
    second_order_rows_tiled_kernel<TB_INVDYN_COUPLED_COSINE><<<(unsigned)blocks, SO_THREADS, smem, st>>>(
        ppoly, breaks, breaks_shared, nseg, dof, grid, grid_shared, G, params, taulim, lim_shared, friction, interp,
        records, W, R_total, row0);
  else
    second_order_rows_tiled_kernel<TB_INVDYN_PENDULUMS><<<(unsigned)blocks, SO_THREADS, smem, st>>>(
        ppoly, breaks, breaks_shared, nseg, dof, grid, grid_shared, G, params, taulim, lim_shared, friction, interp,
        records, W, R_total, row0);
  return check_launch("tb_coeff_second_order");
}

extern "C" int tb_xbound_velocity(const double *ppoly, const double *breaks, int breaks_shared, int B, int nseg, int dof,
                                  const double *grid, int grid_shared, int G, const double *vlim, int lim_shared,
                                  double *records, int W, int R_total, int write_xbound, void *stream) {
  using namespace tb;
  if (!ppoly || !breaks || !grid || !vlim || !records || B <= 0 || nseg <= 0 || dof <= 0 || G <= 0 || R_total < 0 ||
      W < 3 * R_total + 2 || write_xbound < 1 || write_xbound > 3) {
    set_error("tb_xbound_velocity: bad argument");
    return TB_ERR_ARG;
  }
  const long total = (long)B * G;
  const int threads = 128;
  long blocks = (total + threads - 1) / threads;
  if (blocks > 148L * 64) blocks = 148L * 64;
  xbound_varying_kernel<<<(unsigned)blocks, threads, 0, (cudaStream_t)stream>>>(
      ppoly, breaks, breaks_shared, B, nseg, dof, grid, grid_shared, G, vlim, lim_shared, 0, records, W, R_total,
      write_xbound);
  return check_launch("tb_xbound_velocity");
}
