// Warp-level building blocks of the fused PyMOC engine (fp64 throughout).
//
// Layout: one warp owns one ensemble member.  A vertical profile of nz <= 32*LPL levels is
// distributed in contiguous chunks -- lane L holds levels [L*LPL, (L+1)*LPL) in registers --
// so the explicit column step needs only two neighbour shuffles per step and everything
// else is lane-local.  All columns of a member share this map, hence the thermal-wind and
// isopycnal-remap arithmetic that combines basin and north values is lane-local too.
//
// Arithmetic policy (see pmoc_rt.cuh): the once-per-K-steps diagnostics follow the
// reference's NumPy expressions operation by operation (IEEE divide, no contraction);
// the per-step column update uses folded stencil coefficients (three FP64-pipe
// instructions per level and step).  file:line citations are under
// /root/reference/src/pymoc/modules.
#pragma once
#include "pmoc_rt.cuh"

namespace pm {

constexpr double kSv = 1e6;

template <int LPL>
PM_DEV int lev(int j) { return rt::lane() * LPL + j; }
// per-warp shared arrays that are only ever read by their owner use the conflict-free
// lane-major layout: slot j of lane L lives at j*32 + L
PM_DEV int lm(int j) { return j * 32 + rt::lane(); }

// x / c for a constant c with rc = 1/c pre-rounded: product, exact residual, one correction
// (Markstein).  Correctly rounded -- the same bits as the IEEE divide the reference performs --
// whenever no intermediate over/underflows; checked against x / 1e6 on 4e8 random doubles.
PM_DEV double div_const(double x, double c, double rc) {
  const double q = x * rc;
  return rt::fma(rt::fma(-c, q, x), rc, q);
}

// a / b, IEEE.  The compiler's inline divide leaves a zero (or denormal) numerator to a ~60-instruction
// out-of-line routine; zeros are structural here (Psi = 0 at the boundaries, z[-1] = 0, the lowest
// class of the remap), so they are answered directly: 0 / b = +-0 for any finite non-zero b.
PM_DEV double qdiv(double a, double b) {
  if (a == 0.0 && b != 0.0 && fabs(b) < INFINITY) return (std::signbit(a) != std::signbit(b)) ? -0.0 : 0.0;
  if (b == 0.0 && a != 0.0 && a == a) return (std::signbit(a) != std::signbit(b)) ? -INFINITY : INFINITY;
  return a / b;
}

// a / b without branches for a finite a and a finite b that is zero or normal, quotient in the normal range:
// the in-range sequence, with the IEEE results of a zero divisor (+-inf, 0/0 = NaN) selected afterwards.
// (An infinite operand -- a blown-up member -- gives NaN where IEEE gives 0 / inf.)
PM_DEV double sdiv(double a, double b) {
  const bool bz = b == 0.0;
  const double q = rt::div_normal(a, bz ? 1.0 : b);
  const double z = (a != a || a == 0.0) ? NAN : ((std::signbit(a) != std::signbit(b)) ? -INFINITY : INFINITY);
  return bz ? z : q;
}

// registers <- natural-order global/shared array
template <int LPL>
PM_DEV void load_lev(double (&v)[LPL], const double* PM_RESTRICT g, int n, double pad) {
  PM_UNROLL
  for (int j = 0; j < LPL; ++j) {
    const int i = lev<LPL>(j);
    v[j] = i < n ? g[i] : pad;
  }
}
template <int LPL>
PM_DEV void store_lev(const double (&v)[LPL], double* PM_RESTRICT g, int n) {
  PM_UNROLL
  for (int j = 0; j < LPL; ++j) {
    const int i = lev<LPL>(j);
    if (i < n) g[i] = v[j];
  }
}

// exclusive prefix sum of one value per lane
PM_DEV double wscan_excl(double v) {
  const int L = rt::lane();
  PM_UNROLL
  for (int d = 1; d < 32; d <<= 1) {
    const double t = rt::shfl_up(v, d);
    if (L >= d) v = v + t;
  }
  const double prev = rt::shfl_up(v, 1);
  return L == 0 ? 0.0 : prev;
}

// ===================================================================== Column
// Folded coefficients of the explicit step (column.py:235-249).  With d_i = b[i+1]-b[i]:
//   b_i += dt*( -weff_i * (weff_i<0 ? d_i/dzu : d_{i-1}/dzd) / A_i
//               + kappa_i * (d_i/dzu - d_{i-1}/dzd) / (0.5*(dzu+dzd)) )  =  p_i d_i - q_i d_{i-1}
// weff = wA - d(A kappa)/dz is fixed between two streamfunction updates, so p, q are rebuilt
// only then.  Everything state-independent is tabulated once per launch:
//   per block  (GeoTab, lane-major): 1/dzu, 1/dzd, 1/(dzc dzu), 1/(dzc dzd), z
//   per member (ColTab, lane-major): dt kappa, RA = dt/A, dAk
// Boundary and padding levels get p = q = 0.
struct GeoTab {
  const double *zs;                      // natural order, nzp+4 (padded with z[nz-1])
  const double *zl, *rdu, *rdd, *ruu, *rdd2;  // lane-major, nzp each
};
struct ColTab {
  double *kdt, *ra, *dak;  // lane-major, nzp each (per warp): dt*kappa, dt/Area, d(A kappa)/dz
};

// block-cooperative fill of the geometry tables (call before the block barrier)
template <int LPL>
PM_DEV void geo_fill(double* zs, double* zl, double* rdu, double* rdd, double* ruu, double* rdd2,
                     const double* PM_RESTRICT z, int nz, int tid, int nthr, bool folded = true) {
  const int nzp = 32 * LPL;
  for (int i = tid; i < nzp + 4; i += nthr) zs[i] = z[i < nz ? i : nz - 1];
  if (!folded) {
    for (int s = tid; s < nzp; s += nthr) {
      const int i = (s & 31) * LPL + (s >> 5);
      zl[s] = z[i < nz ? i : nz - 1];
    }
    return;
  }
  for (int s = tid; s < nzp; s += nthr) {
    const int L = s & 31, j = s >> 5, i = L * LPL + j;
    double a = 0., b = 0., c = 0., d = 0.;
    if (i >= 1 && i < nz - 1) {
      const double dzu = z[i + 1] - z[i], dzd = z[i] - z[i - 1], dzc = 0.5 * (dzu + dzd);
      a = 1. / dzu;
      b = 1. / dzd;
      c = 1. / (dzc * dzu);
      d = 1. / (dzc * dzd);
    }
    zl[s] = z[i < nz ? i : nz - 1];
    rdu[s] = a;
    rdd[s] = b;
    ruu[s] = c;
    rdd2[s] = d;
  }
}

// per-member tables from the (host-sampled) kappa, d(A kappa)/dz and Area profiles
template <int LPL>
PM_DEV void col_tabulate(const ColTab& T, const GeoTab& G, const double* PM_RESTRICT kappa,
                         const double* PM_RESTRICT dAk, const double* PM_RESTRICT Area, int nz, double dt) {
  PM_UNROLL
  for (int j = 0; j < LPL; ++j) {
    const int i = lev<LPL>(j), s = lm(j);
    double kdt = 0., ra = 0., dk = 0.;
    if (i >= 1 && i < nz - 1) {
      kdt = dt * kappa[i];
      ra = dt / Area[i];
      dk = dAk[i];
    }
    T.kdt[s] = kdt;
    T.ra[s] = ra;
    T.dak[s] = dk;
  }
  rt::syncwarp();
}

template <int LPL>
PM_DEV void col_coeffs(double (&p)[LPL], double (&q)[LPL], const double (&wA)[LPL], const ColTab& T,
                       const GeoTab& G, int nz) {
  PM_UNROLL
  for (int j = 0; j < LPL; ++j) {
    const int i = lev<LPL>(j), s = lm(j);
    double pj = 0.0, qj = 0.0;
    if (i >= 1 && i < nz - 1) {
      const double weff = wA[j] - T.dak[s];
      const double ra = T.ra[s];
      const double kdt = T.kdt[s];
      pj = kdt * G.ruu[s];
      qj = kdt * G.rdd2[s];
      if (weff < 0)
        pj = pj - weff * (ra * G.rdu[s]);
      else
        qj = qj + weff * (ra * G.rdd[s]);
    }
    p[j] = pj;
    q[j] = qj;
  }
}

// The same coefficients straight from the (host-sampled) global profiles, for topologies whose
// per-member tables would cost resident warps: identical expressions, hence identical values.
template <int LPL>
PM_DEV void col_coeffs_global(double (&p)[LPL], double (&q)[LPL], const double (&wA)[LPL],
                              const double* PM_RESTRICT kappa, const double* PM_RESTRICT dAk,
                              const double* PM_RESTRICT Area, double dt, const GeoTab& G, int nz) {
  double kdt[LPL], ra[LPL], dk[LPL];
  PM_UNROLL
  for (int j = 0; j < LPL; ++j) {  // the loads first, so that they overlap
    const int i = lev<LPL>(j);
    const bool in = i >= 1 && i < nz - 1;
    kdt[j] = in ? kappa[i] : 0.0;
    ra[j] = in ? Area[i] : 1.0;
    dk[j] = in ? dAk[i] : 0.0;
  }
  PM_UNROLL
  for (int j = 0; j < LPL; ++j) {
    const int i = lev<LPL>(j), s = lm(j);
    double pj = 0.0, qj = 0.0;
    if (i >= 1 && i < nz - 1) {
      const double weff = wA[j] - dk[j];
      const double rav = rt::div_normal(dt, ra[j]);  // Area: finite, normal
      const double kd = dt * kdt[j];
      pj = kd * G.ruu[s];
      qj = kd * G.rdd2[s];
      if (weff < 0)
        pj = pj - weff * (rav * G.rdu[s]);
      else
        qj = qj + weff * (rav * G.rdd[s]);
    }
    p[j] = pj;
    q[j] = qj;
  }
}

// One explicit step: 2 neighbour shuffles, LPL+1 subtractions, 2*LPL FMAs.
template <int LPL>
PM_DEV void col_step(double (&b)[LPL], const double (&p)[LPL], const double (&q)[LPL]) {
  const double bnext = rt::shfl_down(b[0], 1);
  const double bprev = rt::shfl_up(b[LPL - 1], 1);
  double dm = b[0] - bprev;
  PM_UNROLL
  for (int j = 0; j < LPL; ++j) {
    const double d = (j < LPL - 1 ? b[j + 1 < LPL ? j + 1 : j] : bnext) - b[j];
    b[j] = rt::fma(-q[j], dm, rt::fma(p[j], d, b[j]));
    dm = d;
  }
}

// ---- bit-faithful step ---------------------------------------------------------------------
// The same IEEE operations in the same order as column.py:235-249, with every divide by a
// state-independent number c done as div_const(x, c, 1/c) (correctly rounded, 3 FMAs).  Used
// where the loop sits on structural ties that the folded form would break: in the 'jn' order
// the no-flux bottom condition bbot = b[1] converges to b[0] == b[1] *exactly*, and a one-ulp
// difference flips a flat remap cell into an inverted one (Psib is discontinuous there).
struct ExactGeo {
  const double *dzu, *rdzu, *dzc, *rdzc;  // lane-major, nzp each: cell above each level, centred spacing
};
struct ExactCol {
  double *kap[2], *area, *rarea, *nweff[2];  // lane-major, nzp each (per warp); [variant]
};

template <int LPL>
PM_DEV void geo_fill_exact(double* dzu, double* rdzu, double* dzc, double* rdzc, const double* PM_RESTRICT z, int nz,
                           int tid, int nthr) {
  const int nzp = 32 * LPL;
  for (int s = tid; s < nzp; s += nthr) {
    const int L = s & 31, j = s >> 5, i = L * LPL + j;
    double a = 1., c = 1.;
    if (i < nz - 1) a = z[i + 1] - z[i];
    if (i >= 1 && i < nz - 1) c = 0.5 * ((z[i + 1] - z[i]) + (z[i] - z[i - 1]));
    dzu[s] = a;
    rdzu[s] = 1. / a;
    dzc[s] = c;
    rdzc[s] = 1. / c;
  }
}

template <int LPL>
PM_DEV void col_tabulate_exact(const ExactCol& T, const double* PM_RESTRICT kappa, const double* PM_RESTRICT Area,
                               int nz, int nvar) {
  PM_UNROLL
  for (int j = 0; j < LPL; ++j) {
    const int i = lev<LPL>(j), s = lm(j);
    const bool in = i >= 1 && i < nz - 1;
    const double A = in ? Area[i] : 1.0;
    T.area[s] = A;
    T.rarea[s] = 1.0 / A;
    T.kap[0][s] = in ? kappa[i] : 0.0;
    T.kap[1][s] = in ? kappa[(nvar > 1 ? nz : 0) + i] : 0.0;
  }
  rt::syncwarp();
}

// -weff = -(wA - d(A kappa)/dz) for both kappa variants (column.py:241,245)
template <int LPL>
PM_DEV void col_nweff(const ExactCol& T, const double (&wA)[LPL], const double* PM_RESTRICT dAk, int nz, int nvar) {
  PM_UNROLL
  for (int j = 0; j < LPL; ++j) {
    const int i = lev<LPL>(j), s = lm(j);
    const bool in = i >= 1 && i < nz - 1;
    T.nweff[0][s] = in ? -(wA[j] - dAk[i]) : 0.0;
    T.nweff[1][s] = in ? -(wA[j] - dAk[(nvar > 1 ? nz : 0) + i]) : 0.0;
  }
  rt::syncwarp();
}

// One level of the bit-faithful explicit step (column.py:235-249): g_up / g_dn are the gradients of the cells above
// and below, nweff = -weff, A / rA the Area and its reciprocal.  Every kernel that steps a column this way calls it,
// so that they all round the same operations in the same order.  The operands that callers keep in memory are taken by
// reference: each is then loaded where the arithmetic needs it, not ahead of the level's gradients (register pressure
// of the step loops).
PM_DEV double exact_level(double b, double g_up, double g_dn, const double& dzc, const double& rdzc,
                          const double& nweff, const double& kappa, const double& A, const double& rA, double dt) {
  const double bzz = div_const(g_up - g_dn, dzc, rdzc);
  const double sel = nweff > 0 ? g_up : g_dn;  // weff < 0  <=>  -weff > 0
  const double a = A, ra = rA;  // (read before the product: fewer registers in k_wide_post)
  const double adv = div_const(nweff * sel, a, ra);
  const double tend = adv + kappa * bzz;
  return b + dt * tend;
}

template <int LPL>
PM_DEV void col_step_exact(double (&b)[LPL], const ExactCol& T, int var, const ExactGeo& G, int nz, double dt) {
  // (offsets from one base pointer, not a run-time pick between two pointers: the loads stay LDS)
  const double* kap = T.kap[0] + var * (T.kap[1] - T.kap[0]);
  const double* nweff = T.nweff[0] + var * (T.nweff[1] - T.nweff[0]);
  const double bnext = rt::shfl_down(b[0], 1);
  double bzu[LPL];
  PM_UNROLL
  for (int j = 0; j < LPL; ++j) {
    const int s = lm(j);
    const double up = j < LPL - 1 ? b[j + 1 < LPL ? j + 1 : j] : bnext;
    bzu[j] = div_const(up - b[j], G.dzu[s], G.rdzu[s]);
  }
  const double bzprev = rt::shfl_up(bzu[LPL - 1], 1);
  PM_UNROLL
  for (int j = 0; j < LPL; ++j) {
    const int i = lev<LPL>(j), s = lm(j);
    if (i >= 1 && i < nz - 1) {
      const double bzd = j > 0 ? bzu[j > 0 ? j - 1 : 0] : bzprev;
      b[j] = exact_level(b[j], bzu[j], bzd, G.dzc[s], G.rdzc[s], nweff[s], kap[s], T.area[s], T.rarea[s], dt);
    }
  }
}

// Convective adjustment of one value (column.py:264-271): with convection (cv) a value above bs becomes
// bs + N2min (z[i] - zc), zc the depth of the highest stable level; without, only the surface value is reset to bs.
PM_DEV double convect_level(double v, int i, bool cv, double bs, double n2, double zc, const double* z, int nz) {
  if (cv) return v > bs ? bs + n2 * (z[i] - zc) : v;
  return i == nz - 1 ? bs : v;
}

// Convective adjustment (column.py:264-271).  Strict '>' and un-fused bs + N2min*(z - zconv).
template <int LPL>
PM_DEV void col_convect(double (&b)[LPL], double bs, double N2min, const double* zs, const double* zl, int nz) {
  unsigned mine = 0;
  int top_stable = -1;
  PM_UNROLL
  for (int j = 0; j < LPL; ++j) {
    const int i = lev<LPL>(j);
    if (i < nz) {
      if (b[j] > bs)
        mine |= 1u << j;
      else
        top_stable = i;
    }
  }
  if (rt::ballot(mine != 0)) {
    const int anchor = rt::max_i(top_stable);
    const double zc = zs[anchor >= 0 ? anchor : 0];
    PM_UNROLL
    for (int j = 0; j < LPL; ++j)
      if ((mine >> j) & 1u) b[j] = bs + N2min * (zl[lm(j)] - zc);
  } else {
    PM_UNROLL
    for (int j = 0; j < LPL; ++j)
      if (lev<LPL>(j) == nz - 1) b[j] = bs;
  }
}

// Lateral inflow (column.py:306-313)
template <int LPL>
PM_DEV void col_horadv(double (&b)[LPL], const double* PM_RESTRICT vdx, const double* PM_RESTRICT b_in,
                       const double* PM_RESTRICT Area, int nz, double dt) {
  PM_UNROLL
  for (int j = 0; j < LPL; ++j) {
    const int i = lev<LPL>(j);
    if (i < nz && vdx[i] > 0.0) b[j] = b[j] + dt * vdx[i] * (b_in[i] - b[j]) / Area[i];
  }
}

template <int LPL>
PM_DEV void set_level(double (&b)[LPL], int level, double v) {
  PM_UNROLL
  for (int j = 0; j < LPL; ++j)
    if (lev<LPL>(j) == level) b[j] = v;
}
// value of one level, broadcast to the warp
template <int LPL>
PM_DEV double get_level(const double (&b)[LPL], int level) {
  double mine = 0.0;
  PM_UNROLL
  for (int j = 0; j < LPL; ++j)
    if (lev<LPL>(j) == level) mine = b[j];
  return rt::shfl(mine, level / LPL);
}

// ============================================================== Psi_Thermwind
// Exact solution of Psi'' = (b2-b1)/f, Psi(z0)=Psi(zN)=0 (psi_thermwind.py:123-135) in the form
// SciPy's collocation produces on the un-refined mesh z: Simpson for Psi' with the mid-point
// value gm, cubic-Hermite Simpson for Psi.  For piecewise-linear b's (gm = mean of the ends)
// it is the exact C1 piecewise cubic.  Result in Sv.
template <int LPL>
PM_DEV void tw_solve(double (&psi)[LPL], const double (&b1)[LPL], const double (&b2)[LPL], double f,
                     const double* zs, int nz, const double* PM_RESTRICT gmid) {
  const double rf = 1. / f;
  double g[LPL], T[LPL], part[LPL];
  PM_UNROLL
  for (int j = 0; j < LPL; ++j) g[j] = lev<LPL>(j) < nz ? rf * (b2[j] - b1[j]) : 0.0;
  const double gnext = rt::shfl_down(g[0], 1);
  double run = 0.0;
  PM_UNROLL
  for (int j = 0; j < LPL; ++j) {
    const int i = lev<LPL>(j);
    const double gi = g[j], gi1 = j < LPL - 1 ? g[j + 1 < LPL ? j + 1 : j] : gnext;
    double t = 0.0;
    if (i < nz - 1) {
      const double h = zs[i + 1] - zs[i];
      const double gm = gmid ? rf * gmid[i] : 0.5 * (gi + gi1);
      t = div_const(h, 6., 1. / 6.) * (gi + 4. * gm + gi1);
    }
    T[j] = t;
    part[j] = run;
    run = run + t;
  }
  const double base1 = wscan_excl(run);
  run = 0.0;
  PM_UNROLL
  for (int j = 0; j < LPL; ++j) {
    const int i = lev<LPL>(j);
    const double gi = g[j], gi1 = j < LPL - 1 ? g[j + 1 < LPL ? j + 1 : j] : gnext;
    double cell = 0.0;
    if (i < nz - 1) {
      const double h = zs[i + 1] - zs[i];
      cell = h * (base1 + part[j]) + h * T[j] / 2. - div_const(h * h, 12., 1. / 12.) * (gi1 - gi);
    }
    part[j] = run;
    run = run + cell;
  }
  const double base2 = wscan_excl(run);
  PM_UNROLL
  for (int j = 0; j < LPL; ++j) part[j] = base2 + part[j];
  const double total = get_level<LPL>(part, nz - 1);
  const double z0 = zs[0], H = zs[nz - 1] - zs[0], rH = 1.0 / H;
  PM_UNROLL
  for (int j = 0; j < LPL; ++j) {
    const int i = lev<LPL>(j);
    psi[j] = i < nz ? div_const(part[j] - total * div_const(zs[i] - z0, H, rH), kSv, 1.0 / kSv) : 0.0;
  }
}

// np.linspace(bmin, bmax, nb)[i]  (numpy: arange(nb)*step + start, last element = stop)
struct BGrid {
  double lo, hi, step, rstep;  // rstep = 1/step (for div_const)
  int nb;
  PM_DEV double at(int i) const { return i == nb - 1 ? hi : (double)i * step + lo; }
};

// number of classes with bgrid value <= v (index estimated by division, then corrected against
// the actual grid values)
PM_DEV int bgrid_count_le(const BGrid& G, double v) {
  const int nb = G.nb;
  if (v < G.lo) return 0;
  if (v >= G.hi) return nb;
  if (!(G.step > 0.)) return v >= G.lo ? nb : 0;
  const double r = div_const(v - G.lo, G.step, G.rstep);
  int p = r < (double)(nb - 1) ? (int)r + 1 : nb;
  // one correction each way suffices (see interp_bgrid): the rounding of r and of the nodes is ~1e-13 steps
  if (p < nb && G.at(p) <= v) ++p;
  if (p > 0 && G.at(p - 1) > v) --p;
  return p;
}

// Upwind isopycnal remap (psi_thermwind.py:170-185):
//   psib[i] = sum_c clip((top_c - bgrid_i)/(top_c - bot_c), 0, 1) * u_c,   u_c = -(Psi[c+1]-Psi[c]),
// cell c taking its bottom/top buoyancy from column 2 where u_c < 0 and from column 1 otherwise.
//
// Sorted part.  Where a profile is non-decreasing (which stable stratification and the convective
// adjustment maintain almost everywhere), the cells of column X split for a class value x into
// "entirely above x" (clip = 1), "entirely below" (clip = 0) and at most one straddling cell, so
//   psib(x) = sum_X [ S_X[k] + (bX[k] - x) * w_X[k-1] ],   k = #{levels with bX < x},
// with S_X[k] = sum_{c >= k} [cell c uses X] u_c (a warp suffix scan) and
// w_X[c] = [cell c uses X] u_c / (bX[c+1] - bX[c]).  O(nb + nz) instead of O(nb nz); the sum is
// associated differently from np.sum (relative difference ~1e-16).  Flat cells keep the
// reference's inf/NaN outcomes (SURVEY H3): (top-x)/0 is +inf -> 1 below the cell, -inf -> 0
// above it and 0/0 = NaN on it.  k is not searched for: every level drops a count into the class
// slot where its buoyancy first falls below the class value (integer shared-memory atomics: exact,
// order independent), and a prefix sum over the classes turns the counts into k for both columns.
//
// Exceptional cells.  Profiles are not always sorted: the 'jn' bottom condition bbot = b[1] leaves
// b[0] one rounding above b[1] for many members, and spin-up transients hold inverted layers.  The
// sorted machinery then runs on the running maximum bX' of each profile (sorted by construction)
// with the transport of every cell whose end points differ from the running maximum set to zero,
// and exactly those "exceptional" cells are added class by class with the reference's own
// expression (the direct O(nb E) loop, E = number of exceptional cells).  A NaN anywhere makes
// every cell exceptional.
// Scratch: rs = 6*nzp doubles, psib_s = nb doubles, cnt_s = nb+1 ints, all owned by this warp.

// flat cells sitting exactly on a class value: 0/0 = NaN in the reference (psi_thermwind.py:183)
PM_COLD double remap_flat_fix(double c, double x, int k, int nz, const double* b_s, const double* w_s) {
  for (int cc = k; cc + 1 < nz && b_s[cc + 1] == x; ++cc)
    if (w_s[cc] != 0.0) c = NAN;
  return c;
}

// PMOC_ST_TIE_CELL.  Psib's clip((top-x)/(top-bot), 0, 1) sends a cell's transport u_c to the classes BELOW it when
// the cell is upright or flat ((top-x)/0 = +-inf) and to the classes ABOVE it when it is inverted, so between
// "flat" and "inverted by one ulp" psib jumps by the whole u_c: there the last bit of the state decides.  Flagged:
//   * a cell that IS inverted, by no more than 4 eps (relative, i.e. 4..8 ulp): one rounding away from flat;
//   * the bottom cell within 4 eps of flat, either way: under the 'jn' no-flux condition bbot = b[1] its two
//     levels are the same number one step apart in time, so their difference is the last increment of b[1] --
//     of either sign, and at rounding level once the bottom has equilibrated.
// Not flagged: interior cells that are upright by a few ulp.  Those are the rounded steady state of a column
// relaxing onto bs from below (levels 4, 3, 2, 1 ulp apart); the upwind step is monotone, neither arithmetic
// inverts them, and upright and flat cells contribute identically.
constexpr double kTieEps = 4.0 * 2.220446049250313e-16;
PM_DEV bool remap_tie(double bot, double top, double u, bool bottom) {
  const double a = fabs(top), b = fabs(bot), gap = top - bot;
  return u != 0.0 && fabs(gap) <= kTieEps * (a > b ? a : b) && (gap < 0.0 || bottom);
}

template <int LPL>
PM_DEV BGrid tw_psib(const double (&psi)[LPL], const double (&b1)[LPL], const double (&b2)[LPL], int nz, int nb,
                     double* rs, double* psib_s, int* cnt_s, unsigned* status = nullptr) {
  const int nzp = 32 * LPL, L = rt::lane();
  const double psin = rt::shfl_down(psi[0], 1);
  const double b1n = rt::shfl_down(b1[0], 1), b2n = rt::shfl_down(b2[0], 1);
  double lo = INFINITY, hi = -INFINITY;
  double u[LPL], up1[LPL], up2[LPL], m1[LPL], m2[LPL];
  bool nan = false;
  double r1 = -INFINITY, r2 = -INFINITY;
  PM_UNROLL
  for (int j = 0; j < LPL; ++j) {
    const int i = lev<LPL>(j);
    const bool last = j == LPL - 1;
    const int jn = j + 1 < LPL ? j + 1 : j;
    up1[j] = last ? b1n : b1[jn];
    up2[j] = last ? b2n : b2[jn];
    u[j] = 0.0;
    if (i < nz) {
      lo = b1[j] < lo ? b1[j] : lo;
      lo = b2[j] < lo ? b2[j] : lo;
      hi = b1[j] > hi ? b1[j] : hi;
      hi = b2[j] > hi ? b2[j] : hi;
      nan |= b1[j] != b1[j] || b2[j] != b2[j];
      r1 = b1[j] > r1 ? b1[j] : r1;
      r2 = b2[j] > r2 ? b2[j] : r2;
    }
    m1[j] = r1;
    m2[j] = r2;
    if (i < nz - 1) {
      u[j] = -((last ? psin : psi[jn]) - psi[j]);
      nan |= u[j] != u[j];
    }
  }
  BGrid G;
  G.lo = rt::wmin(lo);
  G.hi = rt::wmax(hi);
  G.nb = nb;
  G.step = (G.hi - G.lo) / (double)(nb - 1);
  G.rstep = 1.0 / G.step;
  const bool allexc = rt::ballot(nan) != 0;
  // running maxima across the lanes (exclusive max-scan of the lane maxima)
  {
    double v1 = r1, v2 = r2;
    PM_UNROLL
    for (int d = 1; d < 32; d <<= 1) {
      const double o1 = rt::shfl_up(v1, d), o2 = rt::shfl_up(v2, d);
      if (L >= d) {
        v1 = o1 > v1 ? o1 : v1;
        v2 = o2 > v2 ? o2 : v2;
      }
    }
    double e1 = rt::shfl_up(v1, 1), e2 = rt::shfl_up(v2, 1);
    if (L == 0) e1 = e2 = -INFINITY;
    PM_UNROLL
    for (int j = 0; j < LPL; ++j) {
      m1[j] = e1 > m1[j] ? e1 : m1[j];
      m2[j] = e2 > m2[j] ? e2 : m2[j];
    }
  }
  const double m1n = rt::shfl_down(m1[0], 1), m2n = rt::shfl_down(m2[0], 1);
  // exceptional cells: an end point below the running maximum of the column the cell is taken from
  unsigned excm = 0;
  int ne = 0;
  bool tie = false;
  PM_UNROLL
  for (int j = 0; j < LPL; ++j) {
    const int i = lev<LPL>(j);
    if (i < nz - 1) {
      const bool last = j == LPL - 1;
      const int jn = j + 1 < LPL ? j + 1 : j;
      const bool from2 = u[j] < 0;
      const double mu = from2 ? (last ? m2n : m2[jn]) : (last ? m1n : m1[jn]);
      const double upv = from2 ? up2[j] : up1[j];
      const double mb = from2 ? m2[j] : m1[j], bv = from2 ? b2[j] : b1[j];
      tie |= remap_tie(bv, upv, u[j], i == 0);
      if (allexc || mu != upv || mb != bv) {
        excm |= 1u << j;
        ++ne;
      }
    }
  }
  if (status != nullptr && rt::ballot(tie) != 0) *status |= 128u;  // PMOC_ST_TIE_CELL
  int incl = ne;
  PM_UNROLL
  for (int d = 1; d < 32; d <<= 1) {
    const int o = rt::shfl_i(incl, L >= d ? L - d : L);
    if (L >= d) incl += o;
  }
  const int E = rt::shfl_i(incl, 31);
  if (E > 0) {
    // the reference's expression, class by class, over the exceptional cells only
    double *ctop = rs, *crinv = rs + nzp, *cu = rs + 2 * nzp;
    int pos = incl - ne;
    PM_UNROLL
    for (int j = 0; j < LPL; ++j) {
      if ((excm >> j) & 1u) {
        const bool from2 = u[j] < 0;
        const double bot = from2 ? b2[j] : b1[j];
        const double top = from2 ? up2[j] : up1[j];
        ctop[pos] = top;
        crinv[pos] = sdiv(1.0, top - bot);
        cu[pos] = u[j];
        ++pos;
      }
    }
    rt::syncwarp();
    constexpr int KB = 8;
    for (int base = 0; base < nb; base += 32 * KB) {
      double bg[KB], acc[KB];
      PM_UNROLL
      for (int k = 0; k < KB; ++k) {
        const int i = base + k * 32 + L;
        bg[k] = G.at(i < nb ? i : nb - 1);
        acc[k] = 0.0;
      }
      for (int c = 0; c < E; ++c) {
        const double top = ctop[c], r = crinv[c], uc = cu[c];
        PM_UNROLL
        for (int k = 0; k < KB; ++k) {
          double t = (top - bg[k]) * r;
          t = t < 0. ? 0. : t;
          t = t > 1. ? 1. : t;
          acc[k] = rt::fma(t, uc, acc[k]);
        }
      }
      PM_UNROLL
      for (int k = 0; k < KB; ++k) {
        const int i = base + k * 32 + L;
        if (i < nb) psib_s[i] = acc[k];
      }
    }
    rt::syncwarp();
    if (allexc) return G;
  }
  {
    double *b1_s = rs, *b2_s = rs + nzp, *w1_s = rs + 2 * nzp, *w2_s = rs + 3 * nzp, *S1_s = rs + 4 * nzp,
           *S2_s = rs + 5 * nzp;
    // suffix sums of the transports taken from each column (exceptional cells carry none)
    double s1[LPL], s2[LPL];
    double q1 = 0.0, q2 = 0.0;
    PM_UNROLL
    for (int j = LPL - 1; j >= 0; --j) {
      const bool from2 = u[j] < 0, ex = (excm >> j) & 1u;
      q1 = q1 + ((from2 || ex) ? 0.0 : u[j]);
      q2 = q2 + ((from2 && !ex) ? u[j] : 0.0);
      s1[j] = q1;
      s2[j] = q2;
    }
    double t1 = q1, t2 = q2;  // inclusive suffix over lanes
    PM_UNROLL
    for (int d = 1; d < 32; d <<= 1) {
      const double o1 = rt::shfl_down(t1, d), o2 = rt::shfl_down(t2, d);
      if (L + d < 32) {
        t1 = t1 + o1;
        t2 = t2 + o2;
      }
    }
    const double e1 = t1 - q1, e2 = t2 - q2;  // lanes above this one
    PM_UNROLL
    for (int j = 0; j < LPL; ++j) {
      const int i = lev<LPL>(j);
      if (i < nz) {
        const bool last = j == LPL - 1;
        const int jn = j + 1 < LPL ? j + 1 : j;
        const bool cell = i < nz - 1 && !((excm >> j) & 1u), from2 = u[j] < 0;
        b1_s[i] = m1[j];
        b2_s[i] = m2[j];
        S1_s[i] = s1[j] + e1;
        S2_s[i] = s2[j] + e2;
        w1_s[i] = (cell && !from2) ? sdiv(u[j], (last ? m1n : m1[jn]) - m1[j]) : 0.0;
        w2_s[i] = (cell && from2) ? sdiv(u[j], (last ? m2n : m2[jn]) - m2[j]) : 0.0;
      }
    }
    rt::syncwarp();
    for (int i = L; i <= nb; i += 32) cnt_s[i] = 0;
    rt::syncwarp();
    PM_UNROLL
    for (int j = 0; j < LPL; ++j) {
      if (lev<LPL>(j) < nz) {
        rt::atomic_add_shared(&cnt_s[bgrid_count_le(G, m1[j])], 1);
        rt::atomic_add_shared(&cnt_s[bgrid_count_le(G, m2[j])], 1 << 16);
      }
    }
    rt::syncwarp();
    const int cpl = (nb + 31) >> 5;  // classes per lane, contiguous
    const int i0 = L * cpl < nb ? L * cpl : nb, i1 = i0 + cpl < nb ? i0 + cpl : nb;
    int run = 0;
    for (int i = i0; i < i1; ++i) run += cnt_s[i];
    int inc2 = run;
    PM_UNROLL
    for (int d = 1; d < 32; d <<= 1) {
      const int o = rt::shfl_i(inc2, L >= d ? L - d : L);
      if (L >= d) inc2 += o;
    }
    run = inc2 - run;  // levels counted in the classes of the lanes below
    for (int i = i0; i < i1; ++i) {
      const double x = G.at(i);
      run += cnt_s[i];
      const int k1 = run & 0xffff, k2 = run >> 16;  // #{levels with bX' < x}
      double c1 = 0.0, c2 = 0.0;
      if (k1 < nz) {
        const double bk = b1_s[k1];
        c1 = S1_s[k1];
        if (k1 > 0 && bk != x) c1 = c1 + (bk - x) * w1_s[k1 - 1];
        if (bk == x) c1 = remap_flat_fix(c1, x, k1, nz, b1_s, w1_s);
      }
      if (k2 < nz) {
        const double bk = b2_s[k2];
        c2 = S2_s[k2];
        if (k2 > 0 && bk != x) c2 = c2 + (bk - x) * w2_s[k2 - 1];
        if (bk == x) c2 = remap_flat_fix(c2, x, k2, nz, b2_s, w2_s);
      }
      psib_s[i] = E > 0 ? psib_s[i] + (c1 + c2) : c1 + c2;
    }
    rt::syncwarp();
  }
  return G;
}

// np.interp(x, bgrid, psib) (numpy/_core/src/multiarray/compiled_base.c: arr_interp) on the
// implicit uniform grid: index by division, then corrected against the actual grid values.
// Written without early exits: the index comes from one multiply-corrected divide (off by at most one
// from the search's answer: the rounding of r and of the grid nodes is ~1e-13 of a grid step), two
// predicated single-step corrections against the actual node values, then both nodes are loaded, the
// segment evaluated and the special cases selected -- so that the interpolations of a lane overlap.
PM_DEV double interp_bgrid(double x, const BGrid& G, const double* psib_s) {
  const int nb = G.nb;
  const bool flat = !(G.step > 0.);  // hi == lo (or NaN): every query sits on the last node
  const double r = div_const(x - G.lo, flat ? 1.0 : G.step, flat ? 1.0 : G.rstep);
  int j = (r >= 0.0 && r < (double)(nb - 1)) ? (int)r : (r >= 0.0 ? nb - 1 : 0);  // (NaN -> 0, unused)
  if (j < nb - 1 && G.at(j + 1) <= x) ++j;
  if (j > 0 && G.at(j) > x) --j;
  if (flat) j = nb - 1;
  const int jj = j < nb - 1 ? j : nb - 2;
  const double xj = G.at(jj), xj1 = G.at(jj + 1), fj = psib_s[jj], fj1 = psib_s[jj + 1];
  const double slope = rt::div_normal(fj1 - fj, flat ? 1.0 : xj1 - xj);  // xj1 - xj: one grid step > 0
  double res = slope * (x - xj) + fj;
  if (res != res) {  // arr_interp's fall-backs for a NaN product (an infinite slope times zero)
    res = slope * (x - xj1) + fj1;
    if (res != res && fj == fj1) res = fj;
  }
  if (xj == x) res = fj;
  if (j == nb - 1) res = fj1;
  if (x < G.lo) res = psib_s[0];
  if (x > G.hi) res = psib_s[nb - 1];
  return x != x ? x : res;
}

// ===================================================================== Psi_SO
// index of the last element <= key in a non-decreasing array (numpy binary_search_with_guess
// result for a key inside the range)
template <class XP>
PM_DEV int search_le(XP a, int n, double key) {
  int lo = 0, hi = n;
  while (lo < hi) {
    const int mid = lo + ((hi - lo) >> 1);
    if (key >= a[mid])
      lo = mid + 1;
    else
      hi = mid;
  }
  return lo - 1;
}

// np.interp(x, xp, fp) for a scalar x, generic (possibly non-uniform) increasing xp
PM_DEV double interp1(double x, const double* xp, const double* fp, int n) {
  if (x != x) return x;
  if (x > xp[n - 1]) return fp[n - 1];
  if (x < xp[0]) return fp[0];
  const int j = search_le(xp, n, x);
  if (j == n - 1) return fp[j];
  if (xp[j] == x) return fp[j];
  const double slope = sdiv(fp[j + 1] - fp[j], xp[j + 1] - xp[j]);
  double res = slope * (x - xp[j]) + fp[j];
  if (res != res) {
    res = slope * (x - xp[j + 1]) + fp[j + 1];
    if (res != res && fp[j] == fp[j + 1]) res = fp[j];
  }
  return res;
}

PM_DEV bool sgn(double v) { return std::signbit(v); }

// scipy.optimize.brentq(lambda y: bs(y) - bval, ya, yb) with the default tolerances --
// statement-for-statement the iteration of scipy/optimize/Zeros/brentq.c (Brent 1973), so a
// multi-root bs(y) resolves to the root the reference finds (SURVEY H7).
PM_COLD double outcrop_brent(double bval, const double* ygrid, const double* bs, int ny, int south, bool* sign_error) {
  const double xtol = 2e-12, rtol = 8.881784197001252e-16;
  double xpre = ygrid[south], xcur = ygrid[ny - 1];
  double xblk = 0., fblk = 0., spre = 0., scur = 0.;
  double fpre = interp1(xpre, ygrid, bs, ny) - bval;
  double fcur = interp1(xcur, ygrid, bs, ny) - bval;
  if (fpre == 0) return xpre;
  if (fcur == 0) return xcur;
  if (sgn(fpre) == sgn(fcur)) {
    *sign_error = true;
    return NAN;
  }
  for (int it = 0; it < 100; ++it) {
    if (fpre != 0 && fcur != 0 && sgn(fpre) != sgn(fcur)) {
      xblk = xpre;
      fblk = fpre;
      spre = scur = xcur - xpre;
    }
    if (fabs(fblk) < fabs(fcur)) {
      xpre = xcur; xcur = xblk; xblk = xpre;
      fpre = fcur; fcur = fblk; fblk = fpre;
    }
    const double delta = (xtol + rtol * fabs(xcur)) / 2;
    const double sbis = (xblk - xcur) / 2;
    if (fcur == 0 || fabs(sbis) < delta) return xcur;
    if (fabs(spre) > delta && fabs(fcur) < fabs(fpre)) {
      double stry;
      if (xpre == xblk) {
        stry = -fcur * (xcur - xpre) / (fcur - fpre);
      } else {
        const double dpre = (fpre - fcur) / (xpre - xcur);
        const double dblk = (fblk - fcur) / (xblk - xcur);
        stry = -fcur * (fblk * dblk - fpre * dpre) / (dblk * dpre * (fblk - fpre));
      }
      const double lim1 = fabs(spre), lim2 = 3 * fabs(sbis) - delta;
      if (2 * fabs(stry) < (lim1 < lim2 ? lim1 : lim2)) {
        spre = scur;
        scur = stry;
      } else {
        spre = sbis;
        scur = sbis;
      }
    } else {
      spre = sbis;
      scur = sbis;
    }
    xpre = xcur;
    fpre = fcur;
    if (fabs(scur) > delta)
      xcur += scur;
    else
      xcur += (sbis > 0 ? delta : -delta);
    fcur = interp1(xcur, ygrid, bs, ny) - bval;
  }
  return xcur;
}

// Unique root of the piecewise-linear bs(y) = bval when bs is non-decreasing north of its
// minimum.  sinv[k] = (y[k+1]-y[k])/(bs[k+1]-bs[k]) is tabulated with the surface scan.
PM_DEV double outcrop_monotone(double bval, const double* ygrid, const double* bs, const double* sinv, int ny,
                               int south) {
  if (bs[south] == bval) return ygrid[south];
  if (bs[ny - 1] == bval) return ygrid[ny - 1];
  int lo = south, hi = ny - 1;  // first index with bs >= bval lies in (south, ny-1]
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (bs[mid] >= bval)
      hi = mid;
    else
      lo = mid;
  }
  if (bs[hi] == bval) return ygrid[hi];
  return ygrid[hi - 1] + (bval - bs[hi - 1]) * sinv[hi - 1];
}

// np.mean(tau + 0*np.linspace(y0, yN, 100)) for a float tau (psi_SO.py:239): numpy's pairwise
// reduction of 100 equal terms (8 accumulators over 96 terms, tree combine, 4 trailing adds).
PM_DEV double mean100(double tau) {
  double r = tau;
  for (int k = 0; k < 11; ++k) r = r + tau;
  double res = ((r + r) + (r + r)) + ((r + r) + (r + r));
  for (int k = 0; k < 4; ++k) res = res + tau;
  return res / 100.0;
}

struct SoPar {
  double tau_ave, f, rho, L, KGM, smax;
  double pre0;  // tau_ave / f / rho * L (psi_SO.py:243, left to right), constant between launches
  const double *sill, *ektap, *toptap, *bottap;  // taper profiles (so_solve: lane-major in shared memory)
  const double* tau_y;                           // tau on the y grid (shared memory) or nullptr for a float tau
  double c;                                      // F2010 phase speed (BVP branch only)
  int with_Ek;
};
struct SoSurf {  // per-refresh scan of bs(y)
  double mn, bsN, y0, yN;
  int south;
  int ndown;  // grid intervals north of the minimum on which bs decreases (adjacent ones counted one by one)
  bool mono;  // ndown == 0
};
constexpr int kSawtoothSegments = 3;  // PMOC_ST_BS_SAWTOOTH: this many decreasing intervals north of the minimum
// block-cooperative copy of the four host-evaluated taper profiles into lane-major shared memory
template <int LPL>
PM_DEV void taper_fill(double* dst, const double* PM_RESTRICT sill, const double* PM_RESTRICT ektap,
                       const double* PM_RESTRICT toptap, const double* PM_RESTRICT bottap, int nz, int tid, int nthr) {
  const int nzp = 32 * LPL;
  for (int s = tid; s < nzp; s += nthr) {
    const int i = (s & 31) * LPL + (s >> 5);
    const bool in = i < nz;
    dst[s] = in ? sill[i] : 0.0;
    dst[nzp + s] = in ? ektap[i] : 0.0;
    dst[2 * nzp + s] = in ? toptap[i] : 0.0;
    dst[3 * nzp + s] = in ? bottap[i] : 0.0;
  }
}

// Scan of the surface buoyancy: minimum / argmin (first occurrence, np.argmin), monotonicity
// north of it, and the inverse segment slopes.  Warp-cooperative; redone only when bs changes.
PM_DEV SoSurf so_scan(const double* ygrid, const double* bs, double* sinv, int ny) {
  SoSurf s;
  {  // mn, south = first occurrence of the minimum, as the scan `if (bs[k] < mn)` from k = 0 finds it (a NaN
     // never wins unless it is bs[0]); lanes take k = lane, lane + 32, ..., then a warp arg-min
    double v = INFINITY;
    int idx = 0x7fffffff;
    for (int k = rt::lane(); k < ny; k += 32) {
      const double x = bs[k];
      if (x < v) { v = x; idx = k; }
    }
    for (int msk = 16; msk > 0; msk >>= 1) {
      const double ov = rt::shfl_xor(v, msk);
      const int oi = rt::shfl_i(idx, rt::lane() ^ msk);
      if (ov < v || (ov == v && oi < idx)) { v = ov; idx = oi; }
    }
    const double b0 = bs[0];
    const bool first = b0 != b0 || idx == 0x7fffffff;  // bs[0] is NaN, or nothing is below +inf
    s.mn = first ? b0 : v;
    s.south = first ? 0 : idx;
  }
  s.ndown = 0;
  for (int k0 = 0; k0 < ny - 1; k0 += 32) {  // (warp-uniform trip count)
    const int k = k0 + rt::lane();
    bool down = false;
    if (k < ny - 1) {
      const double db = bs[k + 1] - bs[k];
      sinv[k] = sdiv(ygrid[k + 1] - ygrid[k], db);
      down = k >= s.south && db < 0;
    }
    s.ndown += rt::popc(rt::ballot(down));
  }
  s.mono = s.ndown == 0;
  s.bsN = bs[ny - 1];
  s.y0 = ygrid[0];
  s.yN = ygrid[ny - 1];
  rt::syncwarp();
  return s;
}

// np.mean(tau(np.linspace(y0, yN, 100))) for tau given on the y grid (psi_SO.py:239):
// numpy's linspace (arange*step + start, last point = stop), np.interp and the pairwise
// reduction of 100 terms (8 accumulators over 96 terms, tree combine, 4 trailing adds).
PM_COLD double tau_mean100(double y0, double yN, const double* ygrid, const double* tau_y, int ny) {
  const double delta = yN - y0, step = delta / 99.0;
  double r[8];
  double res = 0.0;
  for (int p = 0; p < 100; ++p) {
    double yp;
    if (p == 99)
      yp = yN;
    else if (step == 0.0)
      yp = (double)p / 99.0 * delta + y0;
    else
      yp = (double)p * step + y0;
    const double v = interp1(yp, ygrid, tau_y, ny);
    if (p < 8) {
      r[p] = v;
    } else if (p < 96) {
      r[p & 7] = r[p & 7] + v;
    } else {
      if (p == 96) res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
      res = res + v;
    }
  }
  return res / 100.0;
}

// Propagators of u'' = (q0 + q1 s) u across cells of width h, by power series in s:
//   u(h) = A u(0) + B u'(0),  u'(h) = C u(0) + D u'(0),  A D - B C = 1.
// With t_k = a_k h^k the recurrence is t_{k+2} = (Q0 t_k + Q1 t_{k-1}) / ((k+2)(k+1)),
// Q0 = q0 h^2, Q1 = q1 h^3; Bh = B/h.  All terms are positive for a stable stratification.
//
// The trip count is fixed per call from Qmax = max over the warp of |Q0| + |Q1| (every term is bounded by
// Qmax^(k/2) / k!): the smallest multiple of three after which the tail is below 1e-18 of the sums, looked up in
// kSeriesQ.  No convergence test, no divide (1/((k+2)(k+1)) is tabulated) and no register moves (three terms per
// trip rotate through three registers) inside the loop: 9 FP64 instructions per term and level.
#ifdef PMOC_EMU
#define PM_CONST static const
#else
#define PM_CONST static __constant__
#endif
constexpr int kSeriesMax = 99;  // terms tabulated
PM_CONST double kSeriesInv[kSeriesMax] = {
    0.5, 0.16666666666666666, 0.083333333333333329, 0.050000000000000003,
    0.033333333333333333, 0.023809523809523808, 0.017857142857142856, 0.013888888888888888,
    0.011111111111111112, 0.0090909090909090905, 0.007575757575757576, 0.00641025641025641,
    0.0054945054945054949, 0.0047619047619047623, 0.0041666666666666666, 0.0036764705882352941,
    0.0032679738562091504, 0.0029239766081871343, 0.002631578947368421, 0.0023809523809523812,
    0.0021645021645021645, 0.001976284584980237, 0.0018115942028985507, 0.0016666666666666668,
    0.0015384615384615385, 0.0014245014245014246, 0.0013227513227513227, 0.0012315270935960591,
    0.0011494252873563218, 0.0010752688172043011, 0.0010080645161290322, 0.000946969696969697,
    0.00089126559714795004, 0.00084033613445378156, 0.00079365079365079365, 0.00075075075075075074,
    0.00071123755334281653, 0.00067476383265856947, 0.00064102564102564103, 0.00060975609756097561,
    0.00058072009291521487, 0.00055370985603543741, 0.00052854122621564484, 0.00050505050505050505,
    0.00048309178743961351, 0.00046253469010175765, 0.00044326241134751772, 0.00042517006802721087,
    0.00040816326530612246, 0.00039215686274509802, 0.00037707390648567121, 0.00036284470246734398,
    0.00034940600978336826, 0.00033670033670033672, 0.00032467532467532468, 0.00031328320802005011,
    0.00030248033877797946, 0.00029222676797194621, 0.0002824858757062147, 0.00027322404371584699,
    0.00026441036488630354, 0.00025601638504864311, 0.000248015873015873, 0.0002403846153846154,
    0.0002331002331002331, 0.00022614201718679331, 0.00021949078138718174, 0.00021312872975277067,
    0.00020703933747412008, 0.00020120724346076458, 0.00019561815336463224, 0.00019025875190258751,
    0.00018511662347278786, 0.00018018018018018018, 0.00017543859649122806, 0.00017088174982911826,
    0.0001665001665001665, 0.00016228497241155469, 0.00015822784810126583, 0.00015432098765432098,
    0.00015055706112616682, 0.00014692918013517486, 0.00014343086632243257, 0.00014005602240896358,
    0.00013679890560875513, 0.00013365410318096765, 0.00013061650992685477, 0.00012768130745658836,
    0.00012484394506866417, 0.0001221001221001221, 0.00011944577161968466, 0.0001168770453482936,
    0.00011439029970258523, 0.00011198208286674133, 0.00010964912280701755, 0.00010738831615120275,
    0.00010519671786240269, 0.00010307153164296021, 0.00010101010101010101,
};
constexpr int kSeriesSteps = 32;  // trip counts 6, 9, ..., 99
PM_CONST double kSeriesQ[kSeriesSteps] = {  // largest Qmax each trip count serves
    0.00021189593823687914, 0.0071126781656659097, 0.05976755391215325, 0.25608636817847191,
    0.7486299437050602, 1.7217046228815054, 3.3689509837018066, 5.8782970176865499,
    9.4238622023950125, 14.162597418420889, 20.233699163184948, 27.759474637795645,
    36.846863341635874, 47.589171919205832, 60.067791043705142, 74.353784497096072,
    90.509307286529619, 108.58884467139403, 128.64028121036503, 150.70581641647988,
    174.82274590618601, 201.02412660661238, 229.33934305261795, 259.79458981808773,
    292.41328307573838, 327.21641235557291, 364.22284185350316, 403.44956915011363,
    444.91194792769073, 488.62388020105715, 534.59798267940118, 582.84573112698445,
};

// number of three-term trips for a given Qmax (warp-uniform), 0 when the table does not reach (Qmax > 583)
PM_DEV int series_trips(double qmax) {
  int n = 0;
  for (int t = 0; t < kSeriesSteps; ++t)
    if (n == 0 && qmax <= kSeriesQ[t]) n = t + 2;
  return (qmax == qmax) ? n : 0;
}

template <int JC>
PM_DEV void cell_propagators_chunk(const double* Q0, const double* Q1, double* A, double* Bh, double* D, int trips) {
  double ax[JC], ay[JC], az[JC], bx[JC], by[JC], bz[JC], sa[JC], sb[JC], sd[JC], q0[JC], q1[JC];
  PM_UNROLL
  for (int j = 0; j < JC; ++j) {
    q0[j] = Q0[j]; q1[j] = Q1[j];
    ax[j] = 0.; ay[j] = 1.; az[j] = 0.;  // a-series: t_-1, t_0, t_1
    bx[j] = 0.; by[j] = 0.; bz[j] = 1.;  // b-series
    sa[j] = 1.; sb[j] = 1.; sd[j] = 1.;
  }
  for (int g = 0; g < trips; ++g) {
    const int k = 3 * g;
    const double i0 = kSeriesInv[k], i1 = kSeriesInv[k + 1], i2 = kSeriesInv[k + 2];
    const double c0 = (double)(k + 2), c1 = (double)(k + 3), c2 = (double)(k + 4);
    PM_UNROLL
    for (int j = 0; j < JC; ++j) {
      ax[j] = rt::fma(q0[j], ay[j], q1[j] * ax[j]) * i0;  // t_{k+2} from t_k (y), t_{k-1} (x)
      bx[j] = rt::fma(q0[j], by[j], q1[j] * bx[j]) * i0;
      sa[j] = sa[j] + ax[j]; sb[j] = sb[j] + bx[j]; sd[j] = rt::fma(c0, bx[j], sd[j]);
      ay[j] = rt::fma(q0[j], az[j], q1[j] * ay[j]) * i1;  // t_{k+3} from t_{k+1} (z), t_k (y)
      by[j] = rt::fma(q0[j], bz[j], q1[j] * by[j]) * i1;
      sa[j] = sa[j] + ay[j]; sb[j] = sb[j] + by[j]; sd[j] = rt::fma(c1, by[j], sd[j]);
      az[j] = rt::fma(q0[j], ax[j], q1[j] * az[j]) * i2;  // t_{k+4} from t_{k+2} (x), t_{k+1} (z)
      bz[j] = rt::fma(q0[j], bx[j], q1[j] * bz[j]) * i2;
      sa[j] = sa[j] + az[j]; sb[j] = sb[j] + bz[j]; sd[j] = rt::fma(c2, bz[j], sd[j]);
    }
  }
  PM_UNROLL
  for (int j = 0; j < JC; ++j) { A[j] = sa[j]; Bh[j] = sb[j]; D[j] = sd[j]; }
}

// the adaptive form (term-by-term convergence test), for cells beyond the table: N2 h^2 / c^2 > 583
template <int LPL>
PM_COLD bool cell_propagators_adaptive(const double (&Q0)[LPL], const double (&Q1)[LPL], double (&A)[LPL],
                                       double (&Bh)[LPL], double (&D)[LPL]) {
  double am[LPL], ak[LPL], an[LPL], bm[LPL], bk[LPL], bn[LPL];
  for (int j = 0; j < LPL; ++j) {
    am[j] = 0.; ak[j] = 1.; an[j] = 0.;
    bm[j] = 0.; bk[j] = 0.; bn[j] = 1.;
    A[j] = 1.; Bh[j] = 1.; D[j] = 1.;
  }
  for (int k = 0; k < 2000; ++k) {
    const double inv = rt::div_normal(1.0, (double)(k + 2) * (double)(k + 1)), kk = (double)(k + 2);
    bool big = false;
    for (int j = 0; j < LPL; ++j) {
      const double na = (Q0[j] * ak[j] + Q1[j] * am[j]) * inv;
      const double nb = (Q0[j] * bk[j] + Q1[j] * bm[j]) * inv;
      // (an overflowed sum is not converged: inf <= 1e-19 * inf would pass the test)
      big |= !((fabs(na) + fabs(an[j])) <= 1e-19 * fabs(A[j]) && fabs(A[j]) <= 1.79e308);
      big |= !((fabs(nb) + fabs(bn[j])) * kk <= 1e-19 * (fabs(Bh[j]) + fabs(D[j])) && fabs(D[j]) <= 1.79e308);
      A[j] = A[j] + na;
      Bh[j] = Bh[j] + nb;
      D[j] = D[j] + kk * nb;
      am[j] = ak[j]; ak[j] = an[j]; an[j] = na;
      bm[j] = bk[j]; bk[j] = bn[j]; bn[j] = nb;
    }
    if (k >= 3 && rt::ballot(big) == 0) return true;
  }
  return false;
}

template <int LPL>
PM_DEV bool cell_propagators(const double (&Q0)[LPL], const double (&Q1)[LPL], double (&A)[LPL], double (&Bh)[LPL],
                             double (&D)[LPL]) {
  double qm = 0.0;
  PM_UNROLL
  for (int j = 0; j < LPL; ++j) {
    const double q = fabs(Q0[j]) + fabs(Q1[j]);
    qm = (q > qm || q != q) ? q : qm;
  }
  qm = rt::wmax(qm);
  const int trips = series_trips(qm);
  if (trips == 0) return cell_propagators_adaptive<LPL>(Q0, Q1, A, Bh, D);
  // levels in chunks of at most four: 11 live doubles per level
  constexpr int JC = LPL <= 4 ? LPL : (LPL + 1) / 2;
  cell_propagators_chunk<JC>(Q0, Q1, A, Bh, D, trips);
  if constexpr (JC < LPL) cell_propagators_chunk<LPL - JC>(Q0 + JC, Q1 + JC, A + JC, Bh + JC, D + JC, trips);
  return true;
}

// F2010 smoother of Psi_GM (psi_SO.py:308-323): y'' = N2(z)/c^2 (y - T(z)), Dirichlet ends.
// N2 and T are piecewise linear on z (np.interp closures), so with u = y - T each cell obeys
// u'' = q(s) u exactly; matching y' at the nodes gives a symmetric tridiagonal system for the
// nodal values.  This is the converged solution of the ODE the reference hands to its
// adaptive, tol=1e-3 solve_bvp (SURVEY section 0 fact 2: stated tolerance 1e-5), so nothing here
// is tied to the reference's operation order: reciprocals and fused multiply-adds throughout.
//
// The tridiagonal system (rows = levels, LPL per lane) is solved by partitioning: every lane eliminates
// its first LPL-1 rows against the last unknown of the lane below (X_prev) and its own last unknown (X),
//   x_j = y_j - v_j X_prev - w_j X,
// its last row then couples X_prev, X and X_next only: a 32-row tridiagonal system, one row per lane,
// solved by parallel cyclic reduction (five shuffle rounds); the interior unknowns follow.  The system is
// a symmetric M-matrix (diagonally dominant: A, D >= 1), so are its Schur complements: no pivoting.
// In/out: g holds T on entry and the solution y on return (m^3/s).
template <int LPL>
PM_DEV void so_bvp(double (&g)[LPL], const double (&b)[LPL], double c, double ya, double yb, const double* zs, int nz,
                   unsigned* status) {
  static_assert(LPL >= 2, "partitioned solve: at least two levels per lane");
  const int Ln = rt::lane();
  const double rc2 = rt::div_normal(1.0, c * c);
  // N2 (psi_SO.py:154-160) at the own levels and at the level above
  const double bnext = rt::shfl_down(b[0], 1), bprev = rt::shfl_up(b[LPL - 1], 1);
  double n2[LPL], h[LPL], rh[LPL];
  PM_UNROLL
  for (int j = 0; j < LPL; ++j) {
    const int i = lev<LPL>(j);
    h[j] = i < nz - 1 ? zs[i + 1] - zs[i] : 1.0;
    rh[j] = rt::div_normal(1.0, h[j]);
  }
  const double rh_p = rt::shfl_up(rh[LPL - 1], 1), h_p = rt::shfl_up(h[LPL - 1], 1);
  PM_UNROLL
  for (int j = 0; j < LPL; ++j) {
    const int i = lev<LPL>(j);
    const double up = j < LPL - 1 ? b[j + 1 < LPL ? j + 1 : j] : bnext;
    const double dn = j > 0 ? b[j > 0 ? j - 1 : 0] : bprev;
    const double hd = j > 0 ? h[j > 0 ? j - 1 : 0] : h_p, rhd = j > 0 ? rh[j > 0 ? j - 1 : 0] : rh_p;
    double v = 0.0;
    if (i < nz) {
      if (i == 0)
        v = (up - b[j]) * rh[j];
      else if (i == nz - 1)
        v = (b[j] - dn) * rhd;
      else
        v = rt::div_normal(up - dn, h[j] + hd);
    }
    n2[j] = v;
  }
  const double n2next = rt::shfl_down(n2[0], 1), gnext = rt::shfl_down(g[0], 1);
  double Q0[LPL], Q1[LPL], Tp[LPL], A[LPL], Bh[LPL], D[LPL];
  PM_UNROLL
  for (int j = 0; j < LPL; ++j) {
    const int i = lev<LPL>(j);
    const bool cell = i < nz - 1;
    const double n2u = j < LPL - 1 ? n2[j + 1 < LPL ? j + 1 : j] : n2next;
    const double gu = j < LPL - 1 ? g[j + 1 < LPL ? j + 1 : j] : gnext;
    const double s = rc2 * (h[j] * h[j]);
    Q0[j] = cell ? n2[j] * s : 0.0;
    Q1[j] = cell ? (n2u - n2[j]) * s : 0.0;  // slope * h^3
    Tp[j] = cell ? (gu - g[j]) * rh[j] : 0.0;
  }
  if (!cell_propagators<LPL>(Q0, Q1, A, Bh, D)) *status |= 32u;
  double ib[LPL];
  PM_UNROLL
  for (int j = 0; j < LPL; ++j) ib[j] = rt::div_normal(rh[j], Bh[j]);  // 1 / (h Bh): h > 0, Bh >= 1
  const double ib_p = rt::shfl_up(ib[LPL - 1], 1), D_p = rt::shfl_up(D[LPL - 1], 1), Tp_p = rt::shfl_up(Tp[LPL - 1], 1);
  // rows: lo x_{i-1} + di x_i + up x_{i+1} = r (identity rows at the two ends and in the padding)
  double lo[LPL], di[LPL], up[LPL], r[LPL];
  PM_UNROLL
  for (int j = 0; j < LPL; ++j) {
    const int i = lev<LPL>(j);
    lo[j] = 0.; di[j] = 1.; up[j] = 0.; r[j] = 0.;
    if (i == 0)
      r[j] = ya - g[j];
    else if (i == nz - 1)
      r[j] = yb - g[j];
    else if (i < nz) {
      const double ibm = j > 0 ? ib[j > 0 ? j - 1 : 0] : ib_p, Dm = j > 0 ? D[j > 0 ? j - 1 : 0] : D_p;
      const double Tpm = j > 0 ? Tp[j > 0 ? j - 1 : 0] : Tp_p;
      lo[j] = -ibm;
      up[j] = -ib[j];
      di[j] = rt::fma(Dm, ibm, A[j] * ib[j]);
      r[j] = Tp[j] - Tpm;
    }
  }
  // interior rows 0 .. LPL-2 of the lane: Thomas with three right-hand sides (r, lo[0] e_first, up[n-1] e_last)
  constexpr int n = LPL - 1;
  double cp[n], y[n], v[n], w[n];
  {
    double pc = 0., py = 0., pv = 0.;
    PM_UNROLL
    for (int j = 0; j < n; ++j) {
      const double m = rt::div_normal(1.0, rt::fma(-lo[j], pc, di[j]));
      pc = up[j] * m;
      py = rt::fma(-lo[j], py, r[j]) * m;
      pv = (j == 0 ? lo[0] : -lo[j] * pv) * m;
      cp[j] = pc; y[j] = py; v[j] = pv;
    }
    // back substitution; w: the right-hand side up[n-1] e_last has forward image e_last * cp[n-1]
    w[n - 1] = cp[n - 1];
    PM_UNROLL
    for (int j = n - 2; j >= 0; --j) {
      y[j] = rt::fma(-cp[j], y[j + 1], y[j]);
      v[j] = rt::fma(-cp[j], v[j + 1], v[j]);
      w[j] = -cp[j] * w[j + 1];
    }
  }
  // interface row of the lane: a X_prev + bb X + cc X_next = d
  const double y0n = rt::shfl_down(y[0], 1), v0n = rt::shfl_down(v[0], 1), w0n = rt::shfl_down(w[0], 1);
  const double lol = lo[LPL - 1], upl = Ln < 31 ? up[LPL - 1] : 0.0;
  double a = -lol * v[n - 1];
  double bb = rt::fma(-upl, v0n, rt::fma(-lol, w[n - 1], di[LPL - 1]));
  double cc = -upl * w0n;
  double d = rt::fma(-upl, y0n, rt::fma(-lol, y[n - 1], r[LPL - 1]));
  PM_UNROLL
  for (int sft = 1; sft < 32; sft <<= 1) {  // parallel cyclic reduction
    const double am = rt::shfl_up(a, sft), bm = rt::shfl_up(bb, sft), cm = rt::shfl_up(cc, sft), dm = rt::shfl_up(d, sft);
    const double ap = rt::shfl_down(a, sft), bp = rt::shfl_down(bb, sft), cq = rt::shfl_down(cc, sft),
                 dp = rt::shfl_down(d, sft);
    const bool hm = Ln >= sft, hp = Ln + sft < 32;
    const double al = hm ? -a * rt::div_normal(1.0, bm) : 0.0, ga = hp ? -cc * rt::div_normal(1.0, bp) : 0.0;
    bb = rt::fma(ga, ap, rt::fma(al, cm, bb));
    d = rt::fma(ga, dp, rt::fma(al, dm, d));
    a = al * am;
    cc = ga * cq;
  }
  const double X = d * rt::div_normal(1.0, bb);
  double Xp = rt::shfl_up(X, 1);
  if (Ln == 0) Xp = 0.0;
  PM_UNROLL
  for (int j = 0; j < n; ++j) {
    if (lev<LPL>(j) < nz) g[j] = g[j] + rt::fma(-w[j], X, rt::fma(-v[j], Xp, y[j]));
  }
  if (lev<LPL>(LPL - 1) < nz) g[LPL - 1] = g[LPL - 1] + X;
}

// ys(b) for all levels of the lane at once when bs(y) is non-decreasing north of its minimum
// (outcrop_monotone, but branch-free with a fixed trip count so that the LPL searches overlap)
template <int LPL>
PM_DEV void outcrop_monotone_all(double (&yo)[LPL], const double (&b)[LPL], const double* ygrid, const double* bs,
                                 const double* sinv, int ny, const SoSurf& S) {
  int lo[LPL], hi[LPL];
  PM_UNROLL
  for (int j = 0; j < LPL; ++j) {
    lo[j] = S.south;
    hi[j] = ny - 1;
  }
  int span = ny - 1 - S.south, trips = 0;
  while ((1 << trips) < span) ++trips;
  for (int it = 0; it < trips; ++it) {
    PM_UNROLL
    for (int j = 0; j < LPL; ++j) {
      const int mid = (lo[j] + hi[j]) >> 1;
      const bool open = hi[j] - lo[j] > 1, ge = bs[mid] >= b[j];
      hi[j] = (open && ge) ? mid : hi[j];
      lo[j] = (open && !ge) ? mid : lo[j];
    }
  }
  const double bsS = bs[S.south], yS = ygrid[S.south];
  PM_UNROLL
  for (int j = 0; j < LPL; ++j) {
    const int h = hi[j];
    double y = ygrid[h - 1] + (b[j] - bs[h - 1]) * sinv[h - 1];
    if (bs[h] == b[j]) y = ygrid[h];
    if (S.bsN == b[j]) y = S.yN;
    if (bsS == b[j]) y = yS;
    if (b[j] > S.bsN) y = S.yN;
    if (b[j] < S.mn) y = S.y0 - 1e3;
    yo[j] = y;
  }
}

// One level of Psi_SO's explicit branch (psi_SO.py:302-354) for the member's parameters P: level i, taper slot s.
// Shared by so_solve and the block-per-member diagnosis.  exact1 is set when at level 1, with a wind stress
// independent of y, the slope clip or the limiter chose a value made of the member's constants only: Psi_so[1] is
// then reproduced bit for bit whatever the state (PMOC_ST_CARRY_SO1_EXACT).
// Ekman transport, Sv (pre = tau / f / rho * L)
PM_DEV double so_ekman(double pre, const SoPar& P, int s) {
  return div_const(pre * P.sill[s] * P.ektap[s], 1e6, 1.0 / 1e6);
}
// GM transport with the slope sl = z / dy clipped at -smax, before the limiter
PM_DEV double so_gm_clip(double sl, const SoPar& P, int s, int i, bool& exact1) {
  const double ms = -P.smax;
  const double mx = (sl >= ms || sl != sl) ? sl : ms;
  const double g = P.KGM * mx * P.L * P.toptap[s] * P.bottap[s];
  if (i == 1 && !(sl >= ms || sl != sl) && P.tau_y == nullptr) exact1 = true;  // the slope clip: constants only
  return g;
}
// the limiter where the outcrop lies south of the channel (dy > span = yN - y0): GM >= -Ek; then GM in Sv
PM_DEV double so_gm_limit(double gm, double ek, double dy, double span, const SoPar& P, int i, bool& exact1) {
  if (dy > span) {
    const double alt = -ek * 1e6;
    if (i == 1 && !(gm >= alt || gm != gm) && P.tau_y == nullptr) exact1 = true;  // Psi = Ek - (Ek*1e6)/1e6
    gm = (gm >= alt || gm != gm) ? gm : alt;
  }
  return div_const(gm, 1e6, 1.0 / 1e6);
}

// Psi_SO.solve (psi_SO.py:106-140, 218-243, 302-354): outcrop latitudes, Ekman transport, GM
// transport with the explicit slope clip or (BVP) the F2010 smoother.  Sv.  The four taper
// profiles are read lane-major (slot lm(j)) from P.sill/ektap/toptap/bottap.
template <int LPL, bool BVP = false>
PM_DEV void so_solve(double (&psi)[LPL], double (&ek)[LPL], double (&gm)[LPL], double (&ysv)[LPL],
                     const double (&b)[LPL], const double* ygrid, const double* bs, const double* sinv, int ny,
                     const SoSurf& S, const SoPar& P, const double* zs, int nz, unsigned* status,
                     bool* psi1_exact = nullptr) {
  const double pre0 = P.pre0;
  if (S.mono && S.south < ny - 1) {
    outcrop_monotone_all<LPL>(ysv, b, ygrid, bs, sinv, ny, S);
  } else {
    if (!S.mono) *status |= 2u;
    if (S.ndown >= kSawtoothSegments) *status |= 256u;  // PMOC_ST_BS_SAWTOOTH
    PM_UNROLL
    for (int j = 0; j < LPL; ++j) {  // (registers: must stay unrolled; the heavy callee is out of line)
      const double bi = b[j];
      double yo = 0.;
      if (lev<LPL>(j) < nz) {
        if (bi < S.mn)
          yo = S.y0 - 1e3;
        else if (bi > S.bsN)
          yo = S.yN;
        else if (S.mono)
          yo = outcrop_monotone(bi, ygrid, bs, sinv, ny, S.south);
        else {
          bool bad = false;
          yo = outcrop_brent(bi, ygrid, bs, ny, S.south, &bad);
          if (bad) *status |= 4u;
        }
      }
      ysv[j] = yo;
    }
  }
  double dyv[LPL], prev[LPL];
  bool exact1 = false;  // level 1: Psi = Ek + GM came out of state-independent arithmetic (see PMOC_ST_CARRY_SO1_EXACT)
  PM_UNROLL
  for (int j = 0; j < LPL; ++j) prev[j] = pre0;
  if (P.tau_y != nullptr) {  // tau on the y grid: a 100-point mean and two divides per level (kept out of the float-tau path)
    PM_UNROLL
    for (int j = 0; j < LPL; ++j)
      if (lev<LPL>(j) < nz) prev[j] = tau_mean100(ysv[j], S.yN, ygrid, P.tau_y, ny) / P.f / P.rho * P.L;
  }
  PM_UNROLL
  for (int j = 0; j < LPL; ++j) {
    const int i = lev<LPL>(j), s = lm(j);
    const bool in = i < nz;
    const double yo = in ? ysv[j] : 0.0;
    const double e = so_ekman(prev[j], P, s);
    double dy = S.yN - yo;
    dy = 0.1 > dy ? 0.1 : dy;
    const double z = zs[i < nz ? i : nz - 1];
    double g;
    if (BVP)
      g = rt::div_normal(P.KGM * z, dy) * P.L * P.toptap[s] * P.bottap[s];  // dy >= 0.1
    else
      g = so_gm_clip(rt::div_normal(z, dy), P, s, i, exact1);  // dy >= 0.1, |z| <= H: in range
    ek[j] = in ? e : 0.0;
    gm[j] = in ? g : 0.0;
    dyv[j] = in ? dy : 1.0;
    ysv[j] = yo;
  }
  if (BVP) {
    double ya = 0., yb = 0.;
    if (P.with_Ek) {  // bc_GM, psi_SO.py:270-275
      ya = -(get_level<LPL>(ek, 0) * 1e6);
      yb = -(get_level<LPL>(ek, nz - 1) * 1e6);
    }
    so_bvp<LPL>(gm, b, P.c, ya, yb, zs, nz, status);
  }
  PM_UNROLL
  for (int j = 0; j < LPL; ++j) {
    const int i = lev<LPL>(j);
    const double g = so_gm_limit(gm[j], ek[j], dyv[j], S.yN - S.y0, P, i, exact1);
    const bool in = i < nz;
    gm[j] = in ? g : 0.0;
    psi[j] = (in && i != 0) ? ek[j] + g : 0.0;
  }
  if (psi1_exact != nullptr) *psi1_exact = rt::ballot(exact1) != 0;
}

// ====================================================================== SO_ML
// Southern-Ocean mixed layer (SO_ML.py:198-303).  The ny <= 64 surface points are spread
// two per lane (point k lives in lane k/2); everything below is warp-cooperative.
constexpr int kMLP = 2;
constexpr int kMaxNyMl = 32 * kMLP;

// numpy/_core/src/multiarray/compiled_base.c: binary_search_with_guess, statement for
// statement.  For a sorted `arr` the result does not depend on `guess`; for an unsorted
// one (np.interp with a non-monotone b_basin as abscissa, SURVEY a15) it does, and the
// reference's answer is reproduced only by carrying the guess from query to query.
template <class XP>
PM_DEV int search_guess(double key, XP arr, int len, int guess) {
  constexpr int kLikelyInCache = 8;
  int imin = 0, imax = len;
  if (key > arr[len - 1]) return len;
  if (key < arr[0]) return -1;
  if (len <= 4) {
    int i = 1;
    for (; i < len && key >= arr[i]; ++i) {}
    return i - 1;
  }
  if (guess > len - 3) guess = len - 3;
  if (guess < 1) guess = 1;
  if (key < arr[guess]) {
    if (key < arr[guess - 1]) {
      imax = guess - 1;
      if (guess > kLikelyInCache && key >= arr[guess - kLikelyInCache]) imin = guess - kLikelyInCache;
    } else {
      return guess - 1;
    }
  } else {
    if (key < arr[guess + 1]) return guess;
    if (key < arr[guess + 2]) return guess + 1;
    imin = guess + 2;
    if (guess < len - kLikelyInCache - 1 && key < arr[guess + kLikelyInCache]) imax = guess + kLikelyInCache;
  }
  while (imin < imax) {
    const int imid = imin + ((imax - imin) >> 1);
    if (key >= arr[imid])
      imin = imid + 1;
    else
      imax = imid;
  }
  return imin - 1;
}

// value of np.interp(x, xp, fp) once arr_interp's search has returned index k
template <class XP>
PM_DEV double interp_at(double x, XP xp, const double* fp, int n, int k) {
  if (x != x) return x;
  if (k == -1) return fp[0];
  if (k == n) return fp[n - 1];
  if (k == n - 1) return fp[k];
  if (xp[k] == x) return fp[k];
  const double slope = sdiv(fp[k + 1] - fp[k], xp[k + 1] - xp[k]);
  double res = slope * (x - xp[k]) + fp[k];
  if (res != res) {
    res = slope * (x - xp[k + 1]) + fp[k + 1];
    if (res != res && fp[k] == fp[k + 1]) res = fp[k];
  }
  return res;
}

// np.interp(x, xp, fp) for a non-decreasing xp with the index of the previous time step as a first
// guess: j is the last index with xp[j] <= x (what numpy's search returns for a sorted abscissa
// whatever its own guess was), so a verified guess and the binary search agree.
template <class XP>
PM_DEV double interp1_guess(double x, XP xp, const double* fp, int n, int& guess) {
  if (x != x) return x;
  if (x >= xp[n - 1]) return fp[n - 1];  // x == xp[n-1]: the search returns n-1 and arr_interp returns fp[n-1]
  if (x < xp[0]) return fp[0];
  int j = guess < 0 ? 0 : (guess > n - 2 ? n - 2 : guess);
  if (!(xp[j] <= x && x < xp[j + 1])) {
    // the state drifts: try the two neighbouring intervals before searching
    const int up = j + 1 < n - 1 ? j + 1 : j, dn = j > 0 ? j - 1 : 0;
    if (xp[up] <= x && x < xp[up + 1])
      j = up;
    else if (xp[dn] <= x && x < xp[dn + 1])
      j = dn;
    else
      j = search_le(xp, n, x);
  }
  guess = j;
  return interp_at(x, xp, fp, n, j);
}

// natural-order array stored with one pad word after every 2^sh entries (conflict-free for writers that
// own 2^sh consecutive entries each); reads like a pointer
struct PadIdx {
  const double* p;
  int sh;
  PM_DEV double operator[](int i) const { return p[i + (i >> sh)]; }
};

struct MlState {
  double bs[kMLP];                            // surface buoyancy of the lane's points
  int jp[kMLP];                               // np.interp search results of the previous step (predictions)
  double ps[kMLP];                            // Psi_s of the last step (diagnostic)
  double a[kMLP], m[kMLP];                    // Thomas factors of U = tridiag(-s/2, 1+s, -s/2)
  double sfh[kMLP], rv[kMLP], brest[kMLP];    // surflux/h, rest_mask*v_pist/h, b_rest
  double shalf, sdiag;                        // s/2, 1-s
  double h, rh, L, rL, dy, rdy;
  int ny;
  int first_pos;                              // np.argwhere(Psi_b > 0)[0][0], -1 if none
  const double* scan;                         // lane-major [10][32] scan multipliers (shared memory)
};

PM_DEV int mlk(int e) { return rt::lane() * kMLP + e; }

// MlState <-> shared memory (kMlSave doubles owned by the warp), for kernels whose mixed-layer warp
// also carries column state in registers: the mixed layer is parked between its steps.
constexpr int kMlSave = 16 * 32 + 12;
PM_DEV void ml_park(const MlState& S, double* sm, bool all) {
  const int Ln = rt::lane();
  PM_UNROLL
  for (int e = 0; e < kMLP; ++e) {
    sm[(0 + e) * 32 + Ln] = S.bs[e];
    sm[(2 + e) * 32 + Ln] = (double)S.jp[e];
    sm[(4 + e) * 32 + Ln] = S.ps[e];
    if (all) {
      sm[(6 + e) * 32 + Ln] = S.a[e];
      sm[(8 + e) * 32 + Ln] = S.m[e];
      sm[(10 + e) * 32 + Ln] = S.sfh[e];
      sm[(12 + e) * 32 + Ln] = S.rv[e];
      sm[(14 + e) * 32 + Ln] = S.brest[e];
    }
  }
  if (all && Ln == 0) {
    double* u = sm + 16 * 32;
    u[0] = S.shalf; u[1] = S.sdiag; u[2] = S.h; u[3] = S.rh; u[4] = S.L; u[5] = S.rL; u[6] = S.dy; u[7] = S.rdy;
    u[8] = (double)S.ny; u[9] = (double)S.first_pos;
  }
  rt::syncwarp();
}
PM_DEV void ml_unpark(MlState& S, const double* sm, const double* scan) {
  const int Ln = rt::lane();
  PM_UNROLL
  for (int e = 0; e < kMLP; ++e) {
    S.bs[e] = sm[(0 + e) * 32 + Ln];
    S.jp[e] = (int)sm[(2 + e) * 32 + Ln];
    S.ps[e] = sm[(4 + e) * 32 + Ln];
    S.a[e] = sm[(6 + e) * 32 + Ln];
    S.m[e] = sm[(8 + e) * 32 + Ln];
    S.sfh[e] = sm[(10 + e) * 32 + Ln];
    S.rv[e] = sm[(12 + e) * 32 + Ln];
    S.brest[e] = sm[(14 + e) * 32 + Ln];
  }
  const double* u = sm + 16 * 32;
  S.shalf = u[0]; S.sdiag = u[1]; S.h = u[2]; S.rh = u[3]; S.L = u[4]; S.rL = u[5]; S.dy = u[6]; S.rdy = u[7];
  S.ny = (int)u[8]; S.first_pos = (int)u[9];
  S.scan = scan;
}

// State-independent part of SO_ML: flux factors and the factorisation of the Crank-Nicolson
// matrix (SO_ML.py:155-165, 191-196).  inv(U).V.bs is evaluated as a Thomas solve whose two
// first-order recurrences run as warp scans; the multipliers of the scan levels are
// tabulated here (scan_s: 10*32 doubles of shared memory owned by this warp).
PM_DEV void ml_setup(MlState& S, const double* ygrid, int ny, double Ks, double h, double L, double vpist,
                     const double* PM_RESTRICT surflux, const double* PM_RESTRICT rest_mask,
                     const double* PM_RESTRICT b_rest, double dt, double* scan_s) {
  S.ny = ny;
  S.h = h; S.rh = 1.0 / h;
  S.L = L; S.rL = 1.0 / L;
  S.dy = ygrid[1] - ygrid[0];
  S.rdy = 1.0 / S.dy;
  const double s = Ks * dt / (S.dy * S.dy);
  S.shalf = s / 2.;
  S.sdiag = 1 - s;
  S.first_pos = -1;
  PM_UNROLL
  for (int e = 0; e < kMLP; ++e) {
    const int k = mlk(e);
    const bool in = k < ny;
    S.sfh[e] = in ? surflux[k] / h : 0.0;
    S.rv[e] = in ? rest_mask[k] * vpist / h : 0.0;
    S.brest[e] = in ? b_rest[k] : 0.0;
    S.a[e] = 0.0;
    S.m[e] = in ? 1.0 : 0.0;  // identity rows (first, last); padding contributes nothing
    S.ps[e] = 0.0;
    S.jp[e] = 0;
  }
  double aprev = 0.0;
  for (int i = 1; i < ny - 1; ++i) {
    const double mi = 1. / ((1 + s) - S.shalf * aprev);
    aprev = S.shalf * mi;
    PM_UNROLL
    for (int e = 0; e < kMLP; ++e)
      if (mlk(e) == i) {
        S.m[e] = mi;
        S.a[e] = aprev;
      }
  }
  // lane composites: forward y_last = A*y_prev + C, backward x_first = A*x_next + D (same product)
  const int Ln = rt::lane();
  double F = S.a[0] * S.a[1], B = F;
  int lvl = 0;
  for (int d = 1; d < 32; d <<= 1, ++lvl) {
    scan_s[lvl * 32 + Ln] = Ln >= d ? F : 0.0;
    scan_s[(5 + lvl) * 32 + Ln] = Ln + d < 32 ? B : 0.0;
    const double fo = rt::shfl_up(F, d), bo = rt::shfl_down(B, d);
    if (Ln >= d) F = F * fo;
    if (Ln + d < 32) B = B * bo;
  }
  S.scan = scan_s;
  rt::syncwarp();
}

// np.argmin(bs): first occurrence of the minimum, a NaN wins (first NaN).  The doubles are mapped to
// unsigned keys of the same order (-0.0 counted as +0.0, as `<` does) and reduced 32 bits at a time
// with the warp min-reduction; the lowest point index holding the minimum is the answer.
PM_DEV int ml_argmin(const MlState& S) {
  unsigned hi[kMLP], lo[kMLP];
  bool nan = false;
  PM_UNROLL
  for (int e = 0; e < kMLP; ++e) {
    const double x = S.bs[e] + 0.0;
    unsigned long long b;
    static_assert(sizeof(b) == sizeof(x), "binary64");
    memcpy(&b, &x, 8);
    b = (b >> 63) ? ~b : (b | 0x8000000000000000ull);
    const bool in = mlk(e) < S.ny;
    hi[e] = in ? (unsigned)(b >> 32) : 0xffffffffu;
    lo[e] = in ? (unsigned)b : 0xffffffffu;
    nan |= in && x != x;
  }
  if (rt::ballot(nan)) {
    int first = 0x7fffffff;
    PM_UNROLL
    for (int e = kMLP - 1; e >= 0; --e)
      if (mlk(e) < S.ny && S.bs[e] != S.bs[e]) first = mlk(e);
    return rt::min_i(first);
  }
  unsigned h = hi[0];
  PM_UNROLL
  for (int e = 1; e < kMLP; ++e) h = hi[e] < h ? hi[e] : h;
  const unsigned hmin = rt::min_u(h);
  unsigned l = 0xffffffffu;
  PM_UNROLL
  for (int e = 0; e < kMLP; ++e)
    if (hi[e] == hmin && lo[e] < l) l = lo[e];
  const unsigned lmin = rt::min_u(l);
  int idx = 0x7fffffff;
  PM_UNROLL
  for (int e = kMLP - 1; e >= 0; --e)
    if (hi[e] == hmin && lo[e] == lmin && mlk(e) < S.ny) idx = mlk(e);
  return rt::min_i(idx);
}

template <class XP>
PM_DEV void ml_south_bc(MlState& S, double ps1, XP bb_s, unsigned* status) {
  // SO_ML.py:93-98
  if (rt::lane() == 0) {
    if (ps1 > 0) {
      if (S.first_pos >= 0)
        S.bs[0] = bb_s[S.first_pos];
      else
        *status |= 16u;  // the reference raises IndexError here
    } else {
      S.bs[0] = S.bs[1];
    }
  }
}

// SO_ML.advdiff (SO_ML.py:228-274) for one step.  bb_s: b_basin, pm_s: Psi_mod (Psi_b with the
// leading zeros replaced, SO_ML.py:228-230), both natural order in shared memory; bs_s: scratch
// [ny] of this warp.  `sorted`: b_basin is non-decreasing (warp-uniform).
template <class XP>
PM_DEV void ml_step(MlState& S, XP bb_s, const double* pm_s, int nz, bool sorted, double* bs_s, double dt,
                    unsigned* status) {
  const int ny = S.ny, Ln = rt::lane();
  (void)bs_s;
  double ps[kMLP] = {0., 0.};
  if (sorted) {
    PM_UNROLL
    for (int e = 0; e < kMLP; ++e)
      if (mlk(e) < ny) ps[e] = interp1_guess(S.bs[e], bb_s, pm_s, nz, S.jp[e]);
  } else {
    // PMOC_ST_XP_NONMONOTONE: numpy's search carries its result into the next query as the guess
    // (j_k = search_guess(x_k, j_{k-1}), j_{-1} = 0), and for an unsorted abscissa the answer depends
    // on it.  The chain is evaluated speculatively: every lane searches with the guess its
    // predecessor produced in the previous time step, then the guesses actually used are compared
    // with the results actually obtained and the pass repeats until they agree -- which is exactly
    // the sequential chain (lane 0 is always right, each pass fixes at least one more lane), and
    // is one pass when the state moves slowly.
    *status |= 8u;
    int pred = rt::shfl_i(S.jp[kMLP - 1], Ln > 0 ? Ln - 1 : 0);
    int j0 = 0, j1 = 0;
    for (int pass = 0; pass < 33; ++pass) {
      const int g0 = Ln == 0 ? 0 : pred;
      j0 = (mlk(0) < ny && S.bs[0] == S.bs[0]) ? search_guess(S.bs[0], bb_s, nz, g0) : g0;
      j1 = (mlk(1) < ny && S.bs[1] == S.bs[1]) ? search_guess(S.bs[1], bb_s, nz, j0) : j0;
      const int got = rt::shfl_i(j1, Ln > 0 ? Ln - 1 : 0);
      const bool bad = Ln > 0 && got != pred;
      pred = got;
      if (rt::ballot(bad) == 0) break;
    }
    S.jp[0] = j0;
    S.jp[1] = j1;
    if (mlk(0) < ny) ps[0] = interp_at(S.bs[0], bb_s, pm_s, nz, j0);
    if (mlk(1) < ny) ps[1] = interp_at(S.bs[1], bb_s, pm_s, nz, j1);
  }
  const int amin = ml_argmin(S);
  PM_UNROLL
  for (int e = 0; e < kMLP; ++e)
    if (mlk(e) < amin || mlk(e) == 0) ps[e] = 0.0;
  const double ps1 = rt::shfl(ps[1], 0);
  ml_south_bc(S, ps1, bb_s, status);
  // tendencies (SO_ML.py:124-134, 250-259)
  double prev[kMLP], next[kMLP];
  prev[0] = rt::shfl_up(S.bs[1], 1);
  next[0] = S.bs[1];
  prev[1] = S.bs[0];
  next[1] = rt::shfl_down(S.bs[0], 1);
  PM_UNROLL
  for (int e = 0; e < kMLP; ++e) {
    const int k = mlk(e);
    const double flux = S.sfh[e] + S.rv[e] * (S.brest[e] - S.bs[e]);
    double adv = 0.0;
    if (k >= 1 && k < ny - 1) {
      double t = 0.0;
      bool on = false;
      if (ps[e] < 0.) {
        t = -ps[e] * 1e6 * (next[e] - S.bs[e]);
        on = true;
      } else if (ps[e] > 0.) {
        t = -ps[e] * 1e6 * (S.bs[e] - prev[e]);
        on = true;
      }
      if (on) adv = div_const(div_const(div_const(t, S.h, S.rh), S.L, S.rL), S.dy, S.rdy);
    }
    if (k < ny) S.bs[e] = S.bs[e] + dt * (flux + adv);
    S.ps[e] = ps[e];
  }
  if (Ln == 0 && ps1 <= 0) S.bs[0] = S.bs[1];
  // Crank-Nicolson diffusion: rhs = V.bs, then U x = rhs by a scanned Thomas solve
  prev[0] = rt::shfl_up(S.bs[1], 1);
  next[0] = S.bs[1];
  prev[1] = S.bs[0];
  next[1] = rt::shfl_down(S.bs[0], 1);
  double c[kMLP];
  PM_UNROLL
  for (int e = 0; e < kMLP; ++e) {
    const int k = mlk(e);
    double r = S.bs[e];
    if (k >= 1 && k < ny - 1) r = S.shalf * prev[e] + S.sdiag * S.bs[e] + S.shalf * next[e];
    c[e] = k < ny ? r * S.m[e] : 0.0;
  }
  double C = rt::fma(S.a[1], c[0], c[1]);
  int lvl = 0;
  for (int d = 1; d < 32; d <<= 1, ++lvl) {
    const double o = rt::shfl_up(C, d);
    C = rt::fma(S.scan[lvl * 32 + Ln], Ln >= d ? o : 0.0, C);
  }
  double yprev = rt::shfl_up(C, 1);
  if (Ln == 0) yprev = 0.0;
  const double dp0 = rt::fma(S.a[0], yprev, c[0]);
  const double dp1 = rt::fma(S.a[1], dp0, c[1]);
  double D = rt::fma(S.a[0], dp1, dp0);
  lvl = 0;
  for (int d = 1; d < 32; d <<= 1, ++lvl) {
    const double o = rt::shfl_down(D, d);
    D = rt::fma(S.scan[(5 + lvl) * 32 + Ln], Ln + d < 32 ? o : 0.0, D);
  }
  double xnext = rt::shfl_down(D, 1);
  if (Ln == 31) xnext = 0.0;
  const double x1 = rt::fma(S.a[1], xnext, dp1);
  const double x0 = rt::fma(S.a[0], x1, dp0);
  if (mlk(0) < ny) S.bs[0] = x0;
  if (mlk(1) < ny) S.bs[1] = x1;
  ml_south_bc(S, ps1, bb_s, status);
}

// Psi_b -> what ml_step needs: Psi_mod in shared memory (natural order) and the first level
// with Psi_b > 0 (SO_ML.py:94, 228-230).  Returns false when Psi_b has no non-zero entry
// (np.nonzero(...)[0][0] raises IndexError in the reference).
template <int LPL>
PM_DEV bool ml_bind_psi(MlState& S, const double (&psi_b)[LPL], int nz, double* pm_s) {
  int fnz = 0x7fffffff, fpos = 0x7fffffff;
  PM_UNROLL
  for (int j = LPL - 1; j >= 0; --j) {
    const int i = lev<LPL>(j);
    if (i < nz) {
      if (psi_b[j] != 0.0) fnz = i;
      if (psi_b[j] > 0.0) fpos = i;
    }
  }
  fnz = rt::min_i(fnz);
  fpos = rt::min_i(fpos);
  S.first_pos = fpos == 0x7fffffff ? -1 : fpos;
  const bool ok = fnz != 0x7fffffff;
  const double held = ok ? get_level<LPL>(psi_b, fnz) : 0.0;
  PM_UNROLL
  for (int j = 0; j < LPL; ++j) {
    const int i = lev<LPL>(j);
    if (i < nz) pm_s[i] = i < fnz ? held : psi_b[j];
  }
  rt::syncwarp();
  return ok;
}

// b_basin registers -> shared memory (natural order) + is it non-decreasing?
template <int LPL>
PM_DEV bool ml_bind_basin(const double (&b)[LPL], int nz, double* bb_s) {
  const double bnext = rt::shfl_down(b[0], 1);
  bool bad = false;
  PM_UNROLL
  for (int j = 0; j < LPL; ++j) {
    const int i = lev<LPL>(j);
    if (i < nz) bb_s[i] = b[j];
    if (i < nz - 1) {
      const double up = j < LPL - 1 ? b[j + 1 < LPL ? j + 1 : j] : bnext;
      bad |= !(up >= b[j]);
    }
  }
  const bool sorted = rt::ballot(bad) == 0;  // ballot also orders the stores before the reads
  rt::syncwarp();
  return sorted;
}

// ---- the 'jn' bottom-boundary switches (run_JansenNadeau_2018.py:233-254), shared by the warp- and block-per-member
// kernels.  psi_so1, res_b1, res_n1: Psi[1] of Psi_SO, Psi_iso_b and Psi_iso_n; bb0, bb1 / nb0, nb1: levels 0 and 1
// of the basin / northern column before the step; bs0: bs[0] of the mixed layer.
//
// Which of psi_so1, res_b1, res_n1 are rounding noise (bits 0, 1, 2): non-zero and below 1e-12 of mx, the largest
// |Psi| of the three streamfunctions.  psi_so1 is exempt when so1_exact: it came out of state-independent arithmetic
// (PMOC_ST_CARRY_SO1_EXACT).
PM_DEV unsigned jn_noise(double psi_so1, double res_b1, double res_n1, double mx, bool so1_exact) {
  const double tiny = 1e-12 * mx, s1 = fabs(psi_so1), s2 = fabs(res_b1), s3 = fabs(res_n1);
  return ((s1 > 0 && s1 < tiny && !so1_exact) ? 1u : 0u) | ((s2 > 0 && s2 < tiny) ? 2u : 0u) |
         ((s3 > 0 && s3 < tiny) ? 4u : 0u);
}
// the basin's bottom value and kappa variant (both kept when no branch applies, e.g. for a NaN psi_so1)
PM_DEV void jn_switch_basin(double psi_so1, double res_b1, double bb1, double nb0, double bs0, double& bbot, int& var) {
  if (psi_so1 < 0) {
    bbot = bs0;
    var = 1;
  }
  if (res_b1 > 0 && nb0 < bb1 && nb0 < bs0) {
    bbot = nb0;
    var = 1;
  } else if (psi_so1 >= 0) {
    bbot = bb1;
    var = 0;
  }
}
// the northern column's bottom value and kappa variant
PM_DEV void jn_switch_north(double res_n1, double bb0, double nb1, double& bbot, int& var) {
  if (res_n1 < 0 && bb0 < nb1) {
    bbot = bb0;
    var = 1;
  } else {
    bbot = nb1;
    var = 0;
  }
}
// PMOC_ST_NOISE_SWITCH when the outcome of a switch hung on the sign of a noise value (the other operands let it through)
PM_DEV void jn_noise_hit(unsigned noise, double bb0, double bb1, double nb0, double nb1, double bs0, unsigned* status) {
  if (noise != 0 && ((noise & 1u) || ((noise & 2u) && nb0 < bb1 && nb0 < bs0) || ((noise & 4u) && bb0 < nb1)))
    *status |= 64u;  // PMOC_ST_NOISE_SWITCH
}

}  // namespace pm
