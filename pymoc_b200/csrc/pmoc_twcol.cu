// Column + Psi_Thermwind against a fixed northern profile (examples/example_timestepping.py:17-80, BASELINE
// configs[0]), several members per warp.
//
// With 70 levels a warp-per-member mapping leaves a quarter of the lanes idle and pays two 5-stage warp scans, the
// neighbour shuffles and every warp-uniform instruction for ONE member per step -- and this loop re-diagnoses the
// thermal wind every step (K = 1).  Here a member owns an aligned group of G = 8 or 16 lanes (LPL <= 9 levels per
// lane): four or two members per warp share each instruction, the scans take log2 G stages, and the double
// quadrature of Psi'' = (b2 - b1)/f (psi_thermwind.py:123-135) is written for the piecewise-linear profiles it is
// exact for -- trapezoid for Psi', h I1 + h^2 (g_i/3 + g_{i+1}/6) for Psi -- with every state-independent factor
// tabulated: 10 FP64 instructions per level instead of 36.  Same closed form as pm::tw_solve, different association
// (relative difference ~1e-16; C1 has no threshold on Psi).  The column step is the folded stencil of pm::col_step.
// Columns with convection or a gradient bottom condition, other topologies and nz > 144 take the generic kernel.
#include "pmoc_common.cuh"

#include <type_traits>

namespace pmk {

struct TwColArgs {
  pmoc_model m;
  long long it0, nsteps;
  int diagnose_only;
  MemberList list;
};

// Shared memory of k_twcol (in doubles).  Per block: nine level tables of the grid; per member (32 / G a warp): five
// of its own.  Each table has a slot j*G + s for level s*LPL + j.
struct TwcolSmem {
  int nl, off_tab, off_warp0, per_member, per_warp;
  PM_HD constexpr size_t bytes(int wpb) const { return sizeof(double) * (size_t)(off_warp0 + wpb * per_warp); }
};
PM_HD constexpr TwcolSmem twcol_smem(int G, int LPL) {
  TwcolSmem s{};
  s.nl = G * LPL;
  s.off_warp0 = s.off_tab + 9 * s.nl;
  s.per_member = 5 * s.nl;
  s.per_warp = 32 / G * s.per_member;
  return s;
}

// LIST: launched over an active list (a.list.members != NULL); the plain launch compiles without its extra path
template <int G, int LPL, bool LIST>
PM_GLOBAL void PM_LAUNCH_BOUNDS(128, 4) k_twcol(TwColArgs a) {
  constexpr int MPW = 32 / G;   // members per warp
  constexpr TwcolSmem sl = twcol_smem(G, LPL);
  constexpr int NL = sl.nl;     // level slots of a member
  const pmoc_model& M = a.m;
  const int nz = M.nz;
  const int L = rt::lane(), W = rt::warp_in_block(), nthr = rt::warps_per_block() * 32, tid = W * 32 + L;
  const int s = L & (G - 1), grp = L / G;
  double* sm = rt::smem();
  // block tables (all groups of a warp read the same words: broadcast)
  double* tab = sm + sl.off_tab;
  double *t_h = tab, *t_hh = tab + NL, *t_a = tab + 2 * NL, *t_c = tab + 3 * NL, *t_zf = tab + 4 * NL,
         *t_rdu = tab + 5 * NL, *t_rdd = tab + 6 * NL, *t_ruu = tab + 7 * NL, *t_rdd2 = tab + 8 * NL;
  {
    const double* z = M.z;
    const double z0 = z[0], H = z[nz - 1] - z[0];
    for (int idx = tid; idx < NL; idx += nthr) {
      const int j = idx / G, i = (idx % G) * LPL + j;
      double h = 0., ru = 0., rd = 0., uu = 0., dd = 0.;
      if (i < nz - 1) h = z[i + 1] - z[i];
      if (i >= 1 && i < nz - 1) {
        const double dzu = z[i + 1] - z[i], dzd = z[i] - z[i - 1], dzc = 0.5 * (dzu + dzd);
        ru = 1. / dzu; rd = 1. / dzd; uu = 1. / (dzc * dzu); dd = 1. / (dzc * dzd);
      }
      t_h[idx] = h; t_hh[idx] = 0.5 * h; t_a[idx] = h * h / 3.; t_c[idx] = h * h / 6.;
      t_zf[idx] = i < nz ? (z[i] - z0) / H : 0.;
      t_rdu[idx] = ru; t_rdd[idx] = rd; t_ruu[idx] = uu; t_rdd2[idx] = dd;
    }
  }
  rt::syncblock();
  const long long s_raw = (rt::block_idx() * rt::warps_per_block() + W) * MPW + grp, ns = LIST ? a.list.n : M.M;
  const bool live = s_raw < ns;
  const long long slot = live ? s_raw : ns - 1;  // (groups past the end shadow the last slot and store nothing)
  const long long m = LIST ? a.list.members[slot] : slot;
  if (rt::ballot(live) == 0) return;
  auto group_mask = [&]() { return (G == 32 ? 0xffffffffu : ((1u << G) - 1u)) << (grp * G); };
  // per-member tables: the four stream-function independent products of the folded stencil, d(A kappa)/dz
  double* mt = sm + sl.off_warp0 + (size_t)(W * MPW + grp) * sl.per_member;
  double *m_pk = mt, *m_qk = mt + NL, *m_pa = mt + 2 * NL, *m_qa = mt + 3 * NL, *m_dak = mt + 4 * NL;
  const double dt = M.dt;
  double b[LPL], b2[LPL], p[LPL], q[LPL];
  {
    const double *kap = vrow(M.basin.kappa, m), *dak = vrow(M.basin.dAk, m), *area = vrow(M.basin.Area, m);
    const double* fix = vrow(M.tw_b2, m);
    PM_UNROLL
    for (int j = 0; j < LPL; ++j) {
      const int i = s * LPL + j, sl = j * G + s;
      const bool in = i >= 1 && i < nz - 1;
      b[j] = i < nz ? M.basin.b[m * nz + i] : 0.0;
      b2[j] = i < nz ? fix[i] : 0.0;
      const double kdt = in ? dt * kap[i] : 0.0, ra = in ? dt / area[i] : 0.0;
      m_pk[sl] = kdt * t_ruu[sl];
      m_qk[sl] = kdt * t_rdd2[sl];
      m_pa[sl] = ra * t_rdu[sl];
      m_qa[sl] = ra * t_rdd[sl];
      m_dak[sl] = in ? dak[i] : 0.0;
    }
  }
  rt::syncwarp();
  const double rf_sv = 1e-6 / vat(M.tw_f, m);
  const double bs = vat(M.basin.bs, m), bbot = M.basin.bbot[m];
  const int top_s = (nz - 1) / LPL, top_j = (nz - 1) % LPL;
  // Uniform grid (every example: a linspace, spacing equal to 1e-13) and level-independent area: the geometry
  // factors are scalars, (dt/A)/dzu = (dt/A)/dzd and dt kappa/(dzc dzu) = dt kappa/(dzc dzd), so a level reads two
  // table words per step instead of ten (the kernel is otherwise bound by shared-memory reads: ncu
  // short_scoreboard 2.2 warps per issue cycle).  Decided per warp; anything else takes the tabulated path.
  const double h0 = M.z[1] - M.z[0];
  auto odd_of = [&](long long mm) {  // this lane's levels of member mm break the uniform path
    const double* area = vrow(M.basin.Area, mm);
    bool odd = false;
    PM_UNROLL
    for (int j = 0; j < LPL; ++j) {
      const int i = s * LPL + j;
      if (i < nz - 1) odd |= !(fabs(t_h[j * G + s] - h0) <= 1e-13 * fabs(h0));
      if (i >= 1 && i < nz - 1) odd |= area[i] != area[1];
    }
    return odd;
  };
  // The two paths round differently, so with an active list a member takes the decision of its home warp in a run
  // of every member (members m - m % MPW ... + MPW - 1, the last member standing in past the end): each group
  // re-checks those members.  Groups of one warp that then disagree run both paths and keep their own (`mixed`).
  bool fast, mine = true, mixed = false;
  if (!LIST) {
    fast = rt::ballot(odd_of(m)) == 0 && nz >= 3;
  } else {
    bool odd = false;
    for (int q = 0; q < MPW; ++q) {
      const long long mm = m - m % MPW + q;
      odd |= odd_of(mm < M.M ? mm : M.M - 1);
    }
    mine = (rt::ballot(odd) & group_mask()) == 0 && nz >= 3;
    const unsigned all = rt::ballot(mine);
    fast = all == 0xffffffffu;
    mixed = all != 0 && !fast;
  }
  const double u_hh = 0.5 * h0, u_a = h0 * h0 / 3., u_c = h0 * h0 / 6., u_rn = 1.0 / (double)(nz - 1);
  const double u_pa = fast || (LIST && mixed) ? (dt / vrow(M.basin.Area, m)[1]) / h0 : 0.0;

  // folded stencil coefficients from the streamfunction in Sv (column.py:241-248, see pm::col_coeffs)
  auto coeffs_as = [&](const double(&psi)[LPL], auto FAST) {
    constexpr bool fs = decltype(FAST)::value;
    PM_UNROLL
    for (int j = 0; j < LPL; ++j) {
      const int i = s * LPL + j, sl = j * G + s;
      const double weff = rt::fma(psi[j], 1e6, -m_dak[sl]);
      const double dn = weff < 0 ? weff : 0.0, up = weff < 0 ? 0.0 : weff;  // upwind split (NaN goes to the q side)
      if (fs) {
        const bool in = i >= 1 && i < nz - 1;
        const double k = m_pk[sl];  // (== m_qk on a uniform grid; zero outside the interior)
        p[j] = in ? rt::fma(-dn, u_pa, k) : 0.0;
        q[j] = in ? rt::fma(up, u_pa, k) : 0.0;
      } else {
        p[j] = rt::fma(-dn, m_pa[sl], m_pk[sl]);
        q[j] = rt::fma(up, m_qa[sl], m_qk[sl]);
      }
    }
  };
  auto coeffs = [&](const double(&psi)[LPL]) {
    if (fast) {
      coeffs_as(psi, std::true_type{});
    } else if (!LIST || !mixed) {
      coeffs_as(psi, std::false_type{});
    } else {
      double ps[LPL], qs[LPL];
      coeffs_as(psi, std::false_type{});
      PM_UNROLL
      for (int j = 0; j < LPL; ++j) { ps[j] = p[j]; qs[j] = q[j]; }
      coeffs_as(psi, std::true_type{});
      PM_UNROLL
      for (int j = 0; j < LPL; ++j) {
        p[j] = mine ? p[j] : ps[j];
        q[j] = mine ? q[j] : qs[j];
      }
    }
  };
  // Psi_Thermwind.solve for the current state
  auto solve_as = [&](double(&psi)[LPL], auto FAST) {
    constexpr bool fs = decltype(FAST)::value;
    double g[LPL], part[LPL];
    PM_UNROLL
    for (int j = 0; j < LPL; ++j) g[j] = b2[j] - b[j];
    const double gnext = rt::shfl_down_w(g[0], 1, G);
    double run = 0.0;
    PM_UNROLL
    for (int j = 0; j < LPL; ++j) {  // Psi' by the trapezoid rule (exact: g is piecewise linear)
      const double gu = j < LPL - 1 ? g[j + 1 < LPL ? j + 1 : j] : gnext;
      part[j] = run;
      if (fs)
        run = (s * LPL + j < nz - 1) ? rt::fma(u_hh, g[j] + gu, run) : run;
      else
        run = rt::fma(t_hh[j * G + s], g[j] + gu, run);
    }
    double inc = run;
    PM_UNROLL
    for (int d = 1; d < G; d <<= 1) {
      const double o = rt::shfl_up_w(inc, d, G);
      if (s >= d) inc = inc + o;
    }
    const double base1 = inc - run;
    run = 0.0;
    PM_UNROLL
    for (int j = 0; j < LPL; ++j) {  // Psi: h I1 + h^2 (g_i / 3 + g_{i+1} / 6) per cell
      const int sl = j * G + s;
      const double gu = j < LPL - 1 ? g[j + 1 < LPL ? j + 1 : j] : gnext;
      double cell;
      if (fs)
        cell = (s * LPL + j < nz - 1) ? rt::fma(h0, base1 + part[j], rt::fma(u_a, g[j], u_c * gu)) : 0.0;
      else
        cell = rt::fma(t_h[sl], base1 + part[j], rt::fma(t_a[sl], g[j], t_c[sl] * gu));
      part[j] = run;
      run = run + cell;
    }
    inc = run;
    PM_UNROLL
    for (int d = 1; d < G; d <<= 1) {
      const double o = rt::shfl_up_w(inc, d, G);
      if (s >= d) inc = inc + o;
    }
    const double base2 = inc - run;
    double mine = 0.0;
    PM_UNROLL
    for (int j = 0; j < LPL; ++j) {
      part[j] = base2 + part[j];
      if (j == top_j) mine = part[j];
    }
    const double total = rt::shfl_w(mine, top_s, G);
    PM_UNROLL
    for (int j = 0; j < LPL; ++j) {
      const int i = s * LPL + j;
      const double zf = fs ? (double)i * u_rn : t_zf[j * G + s];
      const double x = rf_sv * rt::fma(-total, zf, part[j]);  // in Sv (rf_sv = 1e-6 / f)
      psi[j] = (i > 0 && i < nz - 1) ? x : 0.0;  // Psi(z0) = Psi(zN) = 0 exactly
    }
  };
  auto solve = [&](double(&psi)[LPL]) {
    if (fast) {
      solve_as(psi, std::true_type{});
    } else if (!LIST || !mixed) {
      solve_as(psi, std::false_type{});
    } else {  // (the scans stay inside the G-lane groups: both paths are warp-uniform)
      double pf[LPL];
      solve_as(psi, std::false_type{});
      solve_as(pf, std::true_type{});
      PM_UNROLL
      for (int j = 0; j < LPL; ++j) psi[j] = mine ? pf[j] : psi[j];
    }
  };
  auto store_psi = [&](const double(&psi)[LPL]) {
    if (!live) return;
    PM_UNROLL
    for (int j = 0; j < LPL; ++j) {
      const int i = s * LPL + j;
      if (i < nz) M.Psi_tw[m * nz + i] = psi[j];
    }
  };

  double psi[LPL];
  if (a.diagnose_only) {
    solve(psi);
    store_psi(psi);
    return;
  }
  PM_UNROLL
  for (int j = 0; j < LPL; ++j) {
    const int i = s * LPL + j;
    psi[j] = i < nz ? M.Psi_tw[m * nz + i] : 0.0;  // the loop uses the previous diagnosis until it % K == 0
  }
  coeffs(psi);
  // boundary values of a plain column are invariant under the step: set them once (column.py:230-232)
  PM_UNROLL
  for (int j = 0; j < LPL; ++j) {
    const int i = s * LPL + j;
    if (i == nz - 1) b[j] = bs;
    if (i == 0) b[j] = bbot;
  }
  const long long K = M.K, it_end = a.it0 + a.nsteps;
  const long long last_refresh = ((it_end - 1) / K) * K;
  long long next0 = ((a.it0 + K - 1) / K) * K;  // next iteration with it % K == 0
  for (long long ii = a.it0; ii < it_end; ++ii) {
    {  // pm::col_step: b_i += p_i (b_{i+1} - b_i) - q_i (b_i - b_{i-1})
      const double bnext = rt::shfl_down_w(b[0], 1, G), bprev = rt::shfl_up_w(b[LPL - 1], 1, G);
      double dm = b[0] - bprev;
      PM_UNROLL
      for (int j = 0; j < LPL; ++j) {
        const double d = (j < LPL - 1 ? b[j + 1 < LPL ? j + 1 : j] : bnext) - b[j];
        b[j] = rt::fma(-q[j], dm, rt::fma(p[j], d, b[j]));
        dm = d;
      }
    }
    if (ii == next0) {
      next0 += K;
      solve(psi);
      if (ii == last_refresh) store_psi(psi);
      coeffs(psi);
    }
  }
  bool bad = false;
  PM_UNROLL
  for (int j = 0; j < LPL; ++j) {
    const int i = s * LPL + j;
    if (i < nz) {
      if (live) M.basin.b[m * nz + i] = b[j];
      bad |= !(fabs(b[j]) <= 1.79e308);
    }
  }
  // NaN flag per member: any lane of the group
  unsigned any = rt::ballot(bad);
  const unsigned gmask = group_mask();
  if (live && s == 0 && M.status) M.status[m] |= (any & gmask) ? PMOC_ST_NAN : 0u;
}

template <int G, int LPL>
static int launch_twcol(const TwColArgs& a, void* stream) {
  constexpr int wpb = 4, MPW = 32 / G;
  const long long per_block = (long long)wpb * MPW;
  const long long grid = (a.list.slots(a.m.M) + per_block - 1) / per_block;
  constexpr size_t smem = twcol_smem(G, LPL).bytes(wpb);
  if (a.list.members) return launch(k_twcol<G, LPL, true>, grid, 32 * wpb, smem, stream, a);
  return launch(k_twcol<G, LPL, false>, grid, 32 * wpb, smem, stream, a);
}

}  // namespace pmk

// nz <= 144, column without convection / gradient bottom condition, thermal wind against a fixed profile
bool pmoc_twcol_supported(const pmoc_model* m) {
  const unsigned topo = m->flags & (PMOC_HAS_NORTH | PMOC_HAS_TW | PMOC_ISO | PMOC_HAS_SO | PMOC_HAS_ML | PMOC_HAS_PAC | PMOC_ORDER_JN);
  return topo == PMOC_HAS_TW && m->nz <= 144 && !m->basin.do_conv && !m->basin.bzbot.ptr && m->basin.nvar == 1 &&
         m->tw_b2.ptr && m->Psi_tw;
}

int pmoc_launch_twcol(const pmoc_model* m, long long it0, long long nsteps, int diagnose_only, void* stream,
                      pmk::MemberList list) {
  pmk::TwColArgs a;
  a.m = *m;
  a.it0 = it0;
  a.nsteps = nsteps;
  a.diagnose_only = diagnose_only;
  a.list = list;
  const int nz = m->nz;
#define PM_TWCOL(G, N) if (nz <= (G) * (N)) return pmk::launch_twcol<G, N>(a, stream);
  PM_TWCOL(8, 3) PM_TWCOL(8, 5) PM_TWCOL(8, 7) PM_TWCOL(8, 9) PM_TWCOL(16, 6) PM_TWCOL(16, 7) PM_TWCOL(16, 8) PM_TWCOL(16, 9)
#undef PM_TWCOL
  return pmk::fail(PMOC_EUNSUPPORTED, "nz > 144: use the warp-per-member kernel");
}
