// The fused multi-step engine, instantiated for one levels-per-lane value per translation
// unit (compile with -DPM_LPL=<2..8>).
#include "pmoc_common.cuh"

#include <cstdlib>

#ifndef PM_LPL
#error "compile with -DPM_LPL=<levels per lane>"
#endif


namespace pmk {
// Resident warps per SM the register allocation allows: 16 at 128 registers per thread.  The multi-column
// 'post' topologies have shared memory for ~19 members per SM, but compiled for 20 warps (96 registers,
// -DPM_WARPS_MULTI=20) they measured slower: C3 0.63 vs 0.66, two-basin 0.54 vs 0.56 of the roofline.
#ifndef PM_WARPS_MULTI
#define PM_WARPS_MULTI 16
#endif
// The 'jn' kernels (SO_ML, bit-faithful column step) carry more live state: compiled for 12 resident warps
// (168 registers) they spill a quarter of what they spill at 128, and with shared memory for at most 15
// members per SM little occupancy is lost.  Measured on C4: 16 warps/128 regs 0.236 of the roofline,
// 12/168 0.247, 10/168 0.254, 8/250 0.206; on C5 (nz = 46): 0.089, 0.093, 0.088, 0.079.
#ifndef PM_WARPS_JN
#define PM_WARPS_JN 12
#endif
#ifndef PM_WARPS_SINGLE
#define PM_WARPS_SINGLE 16  /* 12 (166 registers, no spills) measured slower on C2: 0.81 vs 0.86 -- the step loop wants the warps */
#endif
#ifndef PM_PAC_BIT
#define PM_PAC_BIT 0u  /* the three-column 'post' topology measured slower with this budget: 0.57 vs 0.62 */
#endif
constexpr int max_warps(unsigned topo) {
  return (topo & (PMOC_HAS_ML | PM_PAC_BIT)) ? PM_WARPS_JN
                              : (((topo & PMOC_HAS_NORTH) && !(topo & PMOC_SO_BVP)) ? PM_WARPS_MULTI : PM_WARPS_SINGLE);
}

// LIST: launched over an active list (a.list.members != NULL).  A separate instantiation, so that the plain launch
// compiles to the same code it had without lists (the member index stays a function of the grid position).
template <int LPL, unsigned TOPO, bool LIST>
PM_GLOBAL void PM_LAUNCH_BOUNDS(32 * max_warps(TOPO), 1) k_model(RunArgs a) {
  constexpr bool NORTH = (TOPO & PMOC_HAS_NORTH) != 0, TW = (TOPO & PMOC_HAS_TW) != 0;
  constexpr bool ISO = (TOPO & PMOC_ISO) != 0, SO = (TOPO & PMOC_HAS_SO) != 0;
  constexpr bool ML = (TOPO & PMOC_HAS_ML) != 0;  // SO_ML + the loop order of run_JansenNadeau_2018.py
  constexpr bool BVP = (TOPO & PMOC_SO_BVP) != 0;  // F2010 smoother of Psi_GM
  constexpr bool PAC = (TOPO & PMOC_HAS_PAC) != 0;  // third column + zonal thermal wind + second Psi_SO
  const pmoc_model& M = a.m;
  const SmemPlan& sp = a.sp;
  const int nz = M.nz, ny = M.ny, nb = M.nb;
  const int L = rt::lane(), W = rt::warp_in_block(), nthr = rt::warps_per_block() * 32;
  double* sm = rt::smem();
  double* ysm = sm + sp.off_y;
  double* ws = sm + sp.off_warp0 + (size_t)sp.per_warp * W;
  pm::geo_fill<LPL>(sm + sp.off_zs, sm + sp.off_zl, sm + sp.off_rdu, sm + sp.off_rdd, sm + sp.off_ruu,
                    sm + sp.off_rdd2, M.z, nz, W * 32 + L, nthr, !ML);
  if (ML)
    pm::geo_fill_exact<LPL>(sm + sp.off_dzu, sm + sp.off_rdzu, sm + sp.off_dzc, sm + sp.off_rdzc, M.z, nz, W * 32 + L,
                            nthr);
  if (SO) {
    for (int i = W * 32 + L; i < sp.nyp; i += nthr) ysm[i] = M.y[i < ny ? i : ny - 1];
    pm::taper_fill<LPL>(sm + sp.off_tap, M.so_sill_taper, M.so_ek_taper, M.so_top_taper, M.so_bot_taper, nz,
                        W * 32 + L, nthr);
  }
  rt::syncblock();
  const pm::GeoTab G = geo_of(sm, sp);
  const double* zs = G.zs;
  const long long slot = rt::block_idx() * rt::warps_per_block() + W;
  if (slot >= (LIST ? a.list.n : M.M)) return;
  const long long m = LIST ? a.list.members[slot] : slot;
  const double dt = M.dt;

  ColRegs<LPL> cb, cn, cp;
  pm::ExactGeo EG{};
  pm::ExactCol xb{}, xn{};
  col_load<LPL>(cb, M.basin, m, nz);
  if (NORTH) col_load<LPL>(cn, M.north, m, nz);
  if (PAC) col_load<LPL>(cp, M.pac, m, nz);
  if (!ML) {
    if (sp.col_tables) {
      cb.tab = coltab_of(ws, sp, 0);
      col_retabulate<LPL>(cb, M.basin, m, G, nz, dt);
      if (NORTH) {
        cn.tab = coltab_of(ws, sp, 1);
        col_retabulate<LPL>(cn, M.north, m, G, nz, dt);
      }
      if (PAC) {
        cp.tab = coltab_of(ws, sp, 2);
        col_retabulate<LPL>(cp, M.pac, m, G, nz, dt);
      }
    }
  } else {
    EG = exactgeo_of(sm, sp);
    xb = exactcol_of(ws, sp, 0);
    xn = exactcol_of(ws, sp, 1);
    pm::col_tabulate_exact<LPL>(xb, vrow(M.basin.kappa, m), vrow(M.basin.Area, m), nz, M.basin.nvar);
    pm::col_tabulate_exact<LPL>(xn, vrow(M.north.kappa, m), vrow(M.north.Area, m), nz, M.north.nvar);
    if (M.basin.nvar < 2) cb.var = 0;
    if (M.north.nvar < 2) cn.var = 0;
  }
  double b2fix[LPL];
  if (TW && !NORTH) pm::load_lev<LPL>(b2fix, vrow(M.tw_b2, m), nz, 0.0);
  const double tw_f = TW ? vat(M.tw_f, m) : 1.0;
  const double zoc_f = PAC ? vat(M.zoc_f, m) : 1.0;
  pm::SoPar so{};
  pm::SoSurf surf{};
  if (SO) {
    so.tau_ave = M.so_tau_on_y ? 0.0 : pm::mean100(vat(M.so_tau, m));
    so.tau_y = nullptr;
    if (M.so_tau_on_y) {
      const double* t = vrow(M.so_tau, m);
      for (int i = L; i < sp.nyp; i += 32) ws[sp.w_tau + i] = t[i < ny ? i : ny - 1];
      so.tau_y = ws + sp.w_tau;
    }
    so.c = BVP ? vat(M.so_c, m) : 0.0;
    so.with_Ek = M.so_bvp_with_Ek;
    so.f = vat(M.so_f, m); so.rho = vat(M.so_rho, m); so.L = vat(M.so_L, m);
    so.KGM = vat(M.so_KGM, m); so.smax = vat(M.so_smax, m);
    so.sill = sm + sp.off_tap; so.ektap = so.sill + sp.nzp; so.toptap = so.sill + 2 * sp.nzp;
    so.bottap = so.sill + 3 * sp.nzp;
    const double* src = vrow(M.so_bs, m);
    if (ML) src = M.ml_bs + m * ny;  // the mixed layer's bs (run_JansenNadeau_2018.py:214)
    for (int i = L; i < sp.nyp; i += 32) ws[sp.w_bs + i] = src[i < ny ? i : ny - 1];
    rt::syncwarp();
    if (!ML) surf = pm::so_scan(ysm, ws + sp.w_bs, ws + sp.w_sinv, ny);  // bs(y) is fixed without a mixed layer
  }
  if (SO) so.pre0 = so.tau_ave / so.f / so.rho * so.L;
  pm::SoPar so2 = so;  // the pac sector's Psi_SO differs in its zonal length only (twobasin_NadeauJansen.py:76-81)
  if (PAC) {
    so2.L = vat(M.so2_L, m);
    so2.pre0 = so2.tau_ave / so2.f / so2.rho * so2.L;
  }
  unsigned status = 0;
  pm::MlState ml{};
  double* const bb_s = ws + (ML ? sp.w_bb : 0);
  double* const pm_s = ws + (ML ? sp.w_pm : 0);
  double psi_so1 = 0., res_b1 = 0., res_n1 = 0.;  // Psi[1] of the three streamfunctions ('jn' switches)
  // which of them are rounding noise (pm::jn_noise); so1_exact: Psi_so[1] came out of state-independent arithmetic
  unsigned noise = 0;
  bool so1_exact = ML && so1_exact_carried(M, m);
  if (ML) {
    pm::ml_setup(ml, ysm, ny, vat(M.ml_Ks, m), vat(M.ml_h, m), vat(M.ml_L, m), vat(M.ml_vpist, m),
                 vrow(M.ml_surflux, m), vrow(M.ml_rest_mask, m), vrow(M.ml_b_rest, m), dt, ws + sp.w_scan);
    PM_UNROLL
    for (int e = 0; e < pm::kMLP; ++e) ml.bs[e] = ws[sp.w_bs + (pm::mlk(e) < ny ? pm::mlk(e) : ny - 1)];
  }

  // folded stencil coefficients of one column from wA (tables in shared memory or the global profiles)
  auto coeffs = [&](ColRegs<LPL>& c, const pmoc_column& d, const double(&wA)[LPL]) {
    if (sp.col_tables) {
      pm::col_coeffs<LPL>(c.p, c.q, wA, c.tab, G, nz);
    } else {
      const long long voff = (long long)c.var * nz;
      pm::col_coeffs_global<LPL>(c.p, c.q, wA, vrow(d.kappa, m) + voff, vrow(d.dAk, m) + voff, vrow(d.Area, m), dt, G, nz);
    }
  };
  // Streamfunctions -> stencil coefficients of the columns (and what SO_ML needs).
  auto apply = [&](const double(&north_leg)[LPL], const double(&iso_n)[LPL], const double(&psi_so)[LPL],
                   const double(&zon_a)[LPL], const double(&zon_p)[LPL], const double(&psi_so2)[LPL]) {
    double wA[LPL];
    if (PAC) {  // twobasin_NadeauJansen.py:104-106
      PM_UNROLL
      for (int j = 0; j < LPL; ++j) wA[j] = (-zon_p[j] - psi_so2[j]) * 1e6;
      coeffs(cp, M.pac, wA);
      PM_UNROLL
      for (int j = 0; j < LPL; ++j) wA[j] = (north_leg[j] + zon_a[j] - psi_so[j]) * 1e6;
    } else {
      PM_UNROLL
      for (int j = 0; j < LPL; ++j) wA[j] = ((TW ? north_leg[j] : 0.0) - (SO ? psi_so[j] : 0.0)) * 1e6;
    }
    if (ML)
      pm::col_nweff<LPL>(xb, wA, vrow(M.basin.dAk, m), nz, M.basin.nvar);
    else
      coeffs(cb, M.basin, wA);
    if (NORTH) {
      PM_UNROLL
      for (int j = 0; j < LPL; ++j) wA[j] = -iso_n[j] * 1e6;
      if (ML)
        pm::col_nweff<LPL>(xn, wA, vrow(M.north.dAk, m), nz, M.north.nvar);
      else
        coeffs(cn, M.north, wA);
    }
    if (ML) {
      psi_so1 = pm::get_level<LPL>(psi_so, 1);
      res_b1 = pm::get_level<LPL>(north_leg, 1);
      res_n1 = pm::get_level<LPL>(iso_n, 1);
      if (!pm::ml_bind_psi<LPL>(ml, psi_so, nz, pm_s)) status |= PMOC_ST_ML_INDEX;
      double mx = 0.0;
      PM_UNROLL
      for (int j = 0; j < LPL; ++j) {
        const double a1 = fabs(north_leg[j]), a2 = fabs(iso_n[j]), a3 = fabs(psi_so[j]);
        mx = a1 > mx ? a1 : mx;
        mx = a2 > mx ? a2 : mx;
        mx = a3 > mx ? a3 : mx;
      }
      noise = pm::jn_noise(psi_so1, res_b1, res_n1, rt::wmax(mx), so1_exact);
    }
  };

  // Diagnose the streamfunctions from the current state and fold them into the stencils.
  auto refresh = [&](bool write) {
    double psi_tw[LPL], iso_b[LPL], iso_n[LPL], psi_so[LPL], zon_a[LPL], zon_p[LPL], psi_so2[LPL];
    PM_UNROLL
    for (int j = 0; j < LPL; ++j) psi_tw[j] = iso_b[j] = iso_n[j] = psi_so[j] = zon_a[j] = zon_p[j] = psi_so2[j] = 0.0;
    if (TW) {
      const double(&b2)[LPL] = NORTH ? cn.b : b2fix;
      pm::tw_solve<LPL>(psi_tw, cb.b, b2, tw_f, zs, nz, nullptr);
      if (write && M.Psi_tw) pm::store_lev<LPL>(psi_tw, M.Psi_tw + m * nz, nz);
      if (ISO) {
        double* psib_s = ws + sp.w_psib;
        const pm::BGrid BG = pm::tw_psib<LPL>(psi_tw, cb.b, b2, nz, nb, ws + sp.w_remap, psib_s,
                                              reinterpret_cast<int*>(ws + sp.w_cnt), &status);
        PM_UNROLL
        for (int j = 0; j < LPL; ++j) {
          const bool ok = pm::lev<LPL>(j) < nz;
          iso_b[j] = ok ? pm::interp_bgrid(cb.b[j], BG, psib_s) : 0.0;
          iso_n[j] = ok ? pm::interp_bgrid(b2[j], BG, psib_s) : 0.0;
        }
        if (write) {
          pm::store_lev<LPL>(iso_b, M.Psi_iso_b + m * nz, nz);
          pm::store_lev<LPL>(iso_n, M.Psi_iso_n + m * nz, nz);
          if (M.psib)
            for (int i = L; i < nb; i += 32) M.psib[m * nb + i] = psib_s[i];
          if (M.bgrid)
            for (int i = L; i < nb; i += 32) M.bgrid[m * nb + i] = BG.at(i);
        }
        rt::syncwarp();
      }
    }
    if (PAC) {  // ZOC.update(b1=Atl.b, b2=Pac.b); ZOC.solve(); ZOC.Psibz()  (twobasin_NadeauJansen.py:117-119)
      double psi_zoc[LPL];
      pm::tw_solve<LPL>(psi_zoc, cb.b, cp.b, zoc_f, zs, nz, nullptr);
      if (write && M.Psi_zoc) pm::store_lev<LPL>(psi_zoc, M.Psi_zoc + m * nz, nz);
      double* psib_s = ws + sp.w_psib;
      const pm::BGrid BG = pm::tw_psib<LPL>(psi_zoc, cb.b, cp.b, nz, nb, ws + sp.w_remap, psib_s,
                                            reinterpret_cast<int*>(ws + sp.w_cnt), &status);
      PM_UNROLL
      for (int j = 0; j < LPL; ++j) {
        const bool ok = pm::lev<LPL>(j) < nz;
        zon_a[j] = ok ? pm::interp_bgrid(cb.b[j], BG, psib_s) : 0.0;
        zon_p[j] = ok ? pm::interp_bgrid(cp.b[j], BG, psib_s) : 0.0;
      }
      if (write) {
        pm::store_lev<LPL>(zon_a, M.Psi_zon_a + m * nz, nz);
        pm::store_lev<LPL>(zon_p, M.Psi_zon_p + m * nz, nz);
        if (M.psib2)
          for (int i = L; i < nb; i += 32) M.psib2[m * nb + i] = psib_s[i];
        if (M.bgrid2)
          for (int i = L; i < nb; i += 32) M.bgrid2[m * nb + i] = BG.at(i);
      }
      rt::syncwarp();
    }
    if (SO) {
      double ek[LPL], gm[LPL], ysv[LPL];
      if (ML) {  // the channel's surface buoyancy is the mixed layer's (run_JansenNadeau_2018.py:214)
        PM_UNROLL
        for (int e = 0; e < pm::kMLP; ++e)
          if (pm::mlk(e) < ny) ws[sp.w_bs + pm::mlk(e)] = ml.bs[e];
        rt::syncwarp();
        surf = pm::so_scan(ysm, ws + sp.w_bs, ws + sp.w_sinv, ny);
      }
      pm::so_solve<LPL, BVP>(psi_so, ek, gm, ysv, cb.b, ysm, ws + sp.w_bs, ws + sp.w_sinv, ny, surf, so, zs, nz,
                             &status, &so1_exact);
      if (write) {
        pm::store_lev<LPL>(psi_so, M.Psi_so + m * nz, nz);
        if (M.Psi_Ek) pm::store_lev<LPL>(ek, M.Psi_Ek + m * nz, nz);
        if (M.Psi_GM) pm::store_lev<LPL>(gm, M.Psi_GM + m * nz, nz);
      }
      if (PAC) {  // SO_Pac.update(b=Pac.b); SO_Pac.solve()  (twobasin_NadeauJansen.py:122-123)
        pm::so_solve<LPL, false>(psi_so2, ek, gm, ysv, cp.b, ysm, ws + sp.w_bs, ws + sp.w_sinv, ny, surf, so2, zs, nz,
                                 &status);
        if (write) {
          pm::store_lev<LPL>(psi_so2, M.Psi_so2 + m * nz, nz);
          if (M.Psi_Ek2) pm::store_lev<LPL>(ek, M.Psi_Ek2 + m * nz, nz);
          if (M.Psi_GM2) pm::store_lev<LPL>(gm, M.Psi_GM2 + m * nz, nz);
        }
      }
    }
    if (ISO)
      apply(iso_b, iso_n, psi_so, zon_a, zon_p, psi_so2);
    else
      apply(psi_tw, iso_n, psi_so, zon_a, zon_p, psi_so2);
    if (ML) {  // the remap scratch overlaid the column tables (plan_smem)
      pm::col_tabulate_exact<LPL>(xb, vrow(M.basin.kappa, m), vrow(M.basin.Area, m), nz, M.basin.nvar);
      pm::col_tabulate_exact<LPL>(xn, vrow(M.north.kappa, m), vrow(M.north.Area, m), nz, M.north.nvar);
    }
  };

  const long long K = M.K, it_end = a.it0 + a.nsteps;
  // carried streamfunctions -> stencils (the loop uses the previous diagnosis until it % K == 0);
  // the 'jn' order diagnoses at the top of iteration it % K == 0 and then needs nothing carried
  const bool dg = a.diagnose_only != 0;
  if (!dg && (!ML || a.it0 % K != 0)) {
    double t1[LPL], t2[LPL], t3[LPL], t4[LPL], t5[LPL], t6[LPL];
    PM_UNROLL
    for (int j = 0; j < LPL; ++j) t1[j] = t2[j] = t3[j] = t4[j] = t5[j] = t6[j] = 0.0;
    if (TW) pm::load_lev<LPL>(t1, (ISO ? M.Psi_iso_b : M.Psi_tw) + m * nz, nz, 0.0);
    if (NORTH) pm::load_lev<LPL>(t2, M.Psi_iso_n + m * nz, nz, 0.0);
    if (SO) pm::load_lev<LPL>(t3, M.Psi_so + m * nz, nz, 0.0);
    if (PAC) {
      pm::load_lev<LPL>(t4, M.Psi_zon_a + m * nz, nz, 0.0);
      pm::load_lev<LPL>(t5, M.Psi_zon_p + m * nz, nz, 0.0);
      pm::load_lev<LPL>(t6, M.Psi_so2 + m * nz, nz, 0.0);
    }
    apply(t1, t2, t3, t4, t5, t6);
  }

  if (!ML && !dg) {
    // boundary values of "plain" columns are invariant under the step: set them once
    // (surface: column.py:230-231, bottom: column.py:232)
    if (!cb.conv) pm::set_level<LPL>(cb.b, nz - 1, cb.bs);
    if (cb.plain) col_bottom<LPL>(cb, zs);
    if (NORTH) {
      if (!cn.conv) pm::set_level<LPL>(cn.b, nz - 1, cn.bs);
      if (cn.plain) col_bottom<LPL>(cn, zs);
    }
    if (PAC) {
      if (!cp.conv) pm::set_level<LPL>(cp.b, nz - 1, cp.bs);
      if (cp.plain) col_bottom<LPL>(cp, zs);
    }
  }
  // One loop for both orders, with a single (inlined) copy of the diagnosis:
  //   'post' (example_twocol_plusSO.py:99-115): step ... step(it % K == 0) -> refresh
  //   'jn'   (run_JansenNadeau_2018.py:201-261): refresh at the top of it % K == 0 -> steps
  // Only the last refresh of a launch writes the diagnostics to HBM.
  const long long last_refresh = ((it_end - 1) / K) * K;
  const bool two_var_b = M.basin.nvar > 1, two_var_n = M.north.nvar > 1;
  long long ii = a.it0;
  // next iteration with it % K == 0 at or after ii: kept incrementally (a 64-bit integer division costs ~100
  // instructions, which at K = 1 was 6 % of the C1 kernel)
  long long next0 = ((ii + K - 1) / K) * K;
  bool refresh_next = dg || (ML && ii < it_end && ii % K == 0);
  bool wr = dg || ii == last_refresh;
  for (;;) {
    if (refresh_next) {
#ifndef PMOC_EMU
      if (a.sync_refresh) __syncthreads();  // (warps past the last slot have exited: they do not count)
#endif
      refresh(wr);
      refresh_next = false;
      if (dg) break;
    }
    if (ii >= it_end) break;
    if (!ML) {
      const long long stop = next0;  // next iteration with it % K == 0
      const bool hits = stop < it_end;
      const int n = (int)((hits ? stop + 1 : it_end) - ii);
      if (hits) next0 = stop + K;
      for (int s = 0; s < n; ++s) {
        col_advance<LPL>(cb, G, nz);
        if (NORTH) col_advance<LPL>(cn, G, nz);
        if (PAC) col_advance<LPL>(cp, G, nz);
      }
      ii += n;
      refresh_next = hits;
      wr = stop == last_refresh;
    } else {
      if (next0 <= ii) next0 += K;  // here ii % K == 0 was just diagnosed (or the launch starts inside an interval)
      long long stop = next0;
      if (stop > it_end) stop = it_end;
      for (; ii < stop; ++ii) {
        // bottom boundary condition and bottom-boundary-layer kappa (:233-254); levels 0 and 1
        // of both columns and bs[0] live in lane 0
        const double bb0 = rt::shfl(cb.b[0], 0), bb1 = rt::shfl(cb.b[1], 0);
        const double nb0 = rt::shfl(cn.b[0], 0), nb1 = rt::shfl(cn.b[1], 0);
        const double bs0 = rt::shfl(ml.bs[0], 0);
        int vb = cb.var, vn = cn.var;
        pm::jn_switch_basin(psi_so1, res_b1, bb1, nb0, bs0, cb.bbot, vb);
        pm::jn_switch_north(res_n1, bb0, nb1, cn.bbot, vn);
        pm::jn_noise_hit(noise, bb0, bb1, nb0, nb1, bs0, &status);
        if (two_var_b) cb.var = vb;
        if (two_var_n) cn.var = vn;
        col_advance_exact<LPL>(cb, xb, EG, G, nz, dt);
        col_advance_exact<LPL>(cn, xn, EG, G, nz, dt);
        const bool sorted = pm::ml_bind_basin<LPL>(cb.b, nz, bb_s);
        pm::ml_step(ml, bb_s, pm_s, nz, sorted, ws + sp.w_bs, dt, &status);
      }
      refresh_next = ii < it_end;  // here ii % K == 0
      wr = ii == last_refresh;
    }
  }
  auto put_status = [&]() {
    if (M.status && L == 0) M.status[m] = status_word(M.status[m], status, ML && so1_exact);
  };
  if (dg) {
    put_status();
    return;
  }
  if (ML) {
    if (L == 0) {
      M.basin.bbot[m] = cb.bbot;
      M.north.bbot[m] = cn.bbot;
      if (M.basin.var) M.basin.var[m] = cb.var;
      if (M.north.var) M.north.var[m] = cn.var;
    }
    PM_UNROLL
    for (int e = 0; e < pm::kMLP; ++e) {
      const int k = pm::mlk(e);
      if (k < ny) {
        M.ml_bs[m * ny + k] = ml.bs[e];
        if (M.ml_Psi_s) M.ml_Psi_s[m * ny + k] = ml.ps[e];
      }
    }
  }

  pm::store_lev<LPL>(cb.b, M.basin.b + m * nz, nz);
  if (NORTH) pm::store_lev<LPL>(cn.b, M.north.b + m * nz, nz);
  if (PAC) pm::store_lev<LPL>(cp.b, M.pac.b + m * nz, nz);
  bool bad = false;
  PM_UNROLL
  for (int j = 0; j < LPL; ++j) {
    if (pm::lev<LPL>(j) < nz) {
      bad |= !(fabs(cb.b[j]) <= 1.79e308);
      if (NORTH) bad |= !(fabs(cn.b[j]) <= 1.79e308);
      if (PAC) bad |= !(fabs(cp.b[j]) <= 1.79e308);
    }
  }
  if (ML) {
    PM_UNROLL
    for (int e = 0; e < pm::kMLP; ++e)
      if (pm::mlk(e) < ny) bad |= !(fabs(ml.bs[e]) <= 1.79e308);
  }
  if (rt::ballot(bad)) status |= PMOC_ST_NAN;
  put_status();
}

template <int LPL>
int launch_model(const RunArgs& ra, void* stream) {
  const unsigned t = ra.m.flags & (PMOC_HAS_NORTH | PMOC_HAS_TW | PMOC_ISO | PMOC_HAS_SO | PMOC_HAS_ML | PMOC_SO_BVP | PMOC_HAS_PAC);
  // Warps (= members) per CTA: the block-level tables are shared by a CTA's warps, so fewer, larger CTAs
  // leave more shared memory for members; take the split with the most resident warps per SM, at most 16
  // (128 registers per thread); four warps per CTA unless another split is strictly better.
  const int cap = max_warps(t);
  auto resident = [&](int w) {
    const size_t need = ra.sp.bytes(w) + 1024;  // + the per-CTA reservation
    if (need > 228 * 1024) return 0;
    int ctas = (int)((228 * 1024) / need);
    if (ctas * w > cap) ctas = cap / w;
    return ctas * w;
  };
  int wpb = kWarpsPerBlock, best = resident(kWarpsPerBlock);  // four warps per CTA unless another split is better
  for (int w = 1; w <= cap; ++w)
    if (resident(w) > best) { best = resident(w); wpb = w; }
  // the F2010 smoother's diagnosis is the longest instruction stream: eight warps per CTA share its fetches
  // (with the barrier below) when that costs no residency.  Measured, C3_bvp: 4 warps 0.515, 8 warps 0.522.
  if ((t & PMOC_SO_BVP) && !(t & PMOC_HAS_ML) && resident(8) == best) wpb = 8;
  if (best == 0) return fail(PMOC_EUNSUPPORTED, "model does not fit the shared memory of one SM");
  if (const char* e = std::getenv("PMOC_WPB")) {  // tuning knob: force the warps per CTA
    const int w = std::atoi(e);
    if (w >= 1 && w <= cap && resident(w) > 0) wpb = w;
  }
  const long long grid = (ra.list.slots(ra.m.M) + wpb - 1) / wpb;
  const int block = 32 * wpb;
  const size_t smem = ra.sp.bytes(wpb);
  // A CTA barrier in front of every diagnosis re-aligns the CTA's warps, which then walk its ~9 000-instruction
  // stream (144 KB of code, against a 32 KB L1.5 instruction cache) together and share the fetches: ncu's
  // no_instruction stall was 1.28 warps per issue cycle without it.  Measured: C3_bvp 0.473 -> 0.515, C3 0.715 ->
  // 0.731, C4 0.253 -> 0.259; the single-column kernels (short diagnosis) lose 1.5 % and keep running free.
  RunArgs ra2 = ra;
  ra2.sync_refresh = (t & PMOC_ISO) != 0;
  if (const char* e = std::getenv("PMOC_REFRESH_SYNC")) ra2.sync_refresh = std::atoi(e);
#define PM_CASE(T)                                                                      \
  case (T):                                                                             \
    return ra.list.members ? launch(k_model<LPL, (T), true>, grid, block, smem, stream, ra2) \
                           : launch(k_model<LPL, (T), false>, grid, block, smem, stream, ra2);
  switch (t) {
    PM_CASE(PMOC_HAS_TW)
    PM_CASE(PMOC_HAS_SO)
    PM_CASE(PMOC_HAS_SO | PMOC_SO_BVP)
    PM_CASE(PMOC_HAS_TW | PMOC_HAS_SO)
    PM_CASE(PMOC_HAS_TW | PMOC_HAS_SO | PMOC_SO_BVP)
    PM_CASE(PMOC_HAS_NORTH | PMOC_HAS_TW | PMOC_ISO)
    PM_CASE(PMOC_HAS_NORTH | PMOC_HAS_TW | PMOC_ISO | PMOC_HAS_SO)
    PM_CASE(PMOC_HAS_NORTH | PMOC_HAS_TW | PMOC_ISO | PMOC_HAS_SO | PMOC_SO_BVP)
    PM_CASE(PMOC_HAS_NORTH | PMOC_HAS_TW | PMOC_ISO | PMOC_HAS_SO | PMOC_HAS_PAC)
    PM_CASE(PMOC_HAS_NORTH | PMOC_HAS_TW | PMOC_ISO | PMOC_HAS_SO | PMOC_HAS_ML)
    PM_CASE(PMOC_HAS_NORTH | PMOC_HAS_TW | PMOC_ISO | PMOC_HAS_SO | PMOC_HAS_ML | PMOC_SO_BVP)
    default: return fail(PMOC_EUNSUPPORTED, "module combination has no fused kernel");
  }
#undef PM_CASE
}

}  // namespace pmk

#define PM_CAT2(a, b) a##b
#define PM_CAT(a, b) PM_CAT2(a, b)
int PM_CAT(pmoc_launch_model_, PM_LPL)(const RunArgs& ra, void* stream) { return launch_model<PM_LPL>(ra, stream); }
