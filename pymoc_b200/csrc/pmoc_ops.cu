// Per-module kernels and the C-ABI entry points of pymoc_b200 (see include/pymoc_b200.h).
#include "pmoc_common.cuh"

#include <cstdlib>

thread_local char pmoc_g_err[256] = "";

namespace pmk {
// ------------------------------------------------------------------------------------------
// per-module kernels
struct ColumnArgs {
  long long M;
  int nz;
  const double* z;
  pmoc_column col;
  pmoc_vec wA, vdx_in, b_in;
  double dt;
  unsigned stages;
};

template <int LPL>
PM_GLOBAL void k_column(ColumnArgs a) {
  const int nz = a.nz, L = rt::lane(), W = rt::warp_in_block(), nthr = rt::warps_per_block() * 32;
  const SmemPlan sp = plan_smem(LPL, 0, 2, 0);
  double* sm = rt::smem();
  pm::geo_fill<LPL>(sm + sp.off_zs, sm + sp.off_zl, sm + sp.off_rdu, sm + sp.off_rdd, sm + sp.off_ruu,
                    sm + sp.off_rdd2, a.z, nz, W * 32 + L, nthr);
  rt::syncblock();
  const pm::GeoTab G = geo_of(sm, sp);
  const long long m = rt::block_idx() * rt::warps_per_block() + W;
  if (m >= a.M) return;
  ColRegs<LPL> c;
  col_load<LPL>(c, a.col, m, nz);
  c.tab = coltab_of(sm + sp.off_warp0 + (size_t)sp.per_warp * W, sp, 0);
  if (a.stages & PMOC_STAGE_CONVECT) pm::col_convect<LPL>(c.b, c.bs, c.N2min, G.zs, G.zl, nz);
  if (a.stages & PMOC_STAGE_VERTADVDIFF) {
    double wA[LPL];
    pm::load_lev<LPL>(wA, vrow(a.wA, m), nz, 0.0);
    col_retabulate<LPL>(c, a.col, m, G, nz, a.dt);
    pm::col_coeffs<LPL>(c.p, c.q, wA, c.tab, G, nz);
    if (!c.conv) pm::set_level<LPL>(c.b, nz - 1, c.bs);  // column.py:230-231
    col_bottom<LPL>(c, G.zs);
    pm::col_step<LPL>(c.b, c.p, c.q);
  }
  if (a.stages & PMOC_STAGE_HORADV)
    pm::col_horadv<LPL>(c.b, vrow(a.vdx_in, m), vrow(a.b_in, m), vrow(a.col.Area, m), nz, a.dt);
  pm::store_lev<LPL>(c.b, a.col.b + m * nz, nz);
}

struct ThermwindArgs {
  long long M;
  int nz, nb;
  const double* z;
  pmoc_vec b1, b2, f, gmid, Psi_in;
  double *Psi, *psib, *bgrid, *iso_b, *iso_n;
};

// Shared memory of k_thermwind (in doubles), per block: z on the warp's level slots and four more.
struct ThermwindSmem {
  int off_zs, nzs;
  PM_HD constexpr size_t bytes() const { return sizeof(double) * (size_t)(off_zs + nzs); }
};
PM_HD constexpr ThermwindSmem thermwind_smem(int LPL) { return ThermwindSmem{0, 32 * LPL + 4}; }

template <int LPL>
PM_GLOBAL void k_thermwind(ThermwindArgs a) {
  const int nz = a.nz, L = rt::lane(), W = rt::warp_in_block(), nthr = rt::warps_per_block() * 32;
  constexpr ThermwindSmem sl = thermwind_smem(LPL);
  double* zs = rt::smem() + sl.off_zs;
  for (int i = W * 32 + L; i < sl.nzs; i += nthr) zs[i] = a.z[i < nz ? i : nz - 1];
  rt::syncblock();
  const long long m = rt::block_idx() * rt::warps_per_block() + W;
  if (m >= a.M) return;
  double b1[LPL], b2[LPL], psi[LPL];
  pm::load_lev<LPL>(b1, vrow(a.b1, m), nz, 0.0);
  pm::load_lev<LPL>(b2, vrow(a.b2, m), nz, 0.0);
  pm::tw_solve<LPL>(psi, b1, b2, vat(a.f, m), zs, nz, a.gmid.ptr ? vrow(a.gmid, m) : nullptr);
  pm::store_lev<LPL>(psi, a.Psi + m * nz, nz);
}

// Shared memory of k_psib (in doubles), per warp: the remap scratch (6 nzp), psib[nb] and the class counters
// (nb + 1 ints).
struct PsibSmem {
  int w_remap, w_psib, w_cnt, per_warp;
  PM_HD constexpr size_t bytes(int wpb) const { return sizeof(double) * (size_t)per_warp * wpb; }
};
PM_HD constexpr PsibSmem psib_smem(int LPL, int nb) {
  PsibSmem s{};
  const int nbp = (nb + 3) & ~3;
  s.w_psib = s.w_remap + 6 * 32 * LPL; s.w_cnt = s.w_psib + nbp; s.per_warp = s.w_cnt + nbp / 2 + 2;
  return s;
}

template <int LPL>
PM_GLOBAL void k_psib(ThermwindArgs a) {
  const int nz = a.nz, nb = a.nb, L = rt::lane(), W = rt::warp_in_block();
  const long long m = rt::block_idx() * rt::warps_per_block() + W;
  if (m >= a.M) return;
  const PsibSmem sl = psib_smem(LPL, nb);
  double* ws = rt::smem() + (size_t)sl.per_warp * W;
  double b1[LPL], b2[LPL], psi[LPL];
  pm::load_lev<LPL>(b1, vrow(a.b1, m), nz, 0.0);
  pm::load_lev<LPL>(b2, vrow(a.b2, m), nz, 0.0);
  pm::load_lev<LPL>(psi, vrow(a.Psi_in, m), nz, 0.0);
  double* psib_s = ws + sl.w_psib;
  const pm::BGrid G =
      pm::tw_psib<LPL>(psi, b1, b2, nz, nb, ws + sl.w_remap, psib_s, reinterpret_cast<int*>(ws + sl.w_cnt));
  for (int i = L; i < nb; i += 32) {
    a.psib[m * nb + i] = psib_s[i];
    if (a.bgrid) a.bgrid[m * nb + i] = G.at(i);
  }
  if (a.iso_b || a.iso_n) {
    double ib[LPL], in_[LPL];
    PM_UNROLL
    for (int j = 0; j < LPL; ++j) {
      const bool ok = pm::lev<LPL>(j) < nz;
      ib[j] = ok ? pm::interp_bgrid(b1[j], G, psib_s) : 0.0;
      in_[j] = ok ? pm::interp_bgrid(b2[j], G, psib_s) : 0.0;
    }
    if (a.iso_b) pm::store_lev<LPL>(ib, a.iso_b + m * nz, nz);
    if (a.iso_n) pm::store_lev<LPL>(in_, a.iso_n + m * nz, nz);
  }
}

struct SoArgs {
  pmoc_model m;
  pmoc_vec b, bs;
  double *Psi, *Psi_Ek, *Psi_GM, *ys;
  uint32_t* status;
};

// Shared memory of k_so (in doubles).  Per block: z (nzp + 4), y and the four tapers (4 nzp); per warp: bs, the
// inverse slopes and tau on y.
struct SoSmem {
  int nzp, nyp, off_zs, off_ys, off_tap, off_warp0, w_bs, w_sinv, w_tau, per_warp;
  PM_HD constexpr size_t bytes(int wpb) const { return sizeof(double) * (size_t)(off_warp0 + per_warp * wpb); }
};
PM_HD constexpr SoSmem so_smem(int LPL, int ny) {
  SoSmem s{};
  s.nzp = 32 * LPL; s.nyp = (ny + 3) & ~3;
  s.off_ys = s.off_zs + s.nzp + 4; s.off_tap = s.off_ys + s.nyp; s.off_warp0 = s.off_tap + 4 * s.nzp;
  s.w_sinv = s.w_bs + s.nyp; s.w_tau = s.w_sinv + s.nyp; s.per_warp = s.w_tau + s.nyp;
  return s;
}

template <int LPL, bool BVP>
PM_GLOBAL void k_so(SoArgs a) {
  const pmoc_model& M = a.m;
  const int nz = M.nz, ny = M.ny, L = rt::lane(), W = rt::warp_in_block(), nthr = rt::warps_per_block() * 32;
  const SoSmem sl = so_smem(LPL, ny);
  double* sm = rt::smem();
  double* zs = sm + sl.off_zs;
  double* ysm = sm + sl.off_ys;
  double* tap = sm + sl.off_tap;
  double* ws = sm + sl.off_warp0 + (size_t)sl.per_warp * W;
  double* bss = ws + sl.w_bs;
  double* sinv = ws + sl.w_sinv;
  double* tau_s = ws + sl.w_tau;
  for (int i = W * 32 + L; i < sl.nzp + 4; i += nthr) zs[i] = M.z[i < nz ? i : nz - 1];
  for (int i = W * 32 + L; i < sl.nyp; i += nthr) ysm[i] = M.y[i < ny ? i : ny - 1];
  pm::taper_fill<LPL>(tap, M.so_sill_taper, M.so_ek_taper, M.so_top_taper, M.so_bot_taper, nz, W * 32 + L, nthr);
  rt::syncblock();
  const long long m = rt::block_idx() * rt::warps_per_block() + W;
  if (m >= M.M) return;
  const double* src = vrow(a.bs, m);
  for (int i = L; i < sl.nyp; i += 32) bss[i] = src[i < ny ? i : ny - 1];
  rt::syncwarp();
  pm::SoPar so{};
  so.tau_ave = M.so_tau_on_y ? 0.0 : pm::mean100(vat(M.so_tau, m));
  if (M.so_tau_on_y) {
    const double* t = vrow(M.so_tau, m);
    for (int i = L; i < sl.nyp; i += 32) tau_s[i] = t[i < ny ? i : ny - 1];
    so.tau_y = tau_s;
    rt::syncwarp();
  }
  so.f = vat(M.so_f, m); so.rho = vat(M.so_rho, m); so.L = vat(M.so_L, m);
  so.KGM = vat(M.so_KGM, m); so.smax = vat(M.so_smax, m);
  so.pre0 = so.tau_ave / so.f / so.rho * so.L;
  so.sill = tap; so.ektap = tap + sl.nzp; so.toptap = tap + 2 * sl.nzp; so.bottap = tap + 3 * sl.nzp;
  so.c = BVP ? vat(M.so_c, m) : 0.0;
  so.with_Ek = M.so_bvp_with_Ek;
  double b[LPL], psi[LPL], ek[LPL], gm[LPL], ysv[LPL];
  pm::load_lev<LPL>(b, vrow(a.b, m), nz, 0.0);
  unsigned status = 0;
  const pm::SoSurf surf = pm::so_scan(ysm, bss, sinv, ny);
  pm::so_solve<LPL, BVP>(psi, ek, gm, ysv, b, ysm, bss, sinv, ny, surf, so, zs, nz, &status);
  pm::store_lev<LPL>(psi, a.Psi + m * nz, nz);
  if (a.Psi_Ek) pm::store_lev<LPL>(ek, a.Psi_Ek + m * nz, nz);
  if (a.Psi_GM) pm::store_lev<LPL>(gm, a.Psi_GM + m * nz, nz);
  if (a.ys) pm::store_lev<LPL>(ysv, a.ys + m * nz, nz);
  if (a.status && L == 0) a.status[m] |= status;
}

struct MlArgs {
  pmoc_model m;
  pmoc_vec b_basin, Psi_b;
  double dt;
  uint32_t* status;
};

// Shared memory of k_ml (in doubles).  Per block: y; per warp: b_basin and Psi_b on the levels, bs on y and the
// scratch of pm::ml_setup.
struct MlSmem {
  int nyp, off_ys, off_warp0, w_bb, w_pm, w_bs, w_scan, per_warp;
  PM_HD constexpr size_t bytes(int wpb) const { return sizeof(double) * (size_t)(off_warp0 + per_warp * wpb); }
};
PM_HD constexpr MlSmem ml_smem(int nz, int ny) {
  MlSmem s{};
  const int nzp = (nz + 3) & ~3;
  s.nyp = (ny + 3) & ~3; s.off_warp0 = s.off_ys + s.nyp;
  s.w_pm = s.w_bb + nzp; s.w_bs = s.w_pm + nzp; s.w_scan = s.w_bs + s.nyp; s.per_warp = s.w_scan + 10 * 32;
  return s;
}

// SO_ML.timestep for every member: one warp per member, b_basin / Psi_b staged in shared memory
PM_GLOBAL void k_ml(MlArgs a) {
  const pmoc_model& M = a.m;
  const int nz = M.nz, ny = M.ny, L = rt::lane(), W = rt::warp_in_block(), nthr = rt::warps_per_block() * 32;
  const MlSmem sl = ml_smem(nz, ny);
  double* sm = rt::smem();
  double* ysm = sm + sl.off_ys;
  double* ws = sm + sl.off_warp0 + (size_t)sl.per_warp * W;
  double *bb_s = ws + sl.w_bb, *pm_s = ws + sl.w_pm, *bs_s = ws + sl.w_bs, *scan_s = ws + sl.w_scan;
  for (int i = W * 32 + L; i < sl.nyp; i += nthr) ysm[i] = M.y[i < ny ? i : ny - 1];
  rt::syncblock();
  const long long m = rt::block_idx() * rt::warps_per_block() + W;
  if (m >= M.M) return;
  const double* bb = vrow(a.b_basin, m);
  const double* pb = vrow(a.Psi_b, m);
  int fnz = 0x7fffffff, fpos = 0x7fffffff;
  bool bad = false;
  for (int i = L; i < nz; i += 32) {
    const double v = pb[i];
    bb_s[i] = bb[i];
    pm_s[i] = v;
    if (v != 0.0 && i < fnz) fnz = i;
    if (v > 0.0 && i < fpos) fpos = i;
    if (i < nz - 1) bad |= !(bb[i + 1] >= bb[i]);
  }
  fnz = rt::min_i(fnz);
  fpos = rt::min_i(fpos);
  const bool sorted = rt::ballot(bad) == 0;
  rt::syncwarp();
  unsigned status = 0;
  if (fnz == 0x7fffffff) {
    status |= PMOC_ST_ML_INDEX;
  } else {
    const double held = pm_s[fnz];
    rt::syncwarp();
    for (int i = L; i < fnz; i += 32) pm_s[i] = held;
  }
  rt::syncwarp();
  pm::MlState S{};
  pm::ml_setup(S, ysm, ny, vat(M.ml_Ks, m), vat(M.ml_h, m), vat(M.ml_L, m), vat(M.ml_vpist, m), vrow(M.ml_surflux, m),
               vrow(M.ml_rest_mask, m), vrow(M.ml_b_rest, m), a.dt, scan_s);
  S.first_pos = fpos == 0x7fffffff ? -1 : fpos;
  PM_UNROLL
  for (int e = 0; e < pm::kMLP; ++e) S.bs[e] = M.ml_bs[m * ny + (pm::mlk(e) < ny ? pm::mlk(e) : ny - 1)];
  pm::ml_step(S, bb_s, pm_s, nz, sorted, bs_s, a.dt, &status);
  PM_UNROLL
  for (int e = 0; e < pm::kMLP; ++e) {
    const int k = pm::mlk(e);
    if (k < ny) {
      M.ml_bs[m * ny + k] = S.bs[e];
      if (M.ml_Psi_s) M.ml_Psi_s[m * ny + k] = S.ps[e];
    }
  }
  if (a.status && L == 0) a.status[m] |= status;
}

// A per-module kernel whose shared memory grows with nb / ny: refuse sizes one block cannot hold.
static int fail_smem(const char* what, int n, size_t bytes) {
  std::snprintf(g_err, sizeof(g_err), "%s = %d needs %zu bytes of shared memory per block, more than the %zu one block can use",
                what, n, bytes, kMaxSmemPerBlock);
  return PMOC_EUNSUPPORTED;
}

static int lpl_for(int nz) { return nz <= 64 ? 2 : (nz + 31) / 32; }

#define PM_DISPATCH_LPL(nz, CALL)                          \
  switch (lpl_for(nz)) {                                   \
    case 2: { constexpr int LPL = 2; CALL; } break;        \
    case 3: { constexpr int LPL = 3; CALL; } break;        \
    case 4: { constexpr int LPL = 4; CALL; } break;        \
    case 5: { constexpr int LPL = 5; CALL; } break;        \
    case 6: { constexpr int LPL = 6; CALL; } break;        \
    case 7: { constexpr int LPL = 7; CALL; } break;        \
    case 8: { constexpr int LPL = 8; CALL; } break;        \
    default: return fail(PMOC_EUNSUPPORTED, "nz > 256 needs the block-per-member kernel"); \
  }

int check_column(const pmoc_column& c, const char* who) {
  if (!c.b || !c.kappa.ptr || !c.dAk.ptr || !c.Area.ptr || !c.bs.ptr || !c.N2min.ptr || !c.bbot || c.nvar < 1)
    return fail(PMOC_EINVAL, who);
  return PMOC_OK;
}

int check_model(const pmoc_model* m) {
  if (!m) return fail(PMOC_EINVAL, "model is NULL");
  if (m->M <= 0 || m->nz < 3 || m->K < 1 || !m->z) return fail(PMOC_EINVAL, "bad M / nz / K / z");
  const unsigned f = m->flags;
  if (check_column(m->basin, "basin column incomplete")) return PMOC_EINVAL;
  if ((f & PMOC_HAS_NORTH) && check_column(m->north, "north column incomplete")) return PMOC_EINVAL;
  if ((f & PMOC_HAS_NORTH) && !((f & PMOC_HAS_TW) && (f & PMOC_ISO)))
    return fail(PMOC_EINVAL, "a north column needs PMOC_HAS_TW | PMOC_ISO");
  if ((f & PMOC_ISO) && !(f & PMOC_HAS_TW)) return fail(PMOC_EINVAL, "PMOC_ISO needs PMOC_HAS_TW");
  if (f & PMOC_HAS_TW) {
    if (!m->tw_f.ptr) return fail(PMOC_EINVAL, "tw_f missing");
    if (!(f & PMOC_HAS_NORTH) && !m->tw_b2.ptr) return fail(PMOC_EINVAL, "tw_b2 missing");
    if ((f & PMOC_ISO) && (!m->Psi_iso_b || !m->Psi_iso_n || m->nb < 2))
      return fail(PMOC_EINVAL, "Psi_iso_b / Psi_iso_n / nb missing");
    if (!(f & PMOC_ISO) && !m->Psi_tw) return fail(PMOC_EINVAL, "Psi_tw missing");
  }
  if (f & PMOC_HAS_SO) {
    if (!m->y || m->ny < 2 || !m->so_tau.ptr || !m->so_f.ptr || !m->so_rho.ptr || !m->so_L.ptr || !m->so_KGM.ptr ||
        !m->so_smax.ptr || !m->so_sill_taper || !m->so_ek_taper || !m->so_top_taper || !m->so_bot_taper || !m->Psi_so)
      return fail(PMOC_EINVAL, "Psi_SO parameters incomplete");
    if (!(f & PMOC_HAS_ML) && !m->so_bs.ptr) return fail(PMOC_EINVAL, "so_bs missing");
  }
  if (f & PMOC_HAS_PAC) {
    const unsigned need = PMOC_HAS_NORTH | PMOC_HAS_TW | PMOC_ISO | PMOC_HAS_SO;
    if ((f & need) != need || (f & (PMOC_HAS_ML | PMOC_ORDER_JN)))
      return fail(PMOC_EINVAL, "the two-basin topology needs basin + north + thermal wind (iso) + Psi_SO, order 'post'");
    if (check_column(m->pac, "pac column incomplete")) return PMOC_EINVAL;
    if (!m->zoc_f.ptr || !m->so2_L.ptr || !m->Psi_zon_a || !m->Psi_zon_p || !m->Psi_so2)
      return fail(PMOC_EINVAL, "zoc_f / so2_L / Psi_zon_a / Psi_zon_p / Psi_so2 missing");
    if (m->so_c.ptr) return fail(PMOC_EUNSUPPORTED, "the two-basin topology has no F2010 smoother kernel");
    if (m->nz > PMOC_MAX_NZ_WARP) return fail(PMOC_EUNSUPPORTED, "the two-basin topology needs nz <= 256");
  }
  if (((f & PMOC_HAS_ML) != 0) != ((f & PMOC_ORDER_JN) != 0))
    return fail(PMOC_EUNSUPPORTED, "SO_ML is stepped by the 'jn' loop order only (and that order needs SO_ML)");
  if (f & PMOC_HAS_ML) {
    const unsigned need = PMOC_HAS_NORTH | PMOC_HAS_TW | PMOC_ISO | PMOC_HAS_SO;
    if ((f & need) != need) return fail(PMOC_EINVAL, "the 'jn' order needs basin + north + thermal wind (iso) + Psi_SO");
    if (m->ny < 3 || m->ny > PMOC_MAX_NY_ML) return fail(PMOC_EUNSUPPORTED, "SO_ML needs 3 <= ny <= 64");
    if (!m->ml_bs || !m->ml_Ks.ptr || !m->ml_h.ptr || !m->ml_L.ptr || !m->ml_vpist.ptr || !m->ml_surflux.ptr ||
        !m->ml_rest_mask.ptr || !m->ml_b_rest.ptr)
      return fail(PMOC_EINVAL, "SO_ML parameters incomplete");
    if (!m->basin.do_conv || !m->north.do_conv) return fail(PMOC_EINVAL, "the 'jn' order steps both columns with do_conv");
    if (m->basin.bzbot.ptr || m->north.bzbot.ptr) return fail(PMOC_EINVAL, "the 'jn' order sets bbot; bzbot must be NULL");
    if ((m->basin.nvar > 1 && !m->basin.var) || (m->north.nvar > 1 && !m->north.var))
      return fail(PMOC_EINVAL, "kappa variants need the var arrays");
  }
  return PMOC_OK;
}

int run_model(const pmoc_model* m, long long it0, long long nsteps, int diagnose_only, void* stream,
              MemberList list = MemberList{nullptr, 0}) {
  if (int rc = check_model(m)) return rc;
  if (nsteps < 0 || it0 < 0) return fail(PMOC_EINVAL, "negative it0 / nsteps");
  if (!diagnose_only && nsteps == 0) return PMOC_OK;
  if (m->nz > PMOC_MAX_NZ_WARP) return pmoc_run_model_wide(m, it0, nsteps, diagnose_only, stream, list);
  if (pmoc_twcol_supported(m) && !std::getenv("PMOC_NO_TWCOL"))
    return pmoc_launch_twcol(m, it0, nsteps, diagnose_only, stream, list);
  RunArgs ra;
  ra.m = *m;
  ra.m.flags &= ~PMOC_SO_BVP;
  if ((m->flags & PMOC_HAS_SO) && m->so_c.ptr) ra.m.flags |= PMOC_SO_BVP;
  ra.it0 = it0;
  ra.nsteps = nsteps;
  ra.diagnose_only = diagnose_only;
  ra.sync_refresh = 0;
  ra.list = list;
  const int lpl = lpl_for(m->nz);
  ra.sp = plan_smem(lpl, m->ny, m->nb, ra.m.flags);
  switch (lpl) {
    case 2: return pmoc_launch_model_2(ra, stream);
    case 3: return pmoc_launch_model_3(ra, stream);
    case 4: return pmoc_launch_model_4(ra, stream);
    case 5: return pmoc_launch_model_5(ra, stream);
    case 6: return pmoc_launch_model_6(ra, stream);
    case 7: return pmoc_launch_model_7(ra, stream);
    case 8: return pmoc_launch_model_8(ra, stream);
    default: return fail(PMOC_EUNSUPPORTED, "nz > 256 needs the block-per-member kernel");
  }
}

}  // namespace pmk

// ==========================================================================================
extern "C" {

int pmoc_abi_version(void) { return PMOC_ABI_VERSION; }
const char* pmoc_last_error(void) { return g_err; }

int pmoc_device_info(int* sm_count, int* cc_major, int* cc_minor) {
#ifdef PMOC_EMU
  if (sm_count) *sm_count = 0;
  if (cc_major) *cc_major = 0;
  if (cc_minor) *cc_minor = 0;
  return PMOC_OK;
#else
  int dev = 0;
  PM_CUDA_OK(cudaGetDevice(&dev));
  cudaDeviceProp p;
  PM_CUDA_OK(cudaGetDeviceProperties(&p, dev));
  if (sm_count) *sm_count = p.multiProcessorCount;
  if (cc_major) *cc_major = p.major;
  if (cc_minor) *cc_minor = p.minor;
  return PMOC_OK;
#endif
}

uint64_t pmoc_model_scratch_bytes(const pmoc_model* m) {
  if (!m || m->nz <= PMOC_MAX_NZ_WARP) return 0;
  return sizeof(double) * ((uint64_t)4 * m->nz + (uint64_t)m->M * 6 * m->nz);
}

int pmoc_model_diagnose(const pmoc_model* m, void* stream) { return run_model(m, 0, 0, 1, stream); }

int pmoc_model_run(const pmoc_model* m, int64_t it0, int64_t nsteps, void* stream) {
  return run_model(m, it0, nsteps, 0, stream);
}

int pmoc_model_run_members(const pmoc_model* m, const int64_t* members, int64_t n, int64_t it0, int64_t nsteps,
                           void* stream) {
  if (m && (n < 0 || n > m->M)) return fail(PMOC_EINVAL, "member count outside [0, M]");
  if (n > 0 && !members) return fail(PMOC_EINVAL, "member list is NULL");
  if (n == 0 && nsteps > 0) nsteps = 0;  // an empty list validates the model and launches nothing
  return run_model(m, it0, nsteps, 0, stream, MemberList{members, n});
}

int pmoc_column_timestep(int64_t M, int32_t nz, const double* z, const pmoc_column* col, pmoc_vec wA, pmoc_vec vdx_in,
                         pmoc_vec b_in, double dt, uint32_t stages, void* stream) {
  if (M <= 0 || nz < 3 || !z || !col) return fail(PMOC_EINVAL, "bad M / nz / z / col");
  if (check_column(*col, "column incomplete")) return PMOC_EINVAL;
  if ((stages & PMOC_STAGE_VERTADVDIFF) && !wA.ptr) return fail(PMOC_EINVAL, "wA missing");
  if ((stages & PMOC_STAGE_HORADV) && (!vdx_in.ptr || !b_in.ptr)) return fail(PMOC_EINVAL, "vdx_in / b_in missing");
  ColumnArgs a{M, nz, z, *col, wA, vdx_in, b_in, dt, stages};
  PM_DISPATCH_LPL(nz, return launch(k_column<LPL>, blocks_for(M), 32 * kWarpsPerBlock,
                                    plan_smem(LPL, 0, 2, 0).bytes(kWarpsPerBlock), stream, a));
  return PMOC_OK;
}

int pmoc_thermwind_solve(int64_t M, int32_t nz, const double* z, pmoc_vec b1, pmoc_vec b2, pmoc_vec f, pmoc_vec gmid,
                         double* Psi, void* stream) {
  if (M <= 0 || nz < 3 || !z || !b1.ptr || !b2.ptr || !f.ptr || !Psi) return fail(PMOC_EINVAL, "bad thermwind arguments");
  ThermwindArgs a{};
  a.M = M; a.nz = nz; a.z = z; a.b1 = b1; a.b2 = b2; a.f = f; a.gmid = gmid; a.Psi = Psi;
  PM_DISPATCH_LPL(nz, return launch(k_thermwind<LPL>, blocks_for(M), 32 * kWarpsPerBlock, thermwind_smem(LPL).bytes(),
                                    stream, a));
  return PMOC_OK;
}

int pmoc_thermwind_psib(int64_t M, int32_t nz, int32_t nb, pmoc_vec Psi, pmoc_vec b1, pmoc_vec b2, double* psib,
                        double* bgrid, double* iso_b, double* iso_n, void* stream) {
  if (M <= 0 || nz < 3 || nb < 2 || !Psi.ptr || !b1.ptr || !b2.ptr || !psib) return fail(PMOC_EINVAL, "bad psib arguments");
  ThermwindArgs a{};
  a.M = M; a.nz = nz; a.nb = nb; a.Psi_in = Psi; a.b1 = b1; a.b2 = b2;
  a.psib = psib; a.bgrid = bgrid; a.iso_b = iso_b; a.iso_n = iso_n;
  PM_DISPATCH_LPL(nz, {
    const size_t smem = psib_smem(LPL, nb).bytes(kWarpsPerBlock);
    if (smem > kMaxSmemPerBlock) return fail_smem("nb", nb, smem);
    return launch(k_psib<LPL>, blocks_for(M), 32 * kWarpsPerBlock, smem, stream, a);
  });
  return PMOC_OK;
}

int pmoc_so_solve(const pmoc_model* so, pmoc_vec b, pmoc_vec bs, double* Psi, double* Psi_Ek, double* Psi_GM, double* ys,
                  uint32_t* status, void* stream) {
  if (!so || so->M <= 0 || so->nz < 3 || so->ny < 2 || !so->z || !so->y || !b.ptr || !bs.ptr || !Psi)
    return fail(PMOC_EINVAL, "bad Psi_SO arguments");
  if (!so->so_tau.ptr || !so->so_f.ptr || !so->so_rho.ptr || !so->so_L.ptr || !so->so_KGM.ptr || !so->so_smax.ptr ||
      !so->so_sill_taper || !so->so_ek_taper || !so->so_top_taper || !so->so_bot_taper)
    return fail(PMOC_EINVAL, "Psi_SO parameters incomplete");
  SoArgs a{};
  a.m = *so; a.b = b; a.bs = bs; a.Psi = Psi; a.Psi_Ek = Psi_Ek; a.Psi_GM = Psi_GM; a.ys = ys; a.status = status;
  const bool bvp = so->so_c.ptr != nullptr;
  PM_DISPATCH_LPL(so->nz, {
    const size_t smem = so_smem(LPL, so->ny).bytes(kWarpsPerBlock);
    if (smem > kMaxSmemPerBlock) return fail_smem("ny", so->ny, smem);
    if (bvp) return launch(k_so<LPL, true>, blocks_for(so->M), 32 * kWarpsPerBlock, smem, stream, a);
    return launch(k_so<LPL, false>, blocks_for(so->M), 32 * kWarpsPerBlock, smem, stream, a);
  });
  return PMOC_OK;
}

int pmoc_ml_timestep(const pmoc_model* ml, pmoc_vec b_basin, pmoc_vec Psi_b, double dt, uint32_t* status, void* stream) {
  if (!ml || ml->M <= 0 || ml->nz < 2 || !ml->y || !b_basin.ptr || !Psi_b.ptr) return fail(PMOC_EINVAL, "bad SO_ML arguments");
  if (ml->ny < 3 || ml->ny > PMOC_MAX_NY_ML) return fail(PMOC_EUNSUPPORTED, "SO_ML needs 3 <= ny <= 64");
  if (!ml->ml_bs || !ml->ml_Ks.ptr || !ml->ml_h.ptr || !ml->ml_L.ptr || !ml->ml_vpist.ptr || !ml->ml_surflux.ptr ||
      !ml->ml_rest_mask.ptr || !ml->ml_b_rest.ptr)
    return fail(PMOC_EINVAL, "SO_ML parameters incomplete");
  MlArgs a{};
  a.m = *ml; a.b_basin = b_basin; a.Psi_b = Psi_b; a.dt = dt; a.status = status;
  const size_t smem = ml_smem(ml->nz, ml->ny).bytes(kWarpsPerBlock);
  if (smem > 200 * 1024) return fail(PMOC_EUNSUPPORTED, "nz too large for the stand-alone SO_ML kernel");
  return launch(k_ml, blocks_for(ml->M), 32 * kWarpsPerBlock, smem, stream, a);
}

}  // extern "C"

// Runs to equilibrium (pmoc_model_equilibrate, pmoc_equilibrate_work_bytes) extend the C ABI of this unit and are
// compiled with it.
#include "pmoc_equil.cu"
