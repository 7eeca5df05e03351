// Block-per-member kernels for columns too tall for one warp (256 < nz <= 4096).  Two loop orders:
//  - 'jn' (examples/run_single_global_basin.py / run_JansenNadeau_2018.py): two convecting columns, thermal wind
//    with isopycnal remap, explicit Psi_SO, SO_ML; stepped by k_wide_steps2.
//  - 'post' (example_timestepping.py, example_twocol.py, example_twocol_plusSO.py with the explicit GM closure):
//    one column with thermal wind against a fixed profile and/or Psi_SO, or two columns with the isopycnal remap
//    and optionally Psi_SO; stepped by k_wide_post.
//
// One CTA owns one member.  The step kernels keep the buoyancy profiles and the geometry of the thread's levels in
// registers and -weff / kappa in shared memory for all the steps of a launch (see the comments on the kernels); the
// arithmetic is the bit-faithful step of pm::col_step_exact, level by level.  At the stable time step of such grids
// the streamfunctions are re-diagnosed once in hundreds to tens of thousands of steps (K = 72 000 at nz = 4096 in
// the 'jn' model), so the diagnosis is a separate, plain kernel (k_wide_refresh, shared by both orders) and the host
// loop in pmoc_run_model_wide alternates the two.
#include "pmoc_common.cuh"

#include <cstdlib>
#include <type_traits>

namespace pmk {

constexpr int kWideThreads = 256;

struct WideArgs {
  pmoc_model m;
  long long it0, nsteps;
  double* geo;   // scratch: [4][nz] dzu, 1/dzu, dzc, 1/dzc (shared by all members)
  double* memb;  // scratch: per member [6][nz]: -weff basin v0, v1, -weff north v0, v1, 1/Area basin, 1/Area north
  int force_late;  // test hook (PMOC_WIDE_FORCE_LATE=1): always take the serial schedule of the basin column
  MemberList list;
};

PM_DEV int wtid() { return rt::warp_in_block() * 32 + rt::lane(); }
// The member of this CTA (one CTA per slot of the active list).  LIST (a.list.members != NULL) is a template
// parameter of the kernels, so that a plain launch compiles to the code it had without lists.
template <bool LIST>
PM_DEV long long wide_member(const WideArgs& a) {
  return LIST ? a.list.members[rt::block_idx()] : rt::block_idx();
}
PM_DEV int wnthr() { return rt::warps_per_block() * 32; }

// ---- small block collectives on shared memory ------------------------------------------------
// exclusive prefix (reverse = false) or exclusive suffix (reverse = true) sum of a[0..n) in place;
// red: one double per thread.  Fixed association: chunk by chunk, left to right (right to left).
PM_DEV void block_scan_excl(double* a, int n, double* red, bool reverse) {
  const int T = wnthr(), t = wtid();
  const int chunk = (n + T - 1) / T;
  const int lo = t * chunk < n ? t * chunk : n, hi = lo + chunk < n ? lo + chunk : n;
  double s = 0.0;
  if (!reverse)
    for (int i = lo; i < hi; ++i) s = s + a[i];
  else
    for (int i = hi - 1; i >= lo; --i) s = s + a[i];
  red[t] = s;
  rt::syncblock();
  if (t == 0) {
    double run = 0.0;
    if (!reverse)
      for (int k = 0; k < T; ++k) { const double v = red[k]; red[k] = run; run = run + v; }
    else
      for (int k = T - 1; k >= 0; --k) { const double v = red[k]; red[k] = run; run = run + v; }
  }
  rt::syncblock();
  double run = red[t];
  if (!reverse)
    for (int i = lo; i < hi; ++i) { const double v = a[i]; a[i] = run; run = run + v; }
  else
    for (int i = hi - 1; i >= lo; --i) { const double v = a[i]; a[i] = run; run = run + v; }
  rt::syncblock();
}

// block-wide OR of a predicate / max of an int, through two shared ints
PM_DEV bool block_any(bool p, int* flag) {
  if (wtid() == 0) *flag = 0;
  rt::syncblock();
  if (rt::ballot(p) != 0 && rt::lane() == 0) rt::atomic_add_shared(flag, 1);
  rt::syncblock();
  const bool r = *flag != 0;
  rt::syncblock();
  return r;
}
PM_DEV int block_max(int v, int* slot) {
  if (wtid() == 0) *slot = -0x7fffffff;
  rt::syncblock();
  const int w = rt::max_i(v);
  if (rt::lane() == 0) rt::atomic_max_shared(slot, w);
  rt::syncblock();
  const int r = *slot;
  rt::syncblock();
  return r;
}
PM_DEV int block_min(int v, int* slot) { return -block_max(-v, slot); }
PM_DEV unsigned block_or(unsigned v, int* slot) {
  if (wtid() == 0) *slot = 0;
  rt::syncblock();
  for (unsigned bit = 1; bit <= 256u; bit <<= 1)
    if (rt::ballot((v & bit) != 0) != 0 && rt::lane() == 0) rt::atomic_or_shared(slot, (int)bit);
  rt::syncblock();
  const unsigned r = (unsigned)*slot;
  rt::syncblock();
  return r;
}

// ---- geometry -----------------------------------------------------------------------------------
PM_GLOBAL void k_wide_geo(WideArgs a) {
  const int nz = a.m.nz;
  const double* z = a.m.z;
  for (long long i = rt::block_idx() * wnthr() + wtid(); i < nz; i += (long long)wnthr() * 64) {
    double du = 1., dc = 1.;
    if (i < nz - 1) du = z[i + 1] - z[i];
    if (i >= 1 && i < nz - 1) dc = 0.5 * ((z[i + 1] - z[i]) + (z[i] - z[i - 1]));
    a.geo[i] = du;
    a.geo[nz + i] = 1. / du;
    a.geo[2 * nz + i] = dc;
    a.geo[3 * nz + i] = 1. / dc;
  }
}

// ---- diagnosis of the streamfunctions -----------------------------------------------------------
// Psi_Thermwind.solve (+ Psibz) + Psi_SO.solve for one member per CTA, results to global memory
// (same expressions as pm::tw_solve / tw_psib / interp_bgrid / so_solve, level loops instead of
// register chunks).  The parts follow the model's flags: the thermal wind against the northern column
// or the fixed profile tw_b2, the remap only with PMOC_ISO, Psi_SO on the mixed layer's bs ('jn') or on
// so_bs ('post').  The carry bit of the 'jn' switches (PMOC_ST_CARRY_SO1_EXACT) is 'jn' only.
template <bool LIST>
PM_GLOBAL void k_wide_refresh(WideArgs a) {
  const pmoc_model& M = a.m;
  const bool JN = (M.flags & PMOC_ORDER_JN) != 0, NORTH = (M.flags & PMOC_HAS_NORTH) != 0;
  const bool TW = (M.flags & PMOC_HAS_TW) != 0, ISO = (M.flags & PMOC_ISO) != 0, SO = (M.flags & PMOC_HAS_SO) != 0;
  const int nz = M.nz, ny = SO ? M.ny : 0, nb = ISO ? M.nb : 0, T = wnthr(), t = wtid();
  const long long m = wide_member<LIST>(a);
  double* sm = rt::smem();
  // six level arrays: the two profiles and four work arrays
  double *b1 = sm, *b2 = sm + nz, *A = sm + 2 * nz, *B = sm + 3 * nz, *C = sm + 4 * nz, *P = sm + 5 * nz;
  double* psib_s = sm + 6 * nz;
  const int nbp = (nb + 3) & ~3, nyp = (ny + 3) & ~3;
  int* cnt = reinterpret_cast<int*>(psib_s + nbp);
  double* red = psib_s + nbp + nbp / 2 + 2;
  double* bs_s = red + 64 + T;
  double* sinv = bs_s + nyp;
  double* ysm = sinv + nyp;
  int* ibox = reinterpret_cast<int*>(ysm + nyp);  // 4 ints of broadcast space
  const double* z = M.z;
  unsigned status = 0;

  const double* b2src = NORTH ? M.north.b + m * nz : (TW ? vrow(M.tw_b2, m) : nullptr);
  for (int i = t; i < nz; i += T) {
    b1[i] = M.basin.b[m * nz + i];
    b2[i] = b2src ? b2src[i] : 0.0;
  }
  const double* bsrc = JN ? M.ml_bs + m * ny : (SO ? vrow(M.so_bs, m) : nullptr);
  for (int i = t; i < nyp; i += T) {
    ysm[i] = M.y[i < ny ? i : ny - 1];
    bs_s[i] = bsrc[i < ny ? i : ny - 1];
  }
  rt::syncblock();

  bool exact1 = false;  // ('jn' only, see the end)
  if (TW) {
    // --- thermal wind: Psi'' = (b2-b1)/f (psi_thermwind.py:123-135), see pm::tw_solve.  A = T (Simpson
    // increments of Psi'), B = their exclusive prefix, C = cell integrals -> exclusive prefix, P = Psi (Sv)
    const double rf = 1. / vat(M.tw_f, m);
    for (int i = t; i < nz; i += T) {
      double tt = 0.0;
      if (i < nz - 1) {
        const double gi = rf * (b2[i] - b1[i]), gi1 = rf * (b2[i + 1] - b1[i + 1]);
        const double h = z[i + 1] - z[i], gm = 0.5 * (gi + gi1);
        tt = h / 6. * (gi + 4. * gm + gi1);
      }
      A[i] = tt;
      B[i] = tt;
    }
    rt::syncblock();
    block_scan_excl(B, nz, red + 64, false);
    for (int i = t; i < nz; i += T) {
      double cell = 0.0;
      if (i < nz - 1) {
        const double gi = rf * (b2[i] - b1[i]), gi1 = rf * (b2[i + 1] - b1[i + 1]);
        const double h = z[i + 1] - z[i];
        cell = h * B[i] + h * A[i] / 2. - h * h / 12. * (gi1 - gi);
      }
      C[i] = cell;
    }
    rt::syncblock();
    block_scan_excl(C, nz, red + 64, false);
    {
      const double total = C[nz - 1], z0 = z[0], H = z[nz - 1] - z[0];
      for (int i = t; i < nz; i += T) {
        const double v = pm::div_const(C[i] - total * ((z[i] - z0) / H), pm::kSv, 1.0 / pm::kSv);
        P[i] = v;
        if (M.Psi_tw) M.Psi_tw[m * nz + i] = v;
      }
    }
    rt::syncblock();
  }

  if (ISO) {
    // --- isopycnal remap (psi_thermwind.py:170-208), see pm::tw_psib
    double lo = INFINITY, hi = -INFINITY;
    bool unsorted = false;
    for (int i = t; i < nz; i += T) {
      lo = b1[i] < lo ? b1[i] : lo;
      lo = b2[i] < lo ? b2[i] : lo;
      hi = b1[i] > hi ? b1[i] : hi;
      hi = b2[i] > hi ? b2[i] : hi;
      if (i < nz - 1) {
        const double u = -(P[i + 1] - P[i]);
        unsorted |= !(b1[i + 1] >= b1[i]) || !(b2[i + 1] >= b2[i]) || u != u;
        if (u < 0 ? pm::remap_tie(b2[i], b2[i + 1], u, i == 0) : pm::remap_tie(b1[i], b1[i + 1], u, i == 0)) status |= PMOC_ST_TIE_CELL;
      }
    }
    lo = rt::wmin(lo);
    hi = rt::wmax(hi);
    if (rt::lane() == 0) {
      red[rt::warp_in_block()] = lo;
      red[32 + rt::warp_in_block()] = hi;
    }
    rt::syncblock();
    for (int w = 0; w < rt::warps_per_block(); ++w) {
      const double l = red[w], h2 = red[32 + w];
      lo = (l < lo || lo != lo) ? l : lo;
      hi = (h2 > hi || hi != hi) ? h2 : hi;
    }
    rt::syncblock();
    pm::BGrid G;
    G.lo = lo;
    G.hi = hi;
    G.nb = nb;
    G.step = (hi - lo) / (double)(nb - 1);
    G.rstep = 1.0 / G.step;
    const bool direct = block_any(unsorted, ibox);
    // transport of cell c and the column it is taken from
    auto cell_u = [&](int c) { return -(P[c + 1] - P[c]); };
    if (!direct) {
      // A = S_1, B = S_2: S_X[k] = sum_{c >= k} [cell c uses X] u_c  (exclusive suffix + own)
      for (int i = t; i < nz; i += T) {
        const double u = i < nz - 1 ? cell_u(i) : 0.0;
        A[i] = u < 0 ? 0.0 : u;
        B[i] = u < 0 ? u : 0.0;
      }
      rt::syncblock();
      block_scan_excl(A, nz, red + 64, true);
      block_scan_excl(B, nz, red + 64, true);
      for (int i = t; i < nz; i += T) {
        const double u = i < nz - 1 ? cell_u(i) : 0.0;
        A[i] = A[i] + (u < 0 ? 0.0 : u);
        B[i] = B[i] + (u < 0 ? u : 0.0);
      }
      for (int i = t; i <= nb; i += T) cnt[i] = 0;
      rt::syncblock();
      for (int i = t; i < nz; i += T) {
        rt::atomic_add_shared(&cnt[pm::bgrid_count_le(G, b1[i])], 1);
        rt::atomic_add_shared(&cnt[pm::bgrid_count_le(G, b2[i])], 1 << 16);
      }
      rt::syncblock();
      if (t == 0) {  // inclusive prefix over the classes (nb is a few hundred)
        int run = 0;
        for (int i = 0; i <= nb; ++i) {
          run += cnt[i];
          cnt[i] = run;
        }
      }
      rt::syncblock();
      for (int i = t; i < nb; i += T) {
        const double x = G.at(i);
        const int k1 = cnt[i] & 0xffff, k2 = cnt[i] >> 16;  // #{levels with bX < x}
        double c1 = 0.0, c2 = 0.0;
        if (k1 < nz) {
          const double bk = b1[k1];
          c1 = A[k1];
          if (k1 > 0 && bk != x) {
            const double u = cell_u(k1 - 1);
            c1 = c1 + (bk - x) * (u < 0 ? 0.0 : u / (bk - b1[k1 - 1]));
          }
          if (bk == x)  // flat cells taken from column 1 sitting exactly on the class: 0/0 in the reference
            for (int c = k1; c + 1 < nz && b1[c + 1] == x; ++c)
              if (!(cell_u(c) < 0)) c1 = NAN;
        }
        if (k2 < nz) {
          const double bk = b2[k2];
          c2 = B[k2];
          if (k2 > 0 && bk != x) {
            const double u = cell_u(k2 - 1);
            c2 = c2 + (bk - x) * (u < 0 ? u / (bk - b2[k2 - 1]) : 0.0);
          }
          if (bk == x)
            for (int c = k2; c + 1 < nz && b2[c + 1] == x; ++c)
              if (cell_u(c) < 0) c2 = NAN;
        }
        psib_s[i] = c1 + c2;
      }
    } else {
      // direct path: every class against every cell (inverted cells / NaN)
      for (int i = t; i < nb; i += T) {
        const double bg = G.at(i);
        double acc = 0.0;
        for (int c = 0; c < nz - 1; ++c) {
          const double u = cell_u(c);
          const bool from2 = u < 0;
          const double bot = from2 ? b2[c] : b1[c], top = from2 ? b2[c + 1] : b1[c + 1];
          double f = (top - bg) * (1.0 / (top - bot));
          f = f < 0. ? 0. : f;
          f = f > 1. ? 1. : f;
          acc = rt::fma(f, u, acc);
        }
        psib_s[i] = acc;
      }
    }
    rt::syncblock();
    for (int i = t; i < nb; i += T) {
      if (M.psib) M.psib[m * nb + i] = psib_s[i];
      if (M.bgrid) M.bgrid[m * nb + i] = G.at(i);
    }
    for (int i = t; i < nz; i += T) {
      M.Psi_iso_b[m * nz + i] = pm::interp_bgrid(b1[i], G, psib_s);
      M.Psi_iso_n[m * nz + i] = pm::interp_bgrid(b2[i], G, psib_s);
    }
  }

  if (SO) {
    // --- Psi_SO.solve, explicit GM branch (psi_SO.py:106-140, 218-243, 302-354), see pm::so_solve
    const pm::SoSurf S = pm::so_scan(ysm, bs_s, sinv, ny);  // every warp redundantly, same values
    rt::syncblock();
    if (!S.mono) status |= PMOC_ST_BS_NONMONOTONE;
    if (S.ndown >= pm::kSawtoothSegments) status |= PMOC_ST_BS_SAWTOOTH;
    const double tau_ave = pm::mean100(vat(M.so_tau, m));
    pm::SoPar P{};  // (constant wind stress: tau_y = nullptr; tapers in natural order)
    P.L = vat(M.so_L, m);
    P.KGM = vat(M.so_KGM, m);
    P.smax = vat(M.so_smax, m);
    P.sill = M.so_sill_taper; P.ektap = M.so_ek_taper; P.toptap = M.so_top_taper; P.bottap = M.so_bot_taper;
    const double pre = tau_ave / vat(M.so_f, m) / vat(M.so_rho, m) * P.L;
    for (int i = t; i < nz; i += T) {
      const double bi = b1[i];
      double yo;
      if (bi < S.mn)
        yo = S.y0 - 1e3;
      else if (bi > S.bsN)
        yo = S.yN;
      else if (S.mono && S.south < ny - 1)
        yo = pm::outcrop_monotone(bi, ysm, bs_s, sinv, ny, S.south);
      else {
        bool bad = false;
        yo = pm::outcrop_brent(bi, ysm, bs_s, ny, S.south, &bad);
        if (bad) status |= PMOC_ST_BRENT_SIGN;
      }
      const double e = pm::so_ekman(pre, P, i);
      double dy = S.yN - yo;
      dy = 0.1 > dy ? 0.1 : dy;
      double g = pm::so_gm_clip(pm::qdiv(z[i], dy), P, i, i, exact1);
      g = pm::so_gm_limit(g, e, dy, S.yN - S.y0, P, i, exact1);
      const double v = i == 0 ? 0. : e + g;
      M.Psi_so[m * nz + i] = v;
      if (M.Psi_Ek) M.Psi_Ek[m * nz + i] = e;
      if (M.Psi_GM) M.Psi_GM[m * nz + i] = g;
    }
  }
  const unsigned all = block_or(status, ibox);
  if (!JN) {
    if (t == 0 && M.status) M.status[m] = status_word(M.status[m], all, false);
    return;
  }
  // whether Psi_so[1] came out of state-independent arithmetic, for the step kernel's noise classification
  rt::syncblock();
  if (t == 1 % T) red[0] = exact1 ? 1.0 : 0.0;  // the thread that owns level 1
  rt::syncblock();
  if (t == 0 && M.status) M.status[m] = status_word(M.status[m], all, red[0] != 0.0);
}

// ---- the steps, state and per-level constants resident on chip ---------------------------------
// 256 column threads own LPT consecutive levels each (both columns): the buoyancies, dz, 1/dz and
// 1/dzc of those levels stay in registers for the whole launch; -weff and kappa of the variant in
// use live in shared memory in owner-major order (slot j*256 + t: conflict free, re-read from the
// scratch buffer by their owner when a boundary switch flips the variant).  What the neighbours and
// the mixed layer need is published once per step: the basin profile in natural order with one pad
// word per LPT levels (conflict-free stores, read through pm::PadIdx) and the first/last northern
// level of every thread.  The arithmetic is the bit-faithful step of pm::col_step_exact.
//
// SO_ML runs on a ninth warp of its own, one step behind the columns.  The script's order is
// columns(ii) -> SO_ML(ii) -> columns(ii+1), but columns(ii+1) sees SO_ML(ii) only through
// channel.bs[0] in the bottom-boundary switches of the basin (run_JansenNadeau_2018.py:235-246): its
// bottom value bbot, i.e. levels 0 and 1 of thread 0, and -- only when Psi_SO[1] >= 0, Psi_res_b[1] > 0
// and north.b[0] < basin.b[1] -- the choice of the kappa profile.  So per iteration:
//   phase 1   the mixed-layer warp does SO_ML(ii-1) on the profile published after columns(ii-1) (a single
//             dependent chain of ~900 instructions) WHILE the column warps do columns(ii): the whole northern
//             column, and the basin except the two bottom levels (thread 0 keeps the gradient of cell 1-2);
//   barrier;
//   phase 2   bs[0] is known: the switches are evaluated exactly as written, thread 0 finishes basin levels
//             0 and 1, everything is published;  barrier.
// In the rare "late" case (the kappa choice hangs on bs[0]) the basin column waits for phase 2.  Same
// operations on the same operands as the serial order: bit-identical results; the SO_ML chain, which
// was 60 % of the step with seven warps idle at a barrier, is hidden behind the column work.
//
// PIPE = false (16 levels per thread, nz > 2048): a ninth warp would put three warps on one SM sub-partition
// and cap the kernel at 168 registers, and with 80 doubles of column state per thread the spills then cost more
// than the overlap gains (measured at nz = 4096: 65 ms against 52 ms).  There the eighth column warp runs SO_ML
// after its own column work, its state parked in shared memory: same schedule and barriers, no overlap.
// Measured gain of the pipelined form: nz = 1024 +18 %, nz = 2048 +10 %.
constexpr int kWideCol = 256;

template <int LPT, int SH, bool PIPE, bool LIST>
PM_GLOBAL void PM_LAUNCH_BOUNDS(kWideCol + (PIPE ? 32 : 0), 1) k_wide_steps2(WideArgs a) {
  constexpr int kWideAll = kWideCol + (PIPE ? 32 : 0);
  static_assert((1 << SH) == LPT && LPT >= 2, "LPT = 2^SH >= 2");
  const pmoc_model& M = a.m;
  const int nz = M.nz, ny = M.ny, t = wtid(), W = rt::warp_in_block(), Ln = rt::lane();
  const bool col = t < kWideCol, mlw = W == (PIPE ? kWideCol / 32 : kWideCol / 32 - 1);
  const long long m = wide_member<LIST>(a);
  const double dt = M.dt;
  constexpr int nzp = kWideCol * LPT;
  const int nyp = (ny + 3) & ~3;
  double* sm = rt::smem();
  double *nwb = sm, *nwn = sm + nzp, *kb = sm + 2 * nzp, *kn = sm + 3 * nzp;
  double* bbp = sm + 4 * nzp;            // basin profile, padded natural order: nzp + kWideCol
  double* pm_s = bbp + nzp + kWideCol;   // Psi_mod, natural order
  double* bne = pm_s + nzp;              // north: first/last level of every thread, [2*kWideCol] = level 1
  double* bs_s = bne + 2 * kWideCol + 2;
  double* scan_s = bs_s + nyp;
  double* ysm = scan_s + 320;
  double* dbox = ysm + nyp;                           // [0] = bs[0] of the mixed layer
  int* ibox = reinterpret_cast<int*>(dbox + 8);       // 2 x 8 step flags, then 4 ints for the block collectives
  int* cbox = ibox + 16;
  double* mlp = dbox + 8 + 10;                        // parked mixed layer (PIPE = false), pm::kMlSave
  const pm::PadIdx bbx{bbp, SH};
  const double* z = M.z;
  const int lo = t * LPT;
  double* mem = a.memb + (size_t)m * 6 * nz;
  double *nwb0 = mem, *nwb1 = mem + nz, *nwn0 = mem + 2 * nz, *nwn1 = mem + 3 * nz, *rab = mem + 4 * nz,
         *ran = mem + 5 * nz;
  const double* kapb = vrow(M.basin.kappa, m);
  const double* kapn = vrow(M.north.kappa, m);
  const double* dakb = vrow(M.basin.dAk, m);
  const double* dakn = vrow(M.north.dAk, m);
  const double* Ab = vrow(M.basin.Area, m);
  const double* An = vrow(M.north.Area, m);
  const int nvb = M.basin.nvar > 1 ? nz : 0, nvn = M.north.nvar > 1 ? nz : 0;  // offset of variant 1
  unsigned status = 0;

  int var_b = (M.basin.var && M.basin.nvar > 1) ? M.basin.var[m] : 0;
  int var_n = (M.north.var && M.north.nvar > 1) ? M.north.var[m] : 0;
  double bbot_b = M.basin.bbot[m], bbot_n = M.north.bbot[m];
  const double bs_b = vat(M.basin.bs, m), bs_n = vat(M.north.bs, m);
  const double n2_b = vat(M.basin.N2min, m), n2_n = vat(M.north.N2min, m);

  // ---- load: state, geometry, tables ----
  double bb[LPT], bn[LPT], dzu[LPT], rdzu[LPT], rdzc[LPT];
  double dzu_m = 1., rdzu_m = 1.;  // cell below the thread's first level
  int fnz = 0x7fffffff, fpos = 0x7fffffff;
  bool areas_differ = false;
  double mxl = 0.0;  // largest |Psi| of the three streamfunctions: the scale of rounding noise
  PM_UNROLL
  for (int j = 0; j < LPT; ++j) {
    const int i = lo + j;
    bb[j] = bn[j] = 0.;
    dzu[j] = rdzu[j] = rdzc[j] = 1.;
    if (col) {  // boundary and padding levels: zero -weff and kappa make their update an exact no-op
      const int s = j * kWideCol + t;
      nwb[s] = nwn[s] = kb[s] = kn[s] = 0.0;
    }
    if (col && i < nz) {
      bb[j] = M.basin.b[m * nz + i];
      bn[j] = M.north.b[m * nz + i];
      dzu[j] = a.geo[i];
      rdzu[j] = a.geo[nz + i];
      rdzc[j] = a.geo[3 * nz + i];
      const double pso = M.Psi_so[m * nz + i], ib = M.Psi_iso_b[m * nz + i], in_ = M.Psi_iso_n[m * nz + i];
      pm_s[i] = pso;
      mxl = fmax(mxl, fmax(fabs(pso), fmax(fabs(ib), fabs(in_))));
      if (pso != 0.0 && i < fnz) fnz = i;
      if (pso > 0.0 && i < fpos) fpos = i;
      const bool in = i >= 1 && i < nz - 1;
      const double wAb = (ib - pso) * 1e6, wAn = -in_ * 1e6;
      const double b0 = in ? -(wAb - dakb[i]) : 0.0, b1 = in ? -(wAb - dakb[nvb + i]) : 0.0;
      const double n0 = in ? -(wAn - dakn[i]) : 0.0, n1 = in ? -(wAn - dakn[nvn + i]) : 0.0;
      nwb0[i] = b0; nwb1[i] = b1; nwn0[i] = n0; nwn1[i] = n1;
      const int s = j * kWideCol + t;
      nwb[s] = var_b ? b1 : b0;
      nwn[s] = var_n ? n1 : n0;
      kb[s] = in ? kapb[(var_b ? nvb : 0) + i] : 0.0;
      kn[s] = in ? kapn[(var_n ? nvn : 0) + i] : 0.0;
      if (in) areas_differ |= Ab[i] != Ab[1] || An[i] != An[1];
      rab[i] = 1.0 / Ab[i];
      ran[i] = 1.0 / An[i];
    }
  }
  if (col && lo >= 1 && lo - 1 < nz) {
    dzu_m = a.geo[lo - 1];
    rdzu_m = a.geo[nz + lo - 1];
  }
  for (int i = t; i < nyp; i += kWideAll) ysm[i] = M.y[i < ny ? i : ny - 1];
  mxl = rt::wmax(mxl);
  if (Ln == 0) scan_s[W] = mxl;  // (scan_s is free until ml_setup, behind the barriers below)
  fnz = block_min(fnz, cbox);
  fpos = block_min(fpos, cbox);
  const bool uniA = !block_any(areas_differ, cbox);
  const double A_b = Ab[1], rA_b = 1.0 / A_b, A_n = An[1], rA_n = 1.0 / A_n;
  const double psi_so1 = M.Psi_so[m * nz + 1], res_b1 = M.Psi_iso_b[m * nz + 1], res_n1 = M.Psi_iso_n[m * nz + 1];
  // which of the three are rounding noise, classified from the loaded streamfunctions as k_model does
  for (int w = 0; w < rt::warps_per_block(); ++w) mxl = fmax(mxl, scan_s[w]);
  const bool so1_exact = so1_exact_carried(M, m);
  const unsigned noise = pm::jn_noise(psi_so1, res_b1, res_n1, mxl, so1_exact);
  if (fnz == 0x7fffffff) status |= PMOC_ST_ML_INDEX;
  const double held = pm_s[fnz == 0x7fffffff ? 0 : fnz];
  rt::syncblock();
  for (int i = t; i < nz && i < fnz; i += kWideAll) pm_s[i] = held;

  pm::MlState ml{};  // PIPE: lives in the registers of the mixed-layer warp; otherwise parked in shared memory
  if (mlw) {
    pm::ml_setup(ml, ysm, ny, vat(M.ml_Ks, m), vat(M.ml_h, m), vat(M.ml_L, m), vat(M.ml_vpist, m), vrow(M.ml_surflux, m),
                 vrow(M.ml_rest_mask, m), vrow(M.ml_b_rest, m), dt, scan_s);
    ml.first_pos = fpos == 0x7fffffff ? -1 : fpos;
    PM_UNROLL
    for (int e = 0; e < pm::kMLP; ++e) ml.bs[e] = M.ml_bs[m * ny + (pm::mlk(e) < ny ? pm::mlk(e) : ny - 1)];
    if (Ln == 0) {
      dbox[0] = ml.bs[0];
      for (int k = 0; k < 16; ++k) ibox[k] = (k & 7) == 2 || (k & 7) == 3 ? -1 : 0;
    }
    if (!PIPE) pm::ml_park(ml, mlp, true);
  }
  rt::syncblock();

  // publish the state and the flags the next step needs (buffer q): what the neighbours read, whether
  // anything convects and the highest stable level (column.py:264-267), whether b_basin is sorted
  bool mine_b = false, mine_n = false;  // the thread's own levels hold something that convects
  const bool full = lo + LPT <= nz, owns_top = lo <= nz - 1 && nz - 1 < lo + LPT;
  double* const bbo = bbp + t * (LPT + 1);  // = &bbp[pad(lo)]: pad(lo + j) = lo + j + t
  auto publish_as = [&](int q, auto FULL) {
    constexpr bool fl = decltype(FULL)::value;
    int topb = -1, topn = -1;
    bool anyb = false, anyn = false, bad = false;
    PM_UNROLL
    for (int j = 0; j < LPT; ++j) {
      const int i = lo + j;
      if (fl || i < nz) {
        bbo[j] = bb[j];
        if (bb[j] > bs_b) anyb = true; else topb = i;
        if (bn[j] > bs_n) anyn = true; else topn = i;
        if (j + 1 < LPT && (fl || i + 1 < nz)) bad |= !(bb[j + 1 < LPT ? j + 1 : j] >= bb[j]);
      }
    }
    mine_b = anyb;
    mine_n = anyn;
    const double upb = rt::shfl_down(bb[0], 1);  // first level of the next thread (same warp)
    if (Ln < 31 && lo + LPT < nz) bad |= !(upb >= bb[LPT - 1]);
    bne[2 * t] = bn[0];
    bne[2 * t + 1] = bn[LPT - 1];
    if (t == 0) bne[2 * kWideCol] = bn[1];
    const unsigned mb = rt::ballot(anyb), mn = rt::ballot(anyn), mu = rt::ballot(bad);
    const int wb = rt::max_i(topb), wn = rt::max_i(topn);
    if (Ln == 0) {
      int* f = ibox + 8 * q;
      if (mb) rt::atomic_add_shared(&f[0], 1);
      if (mn) rt::atomic_add_shared(&f[1], 1);
      rt::atomic_max_shared(&f[2], wb);
      rt::atomic_max_shared(&f[3], wn);
      if (mu) rt::atomic_or_shared(&f[4], 1);
    }
  };
  auto publish = [&](int q) {
    if (rt::ballot(!full) == 0)
      publish_as(q, std::true_type{});
    else
      publish_as(q, std::false_type{});
  };
  if (col) publish(0);
  rt::syncblock();

  // the owner re-reads its levels of kappa variant v of one column: -weff of both variants from the scratch buffer
  // (nw0, nw1), kappa from the model (variant 1 at offset nv)
  auto load_variant = [&](double* nw, double* kp, const double* nw0, const double* nw1, const double* kap, int nv,
                          int v) {
    PM_UNROLL
    for (int j = 0; j < LPT; ++j) {
      const int i = lo + j, s = j * kWideCol + t;
      if (i < nz) {
        nw[s] = v ? nw1[i] : nw0[i];
        kp[s] = (i >= 1 && i < nz - 1) ? kap[(v ? nv : 0) + i] : 0.0;
      }
    }
  };
  // one SO_ML step of the mixed-layer warp on the profile published with the flags of buffer q; b_basin sorted?
  // inside the threads and warps: flagged by publish; across the warps: here.  bs[0] goes to dbox[0].
  auto ml_published = [&](pm::MlState& s, int q) {
    bool bad = ibox[8 * q + 4] != 0;
    const int e = (Ln + 1) * 32 * LPT;  // first level of the next warp
    if (Ln < kWideCol / 32 - 1 && e < nz) bad |= !(bbx[e] >= bbx[e - 1]);
    pm::ml_step(s, bbx, pm_s, nz, rt::ballot(bad) == 0, bs_s, dt, &status);
    if (Ln == 0) dbox[0] = s.bs[0];
  };

  int p = 0;
  if constexpr (PIPE) {
    for (long long it = 0; it < a.nsteps; ++it, p ^= 1) {
      // ---------------------------------------------------------------- phase 1
      double gb1 = 0.;   // thread 0: gradient of basin cell 1-2 (kept for the deferred bottom levels)
      // the basin's kappa profile hangs on bs[0] of the SO_ML step still running (block-uniform: every thread,
      // the mixed-layer warp included, evaluates it from the published values)
      const bool late = (psi_so1 >= 0 && res_b1 > 0 && bne[0] < bbp[1] && M.basin.nvar > 1) || a.force_late != 0;
      if (mlw) {
        // SO_ML of the previous iteration, then clear the flags this iteration publishes (last read in the previous one)
        if (it > 0) ml_published(ml, p);
        if (Ln == 0) {
          int* f = ibox + 8 * (p ^ 1);
          f[0] = 0; f[1] = 0; f[2] = -1; f[3] = -1; f[4] = 0;
        }
      } else {
        // what the switches need apart from bs[0]; every thread evaluates them from the published values
        const double bb0 = bbp[0], nb1 = bne[2 * kWideCol];
        int vn = var_n;
        pm::jn_switch_north(res_n1, bb0, nb1, bbot_n, vn);
        if (M.north.nvar < 2) vn = 0;
        int vb = psi_so1 < 0 ? 1 : 0;  // (exact unless late; then phase 2 decides)
        if (M.basin.nvar < 2) vb = 0;
        if (!late && vb != var_b) {
          var_b = vb;
          load_variant(nwb, kb, nwb0, nwb1, kapb, nvb, vb);
        }
        if (vn != var_n) {
          var_n = vn;
          load_variant(nwn, kn, nwn0, nwn1, kapn, nvn, vn);
        }
        // convective adjustment of the own levels and of the two neighbour values
        const int* f = ibox + 8 * p;
        const bool cvb = f[0] != 0, cvn = f[1] != 0;
        const double zcb = z[f[2] >= 0 ? f[2] : 0], zcn = z[f[3] >= 0 ? f[3] : 0];
        if ((cvb && mine_b) || (cvn && mine_n) || owns_top) {
          PM_UNROLL
          for (int j = 0; j < LPT; ++j) {
            const int i = lo + j;
            if (i < nz) {
              bb[j] = pm::convect_level(bb[j], i, cvb, bs_b, n2_b, zcb, z, nz);
              bn[j] = pm::convect_level(bn[j], i, cvn, bs_n, n2_n, zcn, z, nz);
            }
          }
        }
        if (t == 0) bn[0] = bbot_n;  // column.py:232 (the basin's bottom value waits for bs[0]: phase 2)
        double gpb = 0., gpn = 0.;  // gradient of the cell below the current level
        if (lo >= 1 && lo < nz) {
          const double vb_ = pm::convect_level(bbx[lo - 1], lo - 1, cvb, bs_b, n2_b, zcb, z, nz);
          const double vn_ = pm::convect_level(bne[2 * (t - 1) + 1], lo - 1, cvn, bs_n, n2_n, zcn, z, nz);
          gpb = pm::div_const(bb[0] - vb_, dzu_m, rdzu_m);
          gpn = pm::div_const(bn[0] - vn_, dzu_m, rdzu_m);
        }
        double ub = 0., un = 0.;  // level above the thread's last one
        if (lo + LPT < nz) {
          ub = pm::convect_level(bbx[lo + LPT], lo + LPT, cvb, bs_b, n2_b, zcb, z, nz);
          un = pm::convect_level(bne[2 * (t + 1)], lo + LPT, cvn, bs_n, n2_n, zcn, z, nz);
        }
        // the explicit step.  No level tests: at the boundary and padding levels -weff = kappa = 0 and every operand
        // is finite, so b + dt*0 = b.  BASIN: both columns (false: the northern one only); thread 0 leaves basin
        // levels 0 and 1 to phase 2.
        auto step = [&](auto UA, auto BASIN) {
          constexpr bool ua = decltype(UA)::value, basin = decltype(BASIN)::value;
          PM_UNROLL
          for (int j = 0; j < LPT; ++j) {
            const int s = j * kWideCol + t;
            const double upb = j + 1 < LPT ? bb[j + 1 < LPT ? j + 1 : j] : ub;
            const double upn = j + 1 < LPT ? bn[j + 1 < LPT ? j + 1 : j] : un;
            const double gn = pm::div_const(upn - bn[j], dzu[j], rdzu[j]);
            const double dzc = 0.5 * (dzu[j] + (j > 0 ? dzu[j > 0 ? j - 1 : 0] : dzu_m));
            double Ai_b = A_b, rAi_b = rA_b, Ai_n = A_n, rAi_n = rA_n;
            if (!ua) {
              const int i = lo + j < nz ? lo + j : nz - 1;
              Ai_b = Ab[i]; rAi_b = rab[i]; Ai_n = An[i]; rAi_n = ran[i];
            }
            if (basin) {
              const double gb = pm::div_const(upb - bb[j], dzu[j], rdzu[j]);
              if (j >= 2 || t != 0)
                bb[j] = pm::exact_level(bb[j], gb, gpb, dzc, rdzc[j], nwb[s], kb[s], Ai_b, rAi_b, dt);
              else if (j == 1)
                gb1 = gb;
              gpb = gb;
            }
            bn[j] = pm::exact_level(bn[j], gn, gpn, dzc, rdzc[j], nwn[s], kn[s], Ai_n, rAi_n, dt);
            gpn = gn;
          }
        };
        if (!late) {
          if (uniA) step(std::true_type{}, std::true_type{});
          else step(std::false_type{}, std::true_type{});
        } else {
          if (uniA) step(std::true_type{}, std::false_type{});
          else step(std::false_type{}, std::false_type{});
        }
      }
      rt::syncblock();  // SO_ML of the previous iteration is done; every neighbour value of this step has been read
      // ---------------------------------------------------------------- phase 2
      if (col) {
        // the switches as the script writes them, now that bs[0] is known
        const double bb0 = bbp[0], bb1 = bbp[1], nb0 = bne[0], nb1 = bne[2 * kWideCol], bs0 = dbox[0];
        int vb = var_b;
        pm::jn_switch_basin(psi_so1, res_b1, bb1, nb0, bs0, bbot_b, vb);
        pm::jn_noise_hit(noise, bb0, bb1, nb0, nb1, bs0, &status);
        if (M.basin.nvar < 2) vb = 0;
        if (late) {
          // the whole basin column, serially after SO_ML (the values the neighbours need are still the published ones)
          if (vb != var_b) {
            var_b = vb;
            load_variant(nwb, kb, nwb0, nwb1, kapb, nvb, vb);
          }
          const int* f = ibox + 8 * p;
          const bool cvb = f[0] != 0;
          const double zcb = z[f[2] >= 0 ? f[2] : 0];
          if (t == 0) bb[0] = bbot_b;
          double gpb = 0.;
          if (lo >= 1 && lo < nz)
            gpb = pm::div_const(bb[0] - pm::convect_level(bbx[lo - 1], lo - 1, cvb, bs_b, n2_b, zcb, z, nz), dzu_m, rdzu_m);
          const double ub = lo + LPT < nz ? pm::convect_level(bbx[lo + LPT], lo + LPT, cvb, bs_b, n2_b, zcb, z, nz) : 0.;
          PM_UNROLL
          for (int j = 0; j < LPT; ++j) {
            const int s = j * kWideCol + t;
            const double upb = j + 1 < LPT ? bb[j + 1 < LPT ? j + 1 : j] : ub;
            const double gb = pm::div_const(upb - bb[j], dzu[j], rdzu[j]);
            const double dzc = 0.5 * (dzu[j] + (j > 0 ? dzu[j > 0 ? j - 1 : 0] : dzu_m));
            const int i = lo + j < nz ? lo + j : nz - 1;
            // (the Area as a value: bound to a reference, the select would let the compiler read Ab[i] unconditionally)
            bb[j] = pm::exact_level(bb[j], gb, gpb, dzc, rdzc[j], nwb[s], kb[s], double(uniA ? A_b : Ab[i]),
                                    double(uniA ? rA_b : rab[i]), dt);
            gpb = gb;
          }
        } else if (t == 0) {
          // basin levels 0 and 1 (column.py:232, 235-249): b[0] = bbot, then level 1 with the kept gradient above it
          bb[0] = bbot_b;
          const double g0 = pm::div_const(bb[1] - bb[0], dzu[0], rdzu[0]);
          const double dzc = 0.5 * (dzu[1] + dzu[0]);
          const int s = 1 * kWideCol + 0;
          bb[1] = pm::exact_level(bb[1], gb1, g0, dzc, rdzc[1], nwb[s], kb[s], double(uniA ? A_b : Ab[1]),
                                  double(uniA ? rA_b : rab[1]), dt);
        }
      }
      if (late) rt::syncblock();  // the serial basin step read the published neighbour values: only now overwrite them
      if (col) publish(p ^ 1);
      rt::syncblock();
    }
    if (mlw && a.nsteps > 0) ml_published(ml, p);  // SO_ML of the last iteration
    rt::syncblock();

  } else {
    // sixteen levels per thread: the serial schedule (columns, barrier, publish, barrier, SO_ML on the last column warp,
    // barrier) -- the deferral logic of the pipelined form costs registers this variant does not have
    for (long long it = 0; it < a.nsteps; ++it, p ^= 1) {
      if (col) {
        // bottom boundary condition and bottom-boundary-layer kappa; every thread evaluates the switches from the
        // published values
        const double bb0 = bbp[0], bb1 = bbp[1], nb0 = bne[0], nb1 = bne[2 * kWideCol], bs0 = dbox[0];
        int vb = var_b, vn = var_n;
        pm::jn_switch_basin(psi_so1, res_b1, bb1, nb0, bs0, bbot_b, vb);
        pm::jn_switch_north(res_n1, bb0, nb1, bbot_n, vn);
        pm::jn_noise_hit(noise, bb0, bb1, nb0, nb1, bs0, &status);
        if (M.basin.nvar < 2) vb = 0;
        if (M.north.nvar < 2) vn = 0;
        if (vb != var_b) {
          var_b = vb;
          load_variant(nwb, kb, nwb0, nwb1, kapb, nvb, vb);
        }
        if (vn != var_n) {
          var_n = vn;
          load_variant(nwn, kn, nwn0, nwn1, kapn, nvn, vn);
        }
        // convective adjustment of the own levels and of the two neighbour values
        const int* f = ibox + 8 * p;
        const bool cvb = f[0] != 0, cvn = f[1] != 0;
        const double zcb = z[f[2] >= 0 ? f[2] : 0], zcn = z[f[3] >= 0 ? f[3] : 0];
        if ((cvb && mine_b) || (cvn && mine_n) || owns_top) {
          PM_UNROLL
          for (int j = 0; j < LPT; ++j) {
            const int i = lo + j;
            if (i < nz) {
              bb[j] = pm::convect_level(bb[j], i, cvb, bs_b, n2_b, zcb, z, nz);
              bn[j] = pm::convect_level(bn[j], i, cvn, bs_n, n2_n, zcn, z, nz);
            }
          }
        }
        if (t == 0) {  // column.py:232
          bb[0] = bbot_b;
          bn[0] = bbot_n;
        }
        double gpb = 0., gpn = 0.;  // gradient of the cell below the current level
        if (lo >= 1 && lo < nz) {
          const double vb_ = pm::convect_level(bbx[lo - 1], lo - 1, cvb, bs_b, n2_b, zcb, z, nz);
          const double vn_ = pm::convect_level(bne[2 * (t - 1) + 1], lo - 1, cvn, bs_n, n2_n, zcn, z, nz);
          gpb = pm::div_const(bb[0] - vb_, dzu_m, rdzu_m);
          gpn = pm::div_const(bn[0] - vn_, dzu_m, rdzu_m);
        }
        double ub = 0., un = 0.;  // level above the thread's last one
        if (lo + LPT < nz) {
          ub = pm::convect_level(bbx[lo + LPT], lo + LPT, cvb, bs_b, n2_b, zcb, z, nz);
          un = pm::convect_level(bne[2 * (t + 1)], lo + LPT, cvn, bs_n, n2_n, zcn, z, nz);
        }
        // the explicit step.  No level tests: at the boundary and padding levels -weff = kappa = 0 and every operand
        // is finite, so b + dt*0 = b.
        auto step = [&](auto UA) {
          constexpr bool ua = decltype(UA)::value;
          PM_UNROLL
          for (int j = 0; j < LPT; ++j) {
            const int s = j * kWideCol + t;
            const double upb = j + 1 < LPT ? bb[j + 1 < LPT ? j + 1 : j] : ub;
            const double upn = j + 1 < LPT ? bn[j + 1 < LPT ? j + 1 : j] : un;
            const double gb = pm::div_const(upb - bb[j], dzu[j], rdzu[j]);
            const double gn = pm::div_const(upn - bn[j], dzu[j], rdzu[j]);
            const double dzc = 0.5 * (dzu[j] + (j > 0 ? dzu[j > 0 ? j - 1 : 0] : dzu_m));
            double Ai_b = A_b, rAi_b = rA_b, Ai_n = A_n, rAi_n = rA_n;
            if (!ua) {
              const int i = lo + j < nz ? lo + j : nz - 1;
              Ai_b = Ab[i]; rAi_b = rab[i]; Ai_n = An[i]; rAi_n = ran[i];
            }
            bb[j] = pm::exact_level(bb[j], gb, gpb, dzc, rdzc[j], nwb[s], kb[s], Ai_b, rAi_b, dt);
            bn[j] = pm::exact_level(bn[j], gn, gpn, dzc, rdzc[j], nwn[s], kn[s], Ai_n, rAi_n, dt);
            gpb = gb;
            gpn = gn;
          }
        };
        if (uniA)
          step(std::true_type{});
        else
          step(std::false_type{});
      }
      rt::syncblock();  // every neighbour value of this step has been read
      publish(p ^ 1);
      rt::syncblock();
      if (mlw) {
        pm::MlState ml;
        pm::ml_unpark(ml, mlp, scan_s);
        ml_published(ml, p ^ 1);
        pm::ml_park(ml, mlp, false);
        if (Ln == 0) {  // read during this step; refilled by the publish of the next one
          int* f = ibox + 8 * p;
          f[0] = 0; f[1] = 0; f[2] = -1; f[3] = -1; f[4] = 0;
        }
      }
      rt::syncblock();
    }

  }
  bool nan = false;
  if (col) {
    PM_UNROLL
    for (int j = 0; j < LPT; ++j) {
      const int i = lo + j;
      if (i < nz) {
        M.basin.b[m * nz + i] = bb[j];
        M.north.b[m * nz + i] = bn[j];
        nan |= !(fabs(bb[j]) <= 1.79e308) || !(fabs(bn[j]) <= 1.79e308);
      }
    }
  }
  if (mlw) {
    if (!PIPE) pm::ml_unpark(ml, mlp, scan_s);
    PM_UNROLL
    for (int e = 0; e < pm::kMLP; ++e) {
      const int k = pm::mlk(e);
      if (k < ny) {
        M.ml_bs[m * ny + k] = ml.bs[e];
        if (M.ml_Psi_s) M.ml_Psi_s[m * ny + k] = ml.ps[e];
        nan |= !(fabs(ml.bs[e]) <= 1.79e308);
      }
    }
  }
  if (block_any(nan, cbox)) status |= PMOC_ST_NAN;
  if (t == 0) {
    M.basin.bbot[m] = bbot_b;
    M.north.bbot[m] = bbot_n;
    if (M.basin.var) M.basin.var[m] = var_b;
    if (M.north.var) M.north.var[m] = var_n;
  }
  const unsigned all = block_or(status, cbox);  // the mixed-layer warp carries SO_ML's bits
  if (t == 0 && M.status) M.status[m] = status_word(M.status[m], all, so1_exact);
}

// Shared memory of k_wide_post (in doubles): -weff and kappa of each column ([NCOL][nzp] each), the first and last
// level of every thread ([2][NCOL][2 * kWideCol]), the convection flags ([3][NCOL][2] ints: any level above bs, top
// stable level) and 4 ints for the block collectives.
struct WidePostSmem {
  int off_nw, off_kp, off_edge, off_flg, off_cbox, size;
  PM_HD constexpr size_t bytes() const { return sizeof(double) * (size_t)size; }
};
PM_HD constexpr WidePostSmem wide_post_smem(int LPT, int NCOL) {
  WidePostSmem s{};
  s.off_kp = s.off_nw + NCOL * kWideCol * LPT; s.off_edge = s.off_kp + NCOL * kWideCol * LPT;
  s.off_flg = s.off_edge + 4 * NCOL * kWideCol; s.off_cbox = s.off_flg + 3 * NCOL; s.size = s.off_cbox + 2;
  return s;
}

// ---- the steps of the 'post' order (example_twocol_plusSO.py:99-115) ----------------------------
// NCOL columns (the basin; and the northern column of the two-column models), each advanced by
// Column.timestep(wA, dt, do_conv) with the streamfunctions of the last diagnosis, which the host loop
// re-runs in a launch of its own after every iteration with it % K == 0.  Layout as in k_wide_steps2: 256
// threads own LPT consecutive levels of every column, whose buoyancies, dz, 1/dz and 1/dzc stay in
// registers for the whole launch; -weff and kappa live in shared memory in owner-major order (slot
// j*256 + t).  wA is assembled from the carried streamfunctions at launch exactly as k_model's apply():
// basin (Psi_iso_b or Psi_tw) - Psi_so, north -Psi_iso_n, times 1e6.  The kappa variant is fixed in this
// order.  Per step, every thread publishes its first and last level of each column and the convection
// flags (anything above bs, highest stable level); the edges are double-buffered and the flags triple-
// buffered (read / written / cleared), so a step costs one barrier.  The arithmetic is that of
// pm::col_step_exact, as in the 'jn' kernel.  At LPT = 4 the kernel is compiled for two CTAs per SM (at most 128
// registers; it needs about 125 without spilling, against 150 / 194 left free), the wider ones for one.
template <int LPT, int NCOL, bool LIST>
PM_GLOBAL void PM_LAUNCH_BOUNDS(kWideCol, LPT == 4 ? 2 : 1) k_wide_post(WideArgs a) {
  const pmoc_model& M = a.m;
  const bool TW = (M.flags & PMOC_HAS_TW) != 0, ISO = (M.flags & PMOC_ISO) != 0, SO = (M.flags & PMOC_HAS_SO) != 0;
  const int nz = M.nz, t = wtid(), Ln = rt::lane();
  const long long m = wide_member<LIST>(a);
  const double dt = M.dt;
  constexpr int nzp = kWideCol * LPT;
  constexpr WidePostSmem sl = wide_post_smem(LPT, NCOL);
  double* sm = rt::smem();
  double* nws = sm + sl.off_nw;
  double* kps = sm + sl.off_kp;
  double* edge = sm + sl.off_edge;
  int* flg = reinterpret_cast<int*>(sm + sl.off_flg);
  int* cbox = reinterpret_cast<int*>(sm + sl.off_cbox);
  const double* z = M.z;
  const int lo = t * LPT;
  double* rarea = a.memb + (size_t)m * 6 * nz;       // [NCOL][nz] 1 / Area (non-uniform Area)

  const pmoc_column* col[2] = {&M.basin, &M.north};
  double bs[NCOL], n2[NCOL], bbot[NCOL], bzbot[NCOL], A1[NCOL], rA1[NCOL];
  bool conv[NCOL], hasz[NCOL];
  const double* Ar[NCOL];
  double b[NCOL][LPT], dzu[LPT], rdzu[LPT], rdzc[LPT];
  double dzu_m = 1., rdzu_m = 1.;  // cell below the thread's first level
  bool areas_differ = false;
  PM_UNROLL
  for (int c = 0; c < NCOL; ++c) {
    const pmoc_column& d = *col[c];
    bs[c] = vat(d.bs, m);
    n2[c] = vat(d.N2min, m);
    bbot[c] = d.bbot[m];
    hasz[c] = d.bzbot.ptr != nullptr;
    bzbot[c] = hasz[c] ? vat(d.bzbot, m) : 0.0;
    conv[c] = d.do_conv != 0;
    Ar[c] = vrow(d.Area, m);
    A1[c] = Ar[c][1];
    rA1[c] = 1.0 / A1[c];
    const int var = (d.var && d.nvar > 1) ? d.var[m] : 0;
    const double* kap = vrow(d.kappa, m) + (size_t)var * nz;
    const double* dak = vrow(d.dAk, m) + (size_t)var * nz;
    const double* lega = c == 0 ? (TW ? (ISO ? M.Psi_iso_b : M.Psi_tw) + m * nz : nullptr) : M.Psi_iso_n + m * nz;
    const double* psos = (c == 0 && SO) ? M.Psi_so + m * nz : nullptr;
    PM_UNROLL
    for (int j = 0; j < LPT; ++j) {
      const int i = lo + j, s = j * kWideCol + t;
      b[c][j] = 0.;
      nws[c * nzp + s] = kps[c * nzp + s] = 0.0;  // boundary and padding levels: zero -weff and kappa, an exact no-op
      if (i < nz) {
        b[c][j] = d.b[m * nz + i];
        const bool in = i >= 1 && i < nz - 1;
        // k_model's apply (pmoc_model.cu): the same expressions, so the same wA bits
        const double wA = c == 0 ? ((lega ? lega[i] : 0.0) - (psos ? psos[i] : 0.0)) * 1e6 : -lega[i] * 1e6;
        if (in) {
          nws[c * nzp + s] = -(wA - dak[i]);
          kps[c * nzp + s] = kap[i];
          areas_differ |= Ar[c][i] != A1[c];
        }
        rarea[c * nz + i] = 1.0 / Ar[c][i];
      }
    }
  }
  PM_UNROLL
  for (int j = 0; j < LPT; ++j) {
    const int i = lo + j;
    dzu[j] = rdzu[j] = rdzc[j] = 1.;
    if (i < nz) {
      dzu[j] = a.geo[i];
      rdzu[j] = a.geo[nz + i];
      rdzc[j] = a.geo[3 * nz + i];
    }
  }
  if (lo >= 1 && lo - 1 < nz) {
    dzu_m = a.geo[lo - 1];
    rdzu_m = a.geo[nz + lo - 1];
  }
  if (t < 3 * NCOL) {  // every flag buffer starts empty
    flg[2 * t] = 0;
    flg[2 * t + 1] = -1;
  }
  const bool uniA = !block_any(areas_differ, cbox);  // (its barriers also order the flag reset before the publish)

  // publish the first / last level of every column and the convection flags of this thread's levels
  bool mine[NCOL];  // the thread's own levels hold something above bs
  PM_UNROLL
  for (int c = 0; c < NCOL; ++c) mine[c] = false;
  const bool owns_top = lo <= nz - 1 && nz - 1 < lo + LPT;
  auto publish = [&](int e, int q) {
    PM_UNROLL
    for (int c = 0; c < NCOL; ++c) {
      double* ed = edge + (e * NCOL + c) * 2 * kWideCol;
      ed[2 * t] = b[c][0];
      ed[2 * t + 1] = b[c][LPT - 1];
      if (!conv[c]) continue;
      int top = -1;
      bool any = false;
      PM_UNROLL
      for (int j = 0; j < LPT; ++j)
        if (lo + j < nz) {
          if (b[c][j] > bs[c]) any = true;
          else top = lo + j;
        }
      mine[c] = any;
      const unsigned ma = rt::ballot(any);
      const int wt = rt::max_i(top);
      if (Ln == 0) {
        int* f = flg + (q * NCOL + c) * 2;
        if (ma) rt::atomic_add_shared(&f[0], 1);
        rt::atomic_max_shared(&f[1], wt);
      }
    }
  };
  publish(0, 0);
  rt::syncblock();

  int e = 0, qr = 0;
  for (long long it = 0; it < a.nsteps; ++it) {
    const int qw = qr == 2 ? 0 : qr + 1, qz = qw == 2 ? 0 : qw + 1;
    PM_UNROLL
    for (int c = 0; c < NCOL; ++c) {
      // convective adjustment or the surface value (column.py:230-231) of the own levels and of the two neighbour
      // values, then the bottom condition (column.py:232-233)
      const int* f = flg + (qr * NCOL + c) * 2;
      const bool cv = conv[c] && f[0] != 0;
      const double zc = z[f[1] >= 0 ? f[1] : 0], bsc = bs[c], n2c = n2[c];
      if ((cv && mine[c]) || owns_top) {
        PM_UNROLL
        for (int j = 0; j < LPT; ++j)
          if (lo + j < nz) b[c][j] = pm::convect_level(b[c][j], lo + j, cv, bsc, n2c, zc, z, nz);
      }
      if (t == 0) b[c][0] = hasz[c] ? b[c][1] - bzbot[c] * dzu[0] : bbot[c];
      const double* ed = edge + (e * NCOL + c) * 2 * kWideCol;
      double gp = 0.;  // gradient of the cell below the current level
      if (lo >= 1 && lo < nz)
        gp = pm::div_const(b[c][0] - pm::convect_level(ed[2 * t - 1], lo - 1, cv, bsc, n2c, zc, z, nz), dzu_m, rdzu_m);
      // level above the thread's last one
      const double ub = lo + LPT < nz ? pm::convect_level(ed[2 * t + 2], lo + LPT, cv, bsc, n2c, zc, z, nz) : 0.;
      // the explicit step.  No level tests: at the boundary and padding levels -weff = kappa = 0 and every operand
      // is finite, so b + dt*0 = b.
      const double* nw = nws + c * nzp;
      const double* kp = kps + c * nzp;
      auto step = [&](auto UA) {
        constexpr bool ua = decltype(UA)::value;
        PM_UNROLL
        for (int j = 0; j < LPT; ++j) {
          const int s = j * kWideCol + t;
          const double up = j + 1 < LPT ? b[c][j + 1 < LPT ? j + 1 : j] : ub;
          const double g = pm::div_const(up - b[c][j], dzu[j], rdzu[j]);
          const double dzc = 0.5 * (dzu[j] + (j > 0 ? dzu[j > 0 ? j - 1 : 0] : dzu_m));
          const int i = lo + j < nz ? lo + j : nz - 1;
          b[c][j] = pm::exact_level(b[c][j], g, gp, dzc, rdzc[j], nw[s], kp[s], ua ? A1[c] : Ar[c][i],
                                    ua ? rA1[c] : rarea[c * nz + i], dt);
          gp = g;
        }
      };
      if (uniA) step(std::true_type{});
      else step(std::false_type{});
    }
    publish(e ^ 1, qw);
    if (t == 0) {
      PM_UNROLL
      for (int c = 0; c < NCOL; ++c) {  // last read in the previous step, next written in the next one
        flg[(qz * NCOL + c) * 2] = 0;
        flg[(qz * NCOL + c) * 2 + 1] = -1;
      }
    }
    rt::syncblock();
    e ^= 1;
    qr = qw;
  }

  bool nan = false;
  PM_UNROLL
  for (int c = 0; c < NCOL; ++c) {
    PM_UNROLL
    for (int j = 0; j < LPT; ++j) {
      const int i = lo + j;
      if (i < nz) {
        col[c]->b[m * nz + i] = b[c][j];
        nan |= !(fabs(b[c][j]) <= 1.79e308);
      }
    }
  }
  if (block_any(nan, cbox) && t == 0 && M.status) M.status[m] |= PMOC_ST_NAN;
}

size_t wide_steps2_smem(int lpt, int ny) {
  const int nyp = (ny + 3) & ~3, nzp = kWideCol * lpt;
  return sizeof(double) * (size_t)(6 * nzp + kWideCol + 2 * kWideCol + 2 + 2 * nyp + 320 + 8 + 10 + pm::kMlSave);
}

size_t wide_refresh_smem(int nz, int ny, int nb) {
  const int nbp = (nb + 3) & ~3, nyp = (ny + 3) & ~3;
  return sizeof(double) * (size_t)(6 * nz + nbp + nbp / 2 + 2 + 64 + kWideThreads + 3 * nyp + 4);
}

// Host loop: alternate the diagnosis and step launches in the model's order.
//   'jn'   (run_JansenNadeau_2018.py:201-261): the diagnosis at the top of every iteration with it % K == 0, then
//          the steps up to the next such iteration.
//   'post' (example_twocol_plusSO.py:99-115): the steps of iterations [ii, stop], stop the first multiple of K at
//          or after ii, then the diagnosis when stop < it_end (k_model's next0 / hits rule, so that split launches
//          reproduce one launch bit for bit).
// Over `ctas` members (LIST: the members of the active list); pmoc_run_model_wide has checked the model.
template <bool LIST>
static int wide_loop(WideArgs a, bool post, int diagnose_only, long long nsteps, long long ctas, size_t sm_r,
                     void* stream) {
  if (diagnose_only) return launch(k_wide_refresh<LIST>, ctas, kWideThreads, sm_r, stream, a);
  long long ii = a.it0;
  const long long K = a.m.K, it_end = a.it0 + nsteps;
  if (post) {
    const bool two = (a.m.flags & PMOC_HAS_NORTH) != 0;
    const int lpt = a.m.nz <= 4 * kWideCol ? 4 : a.m.nz <= 8 * kWideCol ? 8 : 16;
    auto kern = lpt == 4 ? (two ? k_wide_post<4, 2, LIST> : k_wide_post<4, 1, LIST>)
              : lpt == 8 ? (two ? k_wide_post<8, 2, LIST> : k_wide_post<8, 1, LIST>)
                         : (two ? k_wide_post<16, 2, LIST> : k_wide_post<16, 1, LIST>);
    const size_t sm_s = wide_post_smem(lpt, two ? 2 : 1).bytes();
    while (ii < it_end) {
      const long long stop = ((ii + K - 1) / K) * K;  // first iteration with it % K == 0 at or after ii
      const bool hits = stop < it_end;
      a.it0 = ii;
      a.nsteps = (hits ? stop + 1 : it_end) - ii;
      if (int rc = launch(kern, ctas, kWideCol, sm_s, stream, a)) return rc;
      ii += a.nsteps;
      if (hits)
        if (int rc = launch(k_wide_refresh<LIST>, ctas, kWideThreads, sm_r, stream, a)) return rc;
    }
    return PMOC_OK;
  }
  while (ii < it_end) {
    if (ii % K == 0) {
      if (int rc = launch(k_wide_refresh<LIST>, ctas, kWideThreads, sm_r, stream, a)) return rc;
      a.m.flags &= ~kFlagPsiPushed;  // the streamfunctions are the diagnosis's own from here on
    }
    long long stop = (ii / K + 1) * K;
    if (stop > it_end) stop = it_end;
    a.it0 = ii;
    a.nsteps = stop - ii;
    int rc;
    if (a.m.nz <= 4 * kWideCol)
      rc = launch(k_wide_steps2<4, 2, true, LIST>, ctas, kWideCol + 32, wide_steps2_smem(4, a.m.ny), stream, a);
    else if (a.m.nz <= 8 * kWideCol)
      rc = launch(k_wide_steps2<8, 3, true, LIST>, ctas, kWideCol + 32, wide_steps2_smem(8, a.m.ny), stream, a);
    else
      rc = launch(k_wide_steps2<16, 4, false, LIST>, ctas, kWideCol, wide_steps2_smem(16, a.m.ny), stream, a);
    if (rc) return rc;
    ii = stop;
  }
  return PMOC_OK;
}
}  // namespace pmk

int pmoc_run_model_wide(const pmoc_model* m, long long it0, long long nsteps, int diagnose_only, void* stream,
                        MemberList list) {
  const unsigned topo = m->flags & (PMOC_HAS_NORTH | PMOC_HAS_TW | PMOC_ISO | PMOC_HAS_SO | PMOC_HAS_ML | PMOC_ORDER_JN);
  const unsigned jn = PMOC_HAS_NORTH | PMOC_HAS_TW | PMOC_ISO | PMOC_HAS_SO | PMOC_HAS_ML | PMOC_ORDER_JN;
  const bool post = topo == PMOC_HAS_TW || topo == PMOC_HAS_SO || topo == (PMOC_HAS_TW | PMOC_HAS_SO) ||
                    topo == (PMOC_HAS_NORTH | PMOC_HAS_TW | PMOC_ISO) ||
                    topo == (PMOC_HAS_NORTH | PMOC_HAS_TW | PMOC_ISO | PMOC_HAS_SO);
  if ((topo != jn && !post) || (m->flags & PMOC_SO_BVP) || m->so_c.ptr || m->so_tau_on_y)
    return fail(PMOC_EUNSUPPORTED, "nz > 256: only the 'jn' topology and the explicit 'post' topologies (one column with "
                                   "thermal wind and/or Psi_SO, two columns with or without Psi_SO) have block-per-member "
                                   "kernels; the F2010 smoother and a wind stress on y do not");
  if (m->nz > PMOC_MAX_NZ_WIDE) return fail(PMOC_EUNSUPPORTED, "nz > 4096");
  if (!m->scratch || m->scratch_bytes < pmoc_model_scratch_bytes(m))
    return fail(PMOC_EINVAL, "nz > 256 needs pmoc_model.scratch of pmoc_model_scratch_bytes() bytes");
  if (!post && (!m->Psi_tw || !m->Psi_iso_b || !m->Psi_iso_n || !m->Psi_so)) return fail(PMOC_EINVAL, "diagnostic buffers missing");
  WideArgs a;
  a.m = *m;
  a.geo = static_cast<double*>(m->scratch);
  a.memb = a.geo + 4 * (size_t)m->nz;
  a.it0 = it0;
  a.nsteps = 0;
  a.force_late = std::getenv("PMOC_WIDE_FORCE_LATE") != nullptr;
  a.list = list;
  const long long ctas = list.slots(m->M);  // one per member of the active list
  const int nb = (m->flags & PMOC_ISO) ? m->nb : 0, ny = (m->flags & PMOC_HAS_SO) ? m->ny : 0;
  const size_t sm_r = wide_refresh_smem(m->nz, ny, nb);
  if (sm_r > kMaxSmemPerBlock) {
    std::snprintf(g_err, sizeof(g_err), "nz = %d, nb = %d, ny = %d: the diagnosis needs %zu bytes of shared memory per "
                  "block, more than the %zu one block can use", m->nz, nb, ny, sm_r, kMaxSmemPerBlock);
    return PMOC_EUNSUPPORTED;
  }
  if (ctas == 0) return PMOC_OK;
  if (int rc = launch(k_wide_geo, 64, kWideThreads, 0, stream, a)) return rc;
  return list.members ? wide_loop<true>(a, post, diagnose_only, nsteps, ctas, sm_r, stream)
                      : wide_loop<false>(a, post, diagnose_only, nsteps, ctas, sm_r, stream);
}
