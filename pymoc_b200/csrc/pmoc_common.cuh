// Shared declarations of the pymoc_b200 translation units (kernels are split per
// levels-per-lane so that the instantiations compile in parallel).
#pragma once
#include "pmoc_device.cuh"
#include "../../include/pymoc_b200.h"

#include <cstdio>
#include <cstring>

extern thread_local char pmoc_g_err[256];
#define g_err pmoc_g_err

namespace pmk {



#define PM_CUDA_OK(expr)                                                                      \
  do {                                                                                        \
    cudaError_t e_ = (expr);                                                                  \
    if (e_ != cudaSuccess) {                                                                  \
      std::snprintf(g_err, sizeof(g_err), "%s: %s", #expr, cudaGetErrorString(e_));           \
      return e_ == cudaErrorNoDevice || e_ == cudaErrorInsufficientDriver ? PMOC_ENODEVICE : PMOC_ECUDA; \
    }                                                                                         \
  } while (0)

static inline int fail(int code, const char* msg) {
  std::snprintf(g_err, sizeof(g_err), "%s", msg);
  return code;
}

PM_DEV double vat(const pmoc_vec& v, long long m) { return v.ptr[m * v.mstride]; }
PM_DEV const double* vrow(const pmoc_vec& v, long long m) { return v.ptr + m * v.mstride; }

constexpr int kWarpsPerBlock = 4;  // per-module kernels; the fused kernel picks its own per launch (launch_model)
constexpr size_t kMaxSmemPerBlock = 227 * 1024;  // dynamic shared memory one block of sm_100 may opt in to

// ------------------------------------------------------------------------------------------
// shared-memory plan (in doubles).  Per block: the grid tables; per warp (= member): the
// column tables and the scratch of the diagnostics.
struct SmemPlan {
  int nzp, nyp, nbp;
  int off_zs, off_zl, off_rdu, off_rdd, off_ruu, off_rdd2, off_y;  // per block
  int off_dzu, off_rdzu, off_dzc, off_rdzc;                        // per block, bit-faithful step only
  int off_tap;                                                      // per block, 4*nzp Psi_SO tapers
  int off_warp0, per_warp;                                          // per warp region
  int w_col[3];                                                     // column tables of basin / north / pac (3 or 4 nzp each)
  int col_tables;                                                   // 0: folded coefficients are built from global memory
  int w_remap, w_psib, w_cnt, w_bs, w_sinv, w_tau;  // w_remap: 6*nzp of remap scratch, w_psib: psib[nb]
  int w_nweff[2], w_bb, w_pm, w_scan;                               // SO_ML / 'jn' order
  PM_HD size_t bytes(int wpb) const { return sizeof(double) * (size_t)(off_warp0 + per_warp * wpb); }
};

// Topologies with a mixed layer run the bit-faithful column step (pm::col_step_exact): their
// block tables are dz / 1/dz instead of the folded reciprocals, and the remap scratch psib[nb]
// overlays per-step arrays that are dead while the streamfunctions are being re-diagnosed.
static PM_HD SmemPlan plan_smem(int LPL, int ny, int nb, unsigned flags) {
  SmemPlan s{};
  const bool exact = (flags & PMOC_HAS_ML) != 0;
  s.nzp = 32 * LPL;
  s.nyp = (ny + 3) & ~3;
  s.nbp = (nb + 3) & ~3;
  int o = 0;
  s.off_zs = o; o += s.nzp + 4;
  s.off_zl = o; o += s.nzp;
  if (!exact) {
    s.off_rdu = o; o += s.nzp;
    s.off_rdd = o; o += s.nzp;
    s.off_ruu = o; o += s.nzp;
    s.off_rdd2 = o; o += s.nzp;
  } else {
    s.off_dzu = o; o += s.nzp;
    s.off_rdzu = o; o += s.nzp;
    s.off_dzc = o; o += s.nzp;
    s.off_rdzc = o; o += s.nzp;
  }
  s.off_y = o; o += s.nyp;
  if (flags & PMOC_HAS_SO) { s.off_tap = o; o += 4 * s.nzp; }
  s.off_warp0 = o;
  int w = 0;
  const int colw = exact ? 4 : 3;  // arrays per column table
  // The folded-step tables (dt*kappa, dt/A, dAk) are read once per diagnosis.  With several columns they would
  // cost resident warps (16 KB per member instead of 12), so those topologies read the profiles from global
  // memory (L2) instead; the single-column kernels are register-limited anyway and keep them.
  s.col_tables = exact || !(flags & PMOC_HAS_NORTH);
  if (s.col_tables) {
    s.w_col[0] = w; w += colw * s.nzp;
    if (flags & PMOC_HAS_NORTH) { s.w_col[1] = w; w += colw * s.nzp; }
    if (flags & PMOC_HAS_PAC) { s.w_col[2] = w; w += colw * s.nzp; }
  }
  if (exact) {
    // psib[nb] + the class counters are live only inside a refresh: they overlay the column tables,
    // which the kernel re-tabulates from global memory (L2) at the end of every refresh
    const int psz = s.nbp + s.nbp / 2 + 2;
    s.w_psib = s.w_col[0];
    s.w_cnt = s.w_col[0] + s.nbp;
    if (w - s.w_col[0] < psz) w = s.w_col[0] + psz;
  }
  if ((flags & PMOC_ISO) && !exact) {
    s.w_remap = w; w += 6 * s.nzp;
    s.w_psib = w; w += s.nbp;
    s.w_cnt = w; w += s.nbp / 2 + 2;
  }
  if (flags & PMOC_HAS_SO) {
    s.w_bs = w; w += s.nyp;
    s.w_sinv = w; w += s.nyp;
    s.w_tau = w; w += s.nyp;
  }
  if (exact) {
    // the remap scratch (6*nzp + nb, live only inside a refresh) overlays the per-step arrays,
    // which are rebuilt at the end of every refresh
    s.w_remap = w;
    s.w_nweff[0] = w; w += 2 * s.nzp;
    s.w_nweff[1] = w; w += 2 * s.nzp;
    s.w_bb = w; w += s.nzp;
    s.w_pm = w; w += s.nzp;
    s.w_scan = w; w += 10 * 32;
  }
  s.per_warp = w;
  return s;
}

PM_DEV pm::GeoTab geo_of(double* sm, const SmemPlan& sp) {
  return pm::GeoTab{sm + sp.off_zs, sm + sp.off_zl, sm + sp.off_rdu, sm + sp.off_rdd, sm + sp.off_ruu,
                    sm + sp.off_rdd2};
}
PM_DEV pm::ColTab coltab_of(double* ws, const SmemPlan& sp, int which) {
  double* t = ws + sp.w_col[which];
  return pm::ColTab{t, t + sp.nzp, t + 2 * sp.nzp};
}
PM_DEV pm::ExactGeo exactgeo_of(double* sm, const SmemPlan& sp) {
  return pm::ExactGeo{sm + sp.off_dzu, sm + sp.off_rdzu, sm + sp.off_dzc, sm + sp.off_rdzc};
}
PM_DEV pm::ExactCol exactcol_of(double* ws, const SmemPlan& sp, int which) {
  double* t = ws + sp.w_col[which];
  double* n = ws + sp.w_nweff[which];
  return pm::ExactCol{{t, t + sp.nzp}, t + 2 * sp.nzp, t + 3 * sp.nzp, {n, n + sp.nzp}};
}

// Active list of a launch (pmoc_model_run_members): slot s steps member members[s], in place; NULL = every member,
// slot s = member s.  Every kernel reads and writes through the real member index, so nothing is gathered.
struct MemberList {
  const int64_t* members;
  long long n;
  PM_HD long long slots(long long M) const { return members ? n : M; }
};

struct RunArgs {
  pmoc_model m;
  SmemPlan sp;
  long long it0, nsteps;
  int diagnose_only;
  int sync_refresh;  // CTA barrier before every diagnosis: the CTA's warps then run its long instruction stream together
  MemberList list;
};

// per-column registers
template <int LPL>
struct ColRegs {
  double b[LPL], p[LPL], q[LPL];
  double bs, N2min, bbot, bzbot;
  bool has_bzbot, conv, plain;  // plain: neither convection nor a gradient bottom condition
  int var;
  pm::ColTab tab;
};

template <int LPL>
PM_DEV void col_load(ColRegs<LPL>& c, const pmoc_column& d, long long m, int nz) {
  pm::load_lev<LPL>(c.b, d.b + m * nz, nz, 0.0);
  c.bs = vat(d.bs, m);
  c.N2min = vat(d.N2min, m);
  c.bbot = d.bbot[m];
  c.has_bzbot = d.bzbot.ptr != nullptr;
  c.bzbot = c.has_bzbot ? vat(d.bzbot, m) : 0.0;
  c.conv = d.do_conv != 0;
  c.plain = !c.conv && !c.has_bzbot;
  c.var = (d.var != nullptr && d.nvar > 1) ? d.var[m] : 0;
}

// (re)build the member's coefficient tables for the kappa variant in use
template <int LPL>
PM_DEV void col_retabulate(ColRegs<LPL>& c, const pmoc_column& d, long long m, const pm::GeoTab& G, int nz,
                           double dt) {
  const long long voff = (long long)c.var * nz;
  pm::col_tabulate<LPL>(c.tab, G, vrow(d.kappa, m) + voff, vrow(d.dAk, m) + voff, vrow(d.Area, m), nz, dt);
}

// bottom boundary condition of vertadvdiff (column.py:232-233)
template <int LPL>
PM_DEV void col_bottom(ColRegs<LPL>& c, const double* zs) {
  if (rt::lane() == 0) {
    if (c.has_bzbot)
      c.b[0] = c.b[LPL > 1 ? 1 : 0] - c.bzbot * (zs[1] - zs[0]);
    else
      c.b[0] = c.bbot;
  }
}

// Column.timestep(wA, dt, do_conv) as the loop calls it (column.py:336-341).  For a "plain"
// column the boundary values are invariant under the step (p = q = 0 there) and are set once
// per launch, so the step is the bare stencil.
template <int LPL>
PM_DEV void col_advance(ColRegs<LPL>& c, const pm::GeoTab& G, int nz) {
  if (!c.plain) {
    if (c.conv) pm::col_convect<LPL>(c.b, c.bs, c.N2min, G.zs, G.zl, nz);
    col_bottom<LPL>(c, G.zs);
  }
  pm::col_step<LPL>(c.b, c.p, c.q);
}

// the same for the bit-faithful step (always convecting columns of the 'jn' order)
template <int LPL>
PM_DEV void col_advance_exact(ColRegs<LPL>& c, const pm::ExactCol& X, const pm::ExactGeo& EG, const pm::GeoTab& G,
                              int nz, double dt) {
  if (c.conv)
    pm::col_convect<LPL>(c.b, c.bs, c.N2min, G.zs, G.zl, nz);
  else
    pm::set_level<LPL>(c.b, nz - 1, c.bs);
  col_bottom<LPL>(c, G.zs);
  pm::col_step_exact<LPL>(c.b, X, c.var, EG, nz, dt);
}

// ------------------------------------------------------------------------------------------
// launch plumbing
#ifdef PMOC_EMU
template <class K, class A>
int launch(K kern, long long grid, int block, size_t smem, void*, const A& args) {
  // the device refuses more dynamic shared memory than one block may opt in to (cudaFuncSetAttribute fails)
  if (smem > kMaxSmemPerBlock)
    return fail(PMOC_ECUDA, "emulated cudaFuncSetAttribute: dynamic shared memory above the per-block limit");
  pmemu::launch(grid, block, smem, [=]() { kern(args); });
  return PMOC_OK;
}
#else
template <class K, class A>
int launch(K kern, long long grid, int block, size_t smem, void* stream, const A& args) {
  if (smem > 48 * 1024)
    PM_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<(unsigned)grid, block, smem, (cudaStream_t)stream>>>(args);
  PM_CUDA_OK(cudaGetLastError());
  return PMOC_OK;
}
#endif


static inline long long blocks_for(long long M) { return (M + kWarpsPerBlock - 1) / kWarpsPerBlock; }
// Internal pmoc_model.flags bit, set by pmoc_host_step for a launch after the caller pushed the carried
// streamfunctions (PMOC_IO_PSI): the 'jn' step kernels then classify them as rounding noise without the
// PMOC_ST_CARRY_SO1_EXACT exemption of an earlier diagnosis, which does not describe them.
constexpr unsigned kFlagPsiPushed = 0x80000000u;

// The carry of the 'jn' switches (PMOC_ST_CARRY_SO1_EXACT): the member's Psi_so[1] came out of state-independent
// arithmetic at the last diagnosis, and the carried streamfunctions are still that diagnosis's own.
PM_DEV bool so1_exact_carried(const pmoc_model& M, long long m) {
  return M.status && (M.status[m] & PMOC_ST_CARRY_SO1_EXACT) && !(M.flags & kFlagPsiPushed);
}
// A member's status word after a kernel: the old bits and the kernel's, the internal carries replaced by `carry`.
PM_DEV unsigned status_word(unsigned old, unsigned bits, bool carry) {
  return ((old | bits) & ~PMOC_ST_CARRY_MASK) | (carry ? PMOC_ST_CARRY_SO1_EXACT : 0u);
}

// the checks pmoc_model_run applies to a model before it dispatches (pmoc_ops.cu)
int check_model(const pmoc_model* m);
// check_model and the argument checks of pmoc_model_equilibrate but its work buffer (pmoc_equil.cu); the host-buffer
// entry points apply them before they copy anything
int check_equilibrate(const pmoc_model* m, int64_t it0, int64_t max_steps, int64_t every, double tol,
                      const void* stopped_at, const void* converged);
}  // namespace pmk
using namespace pmk;

// block-per-member path for nz > PMOC_MAX_NZ_WARP (pmoc_wide.cu)
int pmoc_run_model_wide(const pmoc_model* m, long long it0, long long nsteps, int diagnose_only, void* stream,
                        pmk::MemberList list);

// several members per warp for the column + thermal-wind topology (pmoc_twcol.cu)
bool pmoc_twcol_supported(const pmoc_model* m);
int pmoc_launch_twcol(const pmoc_model* m, long long it0, long long nsteps, int diagnose_only, void* stream,
                      pmk::MemberList list);

// one launcher per levels-per-lane, each in its own translation unit (pmoc_model.cu)
#define PM_DECL_MODEL(n) int pmoc_launch_model_##n(const RunArgs& ra, void* stream);
PM_DECL_MODEL(2) PM_DECL_MODEL(3) PM_DECL_MODEL(4) PM_DECL_MODEL(5) PM_DECL_MODEL(6) PM_DECL_MODEL(7) PM_DECL_MODEL(8)
