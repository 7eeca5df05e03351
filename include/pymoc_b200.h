/* pymoc_b200 -- C ABI of the B200-native PyMOC time-stepping engine.
 *
 * The reference (pymoc 0.0.1rc5) has no FFI: its boundary is the Python class surface
 * Column / Psi_Thermwind / Psi_SO / SO_ML plus the hand-written loops in examples/
 * (SURVEY.md section 8b).  Every entry point below names the reference interface it
 * replaces (path:line under /root/reference).  INTEGRATION.md shows the ctypes stub a
 * maintainer of the reference would add.
 *
 * Conventions
 *  - plain C, no C++/torch types; all floating point is IEEE binary64;
 *  - every pointer is a DEVICE pointer unless the function name ends in _host;
 *  - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); device
 *    entry points are asynchronous on it and allocate nothing;
 *  - every function returns a pmoc_status (0 = ok); no exception crosses the boundary;
 *  - batched over `M` independent ensemble members; a `pmoc_vec` whose `mstride` is 0 is
 *    shared by all members, otherwise member m starts at ptr + m*mstride (in doubles);
 *  - vertical arrays run bottom (z[0] = -H) to surface (z[nz-1] = 0) like the reference.
 */
#ifndef PYMOC_B200_H_
#define PYMOC_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PMOC_ABI_VERSION 3
#define PMOC_MAX_NZ_WARP 256 /* one warp per member up to this many levels */
#define PMOC_MAX_NZ_WIDE 4096 /* one CTA per member up to this many levels: the 'jn' topology and the explicit
                                 'post' topologies (HAS_TW, HAS_SO, HAS_TW|HAS_SO, HAS_NORTH|HAS_TW|ISO and
                                 HAS_NORTH|HAS_TW|ISO|HAS_SO without so_c or so_tau_on_y) */
#define PMOC_MAX_NY_ML 64    /* SO_ML surface points per member */

typedef enum {
  PMOC_OK = 0,
  PMOC_EINVAL = 1,       /* bad sizes / null pointers / inconsistent flags */
  PMOC_EUNSUPPORTED = 2, /* valid request this build has no kernel for */
  PMOC_ECUDA = 3,        /* a CUDA runtime call failed; see pmoc_last_error() */
  PMOC_ENODEVICE = 4     /* no CUDA device: there is no CPU fallback */
} pmoc_status;

typedef struct {
  const double* ptr;
  int64_t mstride; /* doubles between consecutive members; 0 = shared */
} pmoc_vec;

/* per-member status bits written by the model kernels (pmoc_model.status) */
#define PMOC_ST_NAN 1u            /* non-finite buoyancy at the end of the launch */
#define PMOC_ST_BS_NONMONOTONE 2u /* bs(y) not monotone north of argmin at some diagnosis: ys() (psi_SO.py:106-140) has
                                     several roots.  scipy's brentq is followed statement by statement (SURVEY H7),
                                     which reproduces the reference's root for bit-identical bs, but the root it
                                     lands on depends discontinuously on bs: rounding differences are amplified to
                                     O(1) (measured: every member of the C5 lattice that misses 1e-10 carries this
                                     bit), so parity is undefined */
#define PMOC_ST_BRENT_SIGN 4u     /* f(a), f(b) same sign: scipy.optimize.brentq would raise ValueError.  Only a
                                     non-finite bs(y) reaches it: b < min(bs) and b > bs[-1] are answered before the
                                     root search, so a finite bs always brackets a sign change */
#define PMOC_ST_XP_NONMONOTONE 8u /* b_basin not monotone as np.interp abscissa in SO_ML (SURVEY a15):
                                     numpy's guess-carrying search is followed query by query */
#define PMOC_ST_BVP_SERIES 32u    /* F2010 smoother: a cell propagator series did not converge (N2 h^2/c^2 huge) */
#define PMOC_ST_NOISE_SWITCH 64u  /* 'jn' order: the outcome of a bottom-boundary switch depended on the sign of a
                                     streamfunction value that is rounding noise (0 < |Psi[1]| < 1e-12 max|Psi|,
                                     run_JansenNadeau_2018.py:233-254) while the other operands of that switch
                                     let it through: the reference's own branch is then decided by summation
                                     order, parity for this member is undefined */
#define PMOC_ST_ML_INDEX 16u      /* SO_ML needed np.argwhere(Psi_b > 0)[0][0] / np.nonzero(Psi_b)[0][0] of an
                                     all-non-positive / all-zero Psi_b: the reference raises IndexError */
#define PMOC_ST_TIE_CELL 128u     /* isopycnal remap (psi_thermwind.py:177-184): a cell carrying transport is inverted
                                     by no more than 4 eps (relative), or is the bottom cell within 4 eps of flat.  Psib's
                                     clip((top-x)/(top-bot), 0, 1) jumps by the cell's whole transport between "flat"
                                     and "inverted by one ulp", so the reference's own answer is decided by the last
                                     bit of its state there (structural in the 'jn' loop, whose no-flux bottom
                                     condition bbot = b[1] drives b[0] - b[1] to zero); parity is undefined unless
                                     the roundings happen to agree */
#define PMOC_ST_BS_SAWTOOTH 256u  /* (informational, implies BS_NONMONOTONE) bs(y) decreases on >= 3 grid intervals
                                     north of its first minimum, counted one by one whether or not they are adjacent
                                     (one smooth decrease across three intervals counts): typically the reference's
                                     mixed layer has gone grid-scale unstable (SO_ML.py:124-134 explicit upwind
                                     advection + Crank-Nicolson with Ks dt/dy^2 > 1) */
/* Bits that make parity with the reference UNDEFINED for a member (the reference's own result is decided by
 * rounding noise); the others are informational (a rarer but exactly reproduced code path was taken). */
#define PMOC_ST_PARITY_UNDEFINED (PMOC_ST_BS_NONMONOTONE | PMOC_ST_NOISE_SWITCH | PMOC_ST_TIE_CELL)
/* internal, not sticky: the Psi_SO value of level 1 that the 'jn' switches read was produced by state-independent
 * arithmetic (the non-outcropping limiter or the slope clip) and is therefore reproduced bit for bit even when
 * it is rounding noise; carried between launches in the status word.  Streamfunctions pushed through
 * pmoc_host_step (PMOC_IO_PSI) do not carry it: the step kernels classify them from their values alone.
 * The stateless pmoc_model_run_host pushes the status word together with the streamfunctions it carries, so there
 * the carry bit travels with them: the caller hands back both as an earlier call returned them. */
#define PMOC_ST_CARRY_SO1_EXACT 0x80000000u
#define PMOC_ST_CARRY_MASK 0xF0000000u /* bits reserved for such internal carries */

/* ---- one advective-diffusive column: reference class Column, column.py:19-72 ------------ */
typedef struct {
  double* b;      /* [M, nz] buoyancy, updated in place (column.py:249,268,271) */
  pmoc_vec kappa; /* [nvar, nz] diffusivity sampled on z (make_func, column.py:58)       */
  pmoc_vec dAk;   /* [nvar, nz] np.gradient(Area*kappa, z), host-evaluated (column.py:122) */
  pmoc_vec Area;  /* [nz] */
  pmoc_vec bs;    /* scalar: surface buoyancy (column.py:61) */
  pmoc_vec N2min; /* scalar (column.py:65) */
  pmoc_vec bzbot; /* scalar or ptr==NULL -> use bbot (column.py:232-233) */
  double* bbot;   /* [M] bottom buoyancy; the 'jn' loop rewrites it every step */
  int32_t* var;   /* [M] kappa variant in use (0..nvar-1); NULL when nvar == 1 */
  int32_t nvar;
  int32_t do_conv; /* timestep(..., do_conv=True) (column.py:336-341) */
} pmoc_column;

/* ---- coupled model = what an examples/ script wires together -------------------------- */
#define PMOC_HAS_NORTH 1u /* second (northern) column, convecting as flagged              */
#define PMOC_HAS_TW 2u    /* Psi_Thermwind between basin and north / fixed b2             */
#define PMOC_ISO 4u       /* force columns with Psibz() instead of Psi (psi_thermwind.py:187-208) */
#define PMOC_HAS_SO 8u    /* Psi_SO on the basin column                                   */
#define PMOC_HAS_ML 16u   /* SO_ML mixed layer                                            */
#define PMOC_SO_BVP 64u   /* set by the library when so_c.ptr != NULL: F2010 smoother of Psi_GM
                             (psi_SO.py:308-323); callers leave it clear */
#define PMOC_HAS_PAC 128u /* two-basin topology of examples/twobasin_NadeauJansen.py:63-122: a third column
                             ("Pacific", fields pac / zoc_f / so2_L), a second Psi_Thermwind between basin and pac
                             (the zonal overturning in the channel) and a second Psi_SO on the pac column.
                             Needs PMOC_HAS_NORTH | PMOC_HAS_TW | PMOC_ISO | PMOC_HAS_SO, order 'post' */
#define PMOC_ORDER_JN 32u /* loop order + bottom-boundary switches of
                             examples/run_JansenNadeau_2018.py:201-261; otherwise the order of
                             examples/example_twocol_plusSO.py:99-115 */

typedef struct {
  int64_t M;
  int32_t nz, ny, nb; /* nb: isopycnal classes of Psib (psi_thermwind.py:137, default 500) */
  int32_t K;          /* MOC_up_iters */
  uint32_t flags;
  double dt;
  const double* z; /* [nz] shared grid */
  const double* y; /* [ny] shared channel grid (NULL without SO) */

  pmoc_column basin, north;
  pmoc_column pac; /* PMOC_HAS_PAC only (examples/twobasin_NadeauJansen.py:88) */

  /* Psi_Thermwind (psi_thermwind.py:30-70) */
  pmoc_vec tw_f;  /* scalar */
  pmoc_vec tw_b2; /* [nz] fixed northern profile when there is no north column */
  pmoc_vec zoc_f; /* scalar: f of the basin-pac thermal wind, PMOC_HAS_PAC (twobasin_NadeauJansen.py:69) */

  /* Psi_SO (psi_SO.py:17-104) */
  pmoc_vec so_bs;  /* [ny] surface buoyancy (ignored with PMOC_HAS_ML: the mixed layer's bs is used,
                      run_JansenNadeau_2018.py:214) */
  pmoc_vec so_tau; /* scalar wind stress, or [ny] when so_tau_on_y != 0 */
  pmoc_vec so_f, so_rho, so_L, so_KGM, so_smax;
  pmoc_vec so_c; /* scalar F2010 phase speed; ptr==NULL -> explicit GM (psi_SO.py:325-327) */
  pmoc_vec so2_L; /* scalar: zonal length of the pac sector's Psi_SO, which shares every other parameter with
                     the basin sector's (twobasin_NadeauJansen.py:76-81), PMOC_HAS_PAC */
  int32_t so_tau_on_y;
  int32_t so_bvp_with_Ek;
  /* host-evaluated tapers (psi_SO.py:164-216); all-ones when the height is None, the Ekman
     taper with HEk=None has its last element 0 (psi_SO.py:213-216) */
  const double *so_sill_taper, *so_ek_taper, *so_top_taper, *so_bot_taper; /* [nz] shared */

  /* SO_ML (SO_ML.py:17-71) */
  double* ml_bs; /* [M, ny] state */
  pmoc_vec ml_Ks, ml_h, ml_L, ml_vpist;
  pmoc_vec ml_surflux, ml_rest_mask, ml_b_rest; /* [ny] */

  /* diagnostics, all optional (NULL = not wanted) except those the loop carries between
     launches: Psi_iso_b/Psi_iso_n (or Psi_tw without PMOC_ISO) and Psi_so */
  double *Psi_tw, *Psi_iso_b, *Psi_iso_n; /* [M, nz] Sv */
  double *psib, *bgrid;                   /* [M, nb]     */
  double *Psi_so, *Psi_Ek, *Psi_GM;       /* [M, nz] Sv */
  double* ml_Psi_s;                       /* [M, ny] Sv */
  /* PMOC_HAS_PAC: Psi_zon_a / Psi_zon_p / Psi_so2 are carried between launches like Psi_iso_* / Psi_so */
  double *Psi_zoc, *Psi_zon_a, *Psi_zon_p; /* [M, nz] Sv: ZOC.Psi and its Psibz() legs */
  double *psib2, *bgrid2;                  /* [M, nb] of the basin-pac remap */
  double *Psi_so2, *Psi_Ek2, *Psi_GM2;     /* [M, nz] Sv: Psi_SO of the pac sector */
  uint32_t* status;                       /* [M] PMOC_ST_* bits, OR-ed */

  /* device scratch, needed only when nz > PMOC_MAX_NZ_WARP (block-per-member kernels of both orders):
     pmoc_model_scratch_bytes(m) bytes.  The library never allocates device memory itself (except in
     pmoc_model_run_host). */
  void* scratch;
  uint64_t scratch_bytes;
} pmoc_model;

/* library / device ----------------------------------------------------------------------- */
int pmoc_abi_version(void);
const char* pmoc_last_error(void);     /* text of the last PMOC_ECUDA on this thread */
int pmoc_device_info(int* sm_count, int* cc_major, int* cc_minor);
uint64_t pmoc_model_scratch_bytes(const pmoc_model* m); /* 0 when nz <= PMOC_MAX_NZ_WARP */

/* Diagnose all streamfunctions of the model from its current state -- what the scripts do
 * before their loop (examples/example_twocol_plusSO.py:61-80: AMOC.solve(); AMOC.Psibz();
 * SO.solve()).  Needed once before the first pmoc_model_run of an order-'post' model. */
int pmoc_model_diagnose(const pmoc_model* m, void* stream);

/* Advance every member by `nsteps` iterations of the script loop, iteration counter starting
 * at `it0` (streamfunctions are re-diagnosed on iterations with it % K == 0).  Up to
 * PMOC_MAX_NZ_WARP levels one fused kernel: state stays on-chip for all `nsteps`.  Above that (up to
 * PMOC_MAX_NZ_WIDE, the topologies listed there) one CTA per member: step launches alternate with
 * diagnosis launches, the state stays on chip between two diagnoses.  Other topologies above
 * PMOC_MAX_NZ_WARP (the F2010 smoother, tau on y, the two-basin model) return PMOC_EUNSUPPORTED.
 * Replaces the loop bodies
 * examples/example_timestepping.py:73-80, example_twocol.py:85-96,
 * example_twocol_plusSO.py:99-115, run_JansenNadeau_2018.py:201-261,
 * run_single_global_basin.py:172-229. */
int pmoc_model_run(const pmoc_model* m, int64_t it0, int64_t nsteps, void* stream);

/* pmoc_model_run for the listed members only (device list of indices in [0, M), any order, no repeats); the others
 * are untouched.
 * Each listed member ends exactly as pmoc_model_run would leave it -- state, carried streamfunctions, diagnostics
 * and status -- and the state stays in place (nothing is gathered).  n == 0 launches nothing. */
int pmoc_model_run_members(const pmoc_model* m, const int64_t* members, int64_t n, int64_t it0, int64_t nsteps,
                           void* stream);

/* Run [it0, it0 + max_steps) to equilibrium: in chunks of `every` iterations (a multiple of K; max_steps a multiple
 * of K too, else PMOC_EINVAL), after each chunk freeze the members whose state moved by <= tol since the previous
 * check -- |b_now - b_prev| <= tol at every level of every column and, with PMOC_HAS_ML, at every point of the mixed
 * layer's bs -- and step only the others.  A member with a non-finite value is frozen as not converged.  The last
 * chunk may be shorter than `every`.
 *   stopped_at[M] (device): the iteration each member stopped at (it0 + max_steps when it never stopped);
 *   converged[M] (device, uint8): 1 if the criterion was met, 0 if non-finite or still moving at the end.
 * A member frozen at iteration n holds exactly what pmoc_model_run over [it0, n) gives it.  The loop reads the
 * iteration counter only modulo K and every stop is it0 plus a multiple of K, so after the call all members can be
 * run on together from it0 + max_steps: each continues from its own stop.  An order-'post' model must have been
 * diagnosed, as for pmoc_model_run.
 * `work`: caller-provided device memory of pmoc_equilibrate_work_bytes(m) bytes (the snapshot of the state, two
 * active lists, a counter).  The library allocates nothing; the host reads the 8-byte counter back after every
 * check (one copy and one stream synchronisation), so the call returns when the work is done. */
uint64_t pmoc_equilibrate_work_bytes(const pmoc_model* m);
int pmoc_model_equilibrate(const pmoc_model* m, int64_t it0, int64_t max_steps, int64_t every, double tol,
                           int64_t* stopped_at, uint8_t* converged, void* work, uint64_t work_bytes, void* stream);
/* The same run for a consumer whose arrays are in HOST memory: pmoc_host_equilibrate through the persistent handle
 * below, pmoc_model_equilibrate_host as its stateless form.  Same stops, flags and end state as
 * pmoc_model_equilibrate; stopped_at[M] and converged[M] are HOST arrays; synchronous.  The library allocates the
 * work buffer itself, from its private pool, for the duration of the call.  Argument errors are those of
 * pmoc_model_equilibrate (and of pmoc_host_step for push / pull) and are found before anything is copied; topologies
 * pmoc_model_run refuses are refused with its code and text, and the handle stays usable.  The stateless form moves
 * what pmoc_model_run_host moves; the streamfunctions and diagnostics come back whenever the call diagnoses or
 * steps.  pmoc_host_last_bytes counts the classes moved plus 9 bytes per member of results. */
int pmoc_model_equilibrate_host(const pmoc_model* m, int64_t it0, int64_t max_steps, int64_t every, double tol,
                                int64_t* stopped_at, uint8_t* converged);

/* Same as diagnose (when it0 == 0, order 'post') + run, but every pointer in `m` is a HOST pointer: the
 * stateless form of the handle below (open, one step, close), with the same device mirror and block loop.
 * Grids, parameters and the state (PMOC_IO_STATE) go up every call, the carried streamfunctions
 * (PMOC_IO_PSI) when the launch continues an earlier one; the state comes back, the streamfunctions and
 * diagnostics (PMOC_IO_PSI | PMOC_IO_DIAG) when the call diagnoses, and ml_Psi_s when it steps.
 * Synchronous.  This is the call a non-torch consumer binds. */
int pmoc_model_run_host(const pmoc_model* m, int64_t it0, int64_t nsteps);
/* bytes the last pmoc_model_run_host / pmoc_model_equilibrate_host / pmoc_host_open / pmoc_host_step /
 * pmoc_host_equilibrate of this thread copied host->device / device->host */
void pmoc_host_last_bytes(uint64_t* h2d, uint64_t* d2h);

/* Persistent host-buffer handle: the same loop (the examples' `for ii in range(total_iters)` with its
 * diagnostics every Diag_iters, run_JansenNadeau_2018.py:201-261) for a consumer that keeps its arrays in HOST
 * memory and calls in every few iterations.  pmoc_host_open mirrors every array of `m` (HOST pointers, which must
 * stay valid until pmoc_host_close; pin them for full copy bandwidth) on the device once -- grids, parameters,
 * state, carried streamfunctions; the diagnostics start at zero -- from a memory pool private to the library,
 * and keeps three streams.  pmoc_host_step advances
 * iterations [it0, it0 + nsteps) and moves only the array classes asked for, pipelined over blocks of members so
 * that copies overlap the fused kernel:
 *   push: copied host->device before the launch (0 = the device copy is current: nothing goes up);
 *   pull: copied device->host after it.
 * An order-'post' model is diagnosed first when it0 == 0 (the scripts' pre-loop solve()), or when the state is
 * pushed without matching streamfunctions before any diagnosis.  Synchronous; returns pmoc_status. */
#define PMOC_IO_STATE 1u /* b of every column, bs of the mixed layer, bbot / kappa variant of the 'jn' switches, status */
#define PMOC_IO_PSI 2u   /* the streamfunctions the loop carries: Psi_iso_b/n (Psi_tw without PMOC_ISO), Psi_so, zonal legs */
#define PMOC_IO_DIAG 4u  /* everything else a diagnosis writes: Psi_tw, psib, bgrid, Psi_Ek, Psi_GM, Psi_s, ... (pull only) */
typedef struct pmoc_host pmoc_host;
int pmoc_host_open(const pmoc_model* m, pmoc_host** handle);
int pmoc_host_step(pmoc_host* handle, int64_t it0, int64_t nsteps, uint32_t push, uint32_t pull);
/* pmoc_model_equilibrate through the handle (see there): push / pull as in pmoc_host_step, the order-'post'
 * diagnosis under its rule; a later pmoc_host_step from it0 + max_steps continues each member from its own stop. */
int pmoc_host_equilibrate(pmoc_host* handle, int64_t it0, int64_t max_steps, int64_t every, double tol,
                          int64_t* stopped_at, uint8_t* converged, uint32_t push, uint32_t pull);
int pmoc_host_close(pmoc_host* handle);

/* ---- per-module entry points (the reference's method surface), batched over M ----------- */

/* Column.timestep (column.py:315-348).  `stages` selects what runs, in the reference's
 * order: convect -> vertadvdiff -> horadv; vertadvdiff applies the surface condition
 * b[-1]=bs unless do_conv (column.py:230-231). */
#define PMOC_STAGE_CONVECT 1u
#define PMOC_STAGE_VERTADVDIFF 2u
#define PMOC_STAGE_HORADV 4u
int pmoc_column_timestep(int64_t M, int32_t nz, const double* z, const pmoc_column* col, pmoc_vec wA,
                         pmoc_vec vdx_in, pmoc_vec b_in, double dt, uint32_t stages, void* stream);

/* Psi_Thermwind.solve (psi_thermwind.py:125-135): exact double quadrature of the linear BVP.
 * gmid: optional [nz-1] samples of (b2-b1) at the cell mid-points for callable profiles
 * (ptr==NULL -> piecewise-linear b's).  Psi in Sv. */
int pmoc_thermwind_solve(int64_t M, int32_t nz, const double* z, pmoc_vec b1, pmoc_vec b2, pmoc_vec f,
                         pmoc_vec gmid, double* Psi, void* stream);

/* Psi_Thermwind.Psib / Psibz (psi_thermwind.py:137-208).  Outputs optional except psib.
 * PMOC_EUNSUPPORTED when nb needs more shared memory than one block has (nb > 3816 at nz = 256). */
int pmoc_thermwind_psib(int64_t M, int32_t nz, int32_t nb, pmoc_vec Psi, pmoc_vec b1, pmoc_vec b2,
                        double* psib, double* bgrid, double* iso_b, double* iso_n, void* stream);

/* Psi_SO.solve (psi_SO.py:333-354) with ys/calc_Ekman/calc_GM inside.  `so` reuses the
 * Psi_SO fields of pmoc_model (so_*, y, ny, z, nz, M); b is the basin profile.
 * PMOC_EUNSUPPORTED when ny needs more shared memory than one block has (ny > 2136 at nz = 256). */
int pmoc_so_solve(const pmoc_model* so, pmoc_vec b, pmoc_vec bs, double* Psi, double* Psi_Ek, double* Psi_GM,
                  double* ys, uint32_t* status, void* stream);

/* SO_ML.timestep / advdiff (SO_ML.py:198-303).  `ml` reuses the ml_* fields of pmoc_model. */
int pmoc_ml_timestep(const pmoc_model* ml, pmoc_vec b_basin, pmoc_vec Psi_b, double dt, uint32_t* status,
                     void* stream);

/* FP64 roofline probe: a dependent-free DFMA stream on every SM; returns the measured
 * TFLOP/s (2 flops per FMA) in *tflops.  Used by bench.py for the roofline denominator. */
int pmoc_fp64_peak(double* tflops, double* sm_mhz_est, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PYMOC_B200_H_ */
