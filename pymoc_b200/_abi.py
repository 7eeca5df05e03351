"""ctypes mirror of ``include/pymoc_b200.h`` (keep the two in sync; ABI version checked at load)."""
import ctypes as C

ABI_VERSION = 3

OK, EINVAL, EUNSUPPORTED, ECUDA, ENODEVICE = range(5)
STATUS_NAMES = {1: 'EINVAL', 2: 'EUNSUPPORTED', 3: 'ECUDA', 4: 'ENODEVICE'}

HAS_NORTH, HAS_TW, ISO, HAS_SO, HAS_ML, ORDER_JN, SO_BVP, HAS_PAC = 1, 2, 4, 8, 16, 32, 64, 128
STAGE_CONVECT, STAGE_VERTADVDIFF, STAGE_HORADV = 1, 2, 4
IO_STATE, IO_PSI, IO_DIAG = 1, 2, 4
MAX_NZ_WARP, MAX_NZ_WIDE, MAX_NY_ML = 256, 4096, 64  # PMOC_MAX_* of the header
ST_NAN, ST_BS_NONMONOTONE, ST_BRENT_SIGN, ST_XP_NONMONOTONE, ST_ML_INDEX, ST_BVP_SERIES, ST_NOISE_SWITCH = 1, 2, 4, 8, 16, 32, 64
ST_TIE_CELL, ST_BS_SAWTOOTH = 128, 256
ST_PARITY_UNDEFINED = ST_BS_NONMONOTONE | ST_NOISE_SWITCH | ST_TIE_CELL  # the reference's own result hangs on rounding noise
ST_PUBLIC_MASK = 0x0FFFFFFF  # the top bits carry kernel-internal hand-over flags between launches
ST_BIT_NAMES = {1: 'nan', 2: 'bs_nonmonotone', 4: 'brent_sign', 8: 'xp_nonmonotone', 16: 'ml_index', 32: 'bvp_series',
                64: 'noise_switch', 128: 'tie_cell', 256: 'bs_sawtooth'}


def status_census(status):
  """Members per status bit, plus how many carry a parity-undefined bit and how many carry none at all."""
  import numpy as np
  st = np.asarray(status).astype(np.uint32) & np.uint32(ST_PUBLIC_MASK)
  out = {name: int(((st & np.uint32(bit)) != 0).sum()) for bit, name in ST_BIT_NAMES.items()}
  out['parity_undefined'] = int(((st & np.uint32(ST_PARITY_UNDEFINED)) != 0).sum())
  out['clean'] = int((st == 0).sum())
  out['members'] = int(st.size)
  return out

c_double_p = C.POINTER(C.c_double)


class Vec(C.Structure):
  _fields_ = [('ptr', C.c_void_p), ('mstride', C.c_int64)]


class Column(C.Structure):
  _fields_ = [('b', C.c_void_p), ('kappa', Vec), ('dAk', Vec), ('Area', Vec), ('bs', Vec), ('N2min', Vec),
              ('bzbot', Vec), ('bbot', C.c_void_p), ('var', C.c_void_p), ('nvar', C.c_int32), ('do_conv', C.c_int32)]


class Model(C.Structure):
  _fields_ = [
      ('M', C.c_int64), ('nz', C.c_int32), ('ny', C.c_int32), ('nb', C.c_int32), ('K', C.c_int32),
      ('flags', C.c_uint32), ('dt', C.c_double), ('z', C.c_void_p), ('y', C.c_void_p),
      ('basin', Column), ('north', Column), ('pac', Column),
      ('tw_f', Vec), ('tw_b2', Vec), ('zoc_f', Vec),
      ('so_bs', Vec), ('so_tau', Vec), ('so_f', Vec), ('so_rho', Vec), ('so_L', Vec), ('so_KGM', Vec),
      ('so_smax', Vec), ('so_c', Vec), ('so2_L', Vec), ('so_tau_on_y', C.c_int32), ('so_bvp_with_Ek', C.c_int32),
      ('so_sill_taper', C.c_void_p), ('so_ek_taper', C.c_void_p), ('so_top_taper', C.c_void_p),
      ('so_bot_taper', C.c_void_p),
      ('ml_bs', C.c_void_p), ('ml_Ks', Vec), ('ml_h', Vec), ('ml_L', Vec), ('ml_vpist', Vec),
      ('ml_surflux', Vec), ('ml_rest_mask', Vec), ('ml_b_rest', Vec),
      ('Psi_tw', C.c_void_p), ('Psi_iso_b', C.c_void_p), ('Psi_iso_n', C.c_void_p), ('psib', C.c_void_p),
      ('bgrid', C.c_void_p), ('Psi_so', C.c_void_p), ('Psi_Ek', C.c_void_p), ('Psi_GM', C.c_void_p),
      ('ml_Psi_s', C.c_void_p),
      ('Psi_zoc', C.c_void_p), ('Psi_zon_a', C.c_void_p), ('Psi_zon_p', C.c_void_p), ('psib2', C.c_void_p),
      ('bgrid2', C.c_void_p), ('Psi_so2', C.c_void_p), ('Psi_Ek2', C.c_void_p), ('Psi_GM2', C.c_void_p),
      ('status', C.c_void_p), ('scratch', C.c_void_p), ('scratch_bytes', C.c_uint64),
  ]


EXPORTS = ('pmoc_abi_version', 'pmoc_last_error', 'pmoc_device_info', 'pmoc_model_scratch_bytes', 'pmoc_model_diagnose', 'pmoc_model_run',
           'pmoc_model_run_host', 'pmoc_host_last_bytes', 'pmoc_host_open', 'pmoc_host_step', 'pmoc_host_close', 'pmoc_column_timestep', 'pmoc_thermwind_solve', 'pmoc_thermwind_psib',
           'pmoc_so_solve', 'pmoc_ml_timestep', 'pmoc_fp64_peak', 'pmoc_model_run_members', 'pmoc_equilibrate_work_bytes',
           'pmoc_model_equilibrate', 'pmoc_model_equilibrate_host', 'pmoc_host_equilibrate')


def declare(lib):
  """Attach argument / result types to the exported functions of a loaded library."""
  P = C.POINTER
  lib.pmoc_abi_version.restype = C.c_int
  lib.pmoc_abi_version.argtypes = []
  lib.pmoc_last_error.restype = C.c_char_p
  lib.pmoc_last_error.argtypes = []
  lib.pmoc_device_info.argtypes = [P(C.c_int), P(C.c_int), P(C.c_int)]
  lib.pmoc_model_scratch_bytes.argtypes = [P(Model)]
  lib.pmoc_model_diagnose.argtypes = [P(Model), C.c_void_p]
  lib.pmoc_model_run.argtypes = [P(Model), C.c_int64, C.c_int64, C.c_void_p]
  lib.pmoc_model_run_host.argtypes = [P(Model), C.c_int64, C.c_int64]
  lib.pmoc_host_last_bytes.argtypes = [P(C.c_uint64), P(C.c_uint64)]
  lib.pmoc_host_last_bytes.restype = None
  lib.pmoc_host_open.argtypes = [P(Model), P(C.c_void_p)]
  lib.pmoc_host_step.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_uint32, C.c_uint32]
  lib.pmoc_host_close.argtypes = [C.c_void_p]
  lib.pmoc_column_timestep.argtypes = [C.c_int64, C.c_int32, C.c_void_p, P(Column), Vec, Vec, Vec, C.c_double,
                                       C.c_uint32, C.c_void_p]
  lib.pmoc_thermwind_solve.argtypes = [C.c_int64, C.c_int32, C.c_void_p, Vec, Vec, Vec, Vec, C.c_void_p, C.c_void_p]
  lib.pmoc_thermwind_psib.argtypes = [C.c_int64, C.c_int32, C.c_int32, Vec, Vec, Vec, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_void_p]
  lib.pmoc_so_solve.argtypes = [P(Model), Vec, Vec, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                C.c_void_p]
  lib.pmoc_ml_timestep.argtypes = [P(Model), Vec, Vec, C.c_double, C.c_void_p, C.c_void_p]
  lib.pmoc_fp64_peak.argtypes = [P(C.c_double), P(C.c_double), C.c_void_p]
  lib.pmoc_model_run_members.argtypes = [P(Model), C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p]
  lib.pmoc_equilibrate_work_bytes.argtypes = [P(Model)]
  lib.pmoc_model_equilibrate.argtypes = [P(Model), C.c_int64, C.c_int64, C.c_int64, C.c_double, C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_uint64, C.c_void_p]
  lib.pmoc_model_equilibrate_host.argtypes = [P(Model), C.c_int64, C.c_int64, C.c_int64, C.c_double, C.c_void_p,
                                              C.c_void_p]
  lib.pmoc_host_equilibrate.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_double, C.c_void_p, C.c_void_p,
                                        C.c_uint32, C.c_uint32]
  for name in EXPORTS:
    if name not in ('pmoc_last_error', 'pmoc_model_scratch_bytes', 'pmoc_host_last_bytes', 'pmoc_equilibrate_work_bytes'):
      getattr(lib, name).restype = C.c_int
  lib.pmoc_model_scratch_bytes.restype = C.c_uint64
  lib.pmoc_equilibrate_work_bytes.restype = C.c_uint64
  if lib.pmoc_abi_version() != ABI_VERSION:
    raise RuntimeError('pymoc_b200: ABI version mismatch (library %d, python %d)' %
                       (lib.pmoc_abi_version(), ABI_VERSION))
  return lib


class PmocError(RuntimeError):
  pass


def check(lib, rc):
  if rc != OK:
    msg = lib.pmoc_last_error()
    raise PmocError('pymoc_b200: %s: %s' % (STATUS_NAMES.get(rc, rc), msg.decode() if msg else ''))
