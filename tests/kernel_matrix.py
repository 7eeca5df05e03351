"""Every instantiation of the fused warp-per-member kernel and the batched per-module entry points against the
reference, shared by the CPU (warp-emulator) and GPU test files.

Fused kernel: one cell per topology of ``launch_model`` and levels per lane 2..8, each stepping five members of an
eight-member lattice (the last CTA is partly empty for any warps-per-CTA split) across at least two diagnoses, and
checked three ways: against the live oracle, split launches bit for bit, and CTA packing (``PMOC_WPB``) bit for bit.

Per-module entry points: M = 9 members (three four-warp CTAs, the last with one live warp), per-member inputs with a
member stride mixed with shared (stride 0) ones, one NaN sentinel row after the last member of every output; every
member equals its own M = 1 call bit for bit and the oracle's per-module function.
"""
import contextlib
import ctypes
import dataclasses
import os
import re
import types
import warnings

import numpy as np

from helpers import relmax
from oracle import pymoc_oracle as O
from pymoc_b200 import _abi, configs
from pymoc_b200.ensemble import Ensemble, so_tapers, topology_flags
from pymoc_b200.spec import ThermwindSpec, _vec

TOL = 1e-10
BVP_TOL = 1e-9  # solve_bvp tolerance of the converged reference of the F2010 smoother (the reference runs 1e-3)
SIZES = (64, 65, 128, 129, 192, 193, 256)  # levels per lane 2..8: a full last lane slot, then one level into a new one
LPLS = (2, 3, 4, 5, 6, 7, 8)
K = 3
NSTEPS = 2 * K + 1
CUTS = (K, K + 2)  # launch boundaries: on a diagnosis iteration, and between two diagnoses
MEMBERS = (0, 5)  # of an eight-member lattice

H = _abi
# The topologies of launch_model's switch (pymoc_b200/csrc/pmoc_model.cu, PM_CASE lines), one cell builder each.
TOPOLOGIES = {
    'tw': H.HAS_TW,
    'so': H.HAS_SO,
    'so_bvp': H.HAS_SO | H.SO_BVP,
    'tw_so': H.HAS_TW | H.HAS_SO,
    'tw_so_bvp': H.HAS_TW | H.HAS_SO | H.SO_BVP,
    'twocol': H.HAS_NORTH | H.HAS_TW | H.ISO,
    'c3': H.HAS_NORTH | H.HAS_TW | H.ISO | H.HAS_SO,
    'c3_bvp': H.HAS_NORTH | H.HAS_TW | H.ISO | H.HAS_SO | H.SO_BVP,
    'twobasin': H.HAS_NORTH | H.HAS_TW | H.ISO | H.HAS_SO | H.HAS_PAC,
    'jn': H.HAS_NORTH | H.HAS_TW | H.ISO | H.HAS_SO | H.HAS_ML,
    'jn_bvp': H.HAS_NORTH | H.HAS_TW | H.ISO | H.HAS_SO | H.HAS_ML | H.SO_BVP,
}
CELLS = [(name, nz) for name in TOPOLOGIES for nz in SIZES]
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def lpl_for(nz):
  """Levels per lane of the warp kernels (pmoc_ops.cu lpl_for)."""
  return 2 if nz <= 64 else (nz + 31) // 32


def switch_topologies():
  """The topology flags of the PM_CASE lines of launch_model, read from the source."""
  src = open(os.path.join(ROOT, 'pymoc_b200', 'csrc', 'pmoc_model.cu')).read()
  body = src[src.index('switch (t) {'):]
  body = body[:body.index('default:')]
  out = set()
  for expr in re.findall(r'PM_CASE\(([^)]*)\)', body):
    out.add(sum(getattr(_abi, f.strip()[len('PMOC_'):]) for f in expr.split('|')))
  return out


def kernel_topology(spec):
  """(T, levels per lane) that run_model hands to launch_model for ``spec``."""
  t = topology_flags(spec) & ~_abi.ORDER_JN
  if spec.so is not None and spec.so.c is not None:
    t |= _abi.SO_BVP
  return t, lpl_for(spec.nz)


# ------------------------------------------------------------------------------------------------ cells
def regrid(spec, nz):
  """The same model on ``nz`` uniform levels: every z-profile (each column's kappa variants, Area, b0, and tw.b2)
  interpolated, ``dt`` scaled by (dz_new / dz_old)^2 on a finer grid so that the explicit step stays as stable as it
  was (a coarser grid keeps ``dt``: the mixed layer's step does not get more stable with dz)."""
  z0 = spec.z
  z = np.linspace(z0[0], z0[-1], nz)
  on_z = lambda a: np.ascontiguousarray(np.apply_along_axis(lambda r: np.interp(z, z0, r), -1, a))

  def col(c):
    return None if c is None else dataclasses.replace(c, kappa=on_z(c.kappa), Area=on_z(c.Area), b0=on_z(c.b0))

  tw = spec.tw if spec.tw is None or spec.tw.b2 is None else dataclasses.replace(spec.tw, b2=on_z(spec.tw.b2))
  return dataclasses.replace(spec, z=z, dt=spec.dt * min(1., ((z[1] - z[0]) / (z0[1] - z0[0]))**2), basin=col(spec.basin),
                             north=col(spec.north), pac=col(spec.pac), tw=tw)


def _with_f2010(spec, c=0.1):
  so = dataclasses.replace(spec.so, c=_vec(c, 'c'), bvp_with_Ek=True)
  return dataclasses.replace(spec, so=so)


def cell(name, nz):
  """(spec, environment) of one cell: five members of an eight-member lattice of the topology ``name`` on nz levels,
  K = 3.  C1 takes the generic kernel at nz > 144 and as a convecting column (nz = 65); below that the
  several-members-per-warp kernel is switched off."""
  env = {}
  with configs.members(*MEMBERS):
    if name == 'tw':
      spec = configs.c1_timestepping(8, nz=nz)
      spec.dt *= (69. / (nz - 1))**2  # the script's 60 days at its 70 levels
      if nz == 65:
        spec = dataclasses.replace(spec, basin=dataclasses.replace(spec.basin, do_conv=True))
      elif nz <= 144:
        env['PMOC_NO_TWCOL'] = '1'
    elif name in ('so', 'so_bvp', 'tw_so', 'tw_so_bvp'):
      spec = configs.c2_column_so(8, nz=nz, ny=40, dt_days=10. * (199. / (nz - 1))**2)
      if name.startswith('tw_so'):  # column + thermal wind against a fixed northern profile + Psi_SO
        spec = dataclasses.replace(spec, tw=ThermwindSpec.build(spec.z, f=1e-4, b2=0.004 * np.exp(spec.z / 300.)),
                                   iso=False)
    elif name == 'twocol':
      spec = regrid(configs.twocol(8), nz)
    elif name in ('c3', 'c3_bvp'):
      spec = regrid(configs.c3_twocol_so(8), nz)
    elif name == 'twobasin':
      spec = regrid(configs.twobasin(8), nz)
    elif name == 'jn':
      spec = configs.c5_single_global_basin(8, nz=nz, dt_days=30. * (45. / (nz - 1))**2, axes=(2, 2, 1, 2),
                                            kapfac_max=1.)
    elif name == 'jn_bvp':
      spec = regrid(configs.c4_jansen_nadeau(8, axes=(2, 2, 1, 1, 2)), nz)  # tau x kapfac x KGM
    else:
      raise KeyError(name)
  if name.endswith('_bvp'):
    spec = _with_f2010(spec)
  spec.K = K
  return spec, env


def _flat(case):
  """Every number of an oracle case, for telling members apart."""
  out = []
  for k in sorted(case):
    v = case[k]
    if isinstance(v, dict):
      out.append(_flat(v))
    elif isinstance(v, (int, float, np.ndarray)) and not isinstance(v, bool):
      out.append(np.ravel(np.asarray(v, dtype=np.float64)))
  return np.concatenate(out) if out else np.zeros(0)


# ------------------------------------------------------------------------------------------------ oracle
@contextlib.contextmanager
def converged_f2010(tol=BVP_TOL):
  """The oracle with the F2010 smoother's solve_bvp run to ``tol`` (the reference runs it at 1e-3, adaptively): only
  so_gm's call is tightened, the thermal-wind solve is left as the reference runs it."""
  orig_gm, orig_int = O.so_gm, O.integrate
  tight = types.SimpleNamespace(solve_bvp=lambda *a, **k: orig_int.solve_bvp(*a, **{'tol': tol, 'max_nodes': 100000, **k}))

  def so_gm(*a, **k):
    O.integrate = tight
    try:
      return orig_gm(*a, **k)
    finally:
      O.integrate = orig_int

  O.so_gm = so_gm
  try:
    yield
  finally:
    O.so_gm, O.integrate = orig_gm, orig_int


def oracle_task(args):
  """One member through run_coupled: (case, nsteps, converged) -> dict of fields, or the text of what it raised."""
  case, nsteps, converged = args
  warnings.filterwarnings('ignore')
  try:
    with converged_f2010() if converged else contextlib.nullcontext():
      out = O.run_coupled(case, nsteps, O.REFERENCE)
    return {k: v for k, v in out.items() if v is not None}
  except (ValueError, IndexError, FloatingPointError) as e:
    return repr(e)


def oracle_pool():
  """Spawned workers for the oracle (safe next to CUDA), one BLAS thread each."""
  import multiprocessing as mp
  os.environ.setdefault('OMP_NUM_THREADS', '1')
  os.environ.setdefault('OPENBLAS_NUM_THREADS', '1')
  return mp.get_context('spawn').Pool(os.cpu_count() or 1)


# ------------------------------------------------------------------------------------------------ part 1
def _run(backend, spec, launches):
  ens = Ensemble(spec, backend=backend)
  for n in launches:
    ens.run(n)
  return {**ens.state(), **ens.diagnostics()}


def _same(a, b, what):
  assert a.keys() == b.keys(), what
  for k in a:
    assert np.array_equal(a[k], b[k], equal_nan=True), (what, k)


def fused_cell(backend, pool, monkeypatch, name, nz, bitwise=True, adaptive=False):
  """One cell of the fused-kernel matrix; returns its report (worst error, excused members)."""
  spec, env = cell(name, nz)
  assert kernel_topology(spec) == (TOPOLOGIES[name], lpl_for(nz)), (name, nz, kernel_topology(spec))
  cases = [spec.member_case(m) for m in range(spec.M)]
  assert spec.M == MEMBERS[1] - MEMBERS[0]
  vecs = [_flat(c) for c in cases]
  for i in range(len(vecs)):
    for j in range(i):
      assert not np.array_equal(vecs[i], vecs[j]), ('members not distinct', name, nz, i, j)
  bvp = spec.so is not None and spec.so.c is not None
  pending = pool.map_async(oracle_task, [(c, NSTEPS, bvp) for c in cases], chunksize=1)
  loose = pool.map_async(oracle_task, [(c, NSTEPS, False) for c in cases], chunksize=1) if bvp and adaptive else None
  for k, v in env.items():
    monkeypatch.setenv(k, v)
  got = _run(backend, spec, [NSTEPS])
  if bitwise:
    _same(got, _run(backend, spec, [CUTS[0], CUTS[1] - CUTS[0], NSTEPS - CUTS[1]]), (name, nz, 'split launches'))
    for wpb in ('1', '3'):
      monkeypatch.setenv('PMOC_WPB', wpb)
      _same(got, _run(backend, spec, [NSTEPS]), (name, nz, 'PMOC_WPB=' + wpb))
    monkeypatch.delenv('PMOC_WPB')
  st = got['status']
  rep = dict(cell=name, T=TOPOLOGIES[name], nz=nz, lpl=lpl_for(nz), worst=0.0, excused=0)
  for m, want in enumerate(pending.get()):
    if st[m] & _abi.ST_PARITY_UNDEFINED:
      rep['excused'] += 1
      continue
    assert not isinstance(want, str), (name, nz, m, want)
    assert not st[m] & (_abi.ST_NAN | _abi.ST_BRENT_SIGN | _abi.ST_ML_INDEX), (name, nz, m, int(st[m]))
    for key, w in want.items():
      err = relmax(got[key][m], w)
      rep['worst'] = max(rep['worst'], err)
      assert err < TOL, '%s nz=%d member %d field %s: rel err %.3e' % (name, nz, m, key, err)
  assert spec.M - rep['excused'] >= 4, ('vacuous cell', name, nz, rep['excused'])
  if loose is not None:
    rep['vs_adaptive'] = max(relmax(got[k][m], w[k]) for m, w in enumerate(loose.get()) if not isinstance(w, str)
                             and not st[m] & _abi.ST_PARITY_UNDEFINED for k in w)
  print('matrix %-10s T=%3d nz=%3d lpl=%d worst %.2e excused %d%s' % (
      name, rep['T'], nz, rep['lpl'], rep['worst'], rep['excused'],
      ' vs adaptive solve_bvp %.2e' % rep['vs_adaptive'] if 'vs_adaptive' in rep else ''))
  return rep


def matrix_is_complete():
  """The cells cover exactly the (T, levels per lane) pairs of launch_model's switch."""
  assert set(TOPOLOGIES.values()) == switch_topologies()
  ran = {kernel_topology(cell(name, nz)[0]) for name, nz in CELLS}
  assert ran == {(t, l) for t in switch_topologies() for l in LPLS}


def jn_f2010_wide_refused(backend):
  """'jn' with the F2010 smoother above 256 levels has no block-per-member kernel: refused, never run."""
  import pytest
  with configs.members(0, 2):
    spec = _with_f2010(configs.c5_single_global_basin(8, nz=320, dt_days=1., axes=(2, 2, 1, 2), kapfac_max=1.))
  ens = Ensemble(spec, backend=backend)
  with pytest.raises(_abi.PmocError, match="EUNSUPPORTED: nz > 256: only the 'jn' topology"):
    ens.run(3)


# ------------------------------------------------------------------------------------------------ part 2
MOD_M = 9  # three four-warp CTAs, the last with one live warp
MOD_SIZES = (33,) + SIZES


class Batch:
  """Device buffers of one per-module call."""

  def __init__(self, backend):
    self.be, self.lib, self.keep = backend, backend.lib, []

  def buf(self, arr, dtype=np.float64):
    b = self.be.upload(np.ascontiguousarray(arr, dtype=dtype))
    self.keep.append(b)
    return b

  def ptr(self, arr, dtype=np.float64):
    return None if arr is None else self.be.ptr(self.buf(arr, dtype))

  def vec(self, arr):
    """[M, n] rows with member stride n, or one shared row / scalar ([n] or 0-D) with stride 0."""
    if arr is None:
      return _abi.Vec(None, 0)
    a = np.asarray(arr, dtype=np.float64)
    return _abi.Vec(self.ptr(a), a.shape[1] if a.ndim == 2 else 0)

  def out(self, M, n, fill=np.nan, dtype=np.float64):
    """An output of M rows plus one sentinel row."""
    return self.buf(np.full((M + 1, n), fill, dtype=dtype), dtype)

  def get(self, b):
    self.be.sync()
    return self.be.download(b)


def _pick(a, m):
  """Member m's value of a per-member [M, ...] array or a shared one."""
  return None if a is None else (a[m] if np.ndim(a) == 2 else a)


def _sentinel(arrs, M, tag):
  for k, a in arrs.items():
    if a.dtype == np.float64:
      assert np.isnan(a[M]).all(), (tag, k, 'store past the last member')
    else:
      assert (a[M] == 0xA5A5A5A5).all(), (tag, k, 'store past the last member')


def _member_rows(batched, single, M, tag):
  for k in batched:
    for m in range(M):
      assert np.array_equal(batched[k][m], single[m][k][0], equal_nan=True), (tag, k, m, 'differs from its M = 1 call')


def _oracle_rows(batched, want, M, tag, tol=TOL, floor=None):
  """``floor[m]``: smallest scale of member m's errors (psib at nb = 2 is a sum of transports that cancel to rounding
  noise: its error is measured against the transports)."""
  worst = 0.0
  for m in range(M):
    for k, w in want[m].items():
      err = relmax(batched[k][m], w)
      if floor is not None and np.isfinite(err) and err > 0:
        err *= np.nanmax(np.abs(w)) / max(np.nanmax(np.abs(w)), floor[m])
      worst = max(worst, err)
      assert err < tol, (tag, m, k, err)
  return worst


def _grid(nz):
  return np.linspace(-4000., 0., nz)


def _column_call(be, z, inp, stages, do_conv, M):
  c = Batch(be)
  col = _abi.Column()
  b = c.buf(np.vstack([inp['b'][:M], np.full((1, z.size), np.nan)]))
  col.b = be.ptr(b)
  col.kappa, col.dAk, col.Area = c.vec(inp['kappa'][:M]), c.vec(inp['dAk'][:M]), c.vec(inp['Area'])
  col.bs, col.N2min = c.vec(inp['bs'][:M, None]), c.vec(inp['N2min'])
  col.bzbot = c.vec(None if inp['bzbot'] is None else inp['bzbot'][:M, None])
  col.bbot = c.ptr(inp['bbot'][:M])
  col.nvar, col.do_conv = 1, int(do_conv)
  rc = be.lib.pmoc_column_timestep(M, z.size, c.ptr(z), ctypes.byref(col), c.vec(inp['wA'][:M]),
                                   c.vec(inp['vdx'][:M]), c.vec(inp['b_in'][:M]), inp['dt'], stages, be.stream())
  _abi.check(be.lib, rc)
  return {'b': c.get(b)}


def _one(inp, m):
  """Member m's inputs as a one-member batch."""
  return {k: (v[m:m + 1] if isinstance(v, np.ndarray) and v.ndim >= 1 and v.shape[0] == MOD_M else v)
          for k, v in inp.items()}


def column_batched(backend, grid=_grid, stage_masks=(1, 2, 3, 7)):
  """``grid(nz)``: the z levels (uniform by default); ``stage_masks``: the stage masks run at every size."""
  rng = np.random.default_rng(3)
  M = MOD_M
  worst = 0.0
  cases = [(nz, st, dc, False) for nz in MOD_SIZES for st in stage_masks for dc in (False, True)] + [(129, 3, False, True)]
  for nz, stages, do_conv, bzbot in cases:
    z = grid(nz)
    kap = (1e-5 + 3e-4 * np.exp(-z / 1000 - 4))[None, :] * np.linspace(0.5, 1.2, M)[:, None]
    area = 6e13 * (1. + 0.2 * z / 4000.)  # shared (stride 0)
    b = 0.03 * np.exp(z / 300.)[None, :] * np.linspace(0.8, 1.2, M)[:, None] - 0.001
    b[:, -3:] += 0.004 * (np.arange(M) % 3)[:, None]  # some members unstable at the top: convection has work
    inp = dict(b=b, kappa=kap, dAk=np.gradient(area[None, :] * kap, z, axis=-1), Area=area,
               bs=np.linspace(0.025, 0.033, M), N2min=np.array(1.5e-7), bbot=np.linspace(-0.002, 0., M),
               bzbot=np.linspace(1e-7, 5e-7, M) if bzbot else None,
               wA=rng.normal(0, 2e6, (M, nz)), vdx=rng.normal(0, 1e7, (M, nz)), b_in=rng.uniform(-0.002, 0.03, (M, nz)),
               dt=0.3 * np.diff(z).min()**2 / kap.max())
    tag = ('column', nz, stages, do_conv, bzbot)
    got = _column_call(backend, z, inp, stages, do_conv, M)
    _sentinel(got, M, tag)
    _member_rows(got, [_column_call(backend, z, _one(inp, m), stages, do_conv, 1) for m in range(M)], M, tag)
    want = []
    for m in range(M):
      col = O.ColumnState(z, kap[m], area, b[m], inp['bs'][m], inp['bbot'][m], None if not bzbot else inp['bzbot'][m],
                          1.5e-7)
      col.dAk = inp['dAk'][m]
      if stages & 1:
        O.column_convect(col)
      if stages & 2:
        O.column_vertadvdiff(col, inp['wA'][m], inp['dt'], do_conv)
      if stages & 4:
        O.column_horadv(col, inp['vdx'][m], inp['b_in'][m], inp['dt'])
      want.append({'b': col.b})
    worst = max(worst, _oracle_rows(got, want, M, tag))
  return worst


def _tw_call(be, z, inp, M):
  c = Batch(be)
  psi = c.out(M, z.size)
  _abi.check(be.lib, be.lib.pmoc_thermwind_solve(M, z.size, c.ptr(z), c.vec(inp['b1'][:M]), c.vec(inp['b2']),
                                                  c.vec(inp['f'][:M, None]), c.vec(inp['gmid']), be.ptr(psi),
                                                  be.stream()))
  return {'Psi': c.get(psi)}


def thermwind_batched(backend, grid=_grid):
  M, worst = MOD_M, 0.0
  for nz in SIZES:
    for with_gmid in (False, True):
      z = grid(nz)
      b1 = 0.03 * np.exp(z / 300.)[None, :] * np.linspace(0.7, 1.3, M)[:, None]
      b2 = 0.004 * np.exp(z / 500.)  # shared
      g = b2[None, :] - b1
      gmid = np.hstack([0.5 * (g[:, 1:] + g[:, :-1]), np.zeros((M, 1))]) if with_gmid else None
      inp = dict(b1=b1, b2=b2, f=np.linspace(0.8e-4, 1.4e-4, M), gmid=gmid)
      tag = ('thermwind', nz, with_gmid)
      got = _tw_call(backend, z, inp, M)
      _sentinel(got, M, tag)
      _member_rows(got, [_tw_call(backend, z, _one(inp, m), 1) for m in range(M)], M, tag)
      want = [{'Psi': O.thermwind_solve(z, b1[m], b2, inp['f'][m])} for m in range(M)]
      worst = max(worst, _oracle_rows(got, want, M, tag))
  return worst


def _psib_call(be, nz, nb, inp, M):
  c = Batch(be)
  outs = {'psib': c.out(M, nb), 'bgrid': c.out(M, nb), 'iso_b': c.out(M, nz), 'iso_n': c.out(M, nz)}
  rc = be.lib.pmoc_thermwind_psib(M, nz, nb, c.vec(inp['Psi'][:M]), c.vec(inp['b1'][:M]), c.vec(inp['b2']),
                                  *[be.ptr(outs[k]) for k in ('psib', 'bgrid', 'iso_b', 'iso_n')], be.stream())
  _abi.check(be.lib, rc)
  return {k: c.get(v) for k, v in outs.items()}


def _psib_inputs(nz, M, rng):
  z = _grid(nz)
  b1 = 0.03 * np.exp(z / 300.)[None, :] * np.linspace(0.7, 1.3, M)[:, None]
  b1[1, 10:20] = b1[1, 10:20][::-1]  # one member with an inverted region: the remap's direct path
  psi = 10 * np.sin(np.pi * z / 4000.)**2 * np.sign(z + 1500)
  psi = psi[None, :] * np.linspace(0.5, 1.5, M)[:, None] + rng.normal(0, 0.1, (M, nz))
  psi[:, 0] = psi[:, -1] = 0.
  return dict(Psi=psi, b1=b1, b2=0.004 * np.exp(z / 300.))


def psib_batched(backend):
  rng = np.random.default_rng(5)
  M, worst = MOD_M, 0.0
  for nz in SIZES:
    for nb in (2, 37, 500, 1001):
      inp = _psib_inputs(nz, M, rng)
      tag = ('psib', nz, nb)
      got = _psib_call(backend, nz, nb, inp, M)
      _sentinel(got, M, tag)
      _member_rows(got, [_psib_call(backend, nz, nb, _one(inp, m), 1) for m in range(M)], M, tag)
      want = []
      with np.errstate(all='ignore'):
        for m in range(M):
          ib, in_, p, g = O.thermwind_psibz(inp['Psi'][m], inp['b1'][m], inp['b2'], nb)
          want.append({'psib': p, 'bgrid': g, 'iso_b': ib, 'iso_n': in_})
      worst = max(worst, _oracle_rows(got, want, M, tag, floor=np.abs(inp['Psi']).max(axis=1)))
  return worst


def _so_model(c, z, y, inp, M):
  m = _abi.Model()
  m.M, m.nz, m.ny = M, z.size, y.size
  m.z, m.y = c.ptr(z), c.ptr(y)
  m.so_tau, m.so_tau_on_y = c.vec(inp['tau'][:M] if inp['tau'].ndim == 2 else inp['tau'][:M, None]), int(inp['tau'].ndim == 2)
  m.so_f, m.so_rho, m.so_smax = c.vec(inp['f']), c.vec(inp['rho']), c.vec(inp['smax'])  # 0-D shared, [M, 1] per member
  m.so_L, m.so_KGM = c.vec(inp['L'][:M, None]), c.vec(inp['KGM'][:M, None])
  m.so_c = c.vec(None if inp['c'] is None else inp['c'][:M, None])
  m.so_bvp_with_Ek = int(inp['c'] is not None)
  m.so_sill_taper, m.so_ek_taper, m.so_top_taper, m.so_bot_taper = (c.ptr(t) for t in so_tapers(z, **inp.get('H', {})))
  return m


def _so_call(be, z, y, inp, M):
  c = Batch(be)
  m = _so_model(c, z, y, inp, M)
  outs = {k: c.out(M, z.size) for k in ('Psi', 'Psi_Ek', 'Psi_GM', 'ys')}
  status = c.buf(np.array([0] * M + [0xA5A5A5A5], dtype=np.uint32), np.uint32)
  rc = be.lib.pmoc_so_solve(ctypes.byref(m), c.vec(inp['b'][:M]), c.vec(inp['bs'][:M]),
                            *[be.ptr(outs[k]) for k in ('Psi', 'Psi_Ek', 'Psi_GM', 'ys')], be.ptr(status), be.stream())
  _abi.check(be.lib, rc)
  got = {k: c.get(v) for k, v in outs.items()}
  got['status'] = c.get(status).view(np.uint32)[:, None]
  return got


def _so_inputs(nz, ny, tau_on_y, with_c, M, grid=_grid):
  z, y = grid(nz), np.linspace(0, 2e6, ny)
  bs = 0.03 * (y / y[-1])[None, :]**2 * np.linspace(0.8, 1.2, M)[:, None]
  b = 0.03 * np.exp(z / 300.)[None, :] * np.linspace(0.6, 1.1, M)[:, None] - 0.0005
  tau = np.linspace(0.05, 0.25, M)
  if tau_on_y:
    tau = tau[:, None] * np.sin(np.pi * y / y[-1])[None, :]
  return z, y, dict(b=b, bs=bs, tau=tau, f=np.array(1e-4), rho=np.array(1030.), smax=np.array(0.01),
                    L=np.linspace(4e6, 6e6, M), KGM=np.linspace(800., 1200., M),
                    c=np.linspace(0.08, 0.12, M) if with_c else None)


def _so_oracle(args):
  z, y, tau, L, KGM, c, b, bs = args
  with converged_f2010() if c is not None else contextlib.nullcontext():
    p = O.ChannelParams(z, y, tau, f=1e-4, rho=1030., L=L, KGM=KGM, c=c, bvp_with_Ek=c is not None, smax=0.01)
    psi, ek, gm = O.so_solve(p, b, bs)
  return {'Psi': psi, 'Psi_Ek': ek, 'Psi_GM': gm, 'ys': np.array([O.so_outcrop(v, y, bs) for v in b])}


def so_batched(backend, pool, f2010_sizes=SIZES):
  """ny 3 / 40 / 64 in turn, tau a float or a profile on y, without and (at ``f2010_sizes``) with the F2010 smoother."""
  M, worst = MOD_M, {'explicit': 0.0, 'f2010': 0.0}
  k = 0
  for nz in SIZES:
    for tau_on_y in (0, 1):
      for with_c in (False, True) if nz in f2010_sizes else (False,):
        ny = (3, 40, 64)[k % 3]
        k += 1
        z, y, inp = _so_inputs(nz, ny, tau_on_y, with_c, M)
        tag = ('so', nz, ny, tau_on_y, with_c)
        got = _so_call(backend, z, y, inp, M)
        _sentinel(got, M, tag)
        _member_rows(got, [_so_call(backend, z, y, _one(inp, m), 1) for m in range(M)], M, tag)
        assert not got['status'][:M].any(), (tag, got['status'][:M, 0])
        want = pool.map(_so_oracle, [(z, y, inp['tau'][m] if tau_on_y else float(inp['tau'][m]), inp['L'][m],
                                      inp['KGM'][m], inp['c'][m] if with_c else None, inp['b'][m], inp['bs'][m])
                                     for m in range(M)], chunksize=1)
        key = 'f2010' if with_c else 'explicit'
        worst[key] = max(worst[key], _oracle_rows(got, want, M, tag))
  return worst


def _ml_call(be, nz, y, inp, M):
  c = Batch(be)
  m = _abi.Model()
  m.M, m.nz, m.ny = M, nz, y.size
  m.y = c.ptr(y)
  bs = c.buf(np.vstack([inp['bs'][:M], np.full((1, y.size), np.nan)]))
  psi_s = c.out(M, y.size)
  m.ml_bs, m.ml_Psi_s = be.ptr(bs), be.ptr(psi_s)
  m.ml_Ks, m.ml_vpist = c.vec(inp['Ks'][:M, None]), c.vec(inp['v_pist'][:M, None])
  m.ml_h, m.ml_L = c.vec(inp['h']), c.vec(inp['L'])  # shared
  m.ml_surflux, m.ml_rest_mask, m.ml_b_rest = c.vec(inp['surflux']), c.vec(inp['rest_mask']), c.vec(inp['b_rest'][:M])
  status = c.buf(np.array([0] * M + [0xA5A5A5A5], dtype=np.uint32), np.uint32)
  rc = be.lib.pmoc_ml_timestep(ctypes.byref(m), c.vec(inp['b_basin'][:M]), c.vec(inp['Psi_b'][:M]), inp['dt'],
                               be.ptr(status), be.stream())
  _abi.check(be.lib, rc)
  return {'bs': c.get(bs), 'Psi_s': c.get(psi_s), 'status': c.get(status).view(np.uint32)[:, None]}


def ml_batched(backend):
  """Member 4 has a non-monotone b_basin (np.interp with an unsorted abscissa: status bit 8)."""
  rng = np.random.default_rng(7)
  M, worst = MOD_M, 0.0
  for i, nz in enumerate(SIZES):
    ny = (3, 40, 64)[i % 3]
    y = np.linspace(0, 2e6, ny)
    z = _grid(nz)
    bb = 0.03 * np.exp(z / 300.)[None, :] * np.linspace(0.7, 1.3, M)[:, None] - 0.001
    bb[4, nz // 2:nz // 2 + 5] = bb[4, nz // 2:nz // 2 + 5][::-1]
    psi_b = np.linspace(4., -2., nz)[None, :] * np.linspace(0.5, 1.5, M)[:, None] + rng.normal(0, 0.05, (M, nz))
    psi_b[:, :3] = 0.
    surflux = np.zeros(ny)
    surflux[1:max(2, ny // 8)] = -1e-3
    rest = np.zeros(ny)
    rest[ny // 4:-1] = 1.
    inp = dict(b_basin=bb, Psi_b=psi_b, bs=0.025 * (y / y[-1])[None, :]**2 * np.linspace(0.8, 1.2, M)[:, None],
               Ks=np.linspace(200., 600., M), v_pist=np.linspace(1., 2., M) / 86400., h=np.array(50.), L=np.array(4e6),
               surflux=surflux, rest_mask=rest, b_rest=0.02 * (y / y[-1])[None, :] * np.linspace(0.9, 1.1, M)[:, None],
               dt=86400. * 5)
    tag = ('ml', nz, ny)
    got = _ml_call(backend, nz, y, inp, M)
    _sentinel(got, M, tag)
    _member_rows(got, [_ml_call(backend, nz, y, _one(inp, m), 1) for m in range(M)], M, tag)
    assert [bool(s & _abi.ST_XP_NONMONOTONE) for s in got['status'][:M, 0]] == [m == 4 for m in range(M)], got['status']
    want = []
    for m in range(M):
      ml = O.MixedLayerState(y, Ks=inp['Ks'][m], h=50., L=4e6, surflux=surflux, rest_mask=rest,
                             b_rest=inp['b_rest'][m], v_pist=inp['v_pist'][m], bs=inp['bs'][m])
      O.ml_timestep(ml, bb[m], psi_b[m], inp['dt'])
      want.append({'bs': ml.bs, 'Psi_s': ml.Psi_s})
    worst = max(worst, _oracle_rows(got, want, M, tag))
  return worst


# ------------------------------------------------------------------------------------------------ part 3
SMEM_PER_BLOCK = 227 * 1024  # dynamic shared memory one block of sm_100 may opt in to


def psib_smem(nz, nb):
  """Dynamic shared memory of pmoc_thermwind_psib (pmoc_ops.cu): 6 nzp + nbp + nbp/2 + 2 doubles per warp."""
  nzp, nbp = 32 * lpl_for(nz), (nb + 3) & ~3
  return 8 * (6 * nzp + nbp + nbp // 2 + 2) * 4


def so_smem(nz, ny):
  """Dynamic shared memory of pmoc_so_solve (pmoc_ops.cu): z, y, four tapers per block, 3 nyp per warp."""
  nzp, nyp = 32 * lpl_for(nz), (ny + 3) & ~3
  return 8 * (nzp + 4 + nyp + 4 * nzp + 3 * nyp * 4)


def largest_fitting(smem, nz):
  n = 2
  while smem(nz, n + 1) <= SMEM_PER_BLOCK:
    n += 1
  return n


def smem_limits(backend):
  """At nz = 256: the largest nb / ny whose per-module kernel fits one block matches the oracle; one more is refused
  with EUNSUPPORTED by the entry point and with a ValueError by the drop-in class."""
  import pytest

  from pymoc_b200.modules import Psi_SO, Psi_Thermwind
  nz = 256
  nb = largest_fitting(psib_smem, nz)
  assert psib_smem(nz, nb + 1) > SMEM_PER_BLOCK >= psib_smem(nz, nb)
  inp = _psib_inputs(nz, 2, np.random.default_rng(11))
  got = _psib_call(backend, nz, nb, inp, 2)
  with np.errstate(all='ignore'):
    for m in range(2):
      ib, in_, p, g = O.thermwind_psibz(inp['Psi'][m], inp['b1'][m], inp['b2'], nb)
      for k, w in (('psib', p), ('bgrid', g), ('iso_b', ib), ('iso_n', in_)):
        assert relmax(got[k][m], w) < TOL, ('psib', nb, m, k, relmax(got[k][m], w))
  c = Batch(backend)
  rc = backend.lib.pmoc_thermwind_psib(2, nz, nb + 1, c.vec(inp['Psi']), c.vec(inp['b1']), c.vec(inp['b2']),
                                       c.ptr(np.zeros((2, nb + 1))), None, None, None, backend.stream())
  assert rc == _abi.EUNSUPPORTED, rc
  assert ('nb = %d' % (nb + 1)) in backend.lib.pmoc_last_error().decode()
  tw = Psi_Thermwind(z=_grid(nz), b1=inp['b1'][0].copy(), b2=inp['b2'].copy())
  tw.Psi = inp['Psi'][0].copy()
  with np.errstate(all='ignore'):
    assert relmax(tw.Psib(nb), got['psib'][0]) == 0.0
  with pytest.raises(ValueError, match='Psi_Thermwind: nb = %d' % (nb + 1)):
    tw.Psib(nb + 1)
  with pytest.raises(ValueError, match='Psi_Thermwind: nb = %d' % (nb + 1)):
    tw.Psibz(nb + 1)

  ny = largest_fitting(so_smem, nz)
  assert so_smem(nz, ny + 1) > SMEM_PER_BLOCK >= so_smem(nz, ny)
  z, y, inp = _so_inputs(nz, ny, 0, False, 2)
  got = _so_call(backend, z, y, inp, 2)
  for m in range(2):
    p = O.ChannelParams(z, y, float(inp['tau'][m]), f=1e-4, rho=1030., L=inp['L'][m], KGM=inp['KGM'][m], smax=0.01)
    for k, w in zip(('Psi', 'Psi_Ek', 'Psi_GM'), O.so_solve(p, inp['b'][m], inp['bs'][m])):
      assert relmax(got[k][m], w) < TOL, ('so', ny, m, k, relmax(got[k][m], w))
  z, y, inp = _so_inputs(nz, ny + 1, 0, False, 2)
  c = Batch(backend)
  rc = backend.lib.pmoc_so_solve(ctypes.byref(_so_model(c, z, y, inp, 2)), c.vec(inp['b']), c.vec(inp['bs']),
                                 c.ptr(np.zeros((2, nz))), None, None, None, None, backend.stream())
  assert rc == _abi.EUNSUPPORTED, rc
  assert ('ny = %d' % (ny + 1)) in backend.lib.pmoc_last_error().decode()
  so = Psi_SO(z=z, y=y, b=inp['b'][0].copy(), bs=inp['bs'][0].copy(), tau=float(inp['tau'][0]), f=1e-4, L=inp['L'][0],
              KGM=inp['KGM'][0])
  with pytest.raises(ValueError, match='Psi_SO: ny = %d' % (ny + 1)):
    so.solve()
  return nb, ny
