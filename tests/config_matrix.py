"""Every kernel family under the configurations a caller may pass beyond the example scripts' own, against the
reference, shared by the CPU (warp-emulator) and GPU test files.

The cells of ``kernel_matrix`` / ``tall_matrix`` / ``equilibrium_matrix`` run on uniform grids, with depth-independent
basin areas, no Psi_SO taper and most per-member scalars shared by the ensemble.  Here each cell is run again under one
of four variants:

  stretched  the same end points, level spacing varying smoothly from 1.3 to 0.7 times uniform (bottom to top); every
             z-profile interpolated, dt scaled by 0.45 for the thinner top levels;
  area       the basin area of every column shrinking with depth by a fraction a_m that differs per member, member 0
             uniform (one launch holds both outcomes of the kernels' uniform-area test); the other columns keep one
             kappa for the whole ensemble while their Area is per member (the dAk member stride mix);
  tapers     all four Psi_SO tapers set (sill, Ekman, top, bottom), and a per-member smax small enough that the slope
             clip engages;
  strided    every per-member scalar and profile the topology reads given per member (distinct values within 10 %).

Kernel families: the warp-per-member ``k_model`` (every topology of launch_model), the several-members-per-warp
``k_twcol`` (column + thermal wind up to 144 levels), the block-per-member 'post' kernels (``k_wide_post`` /
``k_wide_refresh``) and the block-per-member 'jn' kernels (``k_wide_steps2``, the late schedule too) above 256 levels,
and the per-module entry points on a stretched grid.  Each cell keeps ``kernel_matrix.fused_cell``'s contract and
asserts that its variant took effect: the oracle's answer moves away from the plain cell's, plus the variant's own mark.
"""
import contextlib
import dataclasses

import numpy as np

import equilibrium_matrix as eqm
import kernel_matrix as km
import tall_matrix as tm
from helpers import relmax
from oracle import pymoc_oracle as O
from pymoc_b200 import _abi
from pymoc_b200.ensemble import Ensemble

VARIANTS = ('stretched', 'area', 'tapers', 'strided')
TAPERS = dict(Hsill=800., HEk=150., Htapertop=250., Htaperbot=600.)  # each spans >= 2 levels at nz = 64
EFFECT = 1e-6  # a variant must move the oracle's answer by more than this (max-norm relative) in some field

# family -> (topologies, sizes on the GPU, sizes on the emulator)
FAMILIES = {
    'warp': (tuple(km.TOPOLOGIES), km.SIZES, (64, 256)),
    'twcol': (('tw',), eqm.TWCOL_NZ, eqm.TWCOL_NZ),
    'post': (tm.TOPOLOGIES, (257, 1025, 2049, 4096), (257,)),
    'jn': (('jn',), (257, 1025, 2049, 4096), (257,)),
}
LATE = ('stretched', 'area')  # 'jn' variants also run on the late (serial) schedule: PMOC_WIDE_FORCE_LATE=1
MODULE_SO_SIZES = {'gpu': km.SIZES, 'emu': (64, 129, 256)}


def has_so(name):
  return name.startswith(('so', 'tw_so', 'c3', 'twobasin', 'jn'))


def applies(name, variant):
  return variant != 'tapers' or has_so(name)


def cells(where):
  """(family, topology, nz, variant, late) of every cell, ``where`` 'gpu' or 'emu'.  On the emulator the F2010
  ('_bvp') cells run at 64 levels only: their converged reference takes seconds of solve_bvp per diagnosis."""
  out = []
  for family, (names, gpu, emu) in FAMILIES.items():
    for name in names:
      for nz in gpu if where == 'gpu' else emu:
        if where == 'emu' and name.endswith('_bvp') and nz != 64:
          continue
        for v in VARIANTS:
          if applies(name, v):
            out.append((family, name, nz, v, False))
            if family == 'jn' and v in LATE:
              out.append((family, name, nz, v, True))
  return out


def cell_id(c):
  return '%s-%s-%d-%s%s' % (c[0], c[1], c[2], c[3], '-late' if c[4] else '')


# ------------------------------------------------------------------------------------------------ variants
def stretched_grid(z0, z1, nz):
  """nz levels from z0 to z1, spacing 1.3 times uniform at z0 falling smoothly to 0.7 times at z1."""
  s = np.linspace(0., 1., nz)
  return z0 + (z1 - z0) * (s + 0.3 * np.sin(np.pi * s) / np.pi)


def module_grid(nz):
  return stretched_grid(-4000., 0., nz)


def _per_member(a, M, k, floor=0.):
  """``a`` ([1|M, ...]) as M distinct rows within 8 % of it; ``floor`` adds an offset of the same relative size where
  ``a`` is zero.  ``k`` decorrelates the factors of different fields."""
  a = np.asarray(a, dtype=np.float64)
  f = 1. + 0.08 * np.sin(1.7 * k + 2.1 * np.arange(M))
  f = f.reshape((M,) + (1,) * (a.ndim - 1))
  return np.ascontiguousarray(np.broadcast_to(a, (M,) + a.shape[1:]) * f + (f - 1.) * floor)


def _stretched(family, spec):
  z = stretched_grid(spec.z[0], spec.z[-1], spec.nz)
  return dataclasses.replace(tm._on_grid(spec, z), dt=spec.dt * 0.45)


def area_fraction(M):
  """Per-member fraction by which the area shrinks from the surface to the bottom; member 0: none."""
  return np.linspace(0., 0.4, M)


def _area(family, spec):
  z, M = spec.z, spec.M
  shape = 1. + area_fraction(M)[:, None] * (z - z[-1])[None, :] / (z[-1] - z[0])

  def col(c, shared_kappa):
    if c is None:
      return None
    kappa = np.ascontiguousarray(c.kappa[:1]) if shared_kappa else c.kappa
    return dataclasses.replace(c, kappa=kappa, Area=np.ascontiguousarray(np.broadcast_to(c.Area, (M, z.size)) * shape))

  return dataclasses.replace(spec, basin=col(spec.basin, False), north=col(spec.north, True), pac=col(spec.pac, True))


def smax_of(M):
  return np.geomspace(0.01, 6e-4, M)


def _tapers(family, spec):
  so = dataclasses.replace(spec.so, smax=smax_of(spec.M), **TAPERS)
  return dataclasses.replace(spec, so=so)


def _strided(family, spec):
  M, post = spec.M, spec.order == 'post'
  pm = lambda a, k, floor=0.: _per_member(a, M, k, floor)

  def col(c, k, bzbot):
    if c is None:
      return None
    c = dataclasses.replace(c, bs=pm(c.bs, k, 1e-3), N2min=pm(c.N2min, k + 1), bbot=pm(c.bbot, k + 2, 1e-4))
    if family == 'twcol':  # k_twcol: per-member Area; it takes no bzbot
      return dataclasses.replace(c, Area=pm(c.Area, k + 3))
    if bzbot:
      c = dataclasses.replace(c, bzbot=pm(2e-7, k + 3))
    return c

  out = dict(basin=col(spec.basin, 0, post), north=col(spec.north, 10, False), pac=col(spec.pac, 20, False))
  if spec.tw is not None:
    out['tw'] = dataclasses.replace(spec.tw, f=pm(spec.tw.f, 30),
                                    b2=None if spec.tw.b2 is None else pm(spec.tw.b2, 31, 1e-4))
  if spec.so is not None:
    so = spec.so
    out['so'] = dataclasses.replace(so, f=pm(so.f, 40), rho=pm(so.rho, 41), L=pm(so.L, 42), KGM=pm(so.KGM, 43),
                                    smax=pm(so.smax, 44), bs=pm(so.bs, 45),
                                    c=None if so.c is None else pm(so.c, 46))
  if spec.ml is not None:
    ml = spec.ml
    out['ml'] = dataclasses.replace(ml, Ks=pm(ml.Ks, 50), h=pm(ml.h, 51), L=pm(ml.L, 52), v_pist=pm(ml.v_pist, 53),
                                    surflux=pm(ml.surflux, 54), rest_mask=pm(ml.rest_mask, 55),
                                    b_rest=pm(ml.b_rest, 56))
  if spec.pac is not None:
    out['zoc_f'], out['so_pac_L'] = pm(spec.zoc_f, 60), pm(spec.so_pac_L, 61)
  return dataclasses.replace(spec, **out)


TRANSFORMS = {'stretched': _stretched, 'area': _area, 'tapers': _tapers, 'strided': _strided}


def strided_vecs(family, spec):
  """The pmoc_vec fields of the marshalled model that the 'strided' variant makes per member."""
  cols = [c for c in ('basin', 'north', 'pac') if getattr(spec, c) is not None]
  out = ['%s.%s' % (c, k) for c in cols for k in ('bs', 'N2min')]
  if family == 'twcol':
    out.append('basin.Area')
  elif spec.order == 'post':
    out.append('basin.bzbot')
  if spec.tw is not None:
    out += ['tw_f'] + (['tw_b2'] if spec.tw.b2 is not None else [])
  if spec.so is not None:
    out += ['so_f', 'so_rho', 'so_L', 'so_KGM', 'so_smax', 'so_bs'] + (['so_c'] if spec.so.c is not None else [])
  if spec.ml is not None:
    out += ['ml_Ks', 'ml_h', 'ml_L', 'ml_vpist', 'ml_surflux', 'ml_rest_mask', 'ml_b_rest']
  if spec.pac is not None:
    out += ['zoc_f', 'so2_L']
  return out


def base_spec(family, name, nz):
  if family == 'twcol':
    return eqm.twcol_spec(nz), {}
  return km.cell(name, nz)


def config_spec(family, name, nz, variant):
  base, env = base_spec(family, name, nz)
  return TRANSFORMS[variant](family, base), env, base


# ------------------------------------------------------------------------------------------------ the cell
class Oracle:
  """The spawned oracle pool plus the plain cells' answers, computed once per (family, topology, nz) and shared by
  that cell's variants."""

  def __init__(self, pool):
    self.pool, self.plain = pool, {}

  def run(self, spec):
    bvp = spec.so is not None and spec.so.c is not None
    return self.pool.map_async(km.oracle_task, [(spec.member_case(m), km.NSTEPS, bvp) for m in range(spec.M)],
                               chunksize=1)

  def base(self, key, spec):
    if key not in self.plain:
      self.plain[key] = self.run(spec)
    return self.plain[key]


def _attr(model, path):
  for p in path.split('.'):
    model = getattr(model, p)
  return model


def _clip_engaged(case):
  """Whether the explicit Psi_SO's slope clip (z / width < -smax) acts on some level of the member's first diagnosis."""
  so = case['so']
  bs = case['ml']['bs'] if case.get('ml') is not None else so['bs']
  z, y = case['z'], so['y']
  with np.errstate(all='ignore'):
    width = np.array([max(y[-1] - O.so_outcrop(b, y, bs), 0.1) for b in case['basin']['b0']])
  return bool((z / width < -so['smax']).any())


def _initial(case):
  """The member's initial state under the names of the oracle's fields."""
  out = {'b_' + c: case[c]['b0'] for c in ('basin', 'north', 'pac') if case.get(c) is not None}
  if case.get('ml') is not None:
    out['bs_ml'] = case['ml']['bs']
  return out


def _check_effect(backend, family, name, variant, spec, cases, base_cases, want, plain, compared):
  """The variant took effect: the oracle moves away from the plain cell, and the variant's own mark is there.  State
  fields are compared by what the run added to the initial state: over a few short steps (dt ~ dz^2 at 4096 levels)
  the state itself hardly moves."""
  moved = {}
  for m in compared:
    if isinstance(plain[m], str):
      continue
    init, init0 = _initial(cases[m]), _initial(base_cases[m])
    for k, w in want[m].items():
      if k in plain[m]:
        d = relmax(w - init[k], plain[m][k] - init0[k]) if k in init else relmax(w, plain[m][k])
        moved[k] = max(moved.get(k, 0.), d)
  assert max(moved.values(), default=0.) > EFFECT, ('variant without effect', family, name, variant, moved)
  if variant == 'tapers':
    sectors = ('Psi_Ek', 'Psi_Ek2') if spec.pac is not None else ('Psi_Ek',)
    for m in compared:
      for k in sectors:
        assert want[m][k][0] == 0., (name, variant, m, k, 'Ekman transport at the bottom level')
    if spec.pac is not None:
      assert moved['Psi_so2'] > EFFECT, (name, 'tapers leave the second sector alone', moved['Psi_so2'])
    if spec.so.c is None:
      assert any(_clip_engaged(c) for c in cases), (name, 'slope clip never engages')
  elif variant == 'area':
    for m, c in enumerate(cases):
      for col in ('basin', 'north', 'pac'):
        if c.get(col) is not None:
          a = c[col]['Area']
          assert (np.ptp(a) == 0.) == (m == 0), (name, col, m, 'Area uniform only for member 0')
  elif variant == 'strided':
    model = Ensemble(spec, backend=backend).model
    for path in strided_vecs(family, spec):
      v = _attr(model, path)
      assert v.ptr and v.mstride != 0, (name, path, 'shared', v.mstride)
  return max(moved.values())


def config_cell(backend, oracle, monkeypatch, family, name, nz, variant, late=False, bitwise=True):
  """One cell: the variant of a cell of ``family`` against the live oracle (F2010: converged solve_bvp); returns its
  report line."""
  spec, env, base = config_spec(family, name, nz, variant)
  if family == 'warp':
    assert km.kernel_topology(spec) == (km.TOPOLOGIES[name], km.lpl_for(nz)), (name, nz, km.kernel_topology(spec))
  cases = [spec.member_case(m) for m in range(spec.M)]
  vecs = [km._flat(c) for c in cases]
  for i in range(len(vecs)):
    for j in range(i):
      assert not np.array_equal(vecs[i], vecs[j]), ('members not distinct', family, name, nz, variant, i, j)
  pending = oracle.run(spec)
  plain = oracle.base((family, name, nz), base)
  for k, v in env.items():
    monkeypatch.setenv(k, v)
  if late:
    monkeypatch.setenv('PMOC_WIDE_FORCE_LATE', '1')
  got = km._run(backend, spec, [km.NSTEPS])
  tag = (family, name, nz, variant, late)
  if bitwise:
    km._same(got, km._run(backend, spec, [km.CUTS[0], km.CUTS[1] - km.CUTS[0], km.NSTEPS - km.CUTS[1]]),
             tag + ('split launches',))
    if family == 'warp':
      for wpb in ('1', '3'):
        monkeypatch.setenv('PMOC_WPB', wpb)
        km._same(got, km._run(backend, spec, [km.NSTEPS]), tag + ('PMOC_WPB=' + wpb,))
      monkeypatch.delenv('PMOC_WPB')
  st = got['status']
  want = pending.get()
  worst, compared = 0.0, []
  for m, w in enumerate(want):
    if st[m] & _abi.ST_PARITY_UNDEFINED:
      continue
    assert not isinstance(w, str), tag + (m, w)
    assert not st[m] & (_abi.ST_NAN | _abi.ST_BRENT_SIGN | _abi.ST_ML_INDEX), tag + (m, int(st[m]))
    for key, v in w.items():
      err = relmax(got[key][m], v)
      worst = max(worst, err)
      assert err < km.TOL, '%s member %d field %s: rel err %.3e' % (cell_id((family, name, nz, variant, late)), m, key,
                                                                    err)
    compared.append(m)
  excused = spec.M - len(compared)
  assert excused <= 1, ('vacuous cell', tag, excused)
  moved = _check_effect(backend, family, name, variant, spec, cases, [base.member_case(m) for m in range(base.M)], want,
                        plain.get(), compared)
  print('config %-5s %-9s nz=%4d %-9s%-5s worst %.2e excused %d moved %.1e' % (
      family, name, nz, variant, ' late' if late else '', worst, excused, moved))
  return worst


# ------------------------------------------------------------------------------------------------ completeness
def covers_every_pair(where):
  """The cells cover every (kernel family, topology, applicable variant) triple at every size of their family: the
  warp family every topology of launch_model's switch (read from the source), 'jn' the late schedule too."""
  got = cells(where)
  by = {}
  for f, name, nz, v, late in got:
    by.setdefault((f, name, v, late), set()).add(nz)
  warp = {}
  for f, name, nz, v, late in got:
    if f == 'warp':
      spec = config_spec(f, name, nz, v)[0]
      warp.setdefault((km.kernel_topology(spec)[0], v), set()).add(km.lpl_for(nz))
  for t in km.switch_topologies():
    for v in VARIANTS:
      if v != 'tapers' or t & _abi.HAS_SO:
        assert (t, v) in warp, ('warp', t, v)
        if where == 'gpu':
          assert warp[(t, v)] == set(km.LPLS), ('warp', t, v, warp[(t, v)])
  want = {('warp', n, v, False) for n in km.TOPOLOGIES for v in VARIANTS if v != 'tapers' or has_so(n)}
  want |= {('twcol', 'tw', v, False) for v in ('stretched', 'area', 'strided')}
  want |= {('post', n, v, False) for n in tm.TOPOLOGIES for v in VARIANTS if v != 'tapers' or has_so(n)}
  want |= {('jn', 'jn', v, False) for v in VARIANTS} | {('jn', 'jn', v, True) for v in LATE}
  assert set(by) == want, set(by) ^ want
  sizes = {'twcol': set(eqm.TWCOL_NZ), 'post': {257, 1025, 2049, 4096} if where == 'gpu' else {257}}
  sizes['jn'] = sizes['post']
  for (f, name, v, late), nzs in by.items():
    if f in sizes:
      assert nzs == sizes[f], (f, name, v, late, nzs)
  for f, name, nz, v, late in got:
    if f == 'twcol':  # what k_twcol takes (pmoc_twcol_supported)
      spec, env, _ = config_spec(f, name, nz, v)
      assert spec.nz <= 144 and not spec.basin.do_conv and spec.basin.bzbot is None and spec.basin.kappa.shape[1] == 1
      assert spec.tw.b2 is not None and 'PMOC_NO_TWCOL' not in env


# ------------------------------------------------------------------------------------------------ per-module calls
def column_stretched(backend):
  """pmoc_column_timestep on a stretched grid: every stage mask, with and without convection."""
  return km.column_batched(backend, grid=module_grid, stage_masks=tuple(range(1, 8)))


def thermwind_stretched(backend):
  """pmoc_thermwind_solve on a stretched grid, with and without gmid."""
  return km.thermwind_batched(backend, grid=module_grid)


def _so_oracle(args):
  z, y, tau, L, KGM, c, f, rho, smax, b, bs = args
  with km.converged_f2010() if c is not None else contextlib.nullcontext():
    p = O.ChannelParams(z, y, tau, f=f, rho=rho, L=L, KGM=KGM, c=c, bvp_with_Ek=c is not None, smax=smax, **TAPERS)
    psi, ek, gm = O.so_solve(p, b, bs)
  return {'Psi': psi, 'Psi_Ek': ek, 'Psi_GM': gm, 'ys': np.array([O.so_outcrop(v, y, bs) for v in b])}


def so_stretched(backend, pool, sizes):
  """pmoc_so_solve on a stretched grid, explicit and F2010, with the four tapers set and per-member f / rho / smax
  (member stride 1) next to shared inputs; same member-row and sentinel contract as ``kernel_matrix.so_batched``."""
  M, worst = km.MOD_M, {'explicit': 0.0, 'f2010': 0.0}
  k = 0
  for nz in sizes:
    for with_c in (False, True):
      tau_on_y, ny = k % 2, (3, 40, 64)[k % 3]
      k += 1
      z, y, inp = km._so_inputs(nz, ny, tau_on_y, with_c, M, grid=module_grid)
      inp.update(f=_per_member(1e-4, M, 1)[:, None], rho=_per_member(1030., M, 2)[:, None],
                 smax=smax_of(M)[:, None], H=TAPERS)
      tag = ('so stretched', nz, ny, tau_on_y, with_c)
      got = km._so_call(backend, z, y, inp, M)
      km._sentinel(got, M, tag)
      km._member_rows(got, [km._so_call(backend, z, y, km._one(inp, m), 1) for m in range(M)], M, tag)
      assert not got['status'][:M].any(), (tag, got['status'][:M, 0])
      want = pool.map(_so_oracle, [(z, y, inp['tau'][m] if tau_on_y else float(inp['tau'][m]), inp['L'][m],
                                    inp['KGM'][m], inp['c'][m] if with_c else None, inp['f'][m, 0], inp['rho'][m, 0],
                                    inp['smax'][m, 0], inp['b'][m], inp['bs'][m]) for m in range(M)], chunksize=1)
      key = 'f2010' if with_c else 'explicit'
      worst[key] = max(worst[key], km._oracle_rows(got, want, M, tag))
      assert all(w['Psi_Ek'][0] == 0. for w in want), (tag, 'sill taper')
      if not with_c:
        case = lambda m: dict(z=z, so=dict(y=y, bs=inp['bs'][m], smax=inp['smax'][m, 0]), basin=dict(b0=inp['b'][m]))
        assert any(_clip_engaged(case(m)) for m in range(M)), (tag, 'slope clip never engages')
  return worst
