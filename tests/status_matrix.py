"""Per-member status bits and the rare solver branches behind them, against the reference; shared by the CPU
(warp-emulator) and GPU test files.

Every check builds inputs on which the condition holds at the first diagnosis (or the first step), so that the kernel
and the reference see bit-identical inputs and the expected bits follow from a plain restatement of the kernel's
predicate.  Each call holds members that trigger a bit, near misses that must not, and clean members, and the bits
are asserted member by member.

- Psi_SO's scan of bs(y) (``pm::so_scan``): BS_NONMONOTONE when bs decreases on any grid interval north of its first
  minimum, BS_SAWTOOTH when it does on three or more intervals, consecutive or not.  BRENT_SIGN is never raised for a
  finite bs: the kernel sends b < min(bs) and b > bs[-1] elsewhere before Brent's method, so the bracket
  [y[argmin bs], y[-1]] always holds a sign change; only a non-finite bs reaches it.
- The F2010 smoother's cell propagators (``pm::cell_propagators``): the tabulated trip counts (kSeriesQ, kSeriesInv)
  recomputed from their definitions, both sides of several table rows, the adaptive series above the table, and
  BVP_SERIES where 2000 terms cannot converge.
- SO_ML's first non-zero Psi_b (ML_INDEX).
- Streamfunctions pushed through the host handle ('jn' NOISE_SWITCH): the flags of the step after the push follow
  from the pushed values, not from carry bits of the diagnosis that preceded it.
"""
import dataclasses
import math
import os
import re

import numpy as np

import kernel_matrix as km
from helpers import relmax
from oracle import pymoc_oracle as O
from pymoc_b200 import _abi, configs
from pymoc_b200.ensemble import HostEnsemble

TOL = km.TOL
ROOT = km.ROOT
SO_NY = 40


# ------------------------------------------------------------------------------------------------ bs(y) scan
def bs_profiles(ny=SO_NY):
  """[name] -> bs on ny points: a monotone base, then one feature each north of the minimum."""
  y = np.linspace(0, 2e6, ny)
  base = 0.03 * (y / y[-1])**2 + 0.001
  k = ny // 2
  step = 0.2 * (base[k + 1] - base[k])  # a decrease much smaller than the local rise: every other interval rises
  out = {'monotone': base.copy()}
  p = base.copy()
  p[k + 1] = p[k + 2] = p[k]  # two flat intervals: not a decrease
  out['plateau'] = p
  for n in (1, 2, 3):  # n consecutive decreasing intervals k .. k+n
    p = base.copy()
    for j in range(1, n + 1):
      p[k + j] = p[k] - j * step
    out['down%d' % n] = p
  p = base.copy()
  for kk in (ny // 4, ny // 2, 3 * ny // 4):  # three separate single-interval dips
    p[kk + 1] = p[kk] - 0.2 * (base[kk + 1] - base[kk])
  out['down_separate3'] = p
  out['min_last'] = base[::-1].copy()  # minimum at ny - 1: nothing north of it
  p = base.copy()
  p[3 * ny // 4] = p[0]  # the minimum attained twice: argmin is the first, the dip to the second is north of it
  out['min_twice'] = p
  return y, out


def scan_bits(bs):
  """pm::so_scan's verdict restated: (BS_NONMONOTONE, BS_SAWTOOTH) of one bs profile."""
  south = int(np.argmin(bs))
  ndown = int(np.sum(np.diff(bs)[south:] < 0))
  return (_abi.ST_BS_NONMONOTONE if ndown > 0 else 0) | (_abi.ST_BS_SAWTOOTH if ndown >= 3 else 0)


EXPECTED_SCAN = {'monotone': 0, 'plateau': 0, 'down1': 2, 'down2': 2, 'down3': 2 | 256, 'down_separate3': 2 | 256,
                 'min_last': 0, 'min_twice': 2}


def _bs_inputs(nz, with_c):
  y, prof = bs_profiles()
  names = sorted(prof)
  M = len(names)
  z, _, inp = km._so_inputs(nz, SO_NY, 0, with_c, M)
  inp['bs'] = np.stack([prof[n] for n in names])
  # every member's b spans its bs, so most levels reach the outcrop search (and some fall on either side of it)
  lo, hi = inp['bs'].min(axis=1), inp['bs'][:, -1]
  s = (np.exp(z / 300.) - np.exp(z[0] / 300.)) / (1. - np.exp(z[0] / 300.))
  inp['b'] = (lo - 0.002)[:, None] + (hi - lo + 0.004)[:, None] * s[None, :]
  return z, y, names, inp


def so_bs_scan(backend, pool, nz, with_c):
  """pmoc_so_solve on the bs profiles: the scan bits member by member, BRENT_SIGN never, ys bit for bit against the
  restated brentq wherever the kernel runs Brent's method, Psi / Psi_Ek / Psi_GM / ys against the reference (scipy's
  brentq) at 1e-10.  Returns the worst error."""
  z, y, names, inp = _bs_inputs(nz, with_c)
  M = len(names)
  got = km._so_call(backend, z, y, inp, M)
  km._sentinel(got, M, ('so_bs', nz, with_c))
  st = got['status'][:M, 0]
  for m, n in enumerate(names):
    assert scan_bits(inp['bs'][m]) == EXPECTED_SCAN[n], (n, scan_bits(inp['bs'][m]))
    assert st[m] == EXPECTED_SCAN[n], ('so_bs', nz, with_c, n, int(st[m]), EXPECTED_SCAN[n])
  brent = 0
  for m in range(M):
    if not st[m] and np.argmin(inp['bs'][m]) < SO_NY - 1:
      continue  # monotone north of the minimum: the kernel inverts the segment linearly (checked at 1e-10 below)
    want = np.array([O.so_outcrop(v, y, inp['bs'][m], 'brentq_restated') for v in inp['b'][m]])
    assert np.array_equal(got['ys'][m], want), ('ys', nz, names[m], np.flatnonzero(got['ys'][m] != want))
    brent += 1
  assert brent == 6, brent  # the five non-monotone profiles and the minimum at ny - 1
  want = pool.map(km._so_oracle, [(z, y, float(inp['tau'][m]), inp['L'][m], inp['KGM'][m],
                                   inp['c'][m] if with_c else None, inp['b'][m], inp['bs'][m]) for m in range(M)],
                  chunksize=1)
  return km._oracle_rows(got, want, M, ('so_bs', nz, with_c))


# ------------------------------------------------------------------------------------------------ F2010 series
def series_tables():
  """kSeriesInv and kSeriesQ as pmoc_device.cuh defines them."""
  src = open(os.path.join(ROOT, 'pymoc_b200', 'csrc', 'pmoc_device.cuh')).read()

  def table(name):
    body = re.search(r'%s\[[^\]]*\]\s*=\s*\{([^}]*)\}' % name, src).group(1)
    body = re.sub(r'//[^\n]*', '', body)
    return [float(v) for v in body.replace('\n', ' ').split(',') if v.strip()]

  return table('kSeriesInv'), table('kSeriesQ')


def series_tail(q, first):
  """Bound of what the terms from index ``first`` on add to the sums A, B/h, D (>= 1): term k is at most
  q^(k/2) / k!, and D weighs it by at most k."""
  return sum(k * math.exp(0.5 * k * math.log(q) - math.lgamma(k + 1)) for k in range(first, first + 600))


def series_table_is_consistent():
  """kSeriesInv[k] = 1/((k+2)(k+1)) exactly; row t of kSeriesQ serves t + 2 trips (terms up to index 3 (t+2) + 1):
  at its Qmax the omitted tail is below 1e-18 of the sums, and one trip fewer would not be."""
  inv, qs = series_tables()
  assert len(inv) == 99 and len(qs) == 32
  for k, v in enumerate(inv):
    assert v == 1.0 / ((k + 2) * (k + 1)), (k, v)
  for t, q in enumerate(qs):
    trips = t + 2
    assert series_tail(q, 3 * trips + 2) < 1e-18, (t, q, series_tail(q, 3 * trips + 2))
    assert series_tail(q, 3 * trips - 1) > 1e-18, (t, q, 'one trip fewer would do')
    assert t == 0 or q > qs[t - 1]


def _qraw(z, b):
  """max over cells of |N2| h^2 + |dN2| h^2 (pm::so_bvp's Q0, Q1 before the 1/c^2)."""
  n2 = O.so_n2(z, b)
  h = np.diff(z)
  return float(np.max(np.abs(n2[:-1]) * h * h + np.abs(n2[1:] - n2[:-1]) * h * h))


def smoother_cases(nz):
  """(label, Qmax) of the F2010 sweep: both sides of table rows 13 .. 31, then the adaptive series."""
  _, qs = series_tables()
  out = []
  for t in range(13, 32):
    out += [('row%d-' % t, qs[t] * (1 - 1e-6)), ('row%d+' % t, qs[t] * (1 + 1e-6))]
  return out + [('adaptive600', 600.), ('adaptive5e3', 5e3), ('adaptive5e4', 5e4)]


def so_smoother_sweep(backend, pool, nz, cases=None):
  """pmoc_so_solve with the F2010 smoother, one member per Qmax (c chosen per member), against the converged
  reference (solve_bvp at tol 1e-9); BVP_SERIES absent.  Returns {label: error}."""
  cases = smoother_cases(nz) if cases is None else cases
  M = len(cases)
  z, y, inp = km._so_inputs(nz, SO_NY, 0, True, M)
  inp['c'] = np.array([math.sqrt(_qraw(z, inp['b'][m]) / q) for m, (_, q) in enumerate(cases)])
  got = km._so_call(backend, z, y, inp, M)
  assert not got['status'][:M].any(), [(c[0], int(s)) for c, s in zip(cases, got['status'][:M, 0])]
  want = pool.map(km._so_oracle, [(z, y, float(inp['tau'][m]), inp['L'][m], inp['KGM'][m], inp['c'][m], inp['b'][m],
                                   inp['bs'][m]) for m in range(M)], chunksize=1)
  out = {}
  for m, (label, _) in enumerate(cases):
    out[label] = max(relmax(got[k][m], want[m][k]) for k in ('Psi', 'Psi_Ek', 'Psi_GM'))
    assert out[label] < TOL, ('smoother', nz, label, out[label])
  return out


def so_series_diverges(backend, nz):
  """Qmax ~ 4e6: 2000 terms of the adaptive series cannot converge; the member next to it (Qmax 600) is clean."""
  z, y, inp = km._so_inputs(nz, SO_NY, 0, True, 2)
  inp['c'] = np.array([math.sqrt(_qraw(z, inp['b'][m]) / q) for m, q in enumerate((4e6, 600.))])
  st = km._so_call(backend, z, y, inp, 2)['status'][:2, 0]
  assert [int(s) for s in st] == [_abi.ST_BVP_SERIES, 0], st


# ------------------------------------------------------------------------------------------------ SO_ML
def ml_index(backend, nz=64):
  """pmoc_ml_timestep: ML_INDEX for an all-zero Psi_b (np.nonzero(Psi_b)[0][0] raises IndexError), not for a near
  miss whose only non-zero value is the smallest subnormal; those members match the reference.  The
  np.argwhere(Psi_b > 0) path needs Psi_s[1] > 0, which np.interp of a non-positive Psi_b cannot give (its values
  are convex combinations of Psi_b's): member 4, with Psi_b <= 0 and non-zero, pins that Psi_s[1] <= 0 in both."""
  M, ny = 5, 40
  y, z = np.linspace(0, 2e6, ny), km._grid(nz)
  bb = 0.03 * np.exp(z / 300.)[None, :] * np.linspace(0.8, 1.2, M)[:, None] - 0.001
  psi_b = np.linspace(4., -2., nz)[None, :] * np.ones((M, 1))
  psi_b[:, :3] = 0.
  psi_b[1] = 0.  # all zero: the reference raises
  psi_b[2] = 0.
  psi_b[2, nz // 2] = -5e-324  # near miss: one non-zero value
  psi_b[4] = -np.abs(psi_b[4])  # Psi_b <= 0, non-zero: Psi_s[1] <= 0, so the argwhere path is not taken
  surflux = np.zeros(ny)
  surflux[1:5] = -1e-3
  inp = dict(b_basin=bb, Psi_b=psi_b, bs=0.025 * (y / y[-1])[None, :]**2 * np.linspace(0.8, 1.2, M)[:, None],
             Ks=np.linspace(200., 600., M), v_pist=np.full(M, 1.5 / 86400.), h=np.array(50.), L=np.array(4e6),
             surflux=surflux, rest_mask=np.zeros(ny), b_rest=np.zeros((M, ny)), dt=86400. * 5)
  old = km.MOD_M
  km.MOD_M = M  # (km._one slices members of a MOD_M batch)
  try:
    got = km._ml_call(backend, nz, y, inp, M)
  finally:
    km.MOD_M = old
  st = [int(s) for s in got['status'][:M, 0]]
  assert st == [0, _abi.ST_ML_INDEX, 0, 0, 0], st
  for m in range(M):
    ml = O.MixedLayerState(y, Ks=inp['Ks'][m], h=50., L=4e6, surflux=surflux, rest_mask=0., b_rest=0.,
                           v_pist=inp['v_pist'][m], bs=inp['bs'][m])
    if st[m]:
      try:
        O.ml_timestep(ml, bb[m], psi_b[m], inp['dt'])
        raise AssertionError('the reference did not raise for member %d' % m)
      except IndexError:
        continue
    O.ml_timestep(ml, bb[m], psi_b[m], inp['dt'])
    if m == 4:
      assert ml.Psi_s[1] <= 0 and got['Psi_s'][m][1] <= 0, (ml.Psi_s[1], got['Psi_s'][m][1])
    for k, w in (('bs', ml.bs), ('Psi_s', ml.Psi_s)):
      assert relmax(got[k][m], w) < TOL, (m, k, relmax(got[k][m], w))


# ------------------------------------------------------------------------------------------------ pushed Psi
def _jn_spec(nz, M=4):
  with configs.members(0, M):
    spec = configs.c5_single_global_basin(8, nz=nz, dt_days=30. * (45. / (nz - 1))**2, axes=(2, 2, 1, 2),
                                          kapfac_max=1.)
  # a small slope limit: Psi_so[1] comes out of the slope clip, the state-independent arithmetic whose rounding
  # noise is exempt from NOISE_SWITCH (PMOC_ST_CARRY_SO1_EXACT) while it is the diagnosis's own
  spec = dataclasses.replace(spec, so=dataclasses.replace(spec.so, smax=np.array([1e-4])))
  spec.K = km.K
  return spec


def pushed_psi(backend, host_backend, nz):
  """A 'jn' model run K + 1 steps through the host handle; member 1's Psi_so[1] replaced by rounding noise
  (1e-15 max|Psi|), by an exact 0, or left alone, pushed (PMOC_IO_PSI) and stepped once at it % K != 0: only the
  noise value raises NOISE_SWITCH, on that member only.  Before the push, the handle agrees with Ensemble bit for
  bit (status included, carry bits too)."""
  spec = _jn_spec(nz)
  K = spec.K
  dev = km.Ensemble(spec, backend=backend)
  dev.run(K + 1)
  want = {**dev.state(), **dev.diagnostics()}
  raw = backend.download(dev.buffer('status')).view(np.uint32)
  assert (raw & np.uint32(_abi.ST_PUBLIC_MASK) == 0).all(), raw
  assert (raw & np.uint32(0x80000000)).all(), ('Psi_so[1] not from the slope clip', [hex(v) for v in raw])
  got = {}
  for case in ('noise', 'zero', 'unchanged'):
    h = HostEnsemble(spec, backend=host_backend)
    h.run(K + 1)
    km._same(want, {**h.state(), **h.diagnostics()}, ('HostEnsemble', nz))
    assert np.array_equal(host_backend.download(h.buffer('status')).view(np.uint32), raw), ('carry bits', nz)
    d = h.diagnostics()
    psi = d['Psi_so'].copy()
    mx = max(np.abs(d[k][1]).max() for k in ('Psi_so', 'Psi_iso_b', 'Psi_iso_n'))
    if case == 'noise':
      psi[1, 1] = 1e-15 * mx
    elif case == 'zero':
      psi[1, 1] = 0.
    host_backend.assign(h.buffer('Psi_so'), psi)
    h.run(1, push=h.IO_PSI)
    got[case] = [int(s) for s in h.diagnostics()['status']]
    h.close()
  assert got['noise'] == [0, _abi.ST_NOISE_SWITCH, 0, 0], got
  assert got['zero'] == [0, 0, 0, 0] and got['unchanged'] == [0, 0, 0, 0], got
  return got


# ------------------------------------------------------------------------------------------------ model cells
def _rows(a, M):
  """A [1|M, ...] spec array as M explicit member rows (a copy)."""
  a = np.array(a, dtype=np.float64, copy=True)
  return np.repeat(a, M, axis=0) if a.shape[0] == 1 else a


def _col(c, M, **rows):
  """Column spec ``c`` with the given per-member arrays: name -> function(rows) editing the [M, ...] rows."""
  return dataclasses.replace(c, **{k: f(_rows(getattr(c, k), M)) for k, f in rows.items()})


def model_spec(name, nz, M=5):
  """Members [0, M) of the eight-member lattice of topology ``name`` on nz levels (kernel_matrix's cells), K = 3."""
  with configs.members(0, M):
    if name == 'tw':  # C1; at nz <= 144 the several-members-per-warp kernel (k_twcol) takes it
      spec = configs.c1_timestepping(8, nz=nz)
      spec.dt *= (69. / (nz - 1))**2
    elif name == 'so':
      spec = configs.c2_column_so(8, nz=nz, ny=40, dt_days=10. * (199. / (nz - 1))**2)
    elif name == 'twocol':
      spec = km.regrid(configs.twocol(8), nz)
    elif name == 'c3':
      spec = km.regrid(configs.c3_twocol_so(8), nz)
    elif name == 'twobasin':
      spec = km.regrid(configs.twobasin(8), nz)
    elif name == 'jn':
      spec = configs.c5_single_global_basin(8, nz=nz, dt_days=30. * (45. / (nz - 1))**2, axes=(2, 2, 1, 2),
                                            kapfac_max=1.)
    else:
      raise KeyError(name)
  spec.K = km.K
  assert spec.M == M
  return spec


def _statuses(backend, host_backend, spec, launches, diagnose=False):
  """Run ``spec``: (state + diagnostics of Ensemble, its raw status word).  The same launches split in two and the
  host handle (HostEnsemble) must give the same public status word, bit for bit."""
  def dev(cuts):
    ens = km.Ensemble(spec, backend=backend)
    if diagnose:
      ens.diagnose()
    for n in cuts:
      ens.run(n)
    return ens, {**ens.state(), **ens.diagnostics()}

  ens, out = dev(launches)
  raw = backend.download(ens.buffer('status')).view(np.uint32).ravel()
  assert np.array_equal(out['status'], raw & np.uint32(_abi.ST_PUBLIC_MASK)), (out['status'], raw)
  if sum(launches) > 1:
    n = sum(launches)
    assert np.array_equal(dev([n // 2, n - n // 2])[1]['status'], out['status']), 'split launch'
  if diagnose and spec.order == 'jn':
    return out, raw  # (the host handle diagnoses only inside a 'jn' step)
  h = HostEnsemble(spec, backend=host_backend)
  if diagnose:
    h.diagnose()
    h.run(0)  # pulls the state class, which holds the status word
  for n in launches:
    h.run(n)
  assert np.array_equal(h.diagnostics()['status'], out['status']), ('HostEnsemble', h.diagnostics()['status'])
  h.close()
  return out, raw


def _bits(st, bit):
  return [bool(s & bit) for s in st]


def _forbidden(st):
  """BRENT_SIGN (finite bs) and NAN / ML_INDEX (outside their own cells) are never raised here."""
  assert not any(s & (_abi.ST_BRENT_SIGN | _abi.ST_NAN | _abi.ST_ML_INDEX) for s in st), st


def model_bs_scan(backend, host_backend, name, nz):
  """The bs profiles as Psi_SO's so_bs ('post') or the mixed layer's initial bs ('jn'), one member each: the scan bits
  of the first diagnosis member by member as the restated scan gives them."""
  probe = model_spec(name, nz, 1)
  ny = (probe.ml.y if probe.ml is not None else probe.so.y).size
  _, prof = bs_profiles(ny)
  names = sorted(prof)
  spec = model_spec(name, nz, 8)
  bs = np.stack([prof[n] for n in names])
  if spec.ml is not None:
    spec = dataclasses.replace(spec, ml=dataclasses.replace(spec.ml, bs0=bs))
    out, _ = _statuses(backend, host_backend, spec, [1])  # the 'jn' loop diagnoses at the top of iteration 0
  else:
    spec = dataclasses.replace(spec, so=dataclasses.replace(spec.so, bs=bs))
    out, _ = _statuses(backend, host_backend, spec, [], diagnose=True)
  st = [int(s) for s in out['status']]
  _forbidden(st)
  mask = _abi.ST_BS_NONMONOTONE | _abi.ST_BS_SAWTOOTH
  got = {n: st[m] & mask for m, n in enumerate(names)}
  assert got == {n: scan_bits(prof[n]) for n in names}, (name, nz, got)
  assert got == EXPECTED_SCAN, (name, nz, got)
  return got


def _ulps(x, n):
  """x moved by n units in the last place (n < 0: down)."""
  for _ in range(abs(n)):
    x = np.nextafter(x, np.inf if n > 0 else -np.inf)
  return x


def model_tie_cell(backend, host_backend, name, nz):
  """TIE_CELL of the first diagnosis.  Member 1: one interior cell inverted by 2 ulps (<= 4 eps, flagged); member 2:
  inverted by 16 ulps (> 4 eps, not flagged); member 3: the bottom cell exactly flat (flagged); member 4: an
  interior cell upright by 2 ulps (not flagged); member 0 untouched.  The cell is edited in every column, so the
  remap meets it whichever column the sign of its transport picks."""
  spec = model_spec(name, nz)
  k = nz // 2

  def edit(b):
    b[1, k + 1] = _ulps(b[1, k], -2)
    b[2, k + 1] = _ulps(b[2, k], -16)
    b[3, 1] = b[3, 0]
    b[4, k + 1] = _ulps(b[4, k], 2)
    return b

  cols = {c: _col(getattr(spec, c), spec.M, b0=edit) for c in ('basin', 'north', 'pac') if getattr(spec, c) is not None}
  spec = dataclasses.replace(spec, **cols)
  out, _ = _statuses(backend, host_backend, spec, [], diagnose=True)  # (a step would lose member 3, as the reference does)
  st = [int(s) for s in out['status']]
  _forbidden(st)
  assert _bits(st, _abi.ST_TIE_CELL) == [False, True, False, True, False], (name, nz, st)
  return st


def _unstable(spec, bad, factor=1e6):
  """Member ``bad``'s kappa scaled by ``factor`` in the columns named: dt kappa / dz^2 far above 1/2."""
  def scale(k):
    k[bad] *= factor
    return k
  return scale


def model_nan(backend, host_backend, name, nz, columns=('basin',), nsteps=80):
  """NAN from an instability: member 1's own kappa (in ``columns``) is far beyond the explicit step's limit, so it
  overflows within the launch; K is larger than the launch, so the member's columns meet only through the
  streamfunctions of the first diagnosis and the overflow stays in the columns it starts in.  Member 2 (kappa x 0.5,
  a near miss) and the rest stay finite and unflagged; they equal, bit for bit, a run in which member 1 is a clean
  member."""
  spec = model_spec(name, nz)
  spec.K = 10 * nsteps
  calm = dataclasses.replace(spec, **{c: _col(getattr(spec, c), spec.M, kappa=_unstable(spec, 2, 0.5)) for c in columns})
  bad = dataclasses.replace(calm, **{c: _col(getattr(calm, c), spec.M, kappa=_unstable(calm, 1)) for c in columns})
  out, _ = _statuses(backend, host_backend, bad, [nsteps])
  st = [int(s) for s in out['status']]
  assert _bits(st, _abi.ST_NAN) == [False, True, False, False, False], (name, nz, st)
  # (in the 'jn' loop the overflowing basin column is also SO_ML's unsorted abscissa: XP_NONMONOTONE)
  assert not any(s & ~(_abi.ST_NAN | (_abi.ST_XP_NONMONOTONE if m == 1 else 0)) for m, s in enumerate(st)), st
  ref = km._run(backend, calm, [nsteps])
  for key, v in out.items():
    for m in (0, 2, 3, 4):
      assert np.array_equal(v[m], ref[key][m], equal_nan=True), (name, nz, key, m)
  assert not np.isfinite(np.concatenate([out[k][1].ravel() for k in ('b_basin', 'b_north') if k in out])).all()
  return st


def model_ml_index(backend, host_backend, pool, nz):
  """'jn': member 1 without wind and eddies (tau = KGM = 0) has Psi_so == 0, so SO_ML's np.nonzero(Psi_b)[0][0]
  raises in the reference: ML_INDEX; member 2 (tau = 0, KGM kept) is a near miss.  The others equal a run in which
  member 1 keeps its wind, bit for bit, and the reference raises IndexError for member 1."""
  spec = model_spec('jn', nz)
  tau, kgm = _rows(spec.so.tau, spec.M), _rows(spec.so.KGM, spec.M)
  tau[1] = tau[2] = 0.
  kgm[1] = 0.
  bad = dataclasses.replace(spec, so=dataclasses.replace(spec.so, tau=tau, KGM=kgm))
  tau_ok = tau.copy()
  tau_ok[1] = _rows(spec.so.tau, spec.M)[1]
  kgm_ok = kgm.copy()
  kgm_ok[1] = _rows(spec.so.KGM, spec.M)[1]
  ok = dataclasses.replace(spec, so=dataclasses.replace(spec.so, tau=tau_ok, KGM=kgm_ok))
  pending = pool.map_async(km.oracle_task, [(bad.member_case(1), km.NSTEPS, False)])
  out, _ = _statuses(backend, host_backend, bad, [km.NSTEPS])
  st = [int(s) for s in out['status']]
  assert _bits(st, _abi.ST_ML_INDEX) == [False, True, False, False, False], (nz, st)
  ref = km._run(backend, ok, [km.NSTEPS])
  for key, v in out.items():
    for m in (0, 2, 3, 4):
      assert np.array_equal(v[m], ref[key][m], equal_nan=True), (nz, key, m)
  lost = pending.get()[0]
  assert isinstance(lost, str) and 'IndexError' in lost, lost
  return st
