"""Shared helpers for the parity tests."""
import os

import numpy as np

from golden_io import load_tree

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')

_cache = {}


def golden(name):
  if name not in _cache:
    _cache[name] = load_tree(os.path.join(GOLDEN, name + '.npz'))
  return _cache[name]


def on_stored_levels(tree, arr):
  """``arr`` as the fixture ``tree`` stores it.  Fixtures of tall columns keep the fields on the z grid at the
  levels ``tree['levels']`` only (every third level at nz = 4096, which keeps the file under 1 MB); other
  arrays are stored whole."""
  levels = tree.get('levels')
  if levels is None:
    return arr
  nz = next(iter(tree['members'].values()))['case']['z'].size
  return arr[..., levels] if np.shape(arr)[-1] == nz else arr


def relmax(got, want):
  """max|got-want| / max|want|  (SURVEY.md section 8c: per-field max-norm relative error)."""
  got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
  if got.shape != want.shape:
    return np.inf
  if np.array_equal(got, want, equal_nan=True):
    return 0.0
  if not np.array_equal(np.isnan(got), np.isnan(want)):
    return np.inf
  scale = np.nanmax(np.abs(want))
  return float(np.nanmax(np.abs(got - want)) / (scale if scale > 0 else 1.0))


def spec_from_cases(cases):
  """Stack single-member oracle cases (the golden layout) into a ModelSpec of M members."""
  from pymoc_b200.spec import (ChannelSpec, ColumnSpec, MixedLayerSpec, ModelSpec, ThermwindSpec)
  c0 = cases[0]
  z = c0['z']
  stack = lambda f: np.stack([np.asarray(f(c), dtype=np.float64) for c in cases])

  def col(name):
    if c0[name] is None:
      return None
    g = lambda k: stack(lambda c: c[name][k])
    d0 = c0[name]
    return ColumnSpec.build(z, g('kappa'), g('Area'), g('bs'), g('b0'), bbot=g('bbot'),
                            bzbot=None if d0['bzbot'] is None else g('bzbot'), N2min=g('N2min'),
                            do_conv=d0['do_conv'], var0=int(d0['var0']))

  basin, north = col('basin'), col('north')
  pac = col('pac') if c0.get('pac') is not None else None
  for cs, name in ((basin, 'basin'), (north, 'north'), (pac, 'pac')):
    if cs is not None:
      cs.kappa = np.ascontiguousarray(stack(lambda c: c[name]['kappa']))  # [M, nvar, nz]
  tw = so = ml = None
  if c0['tw'] is not None:
    tw = ThermwindSpec.build(z, f=stack(lambda c: c['tw']['f']),
                             b2=None if c0['tw']['b2'] is None else stack(lambda c: c['tw']['b2']))
  if c0['so'] is not None:
    s0 = c0['so']
    g = lambda k: stack(lambda c: c['so'][k])
    so = ChannelSpec.build(s0['y'], g('bs'), g('tau'), f=g('f'), rho=g('rho'), L=g('L'), KGM=g('KGM'),
                           c=None if s0['c'] is None else g('c'), bvp_with_Ek=bool(s0['bvp_with_Ek']),
                           Hsill=s0['Hsill'], HEk=s0['HEk'], Htapertop=s0['Htapertop'], Htaperbot=s0['Htaperbot'],
                           smax=g('smax'))
  if c0['ml'] is not None:
    g = lambda k: stack(lambda c: c['ml'][k])
    ml = MixedLayerSpec.build(c0['ml']['y'], g('bs'), Ks=g('Ks'), h=g('h'), L=g('L'), surflux=g('surflux'),
                              rest_mask=g('rest_mask'), b_rest=g('b_rest'), v_pist=g('v_pist'))
  return ModelSpec(M=len(cases), z=z, dt=float(c0['dt']), K=int(c0['K']), nb=int(c0['nb']), order=c0['order'],
                   iso=bool(c0['iso']), basin=basin, north=north, tw=tw, so=so, ml=ml, pac=pac,
                   zoc_f=None if pac is None else stack(lambda c: c['zoc_f']),
                   so_pac_L=None if pac is None else stack(lambda c: c['so_pac_L']))
