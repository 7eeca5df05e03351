"""Pin the CPU oracle to the reference (CPU only).

The fixtures under tests/golden/ were produced by the unmodified reference
(tests/golden/make_golden.py).  In its default modes the oracle must reproduce them bit
for bit; in the 'kernel' modes (closed forms the CUDA path uses) the measured gap must
stay far below the 1e-10 parity gate.
"""
import warnings

import numpy as np
import pytest
from scipy import optimize

from helpers import golden, on_stored_levels, relmax
from oracle import pymoc_oracle as O

warnings.filterwarnings('ignore', category=RuntimeWarning)

COUPLED = [('c1', 300), ('c2', 73), ('twocol', 25), ('c3', 25), ('c3_bvp', 25), ('c4', 13), ('c4_literal', 120),
           ('c5', 25), ('twobasin', 25), ('c5_4096_k20', 21)]


@pytest.mark.parametrize('name,nmax', COUPLED)
def test_coupled_loops_bit_exact(name, nmax):
  tree = golden(name)
  for m, d in tree['members'].items():
    for n, want in d['runs'].items():
      if int(n) > nmax:
        continue
      got = O.run_coupled(d['case'], int(n), O.REFERENCE)
      for key, val in want.items():
        assert np.array_equal(on_stored_levels(tree, got[key]), val, equal_nan=True), (name, m, n, key)


@pytest.mark.parametrize('name,n', [('c1', 300), ('c2', 720), ('twocol', 480), ('c3', 480), ('c4', 600), ('c5', 480),
                                    ('twobasin', 480)])
def test_kernel_closed_forms_within_gate(name, n):
  """Exact quadrature / restated Brent / Thomas vs solve_bvp / brentq / inv: << 1e-10."""
  tree = golden(name)
  m, d = next(iter(tree['members'].items()))
  got = O.run_coupled(d['case'], n, O.KERNEL)
  for key, val in d['runs'][str(n)].items():
    assert relmax(got[key], val) < 1e-11, (name, m, key, relmax(got[key], val))


def test_brent_restatement_matches_scipy():
  rng = np.random.default_rng(7)
  for trial in range(300):
    ny = int(rng.integers(5, 60))
    y = np.linspace(0, 2e6, ny)
    bs = (np.sort(rng.random(ny)) * 0.03, 0.03 * (y / y[-1])**2 + 1e-3 * rng.standard_normal(ny),
          np.cumsum(rng.standard_normal(ny)) * 1e-3)[trial % 3]
    for k in range(4):
      bval = rng.uniform(bs.min(), bs[-1]) if k else bs[int(rng.integers(0, ny))]
      if bval < bs.min() or bval > bs[-1]:
        continue
      assert O.so_outcrop(bval, y, bs, 'brentq') == O.so_outcrop(bval, y, bs, 'brentq_restated')


def _col(inp):
  return O.ColumnState(inp['z'], inp['kappa'], inp['Area'], inp['b'], inp['bs'], inp['bbot'], inp['bzbot'],
                       inp['N2min'])


def test_column_units_bit_exact():
  for i, d in golden('units')['column'].items():
    inp, out = d['inp'], d['out']
    for tag, kw in (('plain', {}), ('conv', dict(do_conv=True)),
                    ('conv_hor', dict(do_conv=True, vdx_in=inp['vdx_in'], b_in=inp['b_in'])),
                    ('hor', dict(vdx_in=inp['vdx_in'], b_in=inp['b_in']))):
      col = _col(inp)
      for s in range(3):
        O.column_timestep(col, inp['wA'], inp['dt'], **kw)
        assert np.array_equal(col.b, out[tag][s]), (i, tag, s)
    col = _col(inp)
    O.column_convect(col)
    assert np.array_equal(col.b, out['convect_only'])
    assert np.array_equal(col.dAk, out['dAkappa_dz'])


def test_thermwind_units():
  for i, d in golden('units')['thermwind'].items():
    inp, out = d['inp'], d['out']
    psi = O.thermwind_solve(inp['z'], inp['b1'], inp['b2'], inp['f'], 'bvp')
    assert np.array_equal(psi, out['Psi']), i
    quad = O.thermwind_solve(inp['z'], inp['b1'], inp['b2'], inp['f'], 'quad')
    assert relmax(quad, out['Psi']) < 2e-14, (i, relmax(quad, out['Psi']))
    if 'psib' in out:
      iso_b, iso_n, psib, bgrid = O.thermwind_psibz(out['Psi'], inp['b1'], inp['b2'], 500)
      for got, key in ((psib, 'psib'), (bgrid, 'bgrid'), (iso_b, 'iso_b'), (iso_n, 'iso_n')):
        assert np.array_equal(got, out[key], equal_nan=True), (i, key)
      assert np.array_equal(O.thermwind_psib(out['Psi'], inp['b1'], inp['b2'], 37)[0], out['psib37'], equal_nan=True)


def test_so_units():
  for i, d in golden('units')['so'].items():
    inp, out = d['inp'], d['out']
    kw = {k: inp[k] for k in ('f', 'rho', 'L', 'KGM', 'c', 'bvp_with_Ek', 'Hsill', 'HEk', 'Htapertop', 'Htaperbot',
                              'smax')}
    p = O.ChannelParams(inp['z'], inp['y'], inp['tau'], **kw)
    psi, ek, gm = O.so_solve(p, inp['b'], inp['bs'])
    for got, key in ((psi, 'Psi'), (ek, 'Psi_Ek'), (gm, 'Psi_GM')):
      assert np.array_equal(got, out[key]), (i, key)
    ys = np.array([O.so_outcrop(v, inp['y'], np.asarray(inp['bs']) + 0 * inp['y'], 'brentq_restated')
                   for v in inp['b']])
    assert np.array_equal(ys, out['ys']), i


def test_ml_units():
  for i, d in golden('units')['ml'].items():
    inp, out = d['inp'], d['out']
    kw = {k: inp[k] for k in ('y', 'Ks', 'h', 'L', 'surflux', 'rest_mask', 'b_rest', 'v_pist', 'bs')}
    ml = O.MixedLayerState(**kw)
    th = O.MixedLayerState(**kw)
    for s in range(5):
      O.ml_timestep(ml, inp['b_basin'], inp['Psi_b'], inp['dt'], 'inv')
      assert np.array_equal(ml.bs, out['bs'][s]) and np.array_equal(ml.Psi_s, out['Psi_s'][s]), (i, s)
      O.ml_timestep(th, inp['b_basin'], inp['Psi_b'], inp['dt'], 'thomas')
      assert relmax(th.bs, out['bs'][s]) < 1e-13, (i, s, relmax(th.bs, out['bs'][s]))
