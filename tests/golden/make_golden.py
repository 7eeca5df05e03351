#!/usr/bin/env python
"""Generate the golden fixtures by running the UNMODIFIED reference.

Run in the build container only (it needs ``/root/reference``):

    python tests/golden/make_golden.py

It imports ``pymoc`` from ``/root/reference/src`` (with an empty ``matplotlib`` stub,
because ``psi_thermwind.py:3`` imports pyplot and never uses it), rebuilds the loop
bodies of the example scripts around the reference classes with the script's own
statement order, and writes small ``.npz`` files next to this script.  The fixtures --
not this script -- travel to the GPU box.

numpy / scipy used: see ``versions`` inside every fixture.
"""
import os
import sys
import tempfile

import numpy as np
import scipy

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

_stub = tempfile.mkdtemp(prefix='mpl_stub_')
os.makedirs(os.path.join(_stub, 'matplotlib'))
for _f in ('__init__.py', 'pyplot.py'):
  open(os.path.join(_stub, 'matplotlib', _f), 'w').close()
sys.path.insert(0, _stub)
sys.path.insert(0, '/root/reference/src')

from pymoc.modules import Column, Psi_SO, Psi_Thermwind, SO_ML  # noqa: E402  (the reference)

from golden_io import save_tree  # noqa: E402
from pymoc_b200 import configs  # noqa: E402

VERSIONS = dict(numpy=np.__version__, scipy=scipy.__version__, pymoc='0.0.1rc5')


def _fn(z, arr):
  """Array on the grid -> the callable a script would pass (exact at the nodes)."""
  arr = np.array(arr, dtype=np.float64)
  return lambda x: np.interp(x, z, arr)


def _column(z, d):
  return Column(z=z, kappa=_fn(z, d['kappa'][d['var0']]), Area=_fn(z, d['Area']), b=d['b0'].copy(), bs=d['bs'],
                bbot=d['bbot'], bzbot=d['bzbot'], N2min=d['N2min'])


def _channel(z, so, b):
  kw = {k: so[k] for k in ('f', 'rho', 'L', 'KGM', 'c', 'bvp_with_Ek', 'Hsill', 'HEk', 'Htapertop', 'Htaperbot',
                           'smax')}
  return Psi_SO(z=z, y=so['y'], b=b, bs=so['bs'].copy(), tau=so['tau'], **kw)


def run_reference(case, checkpoints, diag_iters=None):
  """Run the reference loop of ``case`` and snapshot the outputs after each N in
  ``checkpoints`` (ascending).  Statement order follows the cited scripts."""
  z, dt, K, nb = case['z'], case['dt'], case['K'], case['nb']
  basin = _column(z, case['basin'])
  north = _column(z, case['north']) if case['north'] is not None else None
  pac = _column(z, case['pac']) if case.get('pac') is not None else None
  tw, so, ml = case['tw'], case['so'], case['ml']
  snaps = {}
  two = {}  # the second closure pair of the two-basin topology

  def snapshot(n, AMOC, SO, iso, channel):
    s = dict(b_basin=basin.b.copy())
    if north is not None:
      s['b_north'] = north.b.copy()
    if AMOC is not None:
      s['Psi_tw'] = AMOC.Psi.copy()
    if iso is not None:
      s['Psi_iso_b'], s['Psi_iso_n'] = iso[0].copy(), iso[1].copy()
      s['bgrid'] = AMOC.bgrid.copy()
    if SO is not None:
      s['Psi_so'], s['Psi_Ek'], s['Psi_GM'] = SO.Psi.copy(), SO.Psi_Ek.copy(), SO.Psi_GM.copy()
    if channel is not None:
      s['bs_ml'] = channel.bs.copy()
      s['Psi_s'] = channel.Psi_s.copy()
    if pac is not None:
      s['b_pac'] = pac.b.copy()
      s['Psi_zoc'] = two['ZOC'].Psi.copy()
      s['Psi_zon_a'], s['Psi_zon_p'] = two['zon'][0].copy(), two['zon'][1].copy()
      s['bgrid2'] = two['ZOC'].bgrid.copy()
      s['Psi_so2'], s['Psi_Ek2'], s['Psi_GM2'] = two['SO'].Psi.copy(), two['SO'].Psi_Ek.copy(), two['SO'].Psi_GM.copy()
    snaps[str(n)] = s

  if case['order'] == 'post':
    # example_timestepping.py:52-80 / example_twocol.py:58-96 / example_twocol_plusSO.py:61-115
    AMOC = iso = SO = None
    if tw is not None:
      b2 = north.b if north is not None else tw['b2']
      AMOC = Psi_Thermwind(z=z, b1=basin.b, b2=b2, f=tw['f'])
      AMOC.solve()
      if case['iso']:
        iso = AMOC.Psibz(nb)
    if so is not None:
      SO = _channel(z, so, basin.b.copy())
      SO.solve()
    if pac is not None:  # examples/twobasin_NadeauJansen.py:68-81
      two['ZOC'] = Psi_Thermwind(z=z, b1=basin.b, b2=pac.b, f=case['zoc_f'])
      two['ZOC'].solve()
      two['zon'] = two['ZOC'].Psibz(nb)
      two['SO'] = _channel(z, {**so, 'L': case['so_pac_L']}, pac.b.copy())
      two['SO'].solve()
    for ii in range(max(checkpoints)):
      north_leg = (iso[0] if case['iso'] else AMOC.Psi) if AMOC is not None else 0. * z
      south_leg = SO.Psi if SO is not None else 0. * z
      wAb = (north_leg - south_leg) * 1e6
      if pac is not None:  # :104-109
        wAb = (iso[0] + two['zon'][0] - SO.Psi) * 1e6
        wA_Pac = (-two['zon'][1] - two['SO'].Psi) * 1e6
      basin.timestep(wA=wAb, dt=dt, do_conv=case['basin']['do_conv'])
      if north is not None:
        wAN = -iso[1] * 1e6
        north.timestep(wA=wAN, dt=dt, do_conv=case['north']['do_conv'])
      if pac is not None:
        pac.timestep(wA=wA_Pac, dt=dt, do_conv=case['pac']['do_conv'])
        if ii % K == 0:  # :117-123 (after the AMOC update below in the script; the two are independent)
          two['ZOC'].update(b1=basin.b, b2=pac.b)
          two['ZOC'].solve()
          two['zon'] = two['ZOC'].Psibz(nb)
          two['SO'].update(b=pac.b)
          two['SO'].solve()
      if ii % K == 0:
        if AMOC is not None:
          if north is not None:
            AMOC.update(b1=basin.b, b2=north.b)
          else:
            AMOC.update(b1=basin.b)
          AMOC.solve()
          if case['iso']:
            iso = AMOC.Psibz(nb)
        if SO is not None:
          SO.update(b=basin.b)
          SO.solve()
      if ii + 1 in checkpoints:
        snapshot(ii + 1, AMOC, SO, iso, None)
  else:
    # run_JansenNadeau_2018.py:140-261 / run_single_global_basin.py:119-229
    kap = [[_fn(z, k) for k in case[c]['kappa']] for c in ('basin', 'north')]
    AMOC = Psi_Thermwind(z=z, b1=basin.b, b2=north.b, f=tw['f'])
    AMOC.solve()
    PsiSO = _channel(z, so, basin.b)
    PsiSO.solve()
    m = ml
    channel = SO_ML(y=m['y'], h=m['h'], L=m['L'], Ks=m['Ks'], surflux=m['surflux'].copy(),
                    rest_mask=m['rest_mask'].copy(), b_rest=m['b_rest'].copy(), v_pist=m['v_pist'],
                    bs=m['bs'].copy())
    diag = {k: [] for k in ('AMOC', 'AMOC_b', 'b_basin', 'b_north', 'bs_SO', 'bgrid', 'Psi_SO')}
    for ii in range(max(checkpoints)):
      if ii % K == 0:
        AMOC.update(b1=basin.b, b2=north.b)
        AMOC.solve()
        [Psi_res_b, Psi_res_n] = AMOC.Psibz(nb=nb)
        PsiSO.update(b=basin.b, bs=channel.bs)
        PsiSO.solve()
        if diag_iters and ii % diag_iters == 0:  # run_JansenNadeau_2018.py:218-226
          diag['AMOC'].append(AMOC.Psi.copy())
          diag['AMOC_b'].append(AMOC.Psib(nb=nb).copy())
          diag['bgrid'].append(AMOC.bgrid.copy())
          diag['b_basin'].append(basin.b.copy())
          diag['b_north'].append(north.b.copy())
          diag['bs_SO'].append(channel.bs.copy())
          diag['Psi_SO'].append(PsiSO.Psi.copy())
      wAb = (Psi_res_b - PsiSO.Psi) * 1e6
      wAN = -Psi_res_n * 1e6
      if PsiSO.Psi[1] < 0:
        basin.bbot = channel.bs[0]
        basin.kappa = kap[0][1]
      if Psi_res_b[1] > 0 and north.b[0] < basin.b[1] and north.b[0] < channel.bs[0]:
        basin.bbot = north.b[0]
        basin.kappa = kap[0][1]
      elif PsiSO.Psi[1] >= 0:
        basin.bbot = basin.b[1]
        basin.kappa = kap[0][0]
      if Psi_res_n[1] < 0 and basin.b[0] < north.b[1]:
        north.bbot = basin.b[0]
        north.kappa = kap[1][1]
      else:
        north.bbot = north.b[1]
        north.kappa = kap[1][0]
      basin.timestep(wA=wAb, dt=dt, do_conv=True)
      north.timestep(wA=wAN, dt=dt, do_conv=True)
      channel.timestep(b_basin=basin.b, Psi_b=PsiSO.Psi, dt=dt)
      if ii + 1 in checkpoints:
        snapshot(ii + 1, AMOC, PsiSO, [Psi_res_b, Psi_res_n], channel)
    if diag_iters:
      col = lambda k: np.stack(diag[k], axis=-1)
      # positional layout of np.savez(diagfile, ...) at :268-272 and of the pickup at :266-267
      snaps['diagfile'] = {'arr_%d' % i: a for i, a in enumerate(
          [col('AMOC'), col('AMOC_b'), col('b_basin'), col('b_north'), col('bs_SO'), z, col('bgrid'), so['y'],
           col('Psi_SO'), np.float64(so['tau']), np.float64(so['KGM'])])}
      snaps['pickup'] = {'arr_0': basin.b.copy(), 'arr_1': north.b.copy(), 'arr_2': channel.bs.copy()}
  return snaps


def coupled_fixture(fname, spec, members, checkpoints, extra=None, levels=None):
  """``levels``: store the outputs on the z grid at these levels only (tests/helpers.on_stored_levels)."""
  tree = dict(versions=VERSIONS, name=spec.name, members={})
  if extra:
    tree.update(extra)
  if levels is not None:
    tree['levels'] = levels
  for m in members:
    case = spec.member_case(m)
    runs = run_reference(case, checkpoints)
    if levels is not None:
      runs = {n: {k: v[levels] if v.shape == spec.z.shape else v for k, v in s.items()} for n, s in runs.items()}
    tree['members'][str(m)] = dict(case=case, runs=runs)
    print('  %s member %d done' % (fname, m), flush=True)
  save_tree(os.path.join(HERE, fname), tree)


# ----------------------------------------------------------------------- unit vectors
def unit_fixture():
  rng = np.random.default_rng(20181018)
  tree = dict(versions=VERSIONS)

  # --- Column: convect / vertadvdiff / horadv / timestep ------------------------------------
  cols = {}
  z_u = np.asarray(np.linspace(-4000, 0, 80))
  z_n = -4000. * (1. - np.linspace(0, 1, 61)**0.6)
  z_n[-1] = 0.
  variants = [
      dict(z=z_u, kappa=2e-5 + 0 * z_u, Area=6e13 + 0 * z_u, bs=0.02, bbot=-0.001, bzbot=None, N2min=1e-7,
           b=0.02 * np.exp(z_u / 400.) + 1e-3 * rng.standard_normal(80), wA=3e6 * np.sin(z_u / 600.), dt=30 * 86400.),
      dict(z=z_n, kappa=1e-5 + 2e-4 * np.exp(z_n / 300.), Area=5e13 * (1 + 0.3 * z_n / 4000.), bs=0.03, bbot=0.0,
           bzbot=2e-7, N2min=2e-7, b=0.03 * np.exp(z_n / 500.), wA=-2e6 * np.cos(z_n / 900.), dt=10 * 86400.),
      dict(z=np.asarray([-4000.0, -1000.0, -100.0, 0.0]), kappa=2e-5 + np.zeros(4), Area=6e13 + np.zeros(4), bs=0.0,
           bbot=0.0, bzbot=None, N2min=1.5e-7, b=np.asarray([-0.03, -0.02, 0.01, 0.01]), wA=np.zeros(4), dt=86400.),
      dict(z=z_u, kappa=2e-5 + 0 * z_u, Area=6e13 + 0 * z_u, bs=-0.001, bbot=0.0, bzbot=None, N2min=1e-7,
           b=0.004 * np.exp(z_u / 300.), wA=1e6 * np.sin(z_u / 500.), dt=30 * 86400.),  # everything convects
  ]
  for i, v in enumerate(variants):
    z = v['z']
    vdx = 2e4 * (1 + np.sin(z / 700.))
    vdx[::3] = -1.0
    b_in = v['b'] * 0.9 - 1e-4
    out = {}
    for tag, kw in (('plain', dict()), ('conv', dict(do_conv=True)),
                    ('conv_hor', dict(do_conv=True, vdx_in=vdx, b_in=b_in)), ('hor', dict(vdx_in=vdx, b_in=b_in))):
      c = Column(z=z, kappa=_fn(z, v['kappa']), Area=_fn(z, v['Area']), b=v['b'].copy(), bs=v['bs'], bbot=v['bbot'],
                 bzbot=v['bzbot'], N2min=v['N2min'])
      steps = []
      for _ in range(3):
        c.timestep(wA=v['wA'], dt=v['dt'], **kw)
        steps.append(c.b.copy())
      out[tag] = np.array(steps)
    c = Column(z=z, kappa=_fn(z, v['kappa']), Area=_fn(z, v['Area']), b=v['b'].copy(), bs=v['bs'], bbot=v['bbot'],
               bzbot=v['bzbot'], N2min=v['N2min'])
    c.convect()
    out['convect_only'] = c.b.copy()
    out['dAkappa_dz'] = c.dAkappa_dz(z)
    cols[str(i)] = dict(inp=dict(v, vdx_in=vdx, b_in=b_in), out=out)
  tree['column'] = cols

  # --- Psi_Thermwind: solve / Psib / Psibz ---------------------------------------------------
  tws = {}
  z = z_u
  profiles = [
      (0.03 * np.exp(z / 300.), 0.004 * np.exp(z / 300.), 1e-4),
      (0.03 * np.exp(z / 300.) - 0.0004, 0. * z, 1.2e-4),
      (0.02 * np.exp(z / 300.) + (-0.001) * z / z[0], -0.001 * (z / z[0])**2., 1.2e-4),
      (np.sort(0.03 * rng.random(80)), np.sort(0.01 * rng.random(80)), 1e-4),
  ]
  # flat bottom cell (no-flux BBC) and an inversion
  p4 = 0.02 * np.exp(z / 300.)
  p4[0] = p4[1]
  p5 = 0.02 * np.exp(z / 300.)
  p5[10] = p5[12]
  profiles += [(p4, -0.001 * (z / z[0])**2., 1.2e-4), (p5, 0.001 + 0 * z, 1.2e-4)]
  for i, (b1, b2, f) in enumerate(profiles):
    tw = Psi_Thermwind(z=z, b1=b1.copy(), b2=b2.copy(), f=f)
    tw.solve()
    with np.errstate(all='ignore'):
      psib_small = tw.Psib(37)
      psib = tw.Psib(500)
      bz = tw.Psibz(500)
    tws[str(i)] = dict(inp=dict(z=z, b1=b1, b2=b2, f=f), out=dict(Psi=tw.Psi.copy(), psib=psib, bgrid=tw.bgrid.copy(),
                                                                   iso_b=bz[0], iso_n=bz[1], psib37=psib_small))
  for nz in (46, 70, 200, 1024):
    zz = np.asarray(np.linspace(-4500., 0., nz))
    b1 = 0.025 * np.exp(zz / 400.) - 0.0001 * zz / zz[0]
    b2 = 0.0 - 0.0001 * (zz / zz[0])**2.
    tw = Psi_Thermwind(z=zz, b1=b1, b2=b2, f=1.2e-4)
    tw.solve()
    tws['nz%d' % nz] = dict(inp=dict(z=zz, b1=b1, b2=b2, f=1.2e-4), out=dict(Psi=tw.Psi.copy()))
  tree['thermwind'] = tws

  # --- Psi_SO.solve ---------------------------------------------------------------------------
  sos = {}
  z = np.asarray(np.linspace(-4000, 0, 81))
  y = np.asarray(np.linspace(0, 2.0e6, 51))
  b_lin = np.linspace(-0.001, 0.03, 81)
  b_exp = 0.02 * np.exp(z / 300.) - 0.001 * z / z[0]
  bs_q = 0.03 * (y / y[-1])**2
  bs_lin = np.linspace(0.005, 0.02, 51)
  bs_dip = bs_q.copy()
  bs_dip[:6] = [0.002, 0.001, 0.0, -0.0005, -0.001, -0.0008]
  combos = [
      dict(b=b_exp, bs=bs_q, tau=0.13, f=1e-4, L=5e6, KGM=1000.),
      dict(b=b_lin, bs=bs_lin, tau=0.12),
      dict(b=b_exp, bs=bs_dip, tau=0.1, Hsill=1000., HEk=200., Htapertop=300., Htaperbot=500., smax=0.002),
      dict(b=b_exp, bs=bs_q, tau=np.linspace(0.2, 0.12, 51)),
      dict(b=b_lin, bs=bs_lin, tau=0.12, KGM=800., L=4e6, Htapertop=100.),
      dict(b=b_exp, bs=bs_q, tau=0.13, f=1e-4, L=5e6, KGM=1000., c=0.1, bvp_with_Ek=True),
      dict(b=b_exp, bs=bs_q, tau=0.13, f=1e-4, L=5e6, KGM=1000., c=1.0, bvp_with_Ek=False),
  ]
  for i, kw in enumerate(combos):
    so = Psi_SO(z=z, y=y, **{k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in kw.items()})
    so.solve()
    ys = np.array([so.ys(v) for v in so.b(z)])
    inp = dict(z=z, y=y, rho=1030, f=1.2e-4, L=1e7, KGM=1e3, c=None, bvp_with_Ek=False, Hsill=None, HEk=None,
               Htapertop=None, Htaperbot=None, smax=0.01)
    inp.update(kw)
    sos[str(i)] = dict(inp=inp, out=dict(Psi=so.Psi.copy(), Psi_Ek=so.Psi_Ek.copy(), Psi_GM=so.Psi_GM.copy(), ys=ys))
  tree['so'] = sos

  # --- SO_ML.timestep -------------------------------------------------------------------------
  mls = {}
  spec = configs.c4_jansen_nadeau(1)
  case = spec.member_case(0)
  m = case['ml']
  zb = case['z']
  b_basin = case['basin']['b0']
  psi_variants = [
      3.0 * np.sin(np.pi * zb / 4000.)**2 * np.sign(zb + 2500.),  # lower cell negative, upper positive
      -2.0 * np.sin(np.pi * zb / 4000.)**2,
      np.where(zb > -3000., 4.0 * np.sin(np.pi * zb / 3000.)**2, 0.0),  # zeros below 3000 m (blocked isopycnals)
  ]
  for i, psi in enumerate(psi_variants):
    psi = psi.copy()
    psi[0] = 0.
    channel = SO_ML(y=m['y'], h=m['h'], L=m['L'], Ks=m['Ks'] * (1 + i), surflux=m['surflux'].copy(),
                    rest_mask=m['rest_mask'].copy(), b_rest=m['b_rest'].copy(), v_pist=m['v_pist'], bs=m['bs'].copy())
    steps, psis = [], []
    for _ in range(5):
      channel.timestep(b_basin=b_basin, Psi_b=psi, dt=case['dt'])
      steps.append(channel.bs.copy())
      psis.append(channel.Psi_s.copy())
    mls[str(i)] = dict(inp=dict(m, Ks=m['Ks'] * (1 + i), b_basin=b_basin, Psi_b=psi, dt=case['dt']),
                       out=dict(bs=np.array(steps), Psi_s=np.array(psis)))
  tree['ml'] = mls
  save_tree(os.path.join(HERE, 'units.npz'), tree)


def check_callable_sampling():
  """What sampling callables on the grid (north_star) changes, measured on the literal C1 script.

  * kappa / Area callables: nothing -- ``kappa(z)[1:-1] == kappa(z[1:-1])`` bit for bit.
  * a callable *initial* b1 handed to Psi_Thermwind: ``solve_bvp`` evaluates it at the
    collocation mid-points, so the very first Psi (used for step 0 only) differs from the
    one diagnosed from nodal values; afterwards the loop feeds arrays.  The size of that
    start-up difference is printed and stored in c1.npz as ``callable_init_gap``.
  """
  z = np.asarray(np.linspace(-3500, 0, 70))
  kap = lambda zz: 1e-5 + 3e-5 * np.exp(zz / 100) + 3e-4 * np.exp(-zz / 1000 - 4)
  b_fun = lambda zz: 0.03 * np.exp(zz / 300.) - 0.0004
  assert np.array_equal(kap(z)[1:-1], kap(z[1:-1])), 'np.exp is position dependent on this box'
  case = configs.c1_timestepping(1).member_case(0)
  ours = run_reference(case, [25, 300])

  def literal(b1_init, n):
    basin = Column(z=z, kappa=kap, Area=8e13, b=b_fun, bs=0.03, bbot=-0.0004)
    AMOC = Psi_Thermwind(z=z, b1=b1_init)
    AMOC.solve()
    for ii in range(n):
      basin.timestep(wA=AMOC.Psi * 1e6, dt=60 * 86400)
      AMOC.update(b1=basin.b)
      AMOC.solve()
    return basin.b.copy(), AMOC.Psi.copy()

  b, psi = literal(b_fun(z), 25)
  assert np.array_equal(ours['25']['b_basin'], b) and np.array_equal(ours['25']['Psi_tw'], psi), \
      'script loop with nodal initial b1 differs from the case-driven loop'
  gap = {}
  for n in (25, 300):
    b, psi = literal(b_fun, n)
    gap[str(n)] = np.array([np.abs(b - ours[str(n)]['b_basin']).max() / np.abs(b).max(),
                            np.abs(psi - ours[str(n)]['Psi_tw']).max() / np.abs(psi).max()])
    print('callable initial b1 vs nodal: N=%d  rel gap b %.2e  Psi %.2e' % (n, gap[str(n)][0], gap[str(n)][1]))
  return gap


if __name__ == '__main__':
  # `make_golden.py only c4 c5` regenerates just the named coupled fixtures
  only = sys.argv[sys.argv.index('only') + 1:] if 'only' in sys.argv else None
  want = lambda name: only is None or name in only
  if only is None:
    unit_fixture()
    print('units done', flush=True)
    if 'units' in sys.argv[1:]:
      sys.exit(0)
  if want('equi'):  # Column.solve_equi as examples/example_iteration.py:63 calls it (three outer iterations)
    A, bs, bbot = 8e13, 0.03, -0.0004
    z = np.asarray(np.linspace(-3500, 0, 70))
    kappa = lambda zz: 1e-5 + 3e-5 * np.exp(zz / 100) + 3e-4 * np.exp(-zz / 1000 - 4)
    b0 = bs * np.exp(z / 300.) + z / z[0] * bbot
    amoc = Psi_Thermwind(z=z, b1=b0)
    amoc.solve()
    basin = Column(z=z, kappa=kappa, Area=A, b=b0.copy(), bs=bs, bbot=bbot)
    out = {}
    for it in range(3):
      basin.solve_equi(amoc.Psi * 1e6)
      out[str(it)] = dict(wA=amoc.Psi * 1e6, b=basin.b.copy(), bz=basin.bz.copy())
      amoc.update(b1=0.8 * amoc.b1(z) + 0.2 * basin.b)
      amoc.solve()
    save_tree(os.path.join(HERE, 'equi.npz'), dict(versions=VERSIONS, z=z, b0=b0, A=A, bs=bs, bbot=bbot, iters=out))
    print('equi done', flush=True)
  if want('c1'):
    GAP = check_callable_sampling()
    coupled_fixture('c1.npz', configs.c1_timestepping(1), [0], [1, 2, 10, 300, 1200], extra=dict(callable_init_gap=GAP))
  if want('c2'):
    coupled_fixture('c2.npz', configs.c2_column_so(16, ntau=4), [0, 5, 10, 15], [1, 73, 720, 2160])
  if want('twocol'):
    coupled_fixture('twocol.npz', configs.twocol(1), [0], [1, 25, 480])
  if want('c3'):
    coupled_fixture('c3.npz', configs.c3_twocol_so(16, axes=(2, 2, 2, 2)), [0, 7, 9, 15], [1, 25, 480, 2400])
  if want('c3_bvp'):
    coupled_fixture('c3_bvp.npz', configs.c3_twocol_so(1, c=0.1), [0], [1, 25, 240])
  if want('c4'):
    coupled_fixture('c4.npz', configs.c4_jansen_nadeau(32, axes=(2, 2, 2, 2, 2)), [0, 13, 22, 31], [1, 12, 13, 600, 2400])
  if want('c4_literal'):
    coupled_fixture('c4_literal.npz', configs.c4_jansen_nadeau(1), [0], [1, 120, 1200])
  if want('c4_diags'):  # the diagnostics / pickup files of the literal script, 360 iterations, Diag_iters = 120
    spec = configs.c4_jansen_nadeau(1)
    case = spec.member_case(0)
    tree = dict(versions=VERSIONS, name=spec.name, case=case, diag_iters=120, total_iters=360,
                files=run_reference(case, [360], diag_iters=120))
    save_tree(os.path.join(HERE, 'c4_diags.npz'), tree)
  if want('twobasin'):
    coupled_fixture('twobasin.npz', configs.twobasin(8, axes=(2, 2, 2)), [0, 5, 7], [1, 25, 480, 1200])
  if want('c5'):
    coupled_fixture('c5.npz', configs.c5_single_global_basin(1), [0], [1, 24, 25, 480])
  # columns taller than one warp holds (block-per-member kernels): nz=320 over two refreshes, and the
  # BASELINE size nz=4096 at its stable dt (K=72 000 there, so the fixture only sees the first diagnosis)
  if want('c5_wide'):
    coupled_fixture('c5_wide.npz', configs.c5_single_global_basin(4, nz=320, dt_days=1., axes=(2, 2, 1, 1)), [0, 3],
                    [1, 720, 721, 1000])
  if want('c5_4096'):
    coupled_fixture('c5_4096.npz', configs.c5_single_global_basin(1, nz=4096, dt_days=0.01), [0], [1, 40])
  # the same grid with the streamfunctions re-diagnosed every 20 iterations (MOC_up_iters is a free parameter of the
  # script): the block-wide diagnosis kernel is exercised INSIDE a run at nz = 4096, three times in 45 steps.
  # Every third level (0 ... 4095) is stored, which keeps the file under 1 MB.
  if want('c5_4096_k20'):
    spec = configs.c5_single_global_basin(2, nz=4096, dt_days=0.01, axes=(2, 1, 1, 1))
    spec.K = 20
    coupled_fixture('c5_4096_k20.npz', spec, [0, 1], [20, 21, 45], levels=np.arange(0, spec.nz, 3))
