"""Parity checks shared by the CPU (warp-emulator) and GPU (C ABI on cuda:0) test files."""
import json
import os

import numpy as np

from helpers import golden, on_stored_levels, relmax, spec_from_cases
from pymoc_b200.ensemble import Ensemble

# north_star: 1e-10 relative (max-norm per field, SURVEY.md section 8c) on the explicit path
TOL = 1e-10


def run_against_golden(backend, name, nmax, tol=TOL, chunked=False):
  """Run every member of a golden fixture as one ensemble and compare at each checkpoint."""
  tree = golden(name)
  members = list(tree['members'].items())
  ens = Ensemble(spec_from_cases([d['case'] for _, d in members]), backend=backend)
  done, worst = 0, 0.0
  for n in sorted(int(k) for k in members[0][1]['runs']):
    if n > nmax:
      break
    if chunked:  # many short launches: exercises the carried streamfunctions between launches
      while done < n:
        step = min(7, n - done)
        ens.run(step)
        done += step
    else:
      ens.run(n - done)
      done = n
    got = {**ens.state(), **ens.diagnostics()}
    for i, (m, d) in enumerate(members):
      for key, want in d['runs'][str(n)].items():
        if key not in got:
          continue
        err = relmax(on_stored_levels(tree, got[key][i]), want)
        worst = max(worst, err)
        assert err < tol, '%s member %s step %d field %s: rel err %.3e' % (name, m, n, key, err)
    assert not (got['status'] & 1).any(), 'NaN status raised'
  return worst



def diag_and_pickup_files(backend, tmpdir):
  """The --diagfile / --pickup_save_file archives of examples/run_JansenNadeau_2018.py:266-272 for
  the literal script configuration, 360 iterations with Diag_iters = 120, against the files the
  reference writes (golden c4_diags.npz); then a restart from the pickup."""
  import os

  from pymoc_b200 import pickup
  tree = golden('c4_diags')
  ens = Ensemble(spec_from_cases([tree['case']]), backend=backend)
  rec = pickup.DiagRecorder(ens, int(tree['diag_iters'])).run(int(tree['total_iters']))
  dpath, ppath = os.path.join(tmpdir, 'diags.npz'), os.path.join(tmpdir, 'pickup.npz')
  rec.save(dpath, member=0)
  pickup.save_pickup(ens, ppath, member=0)
  got, want = np.load(dpath), tree['files']['diagfile']
  assert sorted(got.files) == sorted(want), (got.files, sorted(want))
  for k in want:
    assert np.shape(got[k]) == np.shape(want[k]), (k, np.shape(got[k]), np.shape(want[k]))
    assert relmax(got[k], want[k]) < TOL, (k, relmax(got[k], want[k]))
  gotp = np.load(ppath)
  for k, v in tree['files']['pickup'].items():
    assert relmax(gotp[k], v) < TOL, k
  # restart: a fresh ensemble picked up from the file continues like the one that wrote it
  # (the scripts restart their iteration counter, so 360 must be -- and is -- a multiple of K)
  again = Ensemble(spec_from_cases([tree['case']]), backend=backend)
  pickup.load_pickup(again, ppath)
  assert again.it == 0
  again.run(24)
  ens.run(24)
  for k, v in ens.state().items():
    assert np.array_equal(v, again.state()[k]), k


def edge_sizes(backend, wide=True):
  """Sizes at the dispatch boundaries of the kernels against the live oracle: levels per lane 2..8 (nz up to
  256) with member counts that do not fill a CTA, the smallest grids, and the block-per-member kernels at
  the boundaries of their levels-per-thread variants."""
  import warnings

  from oracle import pymoc_oracle as O
  from pymoc_b200 import configs
  warnings.filterwarnings('ignore')
  worst = 0.0

  def check(spec, nsteps, members, keys):
    nonlocal worst
    ens = Ensemble(spec, backend=backend)
    ens.run(nsteps)
    got = {**ens.state(), **ens.diagnostics()}
    for m in members:
      want = O.run_coupled(spec.member_case(m), nsteps, O.REFERENCE)
      for key in keys:
        err = relmax(got[key][m], want[key])
        worst = max(worst, err)
        assert err < TOL, (spec.name, spec.nz, m, key, err)

  # column + Psi_SO: every levels-per-lane variant, 3 members (a partly filled CTA), smallest channel grid
  for nz, ny in ((5, 3), (33, 40), (64, 7), (65, 40), (129, 40), (255, 40), (256, 64)):
    with configs.members(0, 3):
      spec = configs.c2_column_so(4, nz=nz, ny=ny, dt_days=0.5)
    check(spec, 2 * spec.K + 3 if spec.K < 40 else 75, (0, 2), ('b_basin', 'Psi_so', 'Psi_Ek', 'Psi_GM'))
  # 'jn' order at the warp kernels' largest grid and at a tiny one
  for nz, dt_days in ((256, 2.), (12, 30.)):
    with configs.members(1, 4):
      spec = configs.c5_single_global_basin(4, nz=nz, dt_days=dt_days, axes=(2, 2, 1, 1), kapfac_max=1.)
    check(spec, 30, (0, 2), ('b_basin', 'b_north', 'bs_ml', 'Psi_iso_b', 'Psi_so'))
  if wide:  # block-per-member kernels: first size, boundaries of the 4 / 8 / 16 levels-per-thread variants
    for nz, dt_days in ((257, 2.), (1024, 0.1), (1025, 0.1), (2049, 0.02)):
      spec = configs.c5_single_global_basin(1, nz=nz, dt_days=dt_days)
      check(spec, 25, (0,), ('b_basin', 'b_north', 'bs_ml', 'Psi_iso_b', 'Psi_so'))
  return worst


# ------------------------------------------------------------------------------------------------
# Bench-lattice samples against the live oracle (VERDICT round 1, item 1): the golden fixtures hold a handful
# of members; the bench steps 32k..262k-member lattices.  These checks draw seeded-random members from the
# BENCH-SIZE lattice (the very members bench.py runs), step them through the kernel as one ensemble and compare
# every one of them with the oracle.  Contract:
#   * a member that carries none of the PMOC_ST_PARITY_UNDEFINED bits must match to `tol` in every field;
#   * a member the oracle loses (NaN state, or the ValueError / IndexError the reference raises) must be
#     flagged by the kernel (PMOC_ST_NAN / BRENT_SIGN / ML_INDEX), and vice versa;
#   * the fraction of members carrying a parity-undefined bit stays below `max_flagged`, and how many of those
#     nevertheless match is reported.
LATTICE_FIELDS = ('b_basin', 'b_north', 'b_pac', 'bs_ml', 'Psi_tw', 'Psi_iso_b', 'Psi_iso_n', 'Psi_so', 'Psi_zon_a',
                  'Psi_zon_p', 'Psi_so2')


def bench_lattice(workload, M):
  """The bench's own builder for `workload` at lattice size M (imports bench.py: same lattice, by construction)."""
  import bench
  return bench.WORKLOADS[workload][0](M)


def sample_cases(workload, M, nsample, seed):
  """`nsample` seeded-random members of the M-member bench lattice of `workload`, as oracle cases."""
  from pymoc_b200 import configs
  rng = np.random.default_rng(seed)
  ms = sorted(int(m) for m in rng.choice(M, size=min(nsample, M), replace=False))
  cases = []
  for m in ms:
    with configs.members(m, m + 1):  # only this member of the lattice is materialised
      cases.append(bench_lattice(workload, M).member_case(0))
  return ms, cases


def _oracle_task(args):
  case, nsteps = args
  import warnings
  warnings.filterwarnings('ignore')
  from oracle import pymoc_oracle as O
  try:
    out = O.run_coupled(case, nsteps, O.REFERENCE)
    return {k: v for k, v in out.items() if v is not None}
  except (ValueError, IndexError, FloatingPointError) as e:  # what the reference raises on a lost member
    return repr(e)


def oracle_many(cases, nsteps, procs=None):
  """The oracle's reference-faithful loop for every case, on the host cores (spawned workers: safe next to CUDA)."""
  import multiprocessing as mp
  import os
  procs = procs or min(len(cases), os.cpu_count() or 1)
  os.environ.setdefault('OMP_NUM_THREADS', '1')  # (inherited by the workers: one BLAS thread each)
  os.environ.setdefault('OPENBLAS_NUM_THREADS', '1')
  if procs <= 1:
    return [_oracle_task((c, nsteps)) for c in cases]
  with mp.get_context('spawn').Pool(procs) as pool:
    return pool.map(_oracle_task, [(c, nsteps) for c in cases], chunksize=1)


def lattice_sample(backend, workload, M, nsample, nsteps, seed=0, tol=TOL, max_flagged=1.0, procs=None, K=None):
  """``K``: override MOC_up_iters of the sampled members (a free parameter of the scripts), e.g. to cross several
  diagnoses at nz = 4096, whose own K is 72 000."""
  from pymoc_b200 import _abi
  ms, cases = sample_cases(workload, M, nsample, seed)
  if K is not None:
    for c in cases:
      c['K'] = int(K)
  ens = Ensemble(spec_from_cases(cases), backend=backend)
  ens.run(nsteps)
  got = {**ens.state(), **ens.diagnostics()}
  want = oracle_many(cases, nsteps, procs)
  st = got['status']
  rep = dict(workload=workload, lattice=M, sampled=len(ms), steps=nsteps, K=int(cases[0]['K']), census=_abi.status_census(st), worst_unflagged=0.0,
             flagged_matching=0, flagged_missing=0, lost_by_both=0)
  for i, m in enumerate(ms):
    undefined = bool(st[i] & _abi.ST_PARITY_UNDEFINED)
    lost_k = bool(st[i] & (_abi.ST_NAN | _abi.ST_BRENT_SIGN | _abi.ST_ML_INDEX))
    w = want[i]
    lost_o = isinstance(w, str) or not all(np.isfinite(w[k]).all() for k in ('b_basin', 'b_north', 'bs_ml') if k in w)
    if lost_o or lost_k:
      # a blow-up is preceded by a noisy state: the step at which each side gives up may differ, the fact may not
      assert undefined or (lost_o and lost_k), '%s member %d: lost by %s only (status %d, oracle %s)' % (
          workload, m, 'the oracle' if lost_o else 'the kernel', st[i], w if isinstance(w, str) else 'finite')
      rep['lost_by_both'] += int(lost_o and lost_k)
      continue
    err = max(relmax(got[k][i], w[k]) for k in LATTICE_FIELDS if k in got and k in w)
    if undefined:
      rep['flagged_matching' if err < tol else 'flagged_missing'] += 1
    else:
      rep['worst_unflagged'] = max(rep['worst_unflagged'], err)
      assert err < tol, '%s lattice member %d (status %d): rel err %.3e after %d steps, not flagged' % (
          workload, m, st[i], err, nsteps)
  nflag = rep['census']['parity_undefined']
  rep['flagged_fraction'] = nflag / len(ms)
  path = os.environ.get('PMOC_LATTICE_REPORT')  # evidence file (one JSON line per sample), see profiles/
  if path:
    with open(path, 'a') as f:
      f.write(json.dumps(dict(rep, backend=type(backend).__name__, tol=tol)) + '\n')
  assert rep['flagged_fraction'] <= max_flagged, '%s: %d of %d sampled members carry a parity-undefined bit' % (
      workload, nflag, len(ms))
  return rep


def f2010_smoother_converged(backend, sizes=(46, 80, 200, 256), bvp_tol=1e-9, tol=2e-9):
  """The F2010 smoother of Psi_GM (psi_SO.py:308-323) against scipy's solve_bvp run to a tight tolerance on a refined
  mesh (the reference runs the same ODE at tol = 1e-3): the kernel's piecewise-exact solution (series propagators +
  partitioned cyclic reduction) is the converged one (measured 6e-14 against tol = 1e-11, which takes scipy minutes).
  Levels per lane 2, 3, 7, 8."""
  import warnings

  from scipy import integrate

  from oracle import pymoc_oracle as O
  from pymoc_b200 import configs
  from pymoc_b200.spec import _vec
  warnings.filterwarnings('ignore')
  worst = 0.0
  for nz in sizes:
    if nz == 80:
      spec = configs.c3_twocol_so(2, c=0.1, axes=(2, 1, 1, 1))
    else:
      spec = configs.c2_column_so(2, nz=nz, ntau=2)
      spec.so.c, spec.so.bvp_with_Ek = _vec(0.1, 'c'), True
    ens = Ensemble(spec, backend=backend)
    ens.run(25 if nz == 80 else 3)  # a state off the initial condition
    state = ens.state()
    ens.set_state(**state)
    ens.diagnose()
    got = ens.diagnostics()
    assert not got['status'].any()
    for m in range(spec.M):
      case = spec.member_case(m)
      so, z, b = case['so'], case['z'], state['b_basin'][m]
      p = O.ChannelParams(z, so['y'], so['tau'], **{k: so[k] for k in so if k not in ('y', 'tau', 'bs')})
      ek = O.so_ekman(p, b, so['bs']) / 1e6
      width = np.array([max(p.y[-1] - O.so_outcrop(bi, p.y, so['bs']), 0.1) for bi in b])
      target, n2 = p.KGM * z / width * p.L, O.so_n2(z, b)
      rhs = lambda x, s: np.vstack((s[1], np.interp(x, z, n2) / p.c**2. * (s[0] - np.interp(x, z, target))))
      ends = lambda sa, sb: np.array([sa[0] + ek[0] * 1e6, sb[0] + ek[-1] * 1e6])
      zz = np.unique(np.concatenate([z, 0.5 * (z[1:] + z[:-1])]))
      res = integrate.solve_bvp(rhs, ends, zz, np.zeros((2, zz.size)), tol=bvp_tol, max_nodes=2000000)
      gm = res.sol(z)[0] / 1e6
      blocked = width > p.y[-1] - p.y[0]
      gm[blocked] = np.maximum(gm[blocked], -ek[blocked])
      worst = max(worst, relmax(got['Psi_GM'][m], gm))
  assert worst < tol, worst
  return worst


def twcol_sizes(backend):
  """The several-members-per-warp kernel of the column + thermal-wind topology (pmoc_twcol.cu): every group width /
  levels-per-lane variant, member counts that leave groups and warps partly empty, K > 1, split launches bit for
  bit, against the live oracle."""
  import warnings

  from oracle import pymoc_oracle as O
  from pymoc_b200 import configs
  warnings.filterwarnings('ignore')
  worst = 0.0
  for nz, M, K in ((24, 9, 1), (40, 5, 1), (56, 3, 2), (70, 7, 1), (73, 3, 1), (100, 3, 1), (128, 5, 7), (144, 2, 1)):
    spec = configs.c1_timestepping(M, nz=nz)
    spec.dt = spec.dt * min(1., (70. / nz)**2)  # the script's 60 days is diffusively stable up to nz ~ 78
    spec.K = K
    ens = Ensemble(spec, backend=backend)
    ens.run(50)
    got = {**ens.state(), **ens.diagnostics()}
    cut = Ensemble(spec, backend=backend)
    cut.run(13)
    cut.run(37)
    assert np.array_equal(cut.state()['b_basin'], got['b_basin']) and np.array_equal(cut.diagnostics()['Psi_tw'], got['Psi_tw'])
    assert not got['status'].any()
    for m in range(M):
      want = O.run_coupled(spec.member_case(m), 50, O.REFERENCE)
      for key in ('b_basin', 'Psi_tw'):
        err = relmax(got[key][m], want[key])
        worst = max(worst, err)
        assert err < TOL, (nz, M, K, m, key, err)
  # the tabulated path: a stretched grid, and a uniform grid with a level-dependent area (mixed with uniform members)
  from pymoc_b200.spec import ColumnSpec, ModelSpec, ThermwindSpec
  for which in ('stretched', 'area'):
    nz, M = 60, 6
    z = -3500. * (1. - np.linspace(0, 1, nz)**0.8) if which == 'stretched' else np.asarray(np.linspace(-3500, 0, nz))
    z[-1] = 0.
    kap = (1e-5 + 3e-5 * np.exp(z / 100) + 3e-4 * np.exp(-z / 1000 - 4))[None, :] * np.linspace(0.5, 1., M)[:, None]
    area = np.full((M, nz), 8e13)
    if which == 'area':
      area[1::2] *= (1. + 0.3 * z / 3500.)[None, :]  # odd members: area shrinking with depth
    dz_min = np.diff(z).min()
    spec = ModelSpec(M=M, z=z, dt=0.3 * dz_min**2 / kap.max(), K=1,
                     basin=ColumnSpec.build(z, kap, area, 0.03, 0.03 * np.exp(z / 300.) - 4e-4, bbot=-4e-4),
                     tw=ThermwindSpec.build(z, f=1.2e-4, b2=0. * z), order='post', iso=False)
    ens = Ensemble(spec, backend=backend)
    ens.run(40)
    got = {**ens.state(), **ens.diagnostics()}
    for m in range(M):
      want = O.run_coupled(spec.member_case(m), 40, O.REFERENCE)
      for key in ('b_basin', 'Psi_tw'):
        err = relmax(got[key][m], want[key])
        worst = max(worst, err)
        assert err < TOL, (which, m, key, err)
  return worst
