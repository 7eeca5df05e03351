"""Member lists and runs to equilibrium, shared by the CPU (warp-emulator) and GPU test files.

``pmoc_model_run_members`` steps a gapped, shuffled subset of an ensemble: the listed members must equal
``Ensemble.run`` bit for bit in every field, the others stay byte-identical.  ``pmoc_model_equilibrate``
(``Ensemble.run_to_equilibrium``) must stop each member where numpy, looking at fixed-length runs cut at every
check, says it stops, leave it exactly as ``run`` to that iteration does, and let ``run`` continue every member from
its own stop.  Topologies: every cell of the warp kernel's matrix (``kernel_matrix``), the several-members-per-warp
kernel of the column + thermal wind model, and the block-per-member kernels of both orders above 256 levels.
"""
import ctypes
import dataclasses

import numpy as np
import pytest

import kernel_matrix as km
from pymoc_b200 import _abi, configs
from pymoc_b200.ensemble import Ensemble

STATE = ('b_basin', 'b_north', 'b_pac', 'bs_ml')
TALL = [(name, nz) for name in ('tw', 'so', 'tw_so', 'twocol', 'c3', 'jn') for nz in (257, 1025)]
TWCOL_NZ = (40, 70, 144)  # k_twcol's 8-lane groups (up to 72 levels) with 5 and 9 levels per lane, 16-lane groups
EVERY_K = 2  # checks every 2 K iterations ...
CHECKS = 8   # ... up to 8 of them
STAGGER = 4  # member m starts STAGGER * m checks into its spin-up


# ------------------------------------------------------------------------------------------------ helpers
def fields(ens):
  """Every field of state() and diagnostics(), the raw status word (with its internal carry bits) included."""
  out = {**ens.state(), **ens.diagnostics()}
  out['status_raw'] = ens.be.download(ens.buffer('status')).view(np.uint32)
  return out


def fresh(backend, spec, env, monkeypatch):
  for k, v in env.items():
    monkeypatch.setenv(k, v)
  ens = Ensemble(spec, backend=backend)
  if spec.order == 'post':
    ens.diagnose()
  return ens


def run_members(ens, members, it0, nsteps):
  lst = ens.be.upload(np.asarray(members, dtype=np.int64))
  rc = ens.lib.pmoc_model_run_members(ctypes.byref(ens.model), ens.be.ptr(lst) if len(members) else None,
                                      len(members), it0, nsteps, ens.be.stream())
  _abi.check(ens.lib, rc)
  ens.be.sync()


def gapped_subset(M, seed):
  """A shuffled subset with gaps: about half the members, never all, never neighbours only."""
  rng = np.random.default_rng(seed)
  keep = [m for m in range(M) if rng.random() < 0.55]
  if len(keep) < 2:
    keep = [0, M - 1]
  if len(keep) == M:
    keep = keep[::2]
  rng.shuffle(keep)
  return [int(m) for m in keep]


def twcol_spec(nz):
  """Column + thermal wind on nz <= 144 levels, 12 members, K = 3, on the several-members-per-warp kernel.  Member 5
  has a depth-dependent Area: the warp of a full run that holds it (members 4..7 with four members per warp, 4 and 5
  with two) takes the tabulated path, the others the uniform one, so a list that mixes them exercises both paths in
  one warp."""
  with configs.members(0, 12):
    spec = configs.c1_timestepping(12, nz=nz)
  spec.dt *= (69. / (nz - 1))**2
  spec.K = 3
  area = np.repeat(np.asarray(spec.basin.Area, dtype=np.float64).reshape(1, -1), spec.M, axis=0)
  area[5] *= 1. + 0.2 * spec.z / 4000.
  return dataclasses.replace(spec, basin=dataclasses.replace(spec.basin, Area=area))


def spec_of(name, nz):
  if name == 'twcol_kernel':
    return twcol_spec(nz), {}
  return km.cell(name, nz)


def _same_rows(a, b, rows, what):
  for k in a:
    for m in rows:
      assert np.array_equal(a[k][m], b[k][m], equal_nan=True), (what, k, m)


# ------------------------------------------------------------------------------------------------ member lists
def subset_exact(backend, monkeypatch, name, nz, seed=1):
  """A gapped, shuffled subset stepped by pmoc_model_run_members (two launches, cut between two diagnoses) equals
  Ensemble.run for its members and leaves the others byte-identical; an empty list changes nothing; the full list
  in identity order equals Ensemble.run."""
  spec, env = spec_of(name, nz)
  nsteps = km.NSTEPS
  ref = fresh(backend, spec, env, monkeypatch)
  ref.run(nsteps)
  want = fields(ref)

  ens = fresh(backend, spec, env, monkeypatch)
  before = fields(ens)
  sub = gapped_subset(spec.M, seed)
  run_members(ens, sub, 0, km.CUTS[1])
  run_members(ens, sub, km.CUTS[1], nsteps - km.CUTS[1])
  got = fields(ens)
  assert got.keys() == want.keys()
  _same_rows(got, want, sub, (name, nz, 'listed member'))
  _same_rows(got, before, [m for m in range(spec.M) if m not in sub], (name, nz, 'unlisted member'))

  run_members(ens, [], 0, nsteps)
  km._same(got, fields(ens), (name, nz, 'empty list'))

  ens = fresh(backend, spec, env, monkeypatch)
  run_members(ens, list(range(spec.M)), 0, nsteps)
  km._same(want, fields(ens), (name, nz, 'full list'))
  return sub


# ------------------------------------------------------------------------------------------------ equilibrium
def numpy_stops(snaps, tol, it_of):
  """(stopped_at, converged) as numpy decides them from the states at every check (snaps[0]: the start)."""
  M = snaps[0]['b_basin'].shape[0]
  stopped, conv = np.full(M, it_of(len(snaps) - 1), dtype=np.int64), np.zeros(M, dtype=bool)
  for m in range(M):
    for c in range(1, len(snaps)):
      keys = [k for k in STATE if k in snaps[c]]
      now = np.concatenate([snaps[c][k][m].ravel() for k in keys])
      prev = np.concatenate([snaps[c - 1][k][m].ravel() for k in keys])
      bad = not np.isfinite(now).all()
      with np.errstate(invalid='ignore'):
        moved = not (np.abs(now - prev) <= tol).all()
      if bad or not moved:
        stopped[m], conv[m] = it_of(c), not bad
        break
  return stopped, conv


def staggered(backend, spec, env, monkeypatch, every):
  """A fresh ensemble whose member m has run STAGGER * m * every iterations (lists of the members still behind).  The
  members of a test lattice relax at nearly the same rate; staggered, they reach any tolerance at different checks.
  Every member's count is a multiple of K, so the ensemble runs on from iteration 0 (the loop reads the counter
  modulo K)."""
  ens = fresh(backend, spec, env, monkeypatch)
  n = STAGGER * every
  for r in range(spec.M - 1):
    run_members(ens, list(range(r + 1, spec.M)), r * n, n)
  return ens


def reference_checks(backend, spec, env, monkeypatch, every, checks, start=fresh):
  """Fixed-length run cut at every check: the fields after 0, every, 2 every, ... iterations."""
  ens = start(backend, spec, env, monkeypatch) if start is fresh else start(backend, spec, env, monkeypatch, every)
  snaps = [fields(ens)]
  for _ in range(checks):
    ens.run(every)
    snaps.append(fields(ens))
  return snaps


def pick_tol(snaps, it_of):
  """A tolerance under which at least three different stop iterations occur and at least one member never
  converges, from the per-member movement between checks of the reference run."""
  cands = set()
  for c in range(1, len(snaps)):
    keys = [k for k in STATE if k in snaps[c]]
    for m in range(snaps[0]['b_basin'].shape[0]):
      d = np.abs(np.concatenate([snaps[c][k][m].ravel() - snaps[c - 1][k][m].ravel() for k in keys]))
      if np.isfinite(d).all():
        cands.add(float(d.max()))
  best = None
  for tol in sorted(cands):
    stopped, conv = numpy_stops(snaps, tol, it_of)
    if len(set(stopped.tolist())) >= 3 and not conv.all():
      score = (len(set(stopped.tolist())), int(conv.sum()))
      if best is None or score > best[0]:
        best = (score, tol)
  assert best is not None, 'no tolerance gives three stop iterations and a member that never converges'
  return best[1]


def equilibrate_exact(backend, monkeypatch, name, nz, resume=None):
  spec, env = spec_of(name, nz)
  K = spec.K
  every, checks = EVERY_K * K, CHECKS
  it_of = lambda c: c * every
  snaps = reference_checks(backend, spec, env, monkeypatch, every, checks, start=staggered)
  tol = pick_tol(snaps, it_of)
  want_stop, want_conv = numpy_stops(snaps, tol, it_of)

  ens = staggered(backend, spec, env, monkeypatch, every)
  got = ens.run_to_equilibrium(every * checks, every, tol)
  assert ens.it == every * checks
  assert np.array_equal(got['stopped_at'], want_stop), (name, nz, got['stopped_at'], want_stop)
  assert np.array_equal(got['converged'], want_conv), (name, nz, got['converged'], want_conv)
  after = fields(ens)
  for m in range(spec.M):
    c = int(want_stop[m]) // every
    _same_rows(after, snaps[c], [m], (name, nz, 'frozen member', m, int(want_stop[m])))

  k = K + 1 if resume is None else resume  # crosses a diagnosis, ends between two
  ens.run(k)
  resumed = fields(ens)
  for s in sorted(set(want_stop.tolist())):
    fixed = staggered(backend, spec, env, monkeypatch, every)
    fixed.run(s + k)
    _same_rows(resumed, fields(fixed), [m for m in range(spec.M) if want_stop[m] == s],
               (name, nz, 'resumed member', s))
  print('equilibrate %-12s nz=%4d tol %.3e stops %s converged %s' % (
      name, nz, tol, got['stopped_at'].tolist(), got['converged'].astype(int).tolist()))
  return got


def nonfinite_member(backend, monkeypatch, name='so', nz=64):
  """Member 2 with a diffusivity 1e100 times its own (kappa dt / dz^2 far above 1/2: the explicit step blows up
  within a few iterations): stopped at the first check that sees a non-finite value, not converged; every other
  member runs on as in a fixed-length run."""
  spec, env = km.cell(name, nz)
  kap = np.repeat(np.asarray(spec.basin.kappa, dtype=np.float64), spec.M // np.shape(spec.basin.kappa)[0], axis=0)
  kap[2] *= 1e100
  spec = dataclasses.replace(spec, basin=dataclasses.replace(spec.basin, kappa=kap))
  every = EVERY_K * spec.K
  snaps = reference_checks(backend, spec, env, monkeypatch, every, 4)
  assert not np.isfinite(snaps[1]['b_basin'][2]).all()
  ens = fresh(backend, spec, env, monkeypatch)
  got = ens.run_to_equilibrium(4 * every, every, 0.0)
  assert got['stopped_at'][2] == every and not got['converged'][2], got
  assert fields(ens)['status'][2] & _abi.ST_NAN
  want_stop, want_conv = numpy_stops(snaps, 0.0, lambda c: c * every)
  assert np.array_equal(got['stopped_at'], want_stop) and np.array_equal(got['converged'], want_conv)
  after = fields(ens)
  _same_rows(after, snaps[-1], [m for m in range(spec.M) if m != 2], ('nonfinite', 'other members'))
  _same_rows(after, snaps[1], [2], ('nonfinite', 'stopped member'))


# ------------------------------------------------------------------------------------------------ arguments
def _call_equilibrate(ens, every, work_bytes=None, stopped=True, max_steps=None):
  need = int(ens.lib.pmoc_equilibrate_work_bytes(ctypes.byref(ens.model)))
  work = ens.be.upload(np.zeros((need + 7) // 8 + 1))
  st = ens.be.upload(np.zeros(ens.M, dtype=np.int64))
  cv = ens.be.upload(np.zeros(ens.M, dtype=np.uint8))
  return ens.lib.pmoc_model_equilibrate(ctypes.byref(ens.model), 0, every if max_steps is None else max_steps, every,
                                        0.0, ens.be.ptr(st) if stopped else None, ens.be.ptr(cv), ens.be.ptr(work),
                                        need if work_bytes is None else work_bytes, ens.be.stream())


def invalid_arguments(backend):
  """every not a multiple of K, max_steps not a multiple of K, a short work buffer, a NULL stopped_at: EINVAL, and
  nothing runs.  A NULL list with members, or more members than M: EINVAL."""
  spec, _ = km.cell('so', 64)
  ens = Ensemble(spec, backend=backend)
  ens.diagnose()
  before = fields(ens)
  K = spec.K
  need = int(ens.lib.pmoc_equilibrate_work_bytes(ctypes.byref(ens.model)))
  assert need == 8 * (1 + 2 * spec.M + spec.M * spec.nz)
  assert _call_equilibrate(ens, K + 1) == _abi.EINVAL
  assert 'multiple of K' in ens.lib.pmoc_last_error().decode()
  assert _call_equilibrate(ens, 2 * K, max_steps=2 * K + 1) == _abi.EINVAL
  assert _call_equilibrate(ens, 2 * K, work_bytes=need - 8) == _abi.EINVAL
  assert 'pmoc_equilibrate_work_bytes' in ens.lib.pmoc_last_error().decode()
  assert _call_equilibrate(ens, 2 * K, stopped=False) == _abi.EINVAL
  assert ens.lib.pmoc_model_run_members(ctypes.byref(ens.model), None, 2, 0, 3, ens.be.stream()) == _abi.EINVAL
  lst = ens.be.upload(np.arange(spec.M + 1, dtype=np.int64))
  assert ens.lib.pmoc_model_run_members(ctypes.byref(ens.model), ens.be.ptr(lst), spec.M + 1, 0, 3,
                                        ens.be.stream()) == _abi.EINVAL
  km._same(before, fields(ens), 'rejected calls changed the ensemble')
  assert _call_equilibrate(ens, 2 * K) == _abi.OK  # the same call with valid arguments runs


def _refused_specs():
  out = [km._with_f2010(km.cell('c3', 257)[0]), km._with_f2010(km.cell('so', 257)[0])]
  spec, _ = km.cell('so', 257)
  tau = np.asarray(spec.so.tau, dtype=np.float64).reshape(-1)[:1, None]
  tau = tau * np.sin(np.pi * spec.so.y / spec.so.y[-1])[None]
  out.append(dataclasses.replace(spec, so=dataclasses.replace(spec.so, tau=tau)))
  with configs.members(0, 2):
    out.append(km.regrid(configs.twobasin(8), 257))
  with configs.members(0, 2):
    out.append(km._with_f2010(configs.c5_single_global_basin(8, nz=320, dt_days=1., axes=(2, 2, 1, 2),
                                                             kapfac_max=1.)))
  return out


def refusals(backend):
  """Topologies pmoc_model_run refuses are refused by both new calls with the same code and text."""
  for spec in _refused_specs():
    ens = Ensemble(spec, backend=backend)
    K = spec.K
    rc = ens.lib.pmoc_model_run(ctypes.byref(ens.model), 0, 2 * K, ens.be.stream())
    text = ens.lib.pmoc_last_error().decode()
    assert rc == _abi.EUNSUPPORTED, (rc, text)
    lst = ens.be.upload(np.arange(spec.M, dtype=np.int64)[::-1].copy())
    rc2 = ens.lib.pmoc_model_run_members(ctypes.byref(ens.model), ens.be.ptr(lst), spec.M, 0, 2 * K, ens.be.stream())
    assert (rc2, ens.lib.pmoc_last_error().decode()) == (rc, text)
    rc3 = _call_equilibrate(ens, 2 * K)
    assert (rc3, ens.lib.pmoc_last_error().decode()) == (rc, text)
    with pytest.raises(_abi.PmocError, match='EUNSUPPORTED'):
      ens.run_to_equilibrium(2 * K, 2 * K, 0.0)
