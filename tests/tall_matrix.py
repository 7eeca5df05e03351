"""The block-per-member kernels of the 'post' loop order (256 < nz <= 4096) against the reference, shared by the
CPU (warp-emulator) and GPU test files.

The five explicit 'post' topologies of ``launch_model`` (column + thermal wind, column + Psi_SO, column + thermal
wind + Psi_SO, two columns, two columns + Psi_SO) run above one warp's 256 levels on ``k_wide_post`` (the steps) and
``k_wide_refresh`` (the diagnosis), which the host loop alternates.  Cells reuse ``kernel_matrix``: five members of
an eight-member lattice, K = 3, 7 steps across two diagnoses, every field the oracle returns at 1e-10.
"""
import ctypes
import dataclasses

import numpy as np
import pytest

import kernel_matrix as km
from pymoc_b200 import _abi, configs
from pymoc_b200.ensemble import Ensemble, HostEnsemble

TOPOLOGIES = ('tw', 'so', 'tw_so', 'twocol', 'c3')
# the first size above the warp kernels, then both sides of each levels-per-thread boundary (4 | 8 | 16)
SIZES = (257, 1024, 1025, 2048, 2049, 4096)
CELLS = [(name, nz) for name in TOPOLOGIES for nz in SIZES]
VARIANT_SIZES = (257, 1025)
VARIANTS = ('c1_k1', 'c1_convecting', 'c2_bzbot', 'c2_stretched')
REFUSED = "EUNSUPPORTED: nz > 256: only the 'jn' topology and the explicit 'post' topologies"
SMEM_PER_BLOCK = km.SMEM_PER_BLOCK
WIDE_THREADS = 256


def split_launches(backend, name, nz):
  """Launches cut at a diagnosis iteration (K) and between two diagnoses (K + 2) equal one launch bit for bit."""
  spec, _ = km.cell(name, nz)
  km._same(km._run(backend, spec, [km.NSTEPS]),
           km._run(backend, spec, [km.CUTS[0], km.CUTS[1] - km.CUTS[0], km.NSTEPS - km.CUTS[1]]),
           (name, nz, 'split launches'))


# ------------------------------------------------------------------------------------------------ variants
def _on_grid(spec, z):
  """``spec`` on the grid ``z`` (same end points): every z-profile interpolated."""
  z0 = spec.z
  on_z = lambda a: np.ascontiguousarray(np.apply_along_axis(lambda r: np.interp(z, z0, r), -1, a))
  col = lambda c: None if c is None else dataclasses.replace(c, kappa=on_z(c.kappa), Area=on_z(c.Area), b0=on_z(c.b0))
  tw = spec.tw if spec.tw is None or spec.tw.b2 is None else dataclasses.replace(spec.tw, b2=on_z(spec.tw.b2))
  return dataclasses.replace(spec, z=z, basin=col(spec.basin), north=col(spec.north), pac=col(spec.pac), tw=tw)


def variant(name, nz):
  """C1 at the script's own K = 1; C1 with a convecting basin (unstable at the top at first); C2 with a gradient
  bottom condition (bzbot); C2 on a stretched grid (levels from 1.3 to 0.7 times the uniform spacing, with a
  depth-dependent Area so that the non-uniform Area path runs too)."""
  base = 'tw' if name.startswith('c1') else 'so'
  spec, env = km.cell(base, nz)
  if name == 'c1_k1':
    spec.K = 1
  elif name == 'c1_convecting':
    b0 = np.array(spec.basin.b0, dtype=np.float64, copy=True)
    b0[..., -max(3, nz // 40):] += 0.004  # above bs: convects in the first step
    spec = dataclasses.replace(spec, basin=dataclasses.replace(spec.basin, do_conv=True, b0=b0))
  elif name == 'c2_bzbot':
    spec = dataclasses.replace(spec, basin=dataclasses.replace(spec.basin, bzbot=np.array([2e-7])))
  elif name == 'c2_stretched':
    s = np.linspace(0., 1., nz)
    z = spec.z[0] + (spec.z[-1] - spec.z[0]) * (s + 0.3 * np.sin(np.pi * s) / np.pi)
    spec = _on_grid(spec, z)
    spec = dataclasses.replace(spec, dt=spec.dt * 0.45,
                               basin=dataclasses.replace(spec.basin, Area=6e13 * (1. + 0.2 * z / 4000.)[None, :]))
  else:
    raise KeyError(name)
  return spec, env


def variant_cell(backend, pool, name, nz):
  spec, _ = variant(name, nz)
  cases = [spec.member_case(m) for m in range(spec.M)]
  pending = pool.map_async(km.oracle_task, [(c, km.NSTEPS, False) for c in cases], chunksize=1)
  got = km._run(backend, spec, [km.NSTEPS])
  worst, excused = 0.0, 0
  for m, want in enumerate(pending.get()):
    if got['status'][m] & _abi.ST_PARITY_UNDEFINED:
      excused += 1
      continue
    assert not isinstance(want, str), (name, nz, m, want)
    assert not got['status'][m] & (_abi.ST_NAN | _abi.ST_BRENT_SIGN), (name, nz, m, int(got['status'][m]))
    for key, w in want.items():
      err = km.relmax(got[key][m], w)
      worst = max(worst, err)
      assert err < km.TOL, '%s nz=%d member %d field %s: rel err %.3e' % (name, nz, m, key, err)
  assert spec.M - excused >= 4, ('vacuous cell', name, nz, excused)
  print('tall variant %-14s nz=%4d worst %.2e excused %d' % (name, nz, worst, excused))
  return worst


# ------------------------------------------------------------------------------------------------ host buffers
def host_entry_points(backend, host_backend, nz):
  """C3 on nz levels, 16 members, K = 3, 13 + 17 steps: pmoc_model_run_host (stateless) and the persistent handle
  (HostEnsemble) equal Ensemble.run bit for bit.  ``host_backend``: a backend whose buffers are host memory."""
  spec = km.regrid(configs.c3_twocol_so(16, axes=(2, 2, 2, 2)), nz)
  spec.K = 3
  dev = Ensemble(spec, backend=backend)
  dev.run(30)
  want = {**dev.state(), **dev.diagnostics()}
  host = Ensemble(spec, backend=host_backend)
  for it0, n in ((0, 13), (13, 17)):
    _abi.check(host.lib, host.lib.pmoc_model_run_host(ctypes.byref(host.model), it0, n))
  km._same(want, {**host.state(), **host.diagnostics()}, ('pmoc_model_run_host', nz))
  h = HostEnsemble(spec, backend=host_backend)
  h.run(13, pull=0)
  h.run(17)
  km._same(want, {**h.state(), **h.diagnostics()}, ('HostEnsemble', nz))
  h.close()
  assert not want['status'].any() and np.isfinite(want['b_basin']).all()


# ------------------------------------------------------------------------------------------------ refusals
def refresh_smem(nz, ny, nb):
  """Dynamic shared memory of the block-per-member diagnosis (pmoc_wide.cu wide_refresh_smem): six level arrays,
  psib[nb] and its class counters, the reductions, bs / 1/slope / y on the channel grid."""
  nbp, nyp = (nb + 3) & ~3, (ny + 3) & ~3
  return 8 * (6 * nz + nbp + nbp // 2 + 2 + 64 + WIDE_THREADS + 3 * nyp + 4)


def refusals(backend):
  """F2010 (C3 and C2), a wind stress on y, a diagnosis that overflows shared memory, nz > 4096 and the two-basin
  topology above 256 levels are refused with EUNSUPPORTED."""
  for spec in (km._with_f2010(km.cell('c3', 257)[0]), km._with_f2010(km.cell('so', 257)[0])):
    with pytest.raises(_abi.PmocError, match=REFUSED):
      Ensemble(spec, backend=backend).run(3)
  spec, _ = km.cell('so', 257)
  tau = np.asarray(spec.so.tau, dtype=np.float64).reshape(-1)[:1, None] * np.sin(np.pi * spec.so.y / spec.so.y[-1])[None]
  spec = dataclasses.replace(spec, so=dataclasses.replace(spec.so, tau=tau))
  with pytest.raises(_abi.PmocError, match=REFUSED):
    Ensemble(spec, backend=backend).run(3)

  spec, _ = km.cell('c3', 4096)
  ny = spec.so.y.size
  nb = 2
  while refresh_smem(4096, ny, nb + 1) <= SMEM_PER_BLOCK:
    nb += 1
  spec.nb = nb
  Ensemble(spec, backend=backend).diagnose()  # the largest fitting nb runs
  spec.nb = nb + 1
  with pytest.raises(_abi.PmocError, match='EUNSUPPORTED: nz = 4096, nb = %d' % (nb + 1)):
    Ensemble(spec, backend=backend).diagnose()

  spec, _ = km.cell('c3', 4097)
  with pytest.raises(_abi.PmocError, match='EUNSUPPORTED: nz > 4096'):
    Ensemble(spec, backend=backend).run(3)
  with configs.members(0, 2):
    spec = km.regrid(configs.twobasin(8), 257)
  with pytest.raises(_abi.PmocError, match='EUNSUPPORTED: the two-basin topology needs nz <= 256'):
    Ensemble(spec, backend=backend).run(3)
  return nb
