"""Host-buffer entry points on the GPU-less build box (CPU only).

pmoc_model_run_host and the pmoc_host_open / step / close handle run their device mirror, copies and block loop
through the warp emulator, whose build stands host calls in for the CUDA runtime (tests/emu/pmoc_emu.h) and
splits the members into blocks of two, pipelined over the three streams.  Results are compared bit for bit with
the device path (Ensemble.run), and the bytes each call moves with the sizes of the ensemble's host buffers.
"""
import ctypes

import numpy as np
import pytest

from emu.emu_backend import EmuBackend
from pymoc_b200 import _abi, configs
from pymoc_b200.ensemble import Ensemble, HostEnsemble

S, P, D = HostEnsemble.IO_STATE, HostEnsemble.IO_PSI, HostEnsemble.IO_DIAG

# 16 members = eight blocks; C4 (K = 12) crosses diagnoses at 12 and 24 in 13 + 17 steps; C5 at nz = 320 runs the
# block-per-member kernels, whose scratch the library allocates per stream (four blocks, stream 0 used twice)
SPECS = {
    'c1': lambda: configs.c1_timestepping(16),
    'c3': lambda: configs.c3_twocol_so(16, axes=(2, 2, 2, 2)),
    'c4': lambda: configs.c4_jansen_nadeau(16, axes=(2, 2, 2, 2, 1)),
    'c5_320': lambda: configs.c5_single_global_basin(8, nz=320, dt_days=1., axes=(2, 2, 2, 1), kapfac_max=1.),
    'twobasin': lambda: configs.twobasin(16, axes=(4, 2, 2)),
}


@pytest.fixture(scope='module')
def emu():
  return EmuBackend()


def _assert_same(want, got, name):
  for part in ('state', 'diagnostics'):
    a, b = getattr(want, part)(), getattr(got, part)()
    assert a.keys() == b.keys()
    for key in a:
      assert np.array_equal(a[key], b[key], equal_nan=True), (name, key)


def _run_host(ens, it0, nsteps):
  """pmoc_model_run_host on the ensemble's host arrays; the (host->device, device->host) bytes it moved."""
  _abi.check(ens.lib, ens.lib.pmoc_model_run_host(ctypes.byref(ens.model), it0, nsteps))
  h2d, d2h = ctypes.c_uint64(), ctypes.c_uint64()
  ens.lib.pmoc_host_last_bytes(ctypes.byref(h2d), ctypes.byref(d2h))
  return h2d.value, d2h.value


def _classes(ens):
  """PMOC_IO_* class of each per-member host buffer of the ensemble."""
  state = ('b_basin', 'b_north', 'b_pac', 'bs_ml', 'bbot_basin', 'bbot_north', 'bbot_pac', 'var_basin', 'var_north',
           'var_pac', 'status')
  carried = ('Psi_iso_b', 'Psi_iso_n', 'Psi_so', 'Psi_zon_a', 'Psi_zon_p', 'Psi_so2') + (() if ens.spec.iso else ('Psi_tw',))
  return {key: S if key in state else P if key in carried else D
          for key in ens._bufs if key != 'scratch'}  # (the library allocates its own scratch)


def _sizes(ens):
  """Bytes of the ensemble's host buffers: 'param' (grids, tapers and parameter vectors), per PMOC_IO_* class, and
  'Psi_s' (the mixed layer's streamfunction, a diagnostic that every stepping launch writes)."""
  n = {'param': sum(b.nbytes for b in ens._keep), S: 0, P: 0, D: 0, 'Psi_s': 0}
  for key, cls in _classes(ens).items():
    n[cls] += ens._bufs[key].nbytes
  if 'Psi_s' in ens._bufs:
    n['Psi_s'] = ens._bufs['Psi_s'].nbytes
  return n


@pytest.mark.parametrize('name', ['c3', 'c4', 'c5_320', 'twobasin'])
def test_host_buffer_entry_point(emu, name):
  """pmoc_model_run_host (host pointers, copies inside) == device path, bit for bit."""
  spec = SPECS[name]()
  dev = Ensemble(spec, backend=emu)
  dev.run(30)
  host = Ensemble(spec, backend=emu)
  _run_host(host, 0, 13)
  _run_host(host, 13, 17)
  _assert_same(dev, host, name)


@pytest.mark.parametrize('name', ['c3', 'c4', 'c5_320', 'twobasin'])
def test_host_handle_matches_device_path(emu, name):
  """The persistent handle == device path, bit for bit: with nothing pulled between calls, and with state +
  streamfunctions pulled and pushed back every call."""
  spec = SPECS[name]()
  dev = Ensemble(spec, backend=emu)
  dev.run(30)
  a = HostEnsemble(spec, backend=emu)
  a.run(13, pull=0)
  assert a.last_bytes() == (0, 0)  # nothing moved: parameters and state are resident
  a.run(17, pull=S | P | D)
  b = HostEnsemble(spec, backend=emu)
  b.run(13, pull=S | P)
  b.run(17, push=S | P, pull=S | P | D)  # the host copy is the truth: up, 17 steps, down
  for ens in (a, b):
    _assert_same(dev, ens, name)
    ens.close()


def test_stateless_bytes_post_order(emu):
  """Order 'post' (C3, K = 24): the state and the parameters go up every call, the carried streamfunctions when
  it0 > 0; the diagnostics come back when the call diagnoses (pre-loop at it0 == 0, or an iteration it % K == 0)."""
  ens = Ensemble(SPECS['c3'](), backend=emu)
  n = _sizes(ens)
  assert _run_host(ens, 0, 5) == (n['param'] + n[S], n[S] + n[P] + n[D])
  assert _run_host(ens, 5, 3) == (n['param'] + n[S] + n[P], n[S])
  assert _run_host(ens, 8, 20) == (n['param'] + n[S] + n[P], n[S] + n[P] + n[D])  # diagnosis at 24
  assert _run_host(ens, 28, 0) == (n['param'] + n[S] + n[P], n[S])


def test_stateless_bytes_jn_order(emu):
  """Order 'jn' (C4, K = 12): the streamfunctions are carried in unless the launch starts with a diagnosis
  (it0 % K == 0); the mixed layer's Psi_s comes back from every launch that steps."""
  ens = Ensemble(SPECS['c4'](), backend=emu)
  n = _sizes(ens)
  assert n['Psi_s'] > 0
  assert _run_host(ens, 0, 5) == (n['param'] + n[S], n[S] + n[P] + n[D])
  assert _run_host(ens, 5, 3) == (n['param'] + n[S] + n[P], n[S] + n['Psi_s'])
  assert _run_host(ens, 8, 6) == (n['param'] + n[S] + n[P], n[S] + n[P] + n[D])  # diagnosis at 12
  assert _run_host(ens, 14, 0) == (n['param'] + n[S] + n[P], n[S])
  assert _run_host(ens, 24, 2) == (n['param'] + n[S], n[S] + n[P] + n[D])


@pytest.mark.parametrize('name', ['c1', 'c3', 'c4', 'twobasin'])
def test_host_handle_bytes_per_class(emu, name):
  """pmoc_host_open uploads grids, parameters, state and carried streamfunctions; pmoc_host_step moves exactly
  the classes asked for (C1: Psi_tw is carried, without the isopycnal remap)."""
  ens = HostEnsemble(SPECS[name](), backend=emu)
  n = _sizes(ens)
  assert ens.last_bytes() == (n['param'] + n[S] + n[P], 0)
  for push, pull in ((0, 0), (S, 0), (P, 0), (0, S), (0, P), (0, D), (S | P, S | P | D)):
    ens.run(2, push=push, pull=pull)
    assert ens.last_bytes() == (sum(n[c] for c in (S, P) if push & c), sum(n[c] for c in (S, P, D) if pull & c)), (push, pull)
  ens.close()


def test_host_handle_diagnostics_start_at_zero(emu):
  """pmoc_host_open zeroes the device copies of the arrays it does not upload: diagnostics pulled before any
  launch wrote them read as zeros (order 'jn': a call without steps does not diagnose)."""
  ens = HostEnsemble(SPECS['c4'](), backend=emu)
  diags = [key for key, cls in _classes(ens).items() if cls == D]
  assert 'Psi_s' in diags and 'psib' in diags
  for key in diags:
    ens._bufs[key][...] = 1.
  ens.run(0, pull=D)
  for key in diags:
    assert not ens._bufs[key].any(), key
  ens.close()
