"""Runs to equilibrium through the host-buffer entry points (HostEnsemble.run_to_equilibrium, the stateless
pmoc_model_equilibrate_host) on cuda:0 with pinned host buffers: against Ensemble.run_to_equilibrium on device
buffers, bit for bit (run with -s for the tolerances and stops)."""
import numpy as np
import pytest

import equilibrium_matrix as eq
import host_equilibrium_matrix as hm
import kernel_matrix as km

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def cuda():
  from pymoc_b200.backend import CudaBackend
  return CudaBackend()


@pytest.fixture(scope='module')
def pinned():
  from pymoc_b200.backend import PinnedHostBackend
  return PinnedHostBackend()


@pytest.mark.parametrize('name', hm.NAMES)
def test_exact(cuda, pinned, monkeypatch, name):
  hm.exact(cuda, pinned, monkeypatch, name)


@pytest.mark.parametrize('name', ['c3', 'c4'])
def test_push_pull(cuda, pinned, monkeypatch, name):
  hm.push_pull(cuda, pinned, monkeypatch, name)


@pytest.mark.parametrize('name', ['c3', 'c4'])
def test_invalid_arguments(cuda, pinned, name):
  hm.invalid_arguments(cuda, pinned, name)


def test_refusals(cuda, pinned):
  hm.refusals(cuda, pinned)


def test_nonfinite_member(cuda, pinned, monkeypatch):
  hm.nonfinite_member(cuda, pinned, monkeypatch)


def test_c4_lattice(cuda, pinned):
  """C4 at 4 096 members, checked every 1 200 iterations up to 12 000 at tol = 1e-4: the handle equals the device
  path bit for bit."""
  from pymoc_b200 import configs
  from pymoc_b200.ensemble import Ensemble, HostEnsemble
  spec = configs.c4_jansen_nadeau(4096)
  dev = Ensemble(spec, backend=cuda)
  want = dev.run_to_equilibrium(12000, 1200, 1e-4)
  host = HostEnsemble(spec, backend=pinned)
  got = host.run_to_equilibrium(12000, 1200, 1e-4)
  assert np.array_equal(want['stopped_at'], got['stopped_at']) and np.array_equal(want['converged'], got['converged'])
  km._same(eq.fields(dev), eq.fields(host), 'C4 lattice')
  print('C4 lattice: %d distinct stops, %.3f converged' % (len(set(want['stopped_at'].tolist())), want['converged'].mean()))
  host.close()
