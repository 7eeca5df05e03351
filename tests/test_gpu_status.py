"""Per-member status bits and the rare solver branches behind them on cuda:0, every size (run with -s for the
per-cell report)."""
import pytest

import kernel_matrix as km
import status_matrix as sm

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def cuda():
  from pymoc_b200.backend import CudaBackend
  from pymoc_b200.modules import _dispatch
  be = CudaBackend()
  _dispatch._set_backend(be)
  yield be
  _dispatch._set_backend(None)


@pytest.fixture(scope='module')
def pool():
  with km.oracle_pool() as p:
    yield p


@pytest.mark.parametrize('with_c', (False, True))
@pytest.mark.parametrize('nz', (64, 129, 256))
def test_so_bs_scan(cuda, pool, nz, with_c):
  print('so bs scan nz=%d F2010=%d: flagged as restated, worst %.2e' % (nz, with_c, sm.so_bs_scan(cuda, pool, nz, with_c)))


@pytest.mark.parametrize('nz', (64, 256))
def test_smoother_sweep(cuda, pool, nz):
  for label, err in sm.so_smoother_sweep(cuda, pool, nz).items():
    print('smoother nz=%d %-12s %.2e' % (nz, label, err))


def test_series_divergence_is_flagged(cuda):
  sm.so_series_diverges(cuda, 64)


def test_ml_index(cuda):
  sm.ml_index(cuda)


@pytest.mark.parametrize('nz', (64, 257, 1025))
def test_pushed_psi_noise_switch(cuda, nz):
  from pymoc_b200.backend import PinnedHostBackend
  print('pushed Psi nz=%d: %r' % (nz, sm.pushed_psi(cuda, PinnedHostBackend(), nz)))


@pytest.mark.parametrize('name,nz', [(n, z) for n in ('so', 'c3', 'jn') for z in (64, 129, 256, 257, 1025)])
def test_model_bs_scan(cuda, name, nz):
  from pymoc_b200.backend import PinnedHostBackend
  print('bs scan %s nz=%d: %r' % (name, nz, sm.model_bs_scan(cuda, PinnedHostBackend(), name, nz)))


@pytest.mark.parametrize('name,nz', [(n, z) for n in ('twocol', 'c3', 'jn') for z in (64, 256, 257, 1025)])
def test_model_tie_cell(cuda, name, nz):
  from pymoc_b200.backend import PinnedHostBackend
  print('tie cell %s nz=%d: %r' % (name, nz, sm.model_tie_cell(cuda, PinnedHostBackend(), name, nz)))


@pytest.mark.parametrize('name,nz,column', [('tw', 40, 'basin'), ('tw', 100, 'basin'), ('so', 64, 'basin'),
                                            ('so', 256, 'basin'), ('twocol', 64, 'north'), ('jn', 64, 'basin'),
                                            ('jn', 256, 'basin'), ('so', 257, 'basin'), ('so', 1025, 'basin'),
                                            ('so', 2049, 'basin'), ('twocol', 257, 'basin'), ('twocol', 257, 'north'),
                                            ('twocol', 1025, 'north'), ('twocol', 2049, 'north'), ('jn', 257, 'basin'),
                                            ('jn', 1025, 'basin')])
def test_model_nan(cuda, name, nz, column):
  from pymoc_b200.backend import PinnedHostBackend
  print('nan %s nz=%d %s: %r' % (name, nz, column, sm.model_nan(cuda, PinnedHostBackend(), name, nz, columns=(column,))))


@pytest.mark.parametrize('nz', (64, 256, 257, 1025))
def test_model_ml_index(cuda, pool, nz):
  from pymoc_b200.backend import PinnedHostBackend
  print('ml index jn nz=%d: %r' % (nz, sm.model_ml_index(cuda, PinnedHostBackend(), pool, nz)))
