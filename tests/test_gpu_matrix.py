"""Every fused-kernel instantiation and the batched per-module entry points on cuda:0 (run with -s for the
per-cell report)."""
import pytest

import kernel_matrix as km

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


@pytest.mark.parametrize('name,nz', km.CELLS)
def test_fused_kernel_cell(cuda, pool, monkeypatch, name, nz):
  km.fused_cell(cuda, pool, monkeypatch, name, nz, adaptive=True)


def test_matrix_covers_launch_model():
  km.matrix_is_complete()


def test_jn_f2010_above_256_levels_is_refused(cuda):
  km.jn_f2010_wide_refused(cuda)


def test_column_batched(cuda):
  print('column worst %.2e' % km.column_batched(cuda))


def test_thermwind_batched(cuda):
  print('thermwind worst %.2e' % km.thermwind_batched(cuda))


def test_psib_batched(cuda):
  print('psib worst %.2e' % km.psib_batched(cuda))


def test_so_batched(cuda, pool):
  print('so worst %r' % km.so_batched(cuda, pool))


def test_ml_batched(cuda):
  print('ml worst %.2e' % km.ml_batched(cuda))


def test_shared_memory_limits(cuda):
  print('largest nb %d, ny %d at nz = 256' % km.smem_limits(cuda))
