"""The block-per-member kernels of the 'post' loop order (256 < nz <= 4096) on cuda:0, every size (run with -s for
the per-cell report)."""
import pytest

import kernel_matrix as km
import tall_matrix as tm

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


@pytest.mark.parametrize('name,nz', tm.CELLS)
def test_tall_cell(cuda, pool, monkeypatch, name, nz):
  km.fused_cell(cuda, pool, monkeypatch, name, nz, bitwise=False)


@pytest.mark.parametrize('name,nz', tm.CELLS)
def test_tall_split_launches(cuda, name, nz):
  tm.split_launches(cuda, name, nz)


@pytest.mark.parametrize('nz', tm.VARIANT_SIZES)
@pytest.mark.parametrize('name', tm.VARIANTS)
def test_tall_variant(cuda, pool, name, nz):
  tm.variant_cell(cuda, pool, name, nz)


@pytest.mark.parametrize('nz', (257, 1024))
def test_tall_host_entry_points(cuda, nz):
  from pymoc_b200.backend import PinnedHostBackend
  tm.host_entry_points(cuda, PinnedHostBackend(), nz)


def test_tall_refusals(cuda):
  print('largest nb of the diagnosis at nz = 4096: %d' % tm.refusals(cuda))
