"""Every kernel family on stretched grids, depth-dependent areas, Psi_SO tapers and per-member parameters, on cuda:0
at every size of each family (config_matrix; run with -s for the per-cell report)."""
import pytest

import config_matrix as cm
import kernel_matrix as km

pytestmark = pytest.mark.gpu
CELLS = cm.cells('gpu')


@pytest.fixture(scope='module')
def cuda():
  from pymoc_b200.backend import CudaBackend
  from pymoc_b200.modules import _dispatch
  be = CudaBackend()
  _dispatch._set_backend(be)
  yield be
  _dispatch._set_backend(None)


@pytest.fixture(scope='module')
def oracle():
  with km.oracle_pool() as p:
    yield cm.Oracle(p)


@pytest.mark.parametrize('family,name,nz,variant,late', CELLS, ids=[cm.cell_id(c) for c in CELLS])
def test_config_cell(cuda, oracle, monkeypatch, family, name, nz, variant, late):
  cm.config_cell(cuda, oracle, monkeypatch, family, name, nz, variant, late)


def test_cells_cover_every_family_and_variant():
  cm.covers_every_pair('gpu')


def test_column_stretched(cuda):
  print('column stretched worst %.2e' % cm.column_stretched(cuda))


def test_thermwind_stretched(cuda):
  print('thermwind stretched worst %.2e' % cm.thermwind_stretched(cuda))


def test_so_stretched_with_tapers(cuda, oracle):
  print('so stretched worst %r' % cm.so_stretched(cuda, oracle.pool, cm.MODULE_SO_SIZES['gpu']))
