"""Every kernel family on stretched grids, depth-dependent areas, Psi_SO tapers and per-member parameters, on the CPU
warp emulator (config_matrix): the warp kernel at 64 and 256 levels (F2010 at 64), k_twcol, the block-per-member
kernels at 257 levels, and the per-module entry points on a stretched grid."""
import pytest

import config_matrix as cm
import kernel_matrix as km
from emu.emu_backend import EmuBackend
from pymoc_b200.modules import _dispatch

CELLS = cm.cells('emu')


@pytest.fixture(scope='module')
def emu():
  be = EmuBackend()
  _dispatch._set_backend(be)
  yield be
  _dispatch._set_backend(None)


@pytest.fixture(scope='module')
def oracle():
  with km.oracle_pool() as p:
    yield cm.Oracle(p)


@pytest.mark.parametrize('family,name,nz,variant,late', CELLS, ids=[cm.cell_id(c) for c in CELLS])
def test_config_cell(emu, oracle, monkeypatch, family, name, nz, variant, late):
  cm.config_cell(emu, oracle, monkeypatch, family, name, nz, variant, late)


def test_cells_cover_every_family_and_variant():
  cm.covers_every_pair('emu')


def test_column_stretched(emu):
  cm.column_stretched(emu)


def test_thermwind_stretched(emu):
  cm.thermwind_stretched(emu)


def test_so_stretched_with_tapers(emu, oracle):
  cm.so_stretched(emu, oracle.pool, cm.MODULE_SO_SIZES['emu'])
