"""The block-per-member kernels of the 'post' loop order (256 < nz <= 4096) on the CPU warp emulator: the same
cells, split launches, variants and refusals as the GPU file (test_gpu_tall.py); the host-buffer entry points at
nz = 257 only."""
import pytest

import kernel_matrix as km
import tall_matrix as tm
from emu.emu_backend import EmuBackend
from pymoc_b200.modules import _dispatch

@pytest.fixture(scope='module')
def emu():
  be = EmuBackend()
  _dispatch._set_backend(be)
  yield be
  _dispatch._set_backend(None)


@pytest.fixture(scope='module')
def pool():
  with km.oracle_pool() as p:
    yield p


@pytest.mark.parametrize('name,nz', tm.CELLS)
def test_tall_cell(emu, pool, monkeypatch, name, nz):
  km.fused_cell(emu, pool, monkeypatch, name, nz, bitwise=False)


@pytest.mark.parametrize('name,nz', tm.CELLS)
def test_tall_split_launches(emu, name, nz):
  tm.split_launches(emu, name, nz)


@pytest.mark.parametrize('nz', tm.VARIANT_SIZES)
@pytest.mark.parametrize('name', tm.VARIANTS)
def test_tall_variant(emu, pool, name, nz):
  tm.variant_cell(emu, pool, name, nz)


def test_tall_host_entry_points(emu):
  tm.host_entry_points(emu, emu, 257)


def test_tall_refusals(emu):
  tm.refusals(emu)
