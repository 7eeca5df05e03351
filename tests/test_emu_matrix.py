"""Every fused-kernel instantiation and the batched per-module entry points on the CPU warp emulator."""
import pytest

import kernel_matrix as km
from emu.emu_backend import EmuBackend
from pymoc_b200.modules import _dispatch

# On the emulator, split launches and CTA packing are checked bit for bit at levels per lane 2, 5 and 8 only (each
# extra run costs seconds), and so are the F2010 smoother's cells and calls (their converged reference takes seconds
# of solve_bvp per diagnosis).  The GPU file runs all of them at every levels-per-lane width.
SPARSE = (64, 129, 256)  # levels per lane 2, 5, 8
CELLS = [(name, nz) for name, nz in km.CELLS if not name.endswith('_bvp') or nz in SPARSE]


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


@pytest.mark.parametrize('name,nz', CELLS)
def test_fused_kernel_cell(emu, pool, monkeypatch, name, nz):
  km.fused_cell(emu, pool, monkeypatch, name, nz, bitwise=nz in SPARSE)


def test_matrix_covers_launch_model():
  km.matrix_is_complete()


def test_jn_f2010_above_256_levels_is_refused(emu):
  km.jn_f2010_wide_refused(emu)


def test_column_batched(emu):
  km.column_batched(emu)


def test_thermwind_batched(emu):
  km.thermwind_batched(emu)


def test_psib_batched(emu):
  km.psib_batched(emu)


def test_so_batched(emu, pool):
  km.so_batched(emu, pool, f2010_sizes=SPARSE)


def test_ml_batched(emu):
  km.ml_batched(emu)


def test_shared_memory_limits(emu):
  km.smem_limits(emu)
