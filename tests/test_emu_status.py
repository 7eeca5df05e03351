"""Per-member status bits and the rare solver branches behind them on the CPU warp emulator (levels per lane 2 and 8,
nz = 257 for the block-per-member kernels); test_gpu_status.py runs every size."""
import pytest

import kernel_matrix as km
import status_matrix as sm
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


def test_bs_profiles_restate_the_scan():
  _, prof = sm.bs_profiles()
  assert {n: sm.scan_bits(p) for n, p in prof.items()} == sm.EXPECTED_SCAN


@pytest.mark.parametrize('with_c', (False, True))
@pytest.mark.parametrize('nz', (64, 256))
def test_so_bs_scan(emu, pool, nz, with_c):
  sm.so_bs_scan(emu, pool, nz, with_c)


def test_series_table_is_consistent():
  sm.series_table_is_consistent()


@pytest.mark.parametrize('nz', (64, 256))
def test_smoother_sweep(emu, pool, nz):
  sm.so_smoother_sweep(emu, pool, nz)


def test_series_divergence_is_flagged(emu):
  sm.so_series_diverges(emu, 64)


def test_ml_index(emu):
  sm.ml_index(emu)


@pytest.mark.parametrize('nz', (64, 257))
def test_pushed_psi_noise_switch(emu, nz):
  sm.pushed_psi(emu, emu, nz)


# model cells: the fused warp kernels at levels per lane 2 (and k_twcol at nz 40 and 100), the block-per-member
# kernels at nz = 257
@pytest.mark.parametrize('name,nz', [(n, z) for n in ('so', 'c3', 'jn') for z in (64, 257)])
def test_model_bs_scan(emu, name, nz):
  sm.model_bs_scan(emu, emu, name, nz)


@pytest.mark.parametrize('name,nz', [(n, z) for n in ('twocol', 'c3', 'jn') for z in (64, 257)])
def test_model_tie_cell(emu, name, nz):
  sm.model_tie_cell(emu, emu, name, nz)


@pytest.mark.parametrize('name,nz,column', [('tw', 40, 'basin'), ('tw', 100, 'basin'), ('so', 64, 'basin'),
                                            ('twocol', 64, 'north'), ('jn', 64, 'basin'), ('so', 257, 'basin'),
                                            ('twocol', 257, 'basin'), ('twocol', 257, 'north'), ('jn', 257, 'basin')])
def test_model_nan(emu, name, nz, column):
  sm.model_nan(emu, emu, name, nz, columns=(column,))


@pytest.mark.parametrize('nz', (64, 257))
def test_model_ml_index(emu, pool, nz):
  sm.model_ml_index(emu, emu, pool, nz)
