"""Member lists (pmoc_model_run_members) and runs to equilibrium (pmoc_model_equilibrate) on cuda:0: every warp-kernel
cell, the several-members-per-warp kernel and the block-per-member kernels at nz = 257 and 1025 (run with -s for
the tolerances and stops of each cell)."""
import pytest

import equilibrium_matrix as eq
import kernel_matrix as km

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def cuda():
  from pymoc_b200.backend import CudaBackend
  return CudaBackend()


@pytest.mark.parametrize('name,nz', km.CELLS)
def test_subset_warp_kernel(cuda, monkeypatch, name, nz):
  eq.subset_exact(cuda, monkeypatch, name, nz)


@pytest.mark.parametrize('nz', eq.TWCOL_NZ)
def test_subset_twcol(cuda, monkeypatch, nz):
  eq.subset_exact(cuda, monkeypatch, 'twcol_kernel', nz, seed=4)


@pytest.mark.parametrize('name,nz', eq.TALL)
def test_subset_tall(cuda, monkeypatch, name, nz):
  eq.subset_exact(cuda, monkeypatch, name, nz)


@pytest.mark.parametrize('name,nz', km.CELLS)
def test_equilibrate_warp_kernel(cuda, monkeypatch, name, nz):
  eq.equilibrate_exact(cuda, monkeypatch, name, nz)


@pytest.mark.parametrize('nz', eq.TWCOL_NZ)
def test_equilibrate_twcol(cuda, monkeypatch, nz):
  eq.equilibrate_exact(cuda, monkeypatch, 'twcol_kernel', nz)


@pytest.mark.parametrize('name,nz', eq.TALL)
def test_equilibrate_tall(cuda, monkeypatch, name, nz):
  eq.equilibrate_exact(cuda, monkeypatch, name, nz)


def test_nonfinite_member(cuda, monkeypatch):
  eq.nonfinite_member(cuda, monkeypatch)


def test_invalid_arguments(cuda):
  eq.invalid_arguments(cuda)


def test_refusals(cuda):
  eq.refusals(cuda)
