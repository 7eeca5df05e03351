"""Member lists (pmoc_model_run_members) and runs to equilibrium (pmoc_model_equilibrate) on the CPU warp emulator:
every warp-kernel cell, the several-members-per-warp kernel and the block-per-member kernels at nz = 257 and 1025."""
import pytest

import equilibrium_matrix as eq
import kernel_matrix as km
from emu.emu_backend import EmuBackend


@pytest.fixture(scope='module')
def emu():
  return EmuBackend()


@pytest.mark.parametrize('name,nz', km.CELLS)
def test_subset_warp_kernel(emu, monkeypatch, name, nz):
  eq.subset_exact(emu, monkeypatch, name, nz)


@pytest.mark.parametrize('nz', eq.TWCOL_NZ)
def test_subset_twcol(emu, monkeypatch, nz):
  # seed 4 lists members of uniform and tabulated home warps side by side
  eq.subset_exact(emu, monkeypatch, 'twcol_kernel', nz, seed=4)


@pytest.mark.parametrize('name,nz', eq.TALL)
def test_subset_tall(emu, monkeypatch, name, nz):
  eq.subset_exact(emu, monkeypatch, name, nz)


@pytest.mark.parametrize('name,nz', km.CELLS)
def test_equilibrate_warp_kernel(emu, monkeypatch, name, nz):
  eq.equilibrate_exact(emu, monkeypatch, name, nz)


@pytest.mark.parametrize('nz', eq.TWCOL_NZ)
def test_equilibrate_twcol(emu, monkeypatch, nz):
  eq.equilibrate_exact(emu, monkeypatch, 'twcol_kernel', nz)


@pytest.mark.parametrize('name,nz', eq.TALL)
def test_equilibrate_tall(emu, monkeypatch, name, nz):
  eq.equilibrate_exact(emu, monkeypatch, name, nz)


def test_nonfinite_member(emu, monkeypatch):
  eq.nonfinite_member(emu, monkeypatch)


def test_invalid_arguments(emu):
  eq.invalid_arguments(emu)


def test_refusals(emu):
  eq.refusals(emu)
