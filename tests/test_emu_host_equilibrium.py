"""Runs to equilibrium through the host-buffer entry points (HostEnsemble.run_to_equilibrium, the stateless
pmoc_model_equilibrate_host) on the CPU warp emulator, whose build runs the device mirror on host stand-ins of the
CUDA runtime in blocks of two members: against Ensemble.run_to_equilibrium on the emulator, bit for bit."""
import pytest

import host_equilibrium_matrix as hm
from emu.emu_backend import EmuBackend


@pytest.fixture(scope='module')
def emu():
  return EmuBackend()


@pytest.mark.parametrize('name', hm.NAMES)
def test_exact(emu, monkeypatch, name):
  hm.exact(emu, emu, monkeypatch, name)


@pytest.mark.parametrize('name', ['c3', 'c4'])
def test_push_pull(emu, monkeypatch, name):
  hm.push_pull(emu, emu, monkeypatch, name)


@pytest.mark.parametrize('name', ['c3', 'c4'])
def test_invalid_arguments(emu, name):
  hm.invalid_arguments(emu, emu, name)


def test_refusals(emu):
  hm.refusals(emu, emu)


def test_nonfinite_member(emu, monkeypatch):
  hm.nonfinite_member(emu, emu, monkeypatch)
