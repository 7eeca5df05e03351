"""Runs to equilibrium through the host-buffer entry points, shared by the CPU (warp-emulator) and GPU test files.

``HostEnsemble.run_to_equilibrium`` (the persistent handle, ``pmoc_host_equilibrate``) and the stateless
``pmoc_model_equilibrate_host`` must equal ``Ensemble.run_to_equilibrium`` (``pmoc_model_equilibrate`` on device
buffers) bit for bit: stops, flags, every field and the raw status word.  Each check takes two backends: ``dev``,
whose buffers the device path steps, and ``host``, whose buffers are host memory (the emulator's numpy arrays, or
pinned memory on the GPU).  The ensembles are the specs of ``test_emu_host`` (16 members: eight blocks of two in the
emulator build), started staggered as in ``equilibrium_matrix`` so that members stop at different checks and some
never stop.  Runs start at iteration ``every``: an order-'post' handle then keeps the streamfunctions it is given.
"""
import ctypes

import numpy as np
import pytest

import equilibrium_matrix as eq
import kernel_matrix as km
from pymoc_b200 import _abi
from pymoc_b200.ensemble import Ensemble, HostEnsemble
from test_emu_host import SPECS, _sizes

S, P, D = _abi.IO_STATE, _abi.IO_PSI, _abi.IO_DIAG
NAMES = ('c1', 'c3', 'c4', 'c5_320', 'twobasin')


# ------------------------------------------------------------------------------------------------ helpers
def _loaded(dev, host_backend, cls):
  """A ``cls`` ensemble (HostEnsemble or Ensemble) on host buffers holding every array of the device ensemble."""
  ens = cls(dev.spec, backend=host_backend)
  for key, buf in dev._bufs.items():
    if key != 'scratch':
      ens.be.assign(ens._bufs[key], dev.be.download(buf))
  return ens


def _host_arrays(ens):
  return {k: ens.be.download(v) for k, v in ens._bufs.items() if k != 'scratch'}


def _identical(a, b):
  return a.keys() == b.keys() and all(a[k].tobytes() == b[k].tobytes() for k in a)


def _stateless(ens, it0, max_steps, every, tol, stopped=True, converged=True):
  """pmoc_model_equilibrate_host on the ensemble's host arrays: (rc, result dict)."""
  st, cv = np.zeros(ens.M, dtype=np.int64), np.zeros(ens.M, dtype=np.uint8)
  rc = ens.lib.pmoc_model_equilibrate_host(ctypes.byref(ens.model), it0, max_steps, every, tol,
                                           st.ctypes.data if stopped else None, cv.ctypes.data if converged else None)
  return rc, {'stopped_at': st, 'converged': cv.astype(bool)}


def _last_bytes(lib):
  h2d, d2h = ctypes.c_uint64(), ctypes.c_uint64()
  lib.pmoc_host_last_bytes(ctypes.byref(h2d), ctypes.byref(d2h))
  return h2d.value, d2h.value


def _same_result(want, got, what):
  assert np.array_equal(want['stopped_at'], got['stopped_at']), (what, want['stopped_at'], got['stopped_at'])
  assert np.array_equal(want['converged'], got['converged']), (what, want['converged'], got['converged'])


def _setup(dev_backend, monkeypatch, name):
  """(spec, every, checks, tol, staggered device ensemble at iteration every)"""
  spec = SPECS[name]()
  spec.K = min(spec.K, 24)  # c5_320 diagnoses every 720 iterations: 24 keeps its staggered runs short
  every, checks = eq.EVERY_K * spec.K, eq.CHECKS
  snaps = eq.reference_checks(dev_backend, spec, {}, monkeypatch, every, checks, start=eq.staggered)
  tol = eq.pick_tol(snaps, lambda c: c * every)
  dev = eq.staggered(dev_backend, spec, {}, monkeypatch, every)
  dev.it = every
  return spec, every, checks, tol, dev


def _nonvacuous(r, what):
  assert len(set(r['stopped_at'].tolist())) >= 2 and not r['converged'].all(), (what, r)


# ------------------------------------------------------------------------------------------------ checks
def exact(dev_backend, host_backend, monkeypatch, name):
  """Both host entry points == Ensemble.run_to_equilibrium bit for bit, and a following run(n) == Ensemble.run(n);
  the bytes moved are the classes asked for plus 9 bytes per member."""
  spec, every, checks, tol, dev = _setup(dev_backend, monkeypatch, name)
  handle = _loaded(dev, host_backend, HostEnsemble)
  handle.it = every
  flat = _loaded(dev, host_backend, Ensemble)
  n = _sizes(handle)
  max_steps = every * checks

  want = dev.run_to_equilibrium(max_steps, every, tol)
  _nonvacuous(want, name)
  want_fields = eq.fields(dev)

  got = handle.run_to_equilibrium(max_steps, every, tol, push=S | P)
  assert handle.it == every + max_steps
  assert handle.last_bytes() == (n[S] + n[P], n[S] + n[P] + n[D] + 9 * spec.M)
  _same_result(want, got, (name, 'handle'))
  km._same(want_fields, eq.fields(handle), (name, 'handle'))

  rc, got = _stateless(flat, every, max_steps, every, tol)
  _abi.check(flat.lib, rc)
  carry = spec.order == 'post'  # (every is a multiple of K: a 'jn' launch from there starts with a diagnosis)
  assert _last_bytes(flat.lib) == (n['param'] + n[S] + (n[P] if carry else 0), n[S] + n[P] + n[D] + 9 * spec.M)
  _same_result(want, got, (name, 'stateless'))
  km._same(want_fields, eq.fields(flat), (name, 'stateless'))

  k = spec.K + 1  # crosses a diagnosis, ends between two
  dev.run(k)
  handle.run(k)
  _abi.check(flat.lib, flat.lib.pmoc_model_run_host(ctypes.byref(flat.model), every + max_steps, k))
  want_fields = eq.fields(dev)
  km._same(want_fields, eq.fields(handle), (name, 'handle, continued'))
  km._same(want_fields, eq.fields(flat), (name, 'stateless, continued'))
  handle.close()
  print('host equilibrate %-9s tol %.3e stops %s' % (name, tol, want['stopped_at'].tolist()))


def push_pull(dev_backend, host_backend, monkeypatch, name):
  """push=IO_STATE with a new host state == set_state + the device call (an order-'post' model is re-diagnosed);
  pull=0 leaves every host array byte-identical, and a later run(0, pull=IO_STATE) brings the frozen states."""
  spec, every, checks, tol, staggered = _setup(dev_backend, monkeypatch, name)
  new_state = staggered.state()
  max_steps = every * checks

  dev = eq.fresh(dev_backend, spec, {}, monkeypatch)
  dev.set_state(**new_state)
  dev.it = every
  want = dev.run_to_equilibrium(max_steps, every, tol)
  want_fields = eq.fields(dev)
  h = HostEnsemble(spec, backend=host_backend)
  n = _sizes(h)
  for key, val in new_state.items():
    h.be.assign(h._bufs[key], val)
  h.it = every
  got = h.run_to_equilibrium(max_steps, every, tol, push=S)
  assert h.last_bytes() == (n[S], n[S] + n[P] + n[D] + 9 * spec.M)
  _same_result(want, got, (name, 'push state'))
  km._same(want_fields, eq.fields(h), (name, 'push state'))
  h.close()

  dev = staggered
  handle = _loaded(dev, host_backend, HostEnsemble)
  handle.it = every
  want = dev.run_to_equilibrium(max_steps, every, tol)
  before = _host_arrays(handle)
  got = handle.run_to_equilibrium(max_steps, every, tol, push=S | P, pull=0)
  assert handle.last_bytes() == (n[S] + n[P], 9 * spec.M)
  _same_result(want, got, (name, 'pull 0'))
  assert _identical(_host_arrays(handle), before), name
  handle.run(0, pull=S)
  assert handle.last_bytes() == (0, n[S])
  km._same(dev.state(), handle.state(), (name, 'pulled after'))
  handle.close()


def _device_text(dev, it0, max_steps, every, tol, stopped=True, converged=True):
  """(rc, text) of pmoc_model_equilibrate on the device ensemble for the same arguments"""
  need = int(dev.lib.pmoc_equilibrate_work_bytes(ctypes.byref(dev.model)))
  work = dev.be.upload(np.zeros((need + 7) // 8))
  st = dev.be.upload(np.zeros(dev.M, dtype=np.int64))
  cv = dev.be.upload(np.zeros(dev.M, dtype=np.uint8))
  rc = dev.lib.pmoc_model_equilibrate(ctypes.byref(dev.model), it0, max_steps, every, tol,
                                      dev.be.ptr(st) if stopped else None, dev.be.ptr(cv) if converged else None,
                                      dev.be.ptr(work), need, dev.be.stream())
  return rc, dev.lib.pmoc_last_error().decode()


def invalid_arguments(dev_backend, host_backend, name):
  """Every invalid argument: EINVAL with pmoc_model_equilibrate's text (pmoc_host_step's for push / pull bits),
  nothing copied either way (the handle is given a garbage state to push, which must not reach the device), and a
  valid call afterwards equals the device path."""
  spec = SPECS[name]()
  K = spec.K
  dev = Ensemble(spec, backend=dev_backend)
  handle = HostEnsemble(spec, backend=host_backend)
  flat = Ensemble(spec, backend=host_backend)
  good = _host_arrays(handle)
  for key in ('b_basin', 'b_north'):
    if key in handle._bufs:
      handle.be.assign(handle._bufs[key], np.full(tuple(handle._bufs[key].shape), 1e300))
  garbage, flat_before = _host_arrays(handle), _host_arrays(flat)
  st, cv = np.zeros(spec.M, dtype=np.int64), np.zeros(spec.M, dtype=np.uint8)
  bad = [dict(every=K + 1), dict(every=0), dict(every=-2 * K), dict(max_steps=2 * K + 1), dict(max_steps=-2 * K),
         dict(it0=-K), dict(tol=float('nan')), dict(tol=-1.), dict(stopped=False), dict(converged=False)]
  for b in bad:
    a = {**dict(it0=0, max_steps=2 * K, every=2 * K, tol=0., stopped=True, converged=True), **b}
    want = _device_text(dev, **a)
    assert want[0] == _abi.EINVAL, (b, want)
    args = (a['it0'], a['max_steps'], a['every'], a['tol'], st.ctypes.data if a['stopped'] else None,
            cv.ctypes.data if a['converged'] else None)
    rc = handle.lib.pmoc_host_equilibrate(handle._handle, *args, S, S | P | D)
    assert (rc, handle.lib.pmoc_last_error().decode()) == want, (name, 'handle', b)
    assert handle.last_bytes() == (0, 0), b
    rc = flat.lib.pmoc_model_equilibrate_host(ctypes.byref(flat.model), *args)
    assert (rc, flat.lib.pmoc_last_error().decode()) == want, (name, 'stateless', b)
    assert _last_bytes(flat.lib) == (0, 0), b
  for push, pull in ((8, 0), (0, 8), (D, 0)):
    rc = handle.lib.pmoc_host_step(handle._handle, 0, 0, push, pull)
    want = (rc, handle.lib.pmoc_last_error().decode())
    assert want[0] == _abi.EINVAL
    rc = handle.lib.pmoc_host_equilibrate(handle._handle, 0, 2 * K, 2 * K, 0., st.ctypes.data, cv.ctypes.data, push, pull)
    assert (rc, handle.lib.pmoc_last_error().decode()) == want, (name, push, pull)
    assert handle.last_bytes() == (0, 0)
  assert _identical(_host_arrays(handle), garbage) and _identical(_host_arrays(flat), flat_before), name

  for key, val in good.items():  # the host state back as it was, nothing pushed: the device copy is untouched
    handle.be.assign(handle._bufs[key], val)
  want = dev.run_to_equilibrium(4 * K, 2 * K, 0.)
  got = handle.run_to_equilibrium(4 * K, 2 * K, 0.)
  _same_result(want, got, (name, 'handle after refusals'))
  km._same(eq.fields(dev), eq.fields(handle), (name, 'handle after refusals'))
  rc, got = _stateless(flat, 0, 4 * K, 2 * K, 0.)
  _abi.check(flat.lib, rc)
  _same_result(want, got, (name, 'stateless after refusals'))
  km._same(eq.fields(dev), eq.fields(flat), (name, 'stateless after refusals'))
  handle.close()


def refusals(dev_backend, host_backend):
  """Topologies pmoc_model_run refuses are refused by both host entry points with its code and text, with and
  without the order-'post' diagnosis first; the handle stays usable."""
  for spec in eq._refused_specs():
    K = spec.K
    dev = Ensemble(spec, backend=dev_backend)
    rc = dev.lib.pmoc_model_run(ctypes.byref(dev.model), 0, 2 * K, dev.be.stream())
    want = (rc, dev.lib.pmoc_last_error().decode())
    assert rc == _abi.EUNSUPPORTED, want
    handle = HostEnsemble(spec, backend=host_backend)
    flat = Ensemble(spec, backend=host_backend)
    st, cv = np.zeros(spec.M, dtype=np.int64), np.zeros(spec.M, dtype=np.uint8)
    for it0 in (0, 2 * K):
      rc = handle.lib.pmoc_host_equilibrate(handle._handle, it0, 2 * K, 2 * K, 0., st.ctypes.data, cv.ctypes.data, 0, S)
      assert (rc, handle.lib.pmoc_last_error().decode()) == want, (spec.name, 'handle', it0)
      rc, _ = _stateless(flat, it0, 2 * K, 2 * K, 0.)
      assert (rc, flat.lib.pmoc_last_error().decode()) == want, (spec.name, 'stateless', it0)
    with pytest.raises(_abi.PmocError, match='EUNSUPPORTED'):
      handle.run_to_equilibrium(2 * K, 2 * K, 0.)
    _abi.check(handle.lib, handle.lib.pmoc_host_step(handle._handle, K, 0, 0, S))  # still usable
    assert handle.last_bytes() == (0, _sizes(handle)[S])
    handle.close()


def nonfinite_member(dev_backend, host_backend, monkeypatch):
  """A member that blows up is frozen at the first check as not converged through both host entry points, exactly
  as on the device path (equilibrium_matrix.nonfinite_member's ensemble)."""
  import dataclasses
  spec, env = km.cell('so', 64)
  for k, v in env.items():
    monkeypatch.setenv(k, v)
  kap = np.repeat(np.asarray(spec.basin.kappa, dtype=np.float64), spec.M // np.shape(spec.basin.kappa)[0], axis=0)
  kap[2] *= 1e100
  spec = dataclasses.replace(spec, basin=dataclasses.replace(spec.basin, kappa=kap))
  every = eq.EVERY_K * spec.K
  dev = eq.fresh(dev_backend, spec, env, monkeypatch)
  want = dev.run_to_equilibrium(4 * every, every, 0.)
  assert want['stopped_at'][2] == every and not want['converged'][2], want
  handle = HostEnsemble(spec, backend=host_backend)
  flat = Ensemble(spec, backend=host_backend)
  got = handle.run_to_equilibrium(4 * every, every, 0.)
  _same_result(want, got, 'nonfinite, handle')
  km._same(eq.fields(dev), eq.fields(handle), 'nonfinite, handle')
  assert eq.fields(handle)['status'][2] & _abi.ST_NAN
  rc, got = _stateless(flat, 0, 4 * every, every, 0.)
  _abi.check(flat.lib, rc)
  _same_result(want, got, 'nonfinite, stateless')
  km._same(eq.fields(dev), eq.fields(flat), 'nonfinite, stateless')
  handle.close()
