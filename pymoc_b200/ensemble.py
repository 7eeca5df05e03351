"""Batched front end: an ensemble of coupled PyMOC models stepped by one fused CUDA kernel.

    spec = configs.c3_twocol_so(M=4096)
    ens = Ensemble(spec)          # evaluates callables' samples on the host, uploads once
    ens.run(2400)                 # 2400 iterations of the script loop for every member
    b = ens.state()['b_basin']    # [M, nz] numpy
    psi = ens.diagnostics()['Psi_so']

It replaces the ``for ii in range(total_iters)`` loops of the reference's example scripts
(SURVEY.md section 2 #5); one :class:`~pymoc_b200.spec.ModelSpec` describes which modules
exist and how they are wired.  All arithmetic happens in ``libpymoc_b200.so``; this module
only marshals arrays.
"""
from __future__ import annotations

import ctypes

import numpy as np

from . import _abi
from .spec import ModelSpec


# ----------------------------------------------------------------------------- host set-up
def so_tapers(z, Hsill=None, HEk=None, Htapertop=None, Htaperbot=None):
  """The four z-profiles that scale Psi_Ek / Psi_GM, evaluated on the host with the
  reference's expressions (psi_SO.py:185-187 bottom taper, :209-216 top taper; with
  ``HEk=None`` the Ekman taper is all ones except a zero at the surface)."""
  z = np.asarray(z, dtype=np.float64)
  ones = np.ones(z.size)

  def bottom(H):
    return ones.copy() if H is None else 1. - np.maximum(z[0] + H - z, 0.)**2. / H**2.

  def top(H):
    return ones.copy() if H is None else 1 - np.maximum(z + H, 0)**2. / H**2.

  ek = top(HEk)
  if HEk is None:
    ek[-1] = 0.
  return bottom(Hsill), ek, top(Htapertop), bottom(Htaperbot)


def topology_flags(spec: ModelSpec) -> int:
  f = 0
  if spec.north is not None:
    f |= _abi.HAS_NORTH
  if spec.tw is not None:
    f |= _abi.HAS_TW
  if spec.iso:
    f |= _abi.ISO
  if spec.so is not None:
    f |= _abi.HAS_SO
  if spec.ml is not None:
    f |= _abi.HAS_ML
  if spec.order == 'jn':
    f |= _abi.ORDER_JN
  if spec.pac is not None:
    f |= _abi.HAS_PAC
  return f


class Ensemble:
  """Device-resident ensemble.  ``backend`` defaults to CUDA (there is no CPU path in the
  package; the test-suite injects its warp emulator here to run the kernel sources on a
  GPU-less box)."""

  def __init__(self, spec: ModelSpec, backend=None, members=None):
    """``members``: optional ``(start, stop)`` slice of the spec's members held by this
    instance (multi-GPU sharding: every rank builds the same spec and keeps its block)."""
    if backend is None:
      from .backend import CudaBackend
      backend = CudaBackend()
    self.be, self.lib, self.spec = backend, backend.lib, spec
    lo, hi = (0, spec.M) if members is None else members
    if not (0 <= lo < hi <= spec.M):
      raise ValueError('bad member range %r for M=%d' % ((lo, hi), spec.M))
    self.lo, self.hi, self.M = lo, hi, hi - lo
    self.it = 0
    self._keep = []  # device buffers referenced by the struct
    self._bufs = {}
    self._diagnosed = False
    self.model = self._marshal()

  # -------------------------------------------------------------------------- marshalling
  def _slice(self, a):
    """Per-member array -> this instance's block (shared arrays pass through)."""
    return a if a.shape[0] == 1 else a[self.lo:self.hi]

  def _vec(self, a, name=None):
    """numpy [1|M, ...] -> pmoc_vec on the device."""
    a = self._slice(np.asarray(a, dtype=np.float64))
    buf = self.be.upload(a)
    self._keep.append(buf)
    if name:
      self._bufs[name] = buf
    per = int(np.prod(a.shape[1:])) if a.ndim > 1 else 1
    return _abi.Vec(self.be.ptr(buf), 0 if a.shape[0] == 1 else per)

  def _shared(self, a):
    buf = self.be.upload(np.asarray(a, dtype=np.float64))
    self._keep.append(buf)
    return self.be.ptr(buf)

  def _state(self, a, name, dtype=np.float64):
    """Per-member state/output buffer, expanded to [M, ...]."""
    a = self._slice(np.asarray(a, dtype=dtype))
    if a.shape[0] == 1 and self.M > 1:
      a = np.repeat(a, self.M, axis=0)
    buf = self.be.upload(np.ascontiguousarray(a))
    self._bufs[name] = buf
    return self.be.ptr(buf)

  def _out(self, shape, name, dtype=np.float64):
    buf = self.be.zeros(shape, dtype)
    self._bufs[name] = buf
    return self.be.ptr(buf)

  def _column(self, c, tag):
    z = self.spec.z
    col = _abi.Column()
    col.b = self._state(c.b0, 'b_' + tag)
    col.kappa = self._vec(c.kappa)
    # d(A kappa)/dz per member and variant, np.gradient exactly as column.py:122
    M_k = max(c.kappa.shape[0], c.Area.shape[0])
    dAk = c.dAkappa_dz(z)
    if dAk.shape[0] != M_k:
      dAk = np.broadcast_to(dAk, (M_k,) + dAk.shape[1:])
    col.dAk = self._vec(np.ascontiguousarray(dAk))
    col.Area = self._vec(c.Area)
    col.bs = self._vec(c.bs)
    col.N2min = self._vec(c.N2min)
    col.bzbot = self._vec(c.bzbot) if c.bzbot is not None else _abi.Vec(None, 0)
    col.bbot = self._state(c.bbot, 'bbot_' + tag)
    col.nvar = c.kappa.shape[1]
    if col.nvar > 1:
      col.var = self._state(np.full((self.M,), c.var0, dtype=np.int32), 'var_' + tag, np.int32)
    col.do_conv = int(c.do_conv)
    return col

  def _marshal(self):
    s, M = self.spec, self.M
    nz = s.nz
    m = _abi.Model()
    m.M, m.nz, m.nb, m.K, m.dt = M, nz, int(s.nb), int(s.K), float(s.dt)
    m.flags = topology_flags(s)
    m.z = self._shared(s.z)
    m.basin = self._column(s.basin, 'basin')
    if s.north is not None:
      m.north = self._column(s.north, 'north')
    if s.tw is not None:
      m.tw_f = self._vec(s.tw.f)
      if s.tw.b2 is not None:
        m.tw_b2 = self._vec(s.tw.b2)
      m.Psi_tw = self._out((M, nz), 'Psi_tw')
      if s.iso:
        m.Psi_iso_b = self._out((M, nz), 'Psi_iso_b')
        m.Psi_iso_n = self._out((M, nz), 'Psi_iso_n')
        m.psib = self._out((M, s.nb), 'psib')
        m.bgrid = self._out((M, s.nb), 'bgrid')
    if s.so is not None:
      so = s.so
      m.ny = so.y.size
      m.y = self._shared(so.y)
      m.so_bs = self._vec(so.bs)
      m.so_tau = self._vec(so.tau)
      m.so_tau_on_y = int(so.tau.ndim == 2)
      for k in ('f', 'rho', 'L', 'KGM', 'smax'):
        setattr(m, 'so_' + k, self._vec(getattr(so, k)))
      if so.c is not None:
        m.so_c = self._vec(so.c)
      m.so_bvp_with_Ek = int(so.bvp_with_Ek)
      sill, ek, top, bot = so_tapers(s.z, so.Hsill, so.HEk, so.Htapertop, so.Htaperbot)
      m.so_sill_taper, m.so_ek_taper = self._shared(sill), self._shared(ek)
      m.so_top_taper, m.so_bot_taper = self._shared(top), self._shared(bot)
      m.Psi_so = self._out((M, nz), 'Psi_so')
      m.Psi_Ek = self._out((M, nz), 'Psi_Ek')
      m.Psi_GM = self._out((M, nz), 'Psi_GM')
    if s.pac is not None:
      m.pac = self._column(s.pac, 'pac')
      m.zoc_f = self._vec(s.zoc_f)
      m.so2_L = self._vec(s.so_pac_L)
      for attr, name, shape in (('Psi_zoc', 'Psi_zoc', (M, nz)), ('Psi_zon_a', 'Psi_zon_a', (M, nz)),
                                ('Psi_zon_p', 'Psi_zon_p', (M, nz)), ('psib2', 'psib2', (M, s.nb)),
                                ('bgrid2', 'bgrid2', (M, s.nb)), ('Psi_so2', 'Psi_so2', (M, nz)),
                                ('Psi_Ek2', 'Psi_Ek2', (M, nz)), ('Psi_GM2', 'Psi_GM2', (M, nz))):
        setattr(m, attr, self._out(shape, name))
    if s.ml is not None:
      ml = s.ml
      m.ml_bs = self._state(ml.bs0, 'bs_ml')
      for k, attr in (('Ks', 'ml_Ks'), ('h', 'ml_h'), ('L', 'ml_L'), ('v_pist', 'ml_vpist'),
                      ('surflux', 'ml_surflux'), ('rest_mask', 'ml_rest_mask'), ('b_rest', 'ml_b_rest')):
        setattr(m, attr, self._vec(getattr(ml, k)))
      m.ml_Psi_s = self._out((M, ml.y.size), 'Psi_s')
    m.status = self._out((M,), 'status', np.uint32)
    need = int(self.lib.pmoc_model_scratch_bytes(ctypes.byref(m)))
    if need:  # columns taller than one warp handles: per-level constants live in device scratch
      m.scratch = self._out(((need + 7) // 8,), 'scratch')
      m.scratch_bytes = need
    return m

  # ------------------------------------------------------------------------------ running
  def diagnose(self):
    """Diagnose every streamfunction from the current state (the scripts' pre-loop
    ``AMOC.solve(); AMOC.Psibz(); SO.solve()``)."""
    with self._guard():
      _abi.check(self.lib, self.lib.pmoc_model_diagnose(ctypes.byref(self.model), self.be.stream()))
    self._diagnosed = True

  def _guard(self):
    """The backend's device made current around a library call (backends without one: no-op)."""
    import contextlib
    g = getattr(self.be, 'guard', None)
    return g() if g is not None else contextlib.nullcontext()

  def run(self, nsteps, sync=True):
    """Advance every member by ``nsteps`` loop iterations (one fused kernel launch)."""
    if self.spec.order == 'post' and not self._diagnosed:
      self.diagnose()
    with self._guard():
      _abi.check(self.lib, self.lib.pmoc_model_run(ctypes.byref(self.model), self.it, int(nsteps), self.be.stream()))
    self.it += int(nsteps)
    if sync:
      self.be.sync()

  def run_to_equilibrium(self, max_steps, every, tol):
    """Spin-up: advance up to ``max_steps`` iterations in chunks of ``every`` (both multiples of K) and freeze each
    member at the first check where no value of its state (every column's b, the mixed layer's bs) moved by more
    than ``tol`` since the previous check; only the members still moving are stepped.  Non-finite members stop as
    not converged.  Returns ``{'stopped_at': int64[M], 'converged': bool[M]}``; a member stopped at ``n`` holds
    exactly what ``run`` to iteration ``n`` gives it, a valid pickup when ``n`` is a multiple of K.  ``self.it``
    moves on by ``max_steps``: the loop reads the iteration counter only modulo K, so a later ``run`` continues
    every member from its own stop."""
    if self.spec.order == 'post' and not self._diagnosed:
      self.diagnose()
    need = int(self.lib.pmoc_equilibrate_work_bytes(ctypes.byref(self.model)))
    work = self.be.upload(np.zeros((need + 7) // 8, dtype=np.float64))
    stopped = self.be.upload(np.zeros(self.M, dtype=np.int64))
    converged = self.be.upload(np.zeros(self.M, dtype=np.uint8))
    with self._guard():
      _abi.check(self.lib, self.lib.pmoc_model_equilibrate(
          ctypes.byref(self.model), self.it, int(max_steps), int(every), float(tol), self.be.ptr(stopped),
          self.be.ptr(converged), self.be.ptr(work), need, self.be.stream()))
    self.it += int(max_steps)
    self.be.sync()
    return {'stopped_at': self.be.download(stopped), 'converged': self.be.download(converged).astype(bool)}

  # -------------------------------------------------------------------------------- output
  def state(self):
    """Prognostic arrays as numpy: b_basin[, b_north][, bs_ml] -- exactly what the reference's
    pickup files hold (examples/run_JansenNadeau_2018.py:266-267)."""
    self.be.sync()
    keys = [k for k in ('b_basin', 'b_north', 'b_pac', 'bs_ml') if k in self._bufs]
    return {k: self.be.download(self._bufs[k]) for k in keys}

  def set_state(self, **arrays):
    """Overwrite prognostic arrays (``b_basin``, ``b_north``, ``b_pac``, ``bs_ml``; [M, n] each) in place
    on the device -- the pickup path (examples/run_JansenNadeau_2018.py:135-138).  Cached
    streamfunctions are discarded: the next run re-diagnoses them."""
    for k, v in arrays.items():
      if k not in ('b_basin', 'b_north', 'b_pac', 'bs_ml') or k not in self._bufs:
        raise KeyError(k)
      v = np.ascontiguousarray(v, dtype=np.float64)
      if v.shape != tuple(self._bufs[k].shape):
        raise ValueError('%s: shape %r, expected %r' % (k, v.shape, tuple(self._bufs[k].shape)))
      self.be.assign(self._bufs[k], v)
    self._diagnosed = False

  def diagnostics(self):
    self.be.sync()
    keys = [k for k in ('Psi_tw', 'Psi_iso_b', 'Psi_iso_n', 'psib', 'bgrid', 'Psi_so', 'Psi_Ek', 'Psi_GM', 'Psi_s',
                        'status', 'bbot_basin', 'bbot_north', 'var_basin', 'var_north', 'Psi_zoc', 'Psi_zon_a',
                        'Psi_zon_p', 'psib2', 'bgrid2', 'Psi_so2', 'Psi_Ek2', 'Psi_GM2') if k in self._bufs]
    out = {k: self.be.download(self._bufs[k]) for k in keys}
    out['status'] = out['status'].view(np.uint32) & np.uint32(_abi.ST_PUBLIC_MASK)
    return out

  def buffer(self, name):
    """The live device buffer behind a state/diagnostic array (for gathers and checkpoints)."""
    return self._bufs[name]


class HostEnsemble(Ensemble):
  """An ensemble whose arrays live in pinned HOST memory, stepped through the persistent host-buffer handle of
  the C ABI (``pmoc_host_open / pmoc_host_step / pmoc_host_close``): grids and parameters go to the GPU once,
  each :meth:`run` moves only the array classes asked for (``push`` before the launch, ``pull`` after it),
  pipelined over blocks of members.  This is the call pattern of a script that keeps the model state on the
  host and looks at diagnostics every ``Diag_iters`` iterations (examples/run_JansenNadeau_2018.py:218-226).

      ens = HostEnsemble(spec)
      for _ in range(total_iters // 120):
        ens.run(120, pull=IO_STATE | IO_PSI)      # state() / diagnostics() then read the host arrays
  """
  IO_STATE, IO_PSI, IO_DIAG = _abi.IO_STATE, _abi.IO_PSI, _abi.IO_DIAG

  def __init__(self, spec: ModelSpec, backend=None, members=None):
    if backend is None:
      from .backend import PinnedHostBackend
      backend = PinnedHostBackend()
    super().__init__(spec, backend=backend, members=members)
    self._handle = ctypes.c_void_p()
    _abi.check(self.lib, self.lib.pmoc_host_open(ctypes.byref(self.model), ctypes.byref(self._handle)))

  def run(self, nsteps, push=0, pull=_abi.IO_STATE | _abi.IO_PSI | _abi.IO_DIAG, sync=True):
    """Advance ``nsteps`` iterations.  ``push``: classes of host arrays copied to the device first (after the
    caller changed them: ``IO_STATE`` for a new state); ``pull``: classes copied back."""
    if self._handle is None:
      raise RuntimeError('HostEnsemble is closed')
    _abi.check(self.lib, self.lib.pmoc_host_step(self._handle, self.it, int(nsteps), int(push), int(pull)))
    self.it += int(nsteps)

  def diagnose(self):
    _abi.check(self.lib, self.lib.pmoc_host_step(self._handle, 0, 0, 0, _abi.IO_PSI | _abi.IO_DIAG))

  def run_to_equilibrium(self, max_steps, every, tol, push=0, pull=_abi.IO_STATE | _abi.IO_PSI | _abi.IO_DIAG):
    """:meth:`Ensemble.run_to_equilibrium` through the handle (``pmoc_host_equilibrate``): the same stops, flags and
    end state, the same returned dict, and ``self.it`` moves on by ``max_steps``.  ``push`` / ``pull`` as in
    :meth:`run`: the classes copied to the device before the run and back after it."""
    if self._handle is None:
      raise RuntimeError('HostEnsemble is closed')
    stopped, converged = np.zeros(self.M, dtype=np.int64), np.zeros(self.M, dtype=np.uint8)
    _abi.check(self.lib, self.lib.pmoc_host_equilibrate(self._handle, self.it, int(max_steps), int(every), float(tol),
                                                        stopped.ctypes.data, converged.ctypes.data, int(push),
                                                        int(pull)))
    self.it += int(max_steps)
    return {'stopped_at': stopped, 'converged': converged.astype(bool)}

  def last_bytes(self):
    """(host->device, device->host) bytes of the last call."""
    h2d, d2h = ctypes.c_uint64(), ctypes.c_uint64()
    self.lib.pmoc_host_last_bytes(ctypes.byref(h2d), ctypes.byref(d2h))
    return int(h2d.value), int(d2h.value)

  def close(self):
    if getattr(self, '_handle', None) is not None and self._handle:
      self.lib.pmoc_host_close(self._handle)
    self._handle = None

  def __del__(self):
    try:
      self.close()
    except Exception:
      pass
