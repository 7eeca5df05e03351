"""Shared plumbing of the drop-in classes: one lazily created CUDA backend, numpy <-> device
marshalling for the per-module C-ABI entry points."""
import ctypes

import numpy as np

from .. import _abi

_backend = None


def backend():
  """The process-wide device backend (CUDA; created on first use, raises without a GPU)."""
  global _backend
  if _backend is None:
    from ..backend import CudaBackend
    _backend = CudaBackend()
  return _backend


def _set_backend(be):
  """Test seam: the CPU-only test-suite injects its warp emulator of the kernel sources."""
  global _backend
  _backend = be


class Call:
  """Collects the device buffers of one kernel call so that they outlive it."""

  def __init__(self):
    self.be = backend()
    self.lib = self.be.lib
    self.keep = []

  def dev(self, arr, dtype=np.float64):
    buf = self.be.upload(np.ascontiguousarray(arr, dtype=dtype))
    self.keep.append(buf)
    return buf

  def ptr(self, arr, dtype=np.float64):
    return self.be.ptr(self.dev(arr, dtype))

  def vec(self, arr):
    """1 member: stride 0."""
    if arr is None:
      return _abi.Vec(None, 0)
    return _abi.Vec(self.ptr(np.atleast_1d(np.asarray(arr, dtype=np.float64))), 0)

  def out(self, shape, dtype=np.float64):
    buf = self.be.zeros(shape, dtype)
    self.keep.append(buf)
    return buf

  def check(self, rc, who=None):
    """Raise on an error return.  ``who``: the drop-in class, whose size limits (the library's EUNSUPPORTED) are
    a ValueError, like its nz limit."""
    if who is not None and rc == _abi.EUNSUPPORTED:
      raise ValueError('pymoc_b200.modules.%s: %s' % (who, self.lib.pmoc_last_error().decode()))
    _abi.check(self.lib, rc)

  def get(self, buf):
    self.be.sync()
    return self.be.download(buf)


def byref(x):
  return ctypes.byref(x)
