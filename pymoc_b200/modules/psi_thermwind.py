"""Drop-in ``Psi_Thermwind`` (reference: src/pymoc/modules/psi_thermwind.py) on the GPU.

``solve`` replaces ``scipy.integrate.solve_bvp`` by the exact double quadrature of the linear
BVP (pmoc_thermwind_solve); callables for b1/b2 are sampled at the nodes and, like the
collocation solver does, at the cell mid-points.  ``Psib``/``Psibz`` run pmoc_thermwind_psib.
"""
import numpy as np

from .. import _abi
from ..utils import make_array, make_func
from ._dispatch import Call


class Psi_Thermwind(object):

  def __init__(self, f=1.2e-4, z=None, sol_init=None, b1=None, b2=0.):
    self.f = f
    if isinstance(z, np.ndarray):
      self.z = z
      nz = np.size(z)
    else:
      raise TypeError('z needs to be numpy array providing grid levels')
    self.b1 = make_func(b1, self.z, 'b1')
    self.b2 = make_func(b2, self.z, 'b2')
    # kept for signature compatibility; the closed-form solve needs no initial guess
    self.sol_init = np.zeros((2, nz)) if sol_init is None else sol_init

  # the reference's formulation of the problem (psi_thermwind.py:72-123), kept for callers that hand it to their
  # own solver; ``solve`` uses the closed form
  def bc(self, ya, yb):
    return np.array([ya[0], yb[0]])

  def ode(self, z, y):
    return np.vstack((y[1], 1. / self.f * (self.b2(z) - self.b1(z))))

  def _profiles(self):
    z = np.ascontiguousarray(self.z, dtype=np.float64)
    if z.size > _abi.MAX_NZ_WARP:
      raise ValueError('pymoc_b200.modules.Psi_Thermwind: the per-method kernels hold one column per warp, nz <= %d '
                       '(got %d); taller columns run through pymoc_b200.ensemble.Ensemble' % (_abi.MAX_NZ_WARP, z.size))
    ones = 0 * z + 1.
    return z, np.asarray(self.b1(z) * ones, dtype=np.float64), np.asarray(self.b2(z) * ones, dtype=np.float64)

  def solve(self):
    z, b1, b2 = self._profiles()
    zm = 0.5 * (z[1:] + z[:-1])
    gmid = np.append(self.b2(zm) - self.b1(zm) + 0 * zm, 0.)
    c = Call()
    out = c.out((1, z.size))
    c.check(c.lib.pmoc_thermwind_solve(1, z.size, c.ptr(z), c.vec(b1), c.vec(b2), c.vec(float(self.f)), c.vec(gmid),
                                       c.be.ptr(out), c.be.stream()))
    self.Psi = c.get(out)[0]

  def _remap(self, nb, want_z):
    z, _, _ = self._profiles()
    b1 = np.asarray(make_array(self.b1, self.z, 'b1'), dtype=np.float64) + 0 * z
    b2 = np.asarray(make_array(self.b2, self.z, 'b2'), dtype=np.float64) + 0 * z
    c = Call()
    psib, bgrid = c.out((1, nb)), c.out((1, nb))
    iso_b = c.out((1, z.size)) if want_z else None
    iso_n = c.out((1, z.size)) if want_z else None
    c.check(c.lib.pmoc_thermwind_psib(1, z.size, int(nb), c.vec(np.asarray(self.Psi, dtype=np.float64)), c.vec(b1),
                                      c.vec(b2), c.be.ptr(psib), c.be.ptr(bgrid), c.be.ptr(iso_b), c.be.ptr(iso_n),
                                      c.be.stream()), 'Psi_Thermwind')
    self.bgrid = c.get(bgrid)[0]
    return c.get(psib)[0], (c.get(iso_b)[0] if want_z else None), (c.get(iso_n)[0] if want_z else None)

  def Psib(self, nb=500):
    return self._remap(nb, False)[0]

  def Psibz(self, nb=500):
    _, iso_b, iso_n = self._remap(nb, True)
    return [iso_b, iso_n]

  def update(self, b1=None, b2=None):
    if b1 is not None:
      self.b1 = make_func(b1, self.z, 'b1')
    if b2 is not None:
      self.b2 = make_func(b2, self.z, 'b2')
