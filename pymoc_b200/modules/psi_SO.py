"""Drop-in ``Psi_SO`` (reference: src/pymoc/modules/psi_SO.py) on the GPU.

``solve`` runs pmoc_so_solve: outcrop inversion ys(b), Ekman and GM transports in one
kernel.  The taper profiles are evaluated on the host with the reference's expressions.
"""
import numpy as np

from .. import _abi
from ..ensemble import so_tapers
from ..utils import make_func
from ._dispatch import Call, byref


class Psi_SO(object):

  def __init__(self, z=None, y=None, b=None, bs=None, tau=None, f=1.2e-4, rho=1030, L=1e7, KGM=1e3, c=None,
               bvp_with_Ek=False, Hsill=None, HEk=None, Htapertop=None, Htaperbot=None, smax=0.01):
    if isinstance(z, np.ndarray):
      self.z = z
    else:
      raise TypeError('z needs to be numpy array providing grid levels')
    if isinstance(y, np.ndarray):
      self.y = y
    else:
      raise TypeError('y needs to be numpy array providing horizontal grid (or boundaries) of ACC')
    self.b = make_func(b, self.z, 'b')
    self.bs = make_func(bs, self.y, 'bs')
    self.tau = make_func(tau, self.y, 'tau')
    self._tau_raw = tau
    self.f, self.rho, self.L, self.KGM, self.c = f, rho, L, KGM, c
    self.bvp_with_Ek = bvp_with_Ek
    self.Hsill, self.HEk, self.Htapertop, self.Htaperbot = Hsill, HEk, Htapertop, Htaperbot
    self.smax = smax

  def _kernel(self, b_profile):
    z = np.ascontiguousarray(self.z, dtype=np.float64)
    y = np.ascontiguousarray(self.y, dtype=np.float64)
    if z.size > _abi.MAX_NZ_WARP:
      raise ValueError('pymoc_b200.modules.Psi_SO: the per-method kernels hold one column per warp, nz <= %d (got %d); '
                       'taller columns run through pymoc_b200.ensemble.Ensemble' % (_abi.MAX_NZ_WARP, z.size))
    c = Call()
    m = _abi.Model()
    m.M, m.nz, m.ny = 1, z.size, y.size
    m.z, m.y = c.ptr(z), c.ptr(y)
    if isinstance(self._tau_raw, float):
      m.so_tau, m.so_tau_on_y = c.vec(self._tau_raw), 0
    else:
      m.so_tau, m.so_tau_on_y = c.vec(self.tau(y) + 0 * y), 1
    for k in ('f', 'rho', 'L', 'KGM', 'smax'):
      setattr(m, 'so_' + k, c.vec(float(getattr(self, k))))
    if self.c is not None:
      m.so_c = c.vec(float(self.c))
    m.so_bvp_with_Ek = int(bool(self.bvp_with_Ek))
    sill, ek, top, bot = so_tapers(z, self.Hsill, self.HEk, self.Htapertop, self.Htaperbot)
    m.so_sill_taper, m.so_ek_taper, m.so_top_taper, m.so_bot_taper = c.ptr(sill), c.ptr(ek), c.ptr(top), c.ptr(bot)
    outs = [c.out((1, z.size)) for _ in range(4)]
    status = c.out((1,), np.uint32)
    c.check(c.lib.pmoc_so_solve(byref(m), c.vec(b_profile), c.vec(self.bs(y) + 0 * y), *[c.be.ptr(o) for o in outs],
                                c.be.ptr(status), c.be.stream()), 'Psi_SO')
    psi, ek_sv, gm_sv, ys = (c.get(o)[0] for o in outs)
    st = int(c.get(status).view(np.uint32)[0])
    if st & _abi.ST_BRENT_SIGN:
      raise ValueError('f(a) and f(b) must have different signs')  # what scipy.optimize.brentq raises
    return psi, ek_sv, gm_sv, ys

  def ys(self, b):
    """Outcrop latitude of buoyancy class ``b`` (psi_SO.py:106-140)."""
    return float(self._kernel(np.full(self.z.size, float(b)))[3][0])

  def solve(self):
    z = np.asarray(self.z, dtype=np.float64)
    self.Psi, self.Psi_Ek, self.Psi_GM, _ = self._kernel(self.b(z) + 0 * z)

  def calc_Ekman(self):
    """Psi_Ek in m^3/s (psi_SO.py:218-243)."""
    z = np.asarray(self.z, dtype=np.float64)
    return self._kernel(self.b(z) + 0 * z)[1] * 1e6

  def calc_GM(self):
    """Psi_GM in m^3/s (psi_SO.py:277-331); like the reference it needs ``self.Psi_Ek``."""
    z = np.asarray(self.z, dtype=np.float64)
    return self._kernel(self.b(z) + 0 * z)[2] * 1e6

  # --- host-side pieces of the reference's method surface (state-independent or O(nz) set-up arithmetic; the
  # kernels evaluate the same expressions inside pmoc_so_solve) -----------------------------------------------
  def calc_N2(self):
    """Buoyancy frequency N^2(z) as a callable (psi_SO.py:142-162): centred differences over the two adjacent
    cells in the interior, one-sided at the two ends; used by the F2010 smoother (``c`` given)."""
    z = np.asarray(self.z, dtype=np.float64)
    b = self.b(z)
    h = z[1:] - z[:-1]
    n2 = np.empty(z.size)
    n2[1:-1] = (b[2:] - b[:-2]) / (h[1:] + h[:-1])
    n2[0] = (b[1] - b[0]) / h[0]
    n2[-1] = (b[-1] - b[-2]) / h[-1]
    return make_func(n2, self.z, 'N2')

  def calc_bottom_taper(self, H, z):
    """Quadratic taper over the lowest ``H`` metres (psi_SO.py:164-187); the scalar 1. when ``H`` is None."""
    if H is None:
      return 1.
    return 1. - np.maximum(z[0] + H - z, 0.)**2. / H**2.

  def calc_top_taper(self, H, z, scalar=True):
    """Quadratic taper over the uppermost ``H`` metres (psi_SO.py:189-216).  With ``H`` None: the scalar 1., or
    (``scalar=False``, the Ekman taper) ones with a zero at the surface."""
    if H is not None:
      return 1 - np.maximum(z + H, 0)**2. / H**2.
    if scalar:
      return 1.
    ones = np.ones(np.size(z))
    ones[-1] = 0.
    return ones

  def bc_GM(self, ya, yb):
    """Boundary residuals of the F2010 smoother (psi_SO.py:245-275): Psi_GM = -Psi_Ek at both ends when
    ``bvp_with_Ek`` (needs ``self.Psi_Ek`` in Sv, as in the reference), zero otherwise."""
    if self.bvp_with_Ek:
      return np.array([ya[0] + self.Psi_Ek[0] * 1e6, yb[0] + self.Psi_Ek[-1] * 1e6])
    return np.array([ya[0], yb[0]])

  def update(self, b=None, bs=None):
    if b is not None:
      self.b = make_func(b, self.z, 'b')
    if bs is not None:
      self.bs = make_func(bs, self.y, 'bs')
