"""Covariance functions evaluated by the CUDA library, behind the reference's names (gpExp/kernels.py).

Two ways in:
  * standalone -- the classes below (same constructor arguments and hyperParam keys as the reference);
  * patched    -- `gpexp_b200.install_as_gpExp()` with the reference importable keeps the reference's OWN classes and
                  constructors and only rebinds the methods in `DEVICE_METHODS` onto them.

`Kernel.evaluate(x1, x2)` keeps the reference's *pairwise* semantics (kernels.py:49-65): two (n,d) arrays, or one of
them (1,d), give an (n,) vector.
"""
import math

import numpy as np

from . import _lib
from ._lib import check, lib
from .device import Device, ptr


# ---- device-side methods: written against `self.hyperParam` / `self.dimension` only, so the same functions serve the
# ---- classes below and the reference's classes once patched -----------------------------------------------------------
def _bind(self, dev=None) -> Device:
    """Make this kernel the current one of the device handle (family + hyper-parameters -> constant bank)."""
    dev = dev or Device.get()
    fam, d, params = self._gpx_spec()
    dev.set_kernel(fam, d, params)
    return dev


def _no_cuda_spec(self):
    raise AttributeError("this kernel has no CUDA implementation")


def _no_derivative(self):
    """Only KernelSquaredExponential has an N-D `derivative` in the reference."""
    raise AttributeError("derivative of %s not implemented" % type(self).__name__)


def _evaluate(self, x1, x2):
    """kernels.py:49-65 with the np.tile broadcast done by the kernel's index arithmetic."""
    assert len(x2.shape) > 1 and len(x1.shape) > 1, "Must supply nd arrays to evaluation function"
    assert x1.shape[1] == self.dimension and x2.shape[1] == self.dimension, \
        (" Incorrect dimension of input points fed to kernel ", x1.shape, x2.shape)
    return self.evaluateF(x1, x2)


def _evaluateF(self, x1, x2):
    n1, n2 = x1.shape[0], x2.shape[0]
    # equal lengths, or a single point on one side; any other mix fails the reference's shape assert as well
    assert n1 == n2 or n1 == 1 or n2 == 1, "__evaluate() received non-equal shaped point sets"
    dev = self._bind()
    a, b = dev.points(x1), dev.points(x2)
    n = max(n1, n2) if min(n1, n2) > 0 else 0
    out = dev.zeros(max(n, 1))
    check(lib.gpx_kernel_pairwise(dev.h, ptr(a.X), n1, a.ld, ptr(b.X), n2, b.ld, ptr(out), dev.stream),
          "gpx_kernel_pairwise")
    return out[:n].cpu().numpy()


# nu -> family.  The reference implements nu = 3/2 only; nu = 1/2 and 5/2 are served here as well (under
# install_as_gpExp() too, where the unmodified reference would raise).  Its 1e-10 tolerance on nu is kept.
_MATERN_NU = ((0.5, _lib.MATERN12), (1.5, _lib.MATERN32), (2.5, _lib.MATERN52))


def _matern_spec(self):
    for nu, family in _MATERN_NU:
        if np.abs(nu - self.nu) < 1e-10:
            return family, self.dimension, [self.hyperParam['rho'], self.hyperParam['signalSize']]
    # the reference leaves `out` unbound for any other nu (kernels.py:85-91)
    raise UnboundLocalError("KernelIsoMatern is implemented for nu = 1/2, 3/2 and 5/2 only")


def _se_spec(self):
    return _lib.SE, self.dimension, [self.hyperParam['cl%d' % i] for i in range(self.dimension)] + [self.hyperParam['signalSize']]


def _se_derivative(self, x1, x2, version=0):
    """out[jj, ii] = dK(x1[jj], x2)/dx1[jj, ii] as the reference computes it (kernels.py:146-181):
    -signalSize * (x1 - x2)/cl^2 * evaluate(x1, x2).  x2 is a single (1, d) point."""
    assert len(x2.shape) > 1 and len(x1.shape) > 1, "Must supply nd arrays to evaluation function"
    assert x2.shape[0] == 1 and x2.shape[1] == self.dimension, "x2 not in correct shape"
    assert x1.shape[0] > 0 and x1.shape[1] == self.dimension, "x1 not in correct shape"
    dev = self._bind()
    a, b = dev.points(x1), dev.points(x2)
    n, d = x1.shape
    ld = max(n * d, 1)
    out = dev.zeros(1, ld)
    check(lib.gpx_se_dgram(dev.h, ptr(b.X), 1, b.ld, ptr(a.X), n, a.ld, ptr(out), ld, dev.stream), "gpx_se_dgram")
    return out[0, : n * d].cpu().numpy().reshape(n, d)


def _mehler_nd_spec(self):
    return _lib.MEHLER, self.dimension, [self.hyperParam[i] for i in range(self.dimension)]


def _mehler_1d_spec(self):
    return _lib.MEHLER, 1, [self.hyperParam['t']]


def _mehler_1d_evaluateF(self, x1, x2):
    assert x1.shape[1] == 1 and x2.shape[1] == 1, "Hermite1d kernel only accepts one dimensional points"
    out = _evaluateF(self, x1, x2)
    if out.size and math.isnan(out[0]):  # kernels.py:288-292
        print("xs ", x1[0, :], x2[0, :])
        print("t", self.hyperParam['t'])
        print('NAN in kernel hermi1d exiting')
        raise SystemExit
    return out


# class name -> {method name: function}: what install_as_gpExp() rebinds on the reference's own classes
DEVICE_METHODS = {
    "Kernel": {"evaluate": _evaluate, "evaluateF": _evaluateF, "_bind": _bind, "_gpx_spec": _no_cuda_spec,
               "_require_derivative": _no_derivative},
    "KernelIsoMatern": {"evaluateF": _evaluateF, "_gpx_spec": _matern_spec},
    "KernelSquaredExponential": {"evaluateF": _evaluateF, "_gpx_spec": _se_spec, "derivative": _se_derivative,
                                 "_require_derivative": lambda self: True},
    "KernelMehlerND": {"evaluateF": _evaluateF, "_gpx_spec": _mehler_nd_spec},
    "KernelMehler1D": {"evaluateF": _mehler_1d_evaluateF, "_gpx_spec": _mehler_1d_spec},
}


def _attach(cls):
    for name, fn in DEVICE_METHODS[cls.__name__].items():
        setattr(cls, name, fn)
    return cls


# ---- standalone classes: the reference's constructor arguments and hyperParam keys are the drop-in contract ------------
@_attach
class Kernel(object):
    """Base class: a dimension and a dict of hyper-parameters (kernels.py:30-47)."""

    nugget = 0.0
    hyperParam = {}

    def __init__(self, hyperParam, dimension, *argc):
        self.hyperParam, self.dimension = hyperParam, dimension

    def updateHyperParameters(self, hyperParamNew):
        unknown = [key for key in hyperParamNew if key not in self.hyperParam]
        assert not unknown, (unknown[0], " is not a valid hyperParameter")
        self.hyperParam = hyperParamNew


@_attach
class KernelIsoMatern(Kernel):
    """Isotropic Matern, nu = 1/2, 3/2 or 5/2; hyper-parameters rho, signalSize (kernels.py:72-91, which has nu = 3/2
    only)."""

    def __init__(self, rho, signalSize, dimension, nu=1.5):
        self.nu = nu  # not a hyper-parameter (kernels.py:76)
        Kernel.__init__(self, {'rho': rho, 'signalSize': signalSize}, dimension)

    def derivativeWrtHypParams(self, x1, x2):
        raise AttributeError("derivativeWrtHypParams not implemented for KernelIsoMatern")


@_attach
class KernelSquaredExponential(Kernel):
    """signalSize * exp(-1/2 sum (x-x')^2 / cl_i^2); one length (isotropic) or d lengths (ARD); hyper-parameters
    cl0 .. cl{d-1}, signalSize (kernels.py:100-123)."""

    def __init__(self, correlationLength, signalSize, dimension):
        lengths = list(correlationLength) * dimension if len(correlationLength) == 1 else list(correlationLength)
        hyper = {'cl%d' % i: length for i, length in enumerate(lengths)}
        hyper['signalSize'] = signalSize
        Kernel.__init__(self, hyper, dimension)


@_attach
class KernelMehlerND(Kernel):
    """Product of 1-D Mehler kernels; hyper-parameters are keyed by the integer axis (kernels.py:183-228)."""

    def __init__(self, tIn, dimension):
        self.oneDKern = [KernelMehler1D(tIn[i], 1) for i in range(dimension)]
        Kernel.__init__(self, {i: tIn[i] for i in range(dimension)}, dimension)

    def updateHyperParameters(self, params):
        for axis in self.hyperParam:
            self.hyperParam[axis] = params[axis]
            self.oneDKern[axis].updateHyperParameters({'t': params[axis]})

    def derivative(self, x1, x2):
        raise AttributeError("derivative of KernelMehlerND not yet implemented")


@_attach
class KernelMehler1D(Kernel):
    """1-D Mehler (Hermite) kernel; hyper-parameter t (kernels.py:250-293)."""

    def __init__(self, tIn, dimension):
        assert dimension == 1, "Mehler Hermite Kernel is only one dimensional"
        Kernel.__init__(self, {'t': tIn}, dimension)
