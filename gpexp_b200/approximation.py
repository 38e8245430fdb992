"""The `Space` record the cost functions consume (API of gpExp/approximation.py:22-36): input dimension, a sampler
`sample(shape)`, a density `probDensity(points)` and an optional heteroscedastic noise function `noiseFunc(points)`.

UniformMeasure and GaussianMeasure are not in the reference: set as `costFunctionGP_IVAR.measure`, they make the IVAR
cost the exact integral of the posterior variance over that measure instead of its Monte-Carlo mean over mcPoints
(squared-exponential and Mehler kernels; a Mehler kernel needs std_q^2 < (1 + t_q) / (2 t_q) in a GaussianMeasure, or
the integral of its prior variance is infinite)."""
from typing import Callable, Optional

import numpy as np


class Space:
    def __init__(self, dimensionIn: int, samplerIn: Optional[Callable], probDensityIn: Optional[Callable],
                 noise: Optional[Callable] = None):
        # positional order and attribute names are the reference's; nothing else lives here
        self.dimension, self.sample, self.probDensity, self.noiseFunc = dimensionIn, samplerIn, probDensityIn, noise
        self.inBoundsBool = None

    def __repr__(self):
        return "Space(dimension=%r, noiseFunc=%s)" % (self.dimension, "set" if self.noiseFunc is not None else "None")


def _finite_vector(name, values):
    v = np.atleast_1d(np.asarray(values, dtype=np.float64)).ravel()
    if v.size == 0 or not np.all(np.isfinite(v)):
        raise ValueError(f"{name} must be non-empty and finite")
    return v


class _ProductMeasure:
    """A product probability measure on R^d given by two per-dimension parameter vectors; a single value stands for
    every dimension."""

    def __init__(self, p0, p1):
        self.p0, self.p1 = p0, p1
        if p0.size != p1.size and 1 not in (p0.size, p1.size):
            raise ValueError(f"{self!r}: the two parameter vectors have {p0.size} and {p1.size} entries")

    def params(self, d: int):
        """(p0, p1) with d entries each; ValueError if the measure was given for another dimension."""
        if max(self.p0.size, self.p1.size) not in (1, d):
            raise ValueError(f"{self!r} has {max(self.p0.size, self.p1.size)} dimensions, the kernel {d}")
        return np.broadcast_to(self.p0, (d,)).copy(), np.broadcast_to(self.p1, (d,)).copy()


class UniformMeasure(_ProductMeasure):
    """Uniform probability measure on the box [lower_q, upper_q] (lower < upper, finite)."""

    def __init__(self, lower, upper):
        lo, hi = _finite_vector("UniformMeasure lower", lower), _finite_vector("UniformMeasure upper", upper)
        super().__init__(lo, hi)
        if not np.all(np.broadcast_to(lo, (max(lo.size, hi.size),)) < np.broadcast_to(hi, (max(lo.size, hi.size),))):
            raise ValueError("UniformMeasure needs lower < upper in every dimension")

    def __repr__(self):
        return "UniformMeasure(lower=%s, upper=%s)" % (self.p0.tolist(), self.p1.tolist())


class GaussianMeasure(_ProductMeasure):
    """Gaussian probability measure with independent coordinates N(mean_q, std_q^2) (std > 0, finite)."""

    def __init__(self, mean, std):
        mu, sd = _finite_vector("GaussianMeasure mean", mean), _finite_vector("GaussianMeasure std", std)
        super().__init__(mu, sd)
        if not np.all(sd > 0.0):
            raise ValueError("GaussianMeasure needs std > 0 in every dimension")

    def __repr__(self):
        return "GaussianMeasure(mean=%s, std=%s)" % (self.p0.tolist(), self.p1.tolist())
