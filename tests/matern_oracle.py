"""CPU oracle of the Matern nu = 1/2 and nu = 5/2 kernels (GPX_MATERN12, GPX_MATERN52).

`MaternSpec` is an oracle `KernelSpec` whose evaluateF / gram / packed_params know the two families; every ref_* / fast_*
function of oracle/gpexp_oracle.py reads a kernel only through those methods and `signal`, so they run unchanged on it.
With r = |x - y|, t = c0 r and c0 = sqrt(2 nu) / rho (the scaling the reference uses for nu = 3/2, kernels.py:87-89):
    nu = 1/2   k = s exp(-t)
    nu = 5/2   k = s (1 + t + t^2 / 3) exp(-t)
"""
from dataclasses import dataclass

import numpy as np

from oracle import gpexp_oracle as orc

MATERN12, MATERN52 = 3, 4
NU = {MATERN12: 0.5, orc.MATERN32: 1.5, MATERN52: 2.5}


def matern_closed_form(nu, r, rho, s):
    """s p(t) exp(-t) for nu in {1/2, 3/2, 5/2}; r an array of distances."""
    t = np.sqrt(2.0 * nu) * np.asarray(r, dtype=np.float64) / rho
    p = {0.5: 1.0, 1.5: 1.0 + t, 2.5: 1.0 + t + t * t / 3.0}[nu]
    return s * p * np.exp(-t)


@dataclass
class MaternSpec(orc.KernelSpec):
    @staticmethod
    def matern12(rho, signal, dim):
        return MaternSpec(MATERN12, dim, rho=float(rho), signal=float(signal))

    @staticmethod
    def matern52(rho, signal, dim):
        return MaternSpec(MATERN52, dim, rho=float(rho), signal=float(signal))

    def _k(self, sq):
        return matern_closed_form(NU[self.family], np.sqrt(sq), self.rho, self.signal)

    def evaluateF(self, x1, x2):
        assert x1.shape == x2.shape
        return self._k(np.sum((x1 - x2) ** 2.0, axis=1))

    def gram(self, X, Y):
        X, Y = np.asarray(X, dtype=np.float64), np.asarray(Y, dtype=np.float64)
        acc = np.zeros((X.shape[0], Y.shape[0]))
        for i in range(self.dim):
            acc += (X[:, i:i + 1] - Y[None, :, i]) ** 2.0
        return self._k(acc)

    def packed_params(self):
        return np.array([self.rho, self.signal])
