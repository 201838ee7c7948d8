"""
CPU restatement of GPflow 2.2.1's Matern12 and Matern32 kernels for the tests, in the style of oracle.tsvgp_oracle.Matern52: the
same expansion-form square_distance and r = sqrt(max(r2, 1e-36)).  Every oracle model takes them as it takes the kernels it
defines (it reads only K, K_diag, variance and lengthscales).

The M-step gradient restatements (oracle.tsvgp_oracle.elbo_gradients, tests/softmax_grad_oracle.elbo_gradients) read dk/dr2 from
oracle.tsvgp_oracle._kernel_dr2, which knows SE and Matern52 only.  kernel_dr2 adds the two kernels here and defers to it for
the others; elbo_gradients and softmax_elbo_gradients run those restatements with it in place.  Matern12's derivative follows the
rule autodiff takes through GPflow's clamp: -k / (2 r) where r2 >= 1e-36, 0 below.
"""
import contextlib

import numpy as np

from oracle import tsvgp_oracle as orc
from tests import softmax_grad_oracle as sgo


class Matern12:
    """gpflow.kernels.Matern12: r = sqrt(max(r2, 1e-36)); variance * exp(-r)."""

    name = "matern12"

    def __init__(self, variance=1.0, lengthscales=1.0):
        self.variance = orc._param(variance)
        self.lengthscales = orc._param(lengthscales)

    def K_r2(self, r2):
        r = np.sqrt(np.maximum(r2, 1e-36))
        return float(self.variance) * np.exp(-r)

    def K(self, X, X2=None):
        return self.K_r2(orc.square_distance(orc.scale(X, self.lengthscales), None if X2 is None else orc.scale(X2, self.lengthscales)))

    def K_diag(self, X):
        return np.full(X.shape[0], float(self.variance))


class Matern32:
    """gpflow.kernels.Matern32: r = sqrt(max(r2, 1e-36)); variance * (1 + sqrt3 r) exp(-sqrt3 r)."""

    name = "matern32"

    def __init__(self, variance=1.0, lengthscales=1.0):
        self.variance = orc._param(variance)
        self.lengthscales = orc._param(lengthscales)

    def K_r2(self, r2):
        r = np.sqrt(np.maximum(r2, 1e-36))
        sqrt3 = np.sqrt(3.0)
        return float(self.variance) * (1.0 + sqrt3 * r) * np.exp(-sqrt3 * r)

    def K(self, X, X2=None):
        return self.K_r2(orc.square_distance(orc.scale(X, self.lengthscales), None if X2 is None else orc.scale(X2, self.lengthscales)))

    def K_diag(self, X):
        return np.full(X.shape[0], float(self.variance))


_ORACLE_DR2 = orc._kernel_dr2


def kernel_dr2(kernel, r2):
    """dK/d(r^2) of Matern12 and Matern32; the oracle's own rule for every other kernel."""
    var = float(kernel.variance)
    if isinstance(kernel, Matern12):
        r2 = np.asarray(r2, dtype=np.float64)
        r = np.sqrt(np.maximum(r2, 1e-36))
        return np.where(r2 >= 1e-36, -0.5 * (var * np.exp(-r)) / r, 0.0)
    if isinstance(kernel, Matern32):
        return -1.5 * var * np.exp(-np.sqrt(3.0) * np.sqrt(np.maximum(r2, 1e-36)))
    return _ORACLE_DR2(kernel, r2)


@contextlib.contextmanager
def _with_kernel_dr2():
    saved = orc._kernel_dr2
    orc._kernel_dr2 = kernel_dr2
    try:
        yield
    finally:
        orc._kernel_dr2 = saved


def elbo_gradients(model, data):
    """oracle.tsvgp_oracle.elbo_gradients for any kernel of this module or the oracle's"""
    with _with_kernel_dr2():
        return orc.elbo_gradients(model, data)


def softmax_elbo_gradients(model, data):
    """tests/softmax_grad_oracle.elbo_gradients for any kernel of this module or the oracle's"""
    with _with_kernel_dr2():
        return sgo.elbo_gradients(model, data)
