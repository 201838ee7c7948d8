"""
The M-step gradients of the whitened sibling (tests/white_grad_oracle.py) against central differences of the unchanged
OracleTSVGPWhite.elbo: kernel variance, every lengthscale, several Z entries and the likelihood parameter, for all four kernels, the
three independent likelihoods, ARD and isotropic lengthscales and one or two latents.  The sites are trained by a few natural-
gradient steps first: at the default Lambda_2 = 1e-10 I the matrix Q = A^-1 - R^-1 is ~0 and most of Gamma_K would go untested.
"""
import numpy as np
import pytest

from oracle import tsvgp_oracle as orc
from tests import matern_oracle as mo
from tests import white_grad_oracle as wgo

KINDS = {"se": orc.SquaredExponential, "matern12": mo.Matern12, "matern32": mo.Matern32, "matern52": orc.Matern52}


class _ExactDiagonal:
    """K(Z) with its diagonal at exactly the variance.  The expansion form leaves r2 ~ 1e-16 |z|^2 on the diagonal, which moves
    Matern-1/2's K_ii by ~1e-8 relative whenever Z or the lengthscales move, and a central difference would read that rounding as a
    slope.  The restatement differentiates this function: it takes no Z or lengthscale gradient from the diagonal."""

    def K(self, X, X2=None):
        K = super().K(X, X2)
        if X2 is None:
            np.fill_diagonal(K, float(self.variance))
        return K


EXACT = {name: type(name, (_ExactDiagonal, cls), {}) for name, cls in KINDS.items()}


def _model(kind, lik_name, ard, L, N=40, M=7, D=3, seed=0):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((N, D))
    Z = rng.standard_normal((M, D))      # off the data: the Matern-1/2 ELBO is not differentiable where z = x
    ls = np.array([0.9, 1.4, 1.1]) if ard else 1.2
    kernel = EXACT[kind](variance=1.4, lengthscales=ls)
    f = np.stack([np.sin(X.sum(1) + 0.7 * l) for l in range(L)], 1)
    if lik_name == "gaussian":
        lik, Y = orc.Gaussian(variance=0.3), f + 0.2 * rng.standard_normal((N, L))
    elif lik_name == "bernoulli":
        lik, Y = orc.Bernoulli(), (f > 0).astype(float)
    else:
        lik, Y = orc.StudentT(scale=0.5, df=4.0), f + 0.2 * rng.standard_normal((N, L))
    m = orc.OracleTSVGPWhite(kernel, lik, orc.InducingPoints(Z), num_latent_gps=L, num_data=3 * N)
    for _ in range(3):
        m.natgrad_step((X, Y), lr=0.6)
    return m, (X, Y)


def _cd(m, data, set_value, x0, h):
    set_value(x0 + h)
    ep = m.elbo(data)
    set_value(x0 - h)
    em = m.elbo(data)
    set_value(x0)
    return (ep - em) / (2.0 * h)


CASES = [("se", "gaussian", True, 1), ("se", "bernoulli", False, 2), ("matern52", "student_t", True, 1),
         ("matern52", "gaussian", False, 2), ("matern32", "bernoulli", True, 1), ("matern32", "student_t", False, 2),
         ("matern12", "gaussian", True, 2), ("matern12", "student_t", True, 1), ("se", "student_t", False, 1)]


@pytest.mark.parametrize("kind,lik_name,ard,L", CASES)
def test_white_gradients_against_central_differences(kind, lik_name, ard, L):
    m, data = _model(kind, lik_name, ard, L)
    # the trained sites make Q = A^-1 - R^-1 far from zero (the data terms of Gamma_K are exercised)
    A = m.kernel.K(np.asarray(m.inducing_variable.Z)) + orc.DEFAULT_JITTER * np.eye(m.num_inducing)
    assert np.max(np.abs(m.lambda_2)) > 1e-2 * np.max(np.abs(A))
    e, g = wgo.elbo_gradients(m, data)
    assert abs(e - m.elbo(data)) <= 1e-12 * abs(e)
    rtol, atol = 2e-6, 1e-8
    k = m.kernel
    v0 = float(k.variance)
    cd = _cd(m, data, lambda v: setattr(k, "variance", orc._param(v)), v0, 1e-6)
    assert g["variance"] == pytest.approx(cd, rel=rtol, abs=atol)
    ls0 = np.array(k.lengthscales, dtype=np.float64).reshape(-1)
    assert g["lengthscales"].shape == ls0.shape
    for d in range(ls0.size):
        def set_ls(v, d=d):
            a = ls0.copy()
            a[d] = v
            k.lengthscales = orc._param(a if ls0.size > 1 else a[0])
        cd = _cd(m, data, set_ls, ls0[d], 1e-6)
        assert g["lengthscales"][d] == pytest.approx(cd, rel=rtol, abs=atol)
    Z0 = np.array(m.inducing_variable.Z)
    for i, d in [(0, 0), (3, 1), (6, 2), (2, 0)]:
        def set_z(v, i=i, d=d):
            Z = Z0.copy()
            Z[i, d] = v
            m.inducing_variable = orc.InducingPoints(Z)
        cd = _cd(m, data, set_z, Z0[i, d], 1e-6)
        assert g["Z"][i, d] == pytest.approx(cd, rel=rtol, abs=atol)
    if lik_name == "bernoulli":
        assert g["likelihood"] is None
    else:
        lik = m.likelihood
        name = "variance" if lik_name == "gaussian" else "scale"
        p0 = float(getattr(lik, name))
        cd = _cd(m, data, lambda v: setattr(lik, name, v), p0, 1e-6)
        assert g["likelihood"] == pytest.approx(cd, rel=rtol, abs=atol)

