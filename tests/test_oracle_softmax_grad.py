"""
The L-latent M-step gradients of tests/softmax_grad_oracle.py on the CPU: against central differences of the reference-order
OracleTSVGP.elbo with the Softmax likelihood and fixed Monte-Carlo draws (then the ELBO is a deterministic function of the
hyperparameters), and, for independent likelihood terms, against the sum of the oracle's one-latent gradients.
"""
import copy

import numpy as np
import pytest

from oracle import tsvgp_oracle as orc
from tests import softmax_grad_oracle as sgo


def _softmax_model(kind, C, ls, num_data, S=7, seed=11):
    rng = np.random.default_rng(seed)
    N, M, D = 90, 8, 3
    X = rng.standard_normal((N, D))
    Z = X[:M] + 0.1 * rng.standard_normal((M, D))
    W = rng.standard_normal((D, C))
    labels = np.argmax(X @ W + 0.5 * rng.standard_normal((N, C)), axis=1).astype(float)[:, None]
    kernel = (orc.SquaredExponential if kind == "se" else orc.Matern52)(variance=1.3, lengthscales=ls)
    lik = orc.Softmax(C, num_monte_carlo_points=S, epsilon=rng.standard_normal((S, N, C)))
    m = orc.OracleTSVGP(kernel, lik, orc.InducingPoints(Z), num_latent_gps=C, num_data=num_data)
    for _ in range(2):
        m.natgrad_step((X, labels), lr=0.5)
    return m, (X, labels)


def _fd(m, data, setter, x0, h):
    def f(x):
        mm = copy.copy(m)
        mm.kernel, mm.inducing_variable = copy.deepcopy(m.kernel), copy.deepcopy(m.inducing_variable)
        setter(mm, x)
        return mm.elbo(data)
    return (f(x0 + h) - f(x0 - h)) / (2 * h)


@pytest.mark.parametrize("kind,C,ls,num_data", [("se", 2, np.array([1.2, 1.6, 2.0]), None),
                                                ("matern52", 5, np.array([1.4, 1.1, 1.9]), 400),
                                                ("se", 5, 1.5, 300),
                                                ("matern52", 2, 1.7, None)])
def test_softmax_gradients_match_central_differences(kind, C, ls, num_data):
    m, data = _softmax_model(kind, C, ls, num_data)
    elbo, g = sgo.elbo_gradients(m, data)
    assert abs(elbo - m.elbo(data)) < 1e-9 * abs(elbo)
    assert g["likelihood"] is None
    tol = dict(rtol=2e-6, atol=1e-6)
    fd = _fd(m, data, lambda mm, x: setattr(mm.kernel, "variance", orc._param(x)), float(m.kernel.variance), 1e-5)
    np.testing.assert_allclose(g["variance"], fd, **tol)
    ls0 = np.atleast_1d(np.asarray(m.kernel.lengthscales, dtype=float))
    assert g["lengthscales"].shape == ls0.shape
    for d in range(ls0.size):
        def set_ls(mm, x, d=d):
            l = ls0.copy(); l[d] = x
            mm.kernel.lengthscales = orc._param(l if ls0.size > 1 else l[0])
        np.testing.assert_allclose(g["lengthscales"][d], _fd(m, data, set_ls, ls0[d], 1e-5), **tol)
    Z0 = np.asarray(m.inducing_variable.Z).copy()
    for (i, d) in [(0, 0), (3, 1), (7, 2), (5, 0)]:
        def set_z(mm, x, i=i, d=d):
            Zn = Z0.copy(); Zn[i, d] = x
            mm.inducing_variable = orc.InducingPoints(Zn)
        np.testing.assert_allclose(g["Z"][i, d], _fd(m, data, set_z, Z0[i, d], 1e-5), **tol)


def test_softmax_gradient_uses_unclipped_h():
    # with few draws some h_l are positive; the gradient of the Monte-Carlo ELBO must see them as they are
    m, (X, Y) = _softmax_model("se", 5, 1.5, None, S=1)
    mu, var = m.predict_f(X)
    _, _, h = m.likelihood.ve_and_grads(mu, var, Y)
    assert np.any(h > -1e-8)
    _, g = sgo.elbo_gradients(m, (X, Y))
    fd = _fd(m, (X, Y), lambda mm, x: setattr(mm.kernel, "variance", orc._param(x)), float(m.kernel.variance), 1e-5)
    np.testing.assert_allclose(g["variance"], fd, rtol=2e-6, atol=1e-6)


@pytest.mark.parametrize("kind,ard", [("se", True), ("matern52", False)])
def test_independent_latents_sum_the_one_latent_oracle(kind, ard):
    rng = np.random.default_rng(4)
    N, M, D, L = 150, 10, 3, 3
    X = rng.standard_normal((N, D))
    Z = X[:M] + 0.1 * rng.standard_normal((M, D))
    Y = np.stack([np.sin(X[:, 0]), np.cos(X[:, 1]), X[:, 2] * X[:, 0]], 1) + 0.2 * rng.standard_normal((N, L))
    kernel = (orc.SquaredExponential if kind == "se" else orc.Matern52)(variance=1.2, lengthscales=np.array([1.1, 1.4, 0.9]) if ard else 1.3)
    lik = orc.Gaussian(variance=0.15)
    m = orc.OracleTSVGP(kernel, lik, orc.InducingPoints(Z), num_latent_gps=L, num_data=600)
    for _ in range(2):
        m.natgrad_step((X, Y), lr=0.6)
    e, g = sgo.elbo_gradients(m, (X, Y))
    assert abs(e - m.elbo((X, Y))) < 1e-10 * abs(e)
    e_sum, g_sum = 0.0, None
    for l in range(L):
        one = orc.OracleTSVGP(kernel, lik, orc.InducingPoints(Z), lambda_1=m.lambda_1[:, l:l + 1],
                              lambda_2_sqrt=m.lambda_2_sqrt[l:l + 1], num_data=600)
        e_l, g_l = orc.elbo_gradients(one, (X, Y[:, l:l + 1]))
        e_sum += e_l
        g_sum = g_l if g_sum is None else {k: g_sum[k] + g_l[k] for k in g_l}
    assert abs(e - e_sum) < 1e-12 * abs(e)
    for k in ("variance", "lengthscales", "Z", "likelihood"):
        np.testing.assert_allclose(g[k], g_sum[k], rtol=1e-11, atol=1e-11 * np.max(np.abs(g_sum[k])))
