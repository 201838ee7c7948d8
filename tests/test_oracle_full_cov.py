"""
The CPU restatement (tests/full_cov_oracle.py) of the full predictive covariance (GPflow's base_conditional with
full_cov=True, white=False) and sample_mvn [GPflow-recalled], pinned by properties: its diagonal is predict_f's variance, it
is symmetric, L latents are L independent single-latent models, and at the reference's Gaussian fixed point it is exact GP
regression's posterior covariance — the whole-matrix extension of the reference's diagonal pin (tests/models/test_tsvgp.py:113-120).
"""
import numpy as np

from oracle import tsvgp_oracle as orc
from tests import full_cov_oracle as fco
from tests.test_oracle_properties import _setup


def _trained(L=1, steps=3, seed=4):
    rng = np.random.default_rng(seed)
    X = rng.uniform(-2.0, 2.0, (60, 2))
    Y = np.stack([np.sin(X.sum(1) * (1.0 + 0.4 * l)) for l in range(L)], 1) + 0.1 * rng.standard_normal((60, L))
    kernel = orc.Matern52(variance=1.3, lengthscales=0.9)
    m = orc.OracleTSVGP(kernel, orc.Gaussian(variance=0.05), orc.InducingPoints(X[:25].copy()), num_latent_gps=L, num_data=120)
    for _ in range(steps):
        m.natgrad_step((X, Y), lr=0.7)
    return m, X, Y


def test_diagonal_is_predict_f_variance_and_symmetric():
    m, X, _ = _trained(L=2)
    Xs = X[:40] + 0.3
    mu_f, cov = fco.predict_f_full_cov(m, Xs)
    mu, var = m.predict_f(Xs)
    assert cov.shape == (2, 40, 40) and mu_f.shape == (40, 2)
    np.testing.assert_array_equal(mu_f, mu)
    assert np.max(np.abs(np.diagonal(cov, axis1=1, axis2=2).T - var)) <= 1e-12
    for l in range(2):
        assert np.max(np.abs(cov[l] - cov[l].T)) <= 1e-14 * np.max(np.abs(cov[l]))


def test_latents_are_independent_models():
    m, X, _ = _trained(L=3)
    Xs = X[::3] - 0.2
    mu, cov = fco.predict_f_full_cov(m, Xs)
    for l in range(3):
        one = orc.OracleTSVGP(m.kernel, m.likelihood, m.inducing_variable, lambda_1=m.lambda_1[:, l:l + 1],
                              lambda_2_sqrt=m.lambda_2_sqrt[l:l + 1])
        mu1, cov1 = fco.predict_f_full_cov(one, Xs)
        np.testing.assert_allclose(mu1[:, 0], mu[:, l], rtol=0, atol=1e-12 * np.max(np.abs(mu)))
        np.testing.assert_allclose(cov1[0], cov[l], rtol=0, atol=1e-12 * np.max(np.abs(cov)))


def test_full_covariance_matches_gpr_at_the_fixed_point():
    # reference tests/models/test_tsvgp.py:20-42 and :113-120 (Z = X, 10 natgrad steps at lr 0.9), whole matrix at X + 1
    rng = np.random.RandomState(123)
    X, Y, kernel, s2 = _setup(rng)
    m = orc.OracleTSVGP(kernel, orc.Gaussian(variance=s2), orc.InducingPoints(X.copy()))
    for _ in range(10):
        m.natgrad_step((X, Y), lr=0.9)
    Xs = X + 1.0
    mu, cov = fco.predict_f_full_cov(m, Xs)
    mu_g, cov_g = fco.gpr_predict_f_full_cov(kernel, X, Y, s2, Xs)
    np.testing.assert_array_almost_equal(mu, mu_g, decimal=4)
    np.testing.assert_array_almost_equal(cov, cov_g, decimal=4)
    # the closed form's diagonal is the diagonal-only closed form
    np.testing.assert_allclose(np.diagonal(cov_g[0]), orc.gpr_predict_f(kernel, X, Y, s2, Xs)[1][:, 0], rtol=1e-12)


def test_sample_mvn_with_given_draws():
    m, X, _ = _trained(L=2)
    Xs = X[:30] * 1.5
    rng = np.random.default_rng(0)
    eps = rng.standard_normal((7, 30, 2))
    mu, cov = fco.predict_f_full_cov(m, Xs)
    for l in range(2):
        C = np.linalg.cholesky(cov[l] + 1e-6 * np.eye(30))
        np.testing.assert_allclose(fco.sample_mvn(mu[:, l], cov[l], eps[:, :, l].T), mu[:, l:l + 1] + C @ eps[:, :, l].T,
                                   rtol=0, atol=1e-13)
    f = fco.predict_f_samples(m, Xs, 7, full_cov=True, epsilon=eps)
    assert f.shape == (7, 30, 2)
    np.testing.assert_allclose(f[:, :, 1], (mu[:, 1:2] + np.linalg.cholesky(cov[1] + 1e-6 * np.eye(30)) @ eps[:, :, 1].T).T,
                               rtol=0, atol=1e-13)
    mu_d, var_d = m.predict_f(Xs)
    np.testing.assert_array_equal(fco.predict_f_samples(m, Xs, 7, full_cov=False, epsilon=eps), mu_d + np.sqrt(var_d) * eps)
    assert fco.predict_f_samples(m, Xs, None, full_cov=False, epsilon=eps[:1]).shape == (30, 2)
