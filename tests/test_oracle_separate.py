"""
CPU: the restatement of separate kernels per latent and of the heteroskedastic likelihood (tests/separate_oracle.py), and the
host mapping of the new GPflow objects.
"""
import numpy as np
import pytest

from oracle import tsvgp_oracle as orc
from tests import separate_oracle as so


def _data(rng, N=300, D=2, M=25, L=2):
    X = rng.standard_normal((N, D))
    Y = np.stack([np.sin(X.sum(1) * (0.7 + 0.4 * l)) for l in range(L)], axis=1) + 0.2 * rng.standard_normal((N, L))
    return X, Y, X[:M].copy()


def _rel(a, b):
    return float(np.max(np.abs(np.asarray(a) - np.asarray(b))) / np.max(np.abs(b)))


def test_separate_with_equal_kernels_is_the_shared_kernel_model():
    rng = np.random.default_rng(0)
    X, Y, Z = _data(rng)
    k = orc.SquaredExponential(variance=1.1, lengthscales=0.4)
    lik = orc.Gaussian(variance=0.1)
    shared = orc.OracleTSVGP(k, lik, orc.InducingPoints(Z), num_latent_gps=2, num_data=900)
    sep = so.OracleSeparateTSVGP(so.SeparateIndependent([k, k]), lik, orc.InducingPoints(Z), num_latent_gps=2, num_data=900)
    for _ in range(2):
        shared.natgrad_step((X, Y), lr=0.6)
        sep.natgrad_step((X, Y), lr=0.6)
    assert _rel(sep.lambda_1, shared.lambda_1) < 1e-14 and _rel(sep.lambda_2, shared.lambda_2) < 1e-14
    assert abs(sep.elbo((X, Y)) - shared.elbo((X, Y))) < 1e-14 * abs(shared.elbo((X, Y)))
    assert abs(sep.prior_kl() - shared.prior_kl()) < 1e-14 * abs(shared.prior_kl())
    for a, b in zip(sep.predict_f(X[:40]), shared.predict_f(X[:40])):
        assert _rel(a, b) < 1e-14


def test_separate_independent_gaussian_is_two_single_latent_models():
    rng = np.random.default_rng(1)
    X, Y, Z = _data(rng, D=3)
    k1, k2 = orc.Matern52(variance=1.3, lengthscales=[0.8, 1.2, 2.0]), orc.SquaredExponential(variance=0.4, lengthscales=0.6)
    lik = orc.Gaussian(variance=0.15)
    sep = so.OracleSeparateTSVGP(so.SeparateIndependent([k1, k2]), lik, orc.InducingPoints(Z), num_latent_gps=2)
    ones = [orc.OracleTSVGP(k, lik, orc.InducingPoints(Z)) for k in (k1, k2)]
    for _ in range(2):
        sep.natgrad_step((X, Y), lr=0.5)
        for l, m in enumerate(ones):
            m.natgrad_step((X, Y[:, l:l + 1]), lr=0.5)
    for l, m in enumerate(ones):
        np.testing.assert_allclose(sep.lambda_1[:, l:l + 1], m.lambda_1, rtol=0, atol=1e-12 * np.max(np.abs(m.lambda_1)))
        np.testing.assert_allclose(sep.lambda_2[l], m.lambda_2[0], rtol=0, atol=1e-12 * np.max(np.abs(m.lambda_2)))
    e = sum(m.elbo((X, Y[:, l:l + 1])) for l, m in enumerate(ones))
    assert abs(sep.elbo((X, Y)) - e) < 1e-12 * abs(e)
    mu, var = sep.predict_f(X[:30])
    for l, m in enumerate(ones):
        mu_l, var_l = m.predict_f(X[:30])
        assert _rel(mu[:, l:l + 1], mu_l) < 1e-13 and _rel(var[:, l:l + 1], var_l) < 1e-13
    # full covariance: one block per latent kernel, its diagonal is predict_f's variance
    _, cov = sep.predict_f_full_cov(X[:30])
    assert cov.shape == (2, 30, 30)
    assert _rel(np.diagonal(cov, axis1=1, axis2=2).T, var) < 1e-12


def _moments(rng, N=50):
    mu = np.stack([rng.standard_normal(N), 0.5 * rng.standard_normal(N)], axis=1)
    var = np.stack([rng.uniform(0.05, 1.0, N), rng.uniform(0.01, 0.5, N)], axis=1)
    y = mu[:, :1] + rng.standard_normal((N, 1))
    return mu, var, y


def test_heteroskedastic_exp_expectation_has_its_closed_form():
    rng = np.random.default_rng(2)
    mu, var, y = _moments(rng)
    lik = so.HeteroskedasticTFPConditional(scale_transform=so.Exp())
    ve = lik.variational_expectations(mu, var, y)
    closed = (-0.5 * np.log(2 * np.pi) - mu[:, 1]
              - 0.5 * (np.square(y[:, 0] - mu[:, 0]) + var[:, 0]) * np.exp(-2 * mu[:, 1] + 2 * var[:, 1]))
    np.testing.assert_allclose(ve, closed, rtol=0, atol=1e-10)


@pytest.mark.parametrize("transform", ["exp", "softplus"])
def test_heteroskedastic_gradients_are_the_derivatives_of_the_quadrature(transform):
    rng = np.random.default_rng(3)
    mu, var, y = _moments(rng, N=20)
    lik = so.HeteroskedasticTFPConditional(scale_transform=so.Exp() if transform == "exp" else so.Softplus())
    _, g, h = lik.ve_and_grads(mu, var, y)
    eps = 1e-6
    for l in range(2):
        d = np.zeros_like(mu)
        d[:, l] = eps
        fd_g = (lik.variational_expectations(mu + d, var, y) - lik.variational_expectations(mu - d, var, y)) / (2 * eps)
        fd_h = (lik.variational_expectations(mu, var + d, y) - lik.variational_expectations(mu, var - d, y)) / (2 * eps)
        np.testing.assert_allclose(g[:, l], fd_g, rtol=1e-6, atol=1e-7)
        np.testing.assert_allclose(h[:, l], fd_h, rtol=1e-6, atol=1e-7)


def test_heteroskedastic_predictive_moments():
    rng = np.random.default_rng(4)
    mu, var, _ = _moments(rng)
    Ey, Vy = so.HeteroskedasticTFPConditional(scale_transform=so.Exp()).predict_mean_and_var(mu, var)
    np.testing.assert_allclose(Ey[:, 0], mu[:, 0], rtol=0, atol=1e-12)
    np.testing.assert_allclose(Vy[:, 0], var[:, 0] + np.exp(2 * mu[:, 1] + 2 * var[:, 1]), rtol=1e-10)


def _host_model(kernel, likelihood, mu, var):
    """A t_SVGP shell without a device context whose predict_f returns the given moments (host arithmetic only)."""
    import tsvgp_b200 as tb
    m = object.__new__(tb.t_SVGP)
    m.kernel, m.likelihood, m.num_latent_gps = kernel, likelihood, 2
    m.predict_f = lambda X, full_cov=False, full_output_cov=False: (mu, var)
    return m


@pytest.mark.parametrize("transform", ["exp", "softplus"])
def test_host_predict_y_and_log_density_match_the_quadrature(transform):
    from tsvgp_b200 import standins as st
    rng = np.random.default_rng(5)
    mu, var, y = _moments(rng, N=30)
    ref = so.HeteroskedasticTFPConditional(scale_transform=so.Exp() if transform == "exp" else so.Softplus())
    lik = st.HeteroskedasticTFPConditional(st.Normal, st.Exp() if transform == "exp" else st.Softplus())
    m = _host_model(st.SeparateIndependent([st.SquaredExponential(), st.SquaredExponential()]), lik, mu, var)
    Ey, Vy = m.predict_y(None)
    Ey_r, Vy_r = ref.predict_mean_and_var(mu, var)
    assert Ey.shape == (30, 1) and _rel(Ey, Ey_r) < 1e-12 and _rel(Vy, Vy_r) < 1e-12
    ld = m.predict_log_density((None, y))
    assert ld.shape == (30,) and _rel(ld, ref.predict_log_density(mu, var, y)) < 1e-12


def test_host_mapping_of_the_new_objects_and_refusals():
    import tsvgp_b200 as tb
    from tsvgp_b200 import _lib, model, standins as st
    k1, k2 = st.Matern52(1.0, 0.7), st.SquaredExponential(0.3, [3.0, 2.0])
    specs = model._kernel_spec(st.SeparateIndependent([k1, k2]), 2)
    assert [s[0] for s in specs] == [_lib.KERNEL_MATERN52, _lib.KERNEL_SE] and [s[1] for s in specs] == [1.0, 0.3]
    np.testing.assert_array_equal(specs[1][2], [3.0, 2.0])
    with pytest.raises(_lib.InvalidArgumentError):
        model._kernel_spec(st.SeparateIndependent([k1, k2]), 3)
    kind, var, ls = model._kernel_spec(st.SharedIndependent(k2, 2), 2)
    assert kind == _lib.KERNEL_SE and var == 0.3 and list(ls) == [3.0, 2.0]
    with pytest.raises(_lib.InvalidArgumentError):
        model._kernel_spec(st.SharedIndependent(k2, 3), 2)
    assert model._likelihood_spec(st.HeteroskedasticTFPConditional(st.Normal, st.Exp())) == (_lib.LIK_HETEROSKEDASTIC, 0.0, 0.0, 20)
    assert model._likelihood_spec(st.HeteroskedasticTFPConditional(st.Normal, st.Softplus(), 7)) == (_lib.LIK_HETEROSKEDASTIC, 1.0, 0.0, 7)

    class StudentT:
        pass

    class Sigmoid:
        pass

    class Lik:   # num_gauss_hermite_points is read when there is no .quadrature
        distribution_class, scale_transform, num_gauss_hermite_points = st.Normal, st.Exp(), 9

    Lik.__name__ = "HeteroskedasticTFPConditional"
    assert model._likelihood_spec(Lik())[3] == 9
    with pytest.raises(NotImplementedError):
        model._likelihood_spec(st.HeteroskedasticTFPConditional(StudentT, st.Exp()))
    with pytest.raises(NotImplementedError):
        model._likelihood_spec(st.HeteroskedasticTFPConditional(st.Normal, Sigmoid()))
    # not built: the whitened sibling with separate kernels (or the heteroskedastic likelihood), M-step gradients with either
    with pytest.raises(NotImplementedError):
        tb.t_SVGP_white(st.SeparateIndependent([k1, k2]), st.Gaussian(), np.zeros((4, 2)), num_latent_gps=2)
    with pytest.raises(NotImplementedError):
        tb.t_SVGP_white(k1, st.HeteroskedasticTFPConditional(), np.zeros((4, 2)), num_latent_gps=2)
    with pytest.raises(NotImplementedError):
        _host_model(st.SeparateIndependent([k1, k2]), st.Gaussian(), None, None).elbo_and_grad()
    with pytest.raises(NotImplementedError):
        _host_model(k1, st.HeteroskedasticTFPConditional(), None, None).elbo_and_grad()


def test_vem_fit_trains_the_kernel_inside_shared_independent():
    # host logic only: a model shell whose elbo_and_grad returns fixed gradients of the shared (unwrapped) kernel
    from tsvgp_b200 import standins as st, vem

    class Shell:
        def __init__(self, kernel):
            self.kernel, self.likelihood, self.inducing_variable = kernel, st.Gaussian(0.1), np.zeros((3, 2))

        def set_data(self, data):
            pass

        def natgrad_step(self, lr):
            pass

        def elbo_and_grad(self):
            return -1.0, {"variance": 1.0, "lengthscales": np.array([1.0, -1.0]), "Z": np.zeros((3, 2)), "likelihood": 1.0}

    inner = st.SquaredExponential(1.0, [1.0, 1.0])
    vem.fit(Shell(st.SharedIndependent(inner, 2)), (None, None), n_iters=1, n_e_steps=1, n_m_steps=3)
    assert inner.variance > 1.0 and inner.lengthscales[0] > 1.0 > inner.lengthscales[1]
    with pytest.raises(NotImplementedError):
        vem.fit(Shell(st.SeparateIndependent([inner, inner])), (None, None), n_iters=1)
