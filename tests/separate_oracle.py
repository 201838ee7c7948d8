"""
CPU restatement of separate kernels per latent and of the heteroskedastic likelihood, for the tests of tsvgp_set_kernels and
TSVGP_LIK_HETEROSKEDASTIC.  TEST INFRASTRUCTURE ONLY, built on the oracle (oracle/tsvgp_oracle.py), whose functions it reuses
unchanged:

  * ``SeparateIndependent``            gpflow.kernels.SeparateIndependent: ``.kernels``, K / K_diag per latent    [GPflow-recalled]
  * ``OracleSeparateTSVGP``            the reference's t_SVGP (tsvgp.py:117-304) with latent l on ``kernel.kernels[l]``: the
                                       conditional is separate_independent_conditional (base_conditional per latent with
                                       Kmm = k_l(Z) + 1e-6 I, Knn = k_l.K_diag), gauss_kl sums the latents' terms, and
                                       natgrad_step follows tsvgp.py:243-304 latent by latent
  * ``HeteroskedasticTFPConditional``  Normal(loc = f_0, scale = T(f_1)) with NDiagGHQuadrature(2, n_gh), on the literal
                                       n_gh x n_gh grid                                                          [GPflow-recalled]
  * ``predict_f_full_cov``             the per-latent full covariance beside tests/full_cov_oracle.py
"""
import numpy as np
from scipy.special import logsumexp

from oracle import tsvgp_oracle as orc
from tests import full_cov_oracle as fco


class SeparateIndependent:
    def __init__(self, kernels):
        self.kernels = list(kernels)

    def K(self, X, X2=None):   # [L, N, N2]
        return np.stack([k.K(X, X2) for k in self.kernels])

    def K_diag(self, X):       # [N, L]
        return np.stack([k.K_diag(X) for k in self.kernels], axis=-1)


class Normal:
    """tfp.distributions.Normal: the class name is what the device model reads."""


class Exp:
    def __call__(self, f):
        return np.exp(f)


class Softplus:
    def __call__(self, f):
        return np.logaddexp(0.0, f)


class HeteroskedasticTFPConditional:
    name = "heteroskedastic"

    def __init__(self, distribution_class=Normal, scale_transform=None, num_gauss_hermite_points=orc.N_GH):
        self.distribution_class = distribution_class
        self.scale_transform = Exp() if scale_transform is None else scale_transform
        self.latent_dim = 2
        self.num_gauss_hermite_points = int(num_gauss_hermite_points)

    def _grid(self, Fmu, Fvar):
        """f = mu + sqrt(v) (z_i, z_j), weights w_i w_j: F0 [N, n, n], F1 [N, n, n], W [n, n], Z0, Z1 [n, n]."""
        z, w = orc.gh_points_and_weights(self.num_gauss_hermite_points)
        Z0, Z1 = np.meshgrid(z, z, indexing="ij")
        W = np.outer(w, w)
        sd = np.sqrt(Fvar)
        F0 = Fmu[:, 0, None, None] + sd[:, 0, None, None] * Z0
        F1 = Fmu[:, 1, None, None] + sd[:, 1, None, None] * Z1
        return F0, F1, W, Z0, Z1, sd

    def _logp(self, F0, F1, Y):
        s = self.scale_transform(F1)
        return -0.5 * np.log(2 * np.pi) - np.log(s) - 0.5 * np.square((Y - F0) / s)

    def _dlogp(self, F0, F1, Y):
        s = self.scale_transform(F1)
        r = Y - F0
        ds = s if isinstance(self.scale_transform, Exp) else 1.0 / (1.0 + np.exp(-F1))   # T'(f_1)
        return r / np.square(s), ds / s * (np.square(r / s) - 1.0)

    def variational_expectations(self, Fmu, Fvar, Y):
        F0, F1, W, *_ = self._grid(Fmu, Fvar)
        return np.sum(W * self._logp(F0, F1, Y.reshape(-1, 1, 1)), axis=(1, 2))

    def ve_and_grads(self, Fmu, Fvar, Y):
        F0, F1, W, Z0, Z1, sd = self._grid(Fmu, Fvar)
        y = Y.reshape(-1, 1, 1)
        ve = np.sum(W * self._logp(F0, F1, y), axis=(1, 2))
        d0, d1 = self._dlogp(F0, F1, y)
        g = np.stack([np.sum(W * d0, axis=(1, 2)), np.sum(W * d1, axis=(1, 2))], axis=-1)
        h = np.stack([np.sum(W * d0 * Z0, axis=(1, 2)) / (2 * sd[:, 0]), np.sum(W * d1 * Z1, axis=(1, 2)) / (2 * sd[:, 1])], axis=-1)
        return ve, g, h

    def predict_mean_and_var(self, Fmu, Fvar):   # QuadratureLikelihood: E[loc], E[scale^2 + loc^2] - E[loc]^2
        F0, F1, W, *_ = self._grid(Fmu, Fvar)
        Ey = np.sum(W * F0, axis=(1, 2))
        Ey2 = np.sum(W * (np.square(self.scale_transform(F1)) + np.square(F0)), axis=(1, 2))
        return Ey[:, None], (Ey2 - np.square(Ey))[:, None]

    def predict_log_density(self, Fmu, Fvar, Y):
        F0, F1, W, *_ = self._grid(Fmu, Fvar)
        return logsumexp(self._logp(F0, F1, Y.reshape(-1, 1, 1)) + np.log(W), axis=(1, 2))


class OracleSeparateTSVGP:
    """t_SVGP with kernel = SeparateIndependent(kernels): latent l is a one-latent OracleTSVGP on kernels[l] for every kernel-
    dependent quantity; the likelihood sees all latents of a point together."""

    def __init__(self, kernel, likelihood, inducing_variable, *, num_latent_gps, num_data=None):
        assert len(kernel.kernels) == num_latent_gps
        self.kernel, self.likelihood, self.num_data = kernel, likelihood, num_data
        self.num_latent_gps = L = num_latent_gps
        self.inducing_variable = inducing_variable if hasattr(inducing_variable, "Z") else orc.InducingPoints(inducing_variable)
        M = self.inducing_variable.num_inducing
        self.lambda_1 = np.zeros((M, L))                                              # tsvgp.py:174
        self.lambda_2_sqrt = np.array([-np.eye(M) * 1e-10 for _ in range(L)])        # tsvgp.py:175-180

    def _latent(self, l):
        return orc.OracleTSVGP(self.kernel.kernels[l], orc.Gaussian(), self.inducing_variable, num_latent_gps=1,
                               lambda_1=self.lambda_1[:, l:l + 1], lambda_2_sqrt=self.lambda_2_sqrt[l:l + 1], num_data=self.num_data)

    @property
    def lambda_2(self):
        return self.lambda_2_sqrt @ np.swapaxes(self.lambda_2_sqrt, -1, -2)

    def get_mean_chol_cov_inducing_posterior(self):
        parts = [self._latent(l).get_mean_chol_cov_inducing_posterior() for l in range(self.num_latent_gps)]
        return np.concatenate([m for m, _ in parts], axis=1), np.concatenate([s for _, s in parts], axis=0)

    def prior_kl(self):   # gauss_kl with K [L, M, M]: the latents' terms, each with its own log det K6_l
        return sum(self._latent(l).prior_kl() for l in range(self.num_latent_gps))

    def predict_f(self, Xnew):
        parts = [self._latent(l).predict_f(Xnew) for l in range(self.num_latent_gps)]
        return np.concatenate([m for m, _ in parts], axis=1), np.concatenate([v for _, v in parts], axis=1)

    def predict_f_full_cov(self, Xnew):
        parts = [fco.predict_f_full_cov(self._latent(l), Xnew) for l in range(self.num_latent_gps)]
        return np.concatenate([m for m, _ in parts], axis=1), np.concatenate([c for _, c in parts], axis=0)

    def predict_f_samples(self, Xnew, num_samples, full_cov=True, *, epsilon):
        eps = np.asarray(epsilon, dtype=np.float64)
        return np.concatenate([fco.predict_f_samples(self._latent(l), Xnew, num_samples, full_cov, epsilon=eps[:, :, l:l + 1])
                               for l in range(self.num_latent_gps)], axis=-1)

    def elbo(self, data):
        X, Y = (np.asarray(a, dtype=np.float64) for a in data)
        f_mean, f_var = self.predict_f(X)
        scale_ = self.num_data / X.shape[0] if self.num_data is not None else 1.0
        return np.sum(self.likelihood.variational_expectations(f_mean, f_var, Y)) * scale_ - self.prior_kl()

    def natgrad_step(self, data, lr=0.1, jitter=1e-9):   # tsvgp.py:234-304, per latent with its own kernel
        X, Y = (np.asarray(a, dtype=np.float64) for a in data)
        mean, var = self.predict_f(X)                                              # :246
        Z = np.asarray(self.inducing_variable.Z)
        _, g_mean, g_var = self.likelihood.ve_and_grads(mean, var, Y)             # :256-259
        g_var = np.minimum(g_var, -1e-8)                                           # :262-263
        M = Z.shape[0]
        Id = np.eye(M)
        scale_ = self.num_data / X.shape[0] if self.num_data is not None else 1.0  # :286-291
        new_l1, new_sqrt = np.empty_like(self.lambda_1), np.empty_like(self.lambda_2_sqrt)
        for l in range(self.num_latent_gps):
            sub = self._latent(l)
            meanZ, _ = sub.predict_f(Z)                                            # :254
            K_uu = orc.Kuu(self.inducing_variable, self.kernel.kernels[l])         # :268
            K_uf = orc.Kuf(self.inducing_variable, self.kernel.kernels[l], X)      # :269
            A = orc.cholesky_solve(orc.cholesky(K_uu + Id * jitter), K_uf).T       # :270-271
            G1 = A.T @ g_mean[:, l:l + 1]                                          # :279
            G2 = ((A * g_var[:, l:l + 1]).T @ A)[None]                             # :280
            grad_mu = orc.gradient_transformation_mean_var_to_expectation(meanZ, (G1, G2))   # :284
            lambda_2 = -0.5 * sub.lambda_2                                         # :293
            new_l1[:, l:l + 1] = (1 - lr) * sub.lambda_1 + lr * scale_ * grad_mu[0]          # :296
            lambda_2 = (1 - lr) * lambda_2 + lr * scale_ * grad_mu[1]              # :297
            new_sqrt[l] = -orc.cholesky(-2.0 * lambda_2[0] + Id * jitter)          # :300
        self.lambda_1, self.lambda_2_sqrt = new_l1, new_sqrt                       # :302-303
