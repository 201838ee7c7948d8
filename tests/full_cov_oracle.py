"""
CPU restatement of the full predictive covariance and of posterior sampling, for the tests of predict_f(full_cov=True) and
predict_f_samples.  TEST INFRASTRUCTURE ONLY, built on the oracle (oracle/tsvgp_oracle.py), whose functions it reuses unchanged:

  * ``base_conditional_full_cov``   gpflow.conditionals.util.base_conditional, full_cov=True, white=False   [GPflow-recalled]
  * ``sample_mvn``                  gpflow.conditionals.util.sample_mvn, full_cov=True                   [GPflow-recalled]
  * ``predict_f_full_cov`` / ``predict_f_samples``   base_SVGP.predict_f (tsvgp.py:97-114) with full_cov=True, and
    GPModel.predict_f_samples, for an ``OracleTSVGP``
  * ``gpr_predict_f_full_cov``      gpflow.models.GPR.predict_f, full_cov=True, in closed form

GPflow cannot be installed here and no reference test exercises full_cov=True (SURVEY §3.3): the GPflow order is restated from
its published source (SURVEY Appendix B).
"""
import numpy as np

from oracle import tsvgp_oracle as orc


def base_conditional_full_cov(Kmn, Kmm, Knn, f, q_sqrt):
    """base_conditional, full_cov=True, white=False, in GPflow's own order.  Knn [N, N] -> fmean [N, L], fvar [L, N, N]."""
    Lm = orc.cholesky(Kmm)
    A = orc.triangular_solve(Lm, Kmn)  # [M,N]
    fvar = Knn - A.T @ A  # [N,N]
    A = orc.triangular_solve(Lm, A, adjoint=True)  # unwhitened
    fmean = A.T @ f  # [N,L]
    Lq = np.tril(q_sqrt)
    fvar_out = np.empty((Lq.shape[0],) + fvar.shape)
    for l in range(Lq.shape[0]):
        LTA = Lq[l].T @ A  # [M,N]
        fvar_out[l] = fvar + LTA.T @ LTA
    return fmean, fvar_out


def sample_mvn(mean, cov, eps, jitter=orc.DEFAULT_JITTER):
    """sample_mvn, full_cov=True: mean + cholesky(cov + jitter I) @ eps.  mean [N], cov [N, N], eps [N, S] -> [N, S].
    GPflow's own draw layout is not restated: draws are never comparable across implementations, only the transform of given
    draws is."""
    chol = orc.cholesky(cov + jitter * np.eye(cov.shape[-1]))
    return mean[:, None] + chol @ eps


def predict_f_full_cov(model, Xnew):
    """OracleTSVGP.predict_f with full_cov=True -> (mean [N, L], cov [L, N, N]).  assert_positive (tsvgp.py:113) is applied to
    the diagonal only: off-diagonal covariances may be <= 0 in any posterior."""
    Xnew = np.asarray(Xnew, dtype=np.float64)
    q_mu, q_sqrt = model.get_mean_chol_cov_inducing_posterior()
    Kmm = orc.Kuu(model.inducing_variable, model.kernel, jitter=orc.DEFAULT_JITTER)
    Kmn = orc.Kuf(model.inducing_variable, model.kernel, Xnew)
    mu, cov = base_conditional_full_cov(Kmn, Kmm, model.kernel.K(Xnew), q_mu, q_sqrt)
    if not np.all(np.diagonal(cov, axis1=-2, axis2=-1) > 0):
        raise FloatingPointError("predict_f: non-positive predictive variance")
    return mu + model._mean_fn(Xnew), cov


def predict_f_samples(model, Xnew, num_samples=None, full_cov=True, *, epsilon):
    """GPModel.predict_f_samples with the standard normals given: epsilon [S, N, L] -> [S, N, L] ([N, L] for num_samples None).
    full_cov: sample_mvn per latent; otherwise mean + sqrt(var) * epsilon."""
    eps = np.asarray(epsilon, dtype=np.float64)
    if full_cov:
        mu, cov = predict_f_full_cov(model, Xnew)
        out = np.stack([sample_mvn(mu[:, l], cov[l], eps[:, :, l].T).T for l in range(mu.shape[1])], axis=-1)
    else:
        mu, var = model.predict_f(Xnew)
        out = mu[None] + np.sqrt(var)[None] * eps
    return out[0] if num_samples is None else out


def gpr_predict_f_full_cov(kernel, X, Y, noise_variance, Xnew):
    """GPR.predict_f, full_cov=True: Kss - Ksx (Kxx + s2 I)^-1 Kxs -> (mean [N, 1], cov [1, N, N])."""
    N = X.shape[0]
    Lm = orc.cholesky(kernel.K(X) + noise_variance * np.eye(N))
    A = orc.triangular_solve(Lm, kernel.K(X, Xnew))
    fmean = A.T @ orc.triangular_solve(Lm, Y)
    return fmean, (kernel.K(Xnew) - A.T @ A)[None]
