"""
CPU restatement of the M-step gradients of the whitened sibling t_SVGP_white (DESIGN §10, "M-step gradients"), on top of the
unchanged oracle.tsvgp_oracle.OracleTSVGPWhite: d ELBO / d kernel variance, lengthscales, Z and the likelihood parameter with the
sites (lambda_1, Lambda_2) held fixed.  For latent l, with A = Kuu + 1e-6 I:

    R  = Lambda_2 + A + 1e-9 I   (the conditional's matrix)     alpha  = R^-1 lambda_1      Q = A^-1 - R^-1
    R0 = Lambda_2 + A            (the KL's matrix, no 1e-9)     alpha0 = R0^-1 lambda_1
    B  = Kuf diag(h) Kfu,  b = Kuf g   (h unclipped)
    Gamma_uf = s (alpha g^T - 2 Q Kuf diag(h))
    Gamma_K  = s [A^-1 B A^-1 - R^-1 B R^-1 - sym(R^-1 b alpha^T)]
               - 1/2 [2 R0^-1 - A^-1 - R0^-1 A R0^-1 + alpha0 alpha0^T - 2 sym(R0^-1 A alpha0 alpha0^T)]

The lengthscale and Z gradients follow from E = Gamma o dK/dr2 exactly as in oracle.tsvgp_oracle.elbo_gradients (E_uu with a zero
diagonal); dK/dr2 comes from tests/matern_oracle.kernel_dr2, which covers all four kernels.  The latents add up.
"""
import numpy as np

from oracle import tsvgp_oracle as orc
from tests import matern_oracle as mo


def _sym(A):
    return 0.5 * (A + A.T)


def _inv_spd(A):
    iL = orc.triangular_solve(orc.cholesky(A), np.eye(A.shape[0]))
    return iL.T @ iL


def elbo_gradients(model, data):
    """-> (elbo, dict(variance=, lengthscales=[D] or [1], Z=[M, D], likelihood=)) of an OracleTSVGPWhite with a Zero mean function
    and any number of latents (Y [N, L]).  `likelihood` is d/d variance (Gaussian), d/d scale (StudentT) or None (Bernoulli)."""
    X, Y = (np.asarray(a, dtype=np.float64) for a in data)
    kernel, lik = model.kernel, model.likelihood
    Z = np.asarray(model.inducing_variable.Z, dtype=np.float64)
    M, D = Z.shape
    N = X.shape[0]
    ls = np.broadcast_to(np.asarray(kernel.lengthscales, dtype=np.float64).reshape(-1), (D,)).copy()
    var = float(kernel.variance)
    s = model.num_data / N if model.num_data is not None else 1.0
    K = kernel.K(Z)
    A = K + orc.DEFAULT_JITTER * np.eye(M)
    Kuf_ = kernel.K(Z, X)
    Kff = kernel.K_diag(X)[:, None]
    # the ELBO exactly as OracleTSVGPWhite.elbo forms it
    mu, v = orc.conditional_from_precision_sites_white(A, Kff, Kuf_, model.lambda_1, model.lambda_2)
    ve, g_all, h_all = lik.ve_and_grads(mu, v, Y)
    elbo = np.sum(ve) * s - orc.kl_from_precision_sites_white(A, model.lambda_1, model.lambda_2)

    Ainv = _inv_spd(A)
    G_uf = np.zeros((M, N))
    G_K = np.zeros((M, M))
    for l in range(model.lambda_2.shape[0]):
        lam1, Lam2 = model.lambda_1[:, l], model.lambda_2[l]
        Rinv = _inv_spd(Lam2 + A + 1e-9 * np.eye(M))
        R0inv = _inv_spd(Lam2 + A)
        alpha, alpha0 = Rinv @ lam1, R0inv @ lam1
        Q = Ainv - Rinv
        g, h = g_all[:, l], h_all[:, l]
        b = Kuf_ @ g
        B = (Kuf_ * h) @ Kuf_.T
        G_uf += s * (np.outer(alpha, g) - 2.0 * (Q @ Kuf_) * h)
        G_K += s * (Ainv @ B @ Ainv - Rinv @ B @ Rinv - _sym(np.outer(Rinv @ b, alpha))) \
            - 0.5 * (2.0 * R0inv - Ainv - R0inv @ A @ R0inv + np.outer(alpha0, alpha0) - 2.0 * _sym(np.outer(R0inv @ A @ alpha0, alpha0)))

    Zs, Xs = Z / ls, X / ls
    E_uf = G_uf * mo.kernel_dr2(kernel, orc.square_distance(Zs, Xs))
    E_uu = G_K * mo.kernel_dr2(kernel, orc.square_distance(Zs, None))
    np.fill_diagonal(E_uu, 0.0)                       # r = 0 on the diagonal: no dependence on Z or the lengthscales
    d_ls = np.empty(D)
    d_Z = np.empty((M, D))
    for d in range(D):
        duf = Zs[:, d:d + 1] - Xs[None, :, d]
        duu = Zs[:, d:d + 1] - Zs[None, :, d]
        d_ls[d] = -(2.0 / ls[d]) * (np.sum(E_uf * duf * duf) + np.sum(E_uu * duu * duu))
        d_Z[:, d] = (2.0 / ls[d]) * (np.sum(E_uf * duf, axis=1) + 2.0 * np.sum(E_uu * duu, axis=1))
    d_var = (np.sum(G_uf * Kuf_) + np.sum(G_K * K)) / var + s * np.sum(h_all)
    if isinstance(lik, orc.Gaussian):
        s2 = float(lik.variance)
        d_lik = s * np.sum(-0.5 / s2 + 0.5 * (np.square(Y - mu) + v) / (s2 * s2))
    elif isinstance(lik, orc.StudentT):
        z, w = orc.gh_points_and_weights(lik.n_gh)
        r_ = Y[..., None] - (mu[..., None] + np.sqrt(v)[..., None] * z)
        sc, df = float(lik.scale), lik.df
        d_lik = s * np.sum((-1.0 / sc + (df + 1.0) * np.square(r_) / (sc * (df * sc * sc + np.square(r_)))) * w)
    else:
        d_lik = None
    if np.asarray(kernel.lengthscales).size == 1:
        d_ls = np.array([np.sum(d_ls)])
    return elbo, dict(variance=d_var, lengthscales=d_ls, Z=d_Z, likelihood=d_lik)
