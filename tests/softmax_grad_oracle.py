"""
CPU restatement of the M-step gradients for L latents sharing one kernel, for the tests of tsvgp_elbo_grad with the Softmax
likelihood and of the augmented blocks at any input dimension.  TEST INFRASTRUCTURE ONLY, built on the oracle
(oracle/tsvgp_oracle.py), whose functions it reuses unchanged:

  * ``elbo_gradients``   oracle.elbo_gradients restated per latent and summed (DESIGN §9, "Coupled likelihood").  Kuf and Kuu
                         are shared, so dELBO/dKuf and dELBO/dKuu are sums of the one-latent expressions with each latent's
                         Q_l, B_l, b_l, alpha_l, m_l; the likelihood enters only through g_l = d ve / d mu_l and h_l = d ve / d v_l
                         of ``likelihood.ve_and_grads`` on [N, L] moments (h unclipped: the clip belongs to natgrad_step).
                         For the Softmax likelihood these are the analytic derivatives of the Monte-Carlo sum for the fixed
                         draws ``likelihood.epsilon`` — what GPflow's GradientTape gives for fixed draws.  The oracle's
                         sums over (inducing point, data point) pairs are taken as products over the points in coordinates
                         relative to the centroid of Z (at D = 784 the pair-by-pair loop would take minutes); the CPU tests
                         tie this form to central differences and to the oracle's own one-latent gradients.
"""
import numpy as np

from oracle import tsvgp_oracle as orc


def elbo_gradients(model, data):
    """-> (elbo, dict(variance=, lengthscales=[D] or [1], Z=[M, D], likelihood=...)) for num_latent_gps = L >= 1, one kernel
    shared by the latents, Zero mean function.  `likelihood` is d/d variance (Gaussian), d/d scale (StudentT), None otherwise."""
    X, Y = (np.asarray(a, dtype=np.float64) for a in data)
    kernel, lik = model.kernel, model.likelihood
    Z = np.asarray(model.inducing_variable.Z)
    M, D = Z.shape
    N = X.shape[0]
    L = model.lambda_1.shape[1]
    ls = np.broadcast_to(np.asarray(kernel.lengthscales, dtype=np.float64).reshape(-1), (D,)).copy()
    var = float(kernel.variance)
    s = model.num_data / N if model.num_data is not None else 1.0
    K = kernel.K(Z)
    K6 = K + orc.DEFAULT_JITTER * np.eye(M)
    Kuf_ = kernel.K(Z, X)
    sym = lambda A: 0.5 * (A + A.T)  # noqa: E731
    alphas, Qs, ms, Us, mu, v, kl = [], [], [], [], np.empty((N, L)), np.empty((N, L)), 0.0
    for l in range(L):
        Lam2 = model.lambda_2_sqrt[l] @ model.lambda_2_sqrt[l].T
        IK = np.eye(M) + Lam2 @ K6
        alpha = np.linalg.solve(IK, model.lambda_1[:, l])     # K6^-1 m_q
        Q = np.linalg.solve(IK, Lam2)                         # (Lam2^-1 + K6)^-1, symmetric
        Q = 0.5 * (Q + Q.T)
        m = K6 @ alpha
        mu[:, l] = Kuf_.T @ alpha
        U = Q @ Kuf_
        v[:, l] = var - np.sum(Kuf_ * U, axis=0)
        kl += 0.5 * (m @ alpha - np.trace(Q @ K6) + np.linalg.slogdet(IK)[1])
        alphas.append(alpha); Qs.append(Q); ms.append(m); Us.append(U)
    ve, g, h = lik.ve_and_grads(mu, v, Y)
    g, h = np.reshape(g, (N, L)), np.reshape(h, (N, L))
    elbo = s * np.sum(ve) - kl
    G_uf, G_K = np.zeros((M, N)), np.zeros((M, M))
    for l in range(L):
        alpha, Q, m = alphas[l], Qs[l], ms[l]
        b = Kuf_ @ g[:, l]
        B = (Kuf_ * h[:, l]) @ Kuf_.T
        G_uf += s * (np.outer(alpha, g[:, l]) - 2.0 * Us[l] * h[:, l])
        G_K += s * (Q @ B @ Q - sym(np.outer(Q @ b, alpha))) - 0.5 * (np.outer(alpha, alpha) - 2.0 * sym(np.outer(Q @ m, alpha))
                                                                      + Q @ K6 @ Q)
    Zs, Xs = Z / ls, X / ls
    E_uf = G_uf * orc._kernel_dr2(kernel, orc.square_distance(Zs, Xs))
    E_uu = G_K * orc._kernel_dr2(kernel, orc.square_distance(Zs, None))
    np.fill_diagonal(E_uu, 0.0)                               # r = 0 on the diagonal: no dependence on Z or the lengthscales
    # the oracle's sums over pairs, sum_n E_in (z_id - x_nd)^k for k = 1, 2, as products over the points (D = 784 would take
    # minutes pair by pair); coordinates relative to the centroid of Zs so that the expansion does not cancel
    o = Zs.mean(axis=0)
    Zc, Xc = Zs - o, Xs - o
    d_ls = np.zeros(D)
    d_Z = np.zeros((M, D))
    for E, P, wz in ((E_uf, Xc, 1.0), (E_uu, Zc, 2.0)):
        S1, EX, EX2 = E.sum(axis=1), E @ P, E @ np.square(P)
        first = Zc * S1[:, None] - EX                                  # sum_n E_in (z_i - p_n)
        second = np.square(Zc) * S1[:, None] - 2.0 * Zc * EX + EX2     # sum_n E_in (z_i - p_n)^2
        d_ls -= (2.0 / ls) * second.sum(axis=0)
        d_Z += (2.0 * wz / ls) * first
    d_var = (np.sum(G_uf * Kuf_) + np.sum(G_K * K)) / var + s * np.sum(h)
    if isinstance(lik, orc.Gaussian):
        s2 = float(lik.variance)
        d_lik = s * np.sum(-0.5 / s2 + 0.5 * (np.square(Y - mu) + v) / (s2 * s2))
    elif isinstance(lik, orc.StudentT):
        z, w = orc.gh_points_and_weights(lik.n_gh)
        F = mu[..., None] + np.sqrt(v)[..., None] * z
        r_ = Y[..., None] - F
        sc, df = float(lik.scale), lik.df
        d_lik = s * np.sum((-1.0 / sc + (df + 1.0) * np.square(r_) / (sc * (df * sc * sc + np.square(r_)))) * w)
    else:
        d_lik = None
    if np.asarray(kernel.lengthscales).size == 1:
        d_ls = np.array([np.sum(d_ls)])
    return elbo, dict(variance=d_var, lengthscales=d_ls, Z=d_Z, likelihood=d_lik)
