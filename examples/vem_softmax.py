"""
10-class classification with variational EM on the B200 path, in the shape of the reference's docs/notebooks/mnist.py:
Matern-5/2 with one lengthscale per input (D = 784), Softmax(10) with 100 Monte-Carlo points, M = 100 inducing inputs and
minibatches of 200 rows; per minibatch a few natural-gradient steps on the sites (E-step) and Adam steps on the kernel and Z
(M-step, `train_Z=True`).  The data are synthetic and seeded — 10 class prototypes (sparse "images" in [0, 1]^784) plus
Gaussian pixel noise — so nothing is downloaded.

    python examples/vem_softmax.py        (needs a B200; there is no CPU fallback)
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import tsvgp_b200 as tb  # noqa: E402
from tsvgp_b200 import standins as st, vem  # noqa: E402


def make_data(n, D=784, C=10, noise=0.3, seed=0, rows_seed=1):
    """n rows of class prototype + noise; -> X [n, D], labels [n, 1] (float class indices)."""
    protos = (np.random.RandomState(seed).rand(C, D) < 0.2).astype(float)   # the classes: fixed by `seed`
    rows = np.random.RandomState(rows_seed)
    y = rows.randint(C, size=n)
    X = protos[y] + noise * rows.randn(n, D)
    return X, y.astype(float)[:, None]


def main(n_train=2000, n_test=1000, M=100, batch=200, S=100, n_epochs=2, n_e_steps=2, n_m_steps=2, lr_natgrad=0.5,
         lr_adam=0.01, fixed_draws=False, verbose=True):
    """-> (ELBO trace of the M-steps, training accuracy, test accuracy).  fixed_draws: every minibatch gets explicit
    Monte-Carlo draws from a seeded generator (set_mc_epsilon), so that a run is reproducible bit for bit."""
    C, D = 10, 784
    X, y = make_data(n_train, D, C)
    Xt, yt = make_data(n_test, D, C, rows_seed=2)
    Z = X[:M].copy()
    kernel = st.Matern52(variance=1.0, lengthscales=np.full(D, 20.0))
    lik = st.Softmax(C, num_monte_carlo_points=S)
    model = tb.t_SVGP(kernel, lik, Z, num_latent_gps=C, num_data=n_train)
    rng, eps_rng = np.random.RandomState(7), np.random.RandomState(8)
    trace = []
    for ep in range(n_epochs):
        order = rng.permutation(n_train)
        for k in range(n_train // batch):
            idx = order[k * batch:(k + 1) * batch]
            if fixed_draws:
                model.set_mc_epsilon(eps_rng.randn(S, batch, C))
            trace += vem.fit(model, (X[idx], y[idx]), n_iters=1, n_e_steps=n_e_steps, n_m_steps=n_m_steps,
                             lr_natgrad=lr_natgrad, lr_adam=lr_adam, train_Z=True)
        if verbose:
            print(f"epoch {ep}  elbo {trace[-1]:12.2f}  kernel variance {kernel.variance:.3f}  "
                  f"lengthscales {np.min(kernel.lengthscales):.2f}..{np.max(kernel.lengthscales):.2f}")
    model.set_mc_epsilon(None)

    def accuracy(A, labels):
        return float(np.mean(np.argmax(model.predict_f(A)[0], axis=1) == labels[:, 0]))

    acc_train, acc_test = accuracy(X, y), accuracy(Xt, yt)
    if verbose:
        print(f"ELBO {trace[0]:.2f} -> {trace[-1]:.2f}; accuracy train {acc_train:.3f}, test {acc_test:.3f} (chance 0.1)")
    model.close()
    return trace, acc_train, acc_test


if __name__ == "__main__":
    main()
