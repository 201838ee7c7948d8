"""
Hyperparameter learning with the two site parameterisations side by side: variational EM on `t_SVGP` (sites in the dual
parameterisation) and on `t_SVGP_white` (sites in the K-scaled, whitened one), from the same start on the toy data of the
reference's docs/notebooks/regression_1D.py.  The two models have the same optimum q(u) for fixed hyperparameters, but their
ELBO surfaces over the hyperparameters differ once the sites are held fixed in the M-step, so the EM paths differ too.  Prints
both ELBO traces and the learned hyperparameters.

    python examples/vem_white_vs_dense.py        (needs a B200; there is no CPU fallback)
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import tsvgp_b200 as tb  # noqa: E402
from tsvgp_b200 import standins as st, vem  # noqa: E402


def _run(cls, X, Y, Z, n_iters):
    kernel = st.SquaredExponential(variance=0.3, lengthscales=0.3)   # deliberately poor initial hyperparameters, as in
    lik = st.Gaussian(variance=1.0)                                  # examples/vem_regression_1d.py
    model = cls(kernel, lik, Z.copy(), num_data=X.shape[0])
    for _ in range(5):                                               # regression_1D.py: nit = 5 natural-gradient steps, lr 0.9
        model.natgrad_step((X, Y), lr=0.9)
    e0 = model.elbo((X, Y))
    trace = vem.fit(model, (X, Y), n_iters=n_iters, n_e_steps=4, n_m_steps=10, lr_natgrad=0.9, lr_adam=0.05)
    for _ in range(4):
        model.natgrad_step(lr=0.9)
    e1 = model.elbo()
    model.close()
    return dict(elbo_start=e0, elbo_end=e1, trace=np.asarray(trace), variance=float(kernel.variance),
                lengthscale=float(kernel.lengthscales), noise=float(lik.variance))


def main(n_iters=15, verbose=True):
    rng = np.random.RandomState(123)
    N, M = 200, 20
    X = rng.rand(N, 1) * 2 - 1
    Y = np.sin(15 * X) + 0.3 * rng.randn(N, 1)                       # true noise variance 0.09
    Z = np.linspace(X.min(), X.max(), M).reshape(-1, 1)
    out = {"t_SVGP": _run(tb.t_SVGP, X, Y, Z, n_iters), "t_SVGP_white": _run(tb.t_SVGP_white, X, Y, Z, n_iters)}
    if verbose:
        for name, r in out.items():
            print(f"{name}: ELBO trace (every 10th M-step) {np.array2string(r['trace'][::10], precision=2)}")
        for name, r in out.items():
            print(f"{name:13s} ELBO {r['elbo_start']:10.3f} -> {r['elbo_end']:10.3f}   variance {r['variance']:.3f}  "
                  f"lengthscale {r['lengthscale']:.3f}  noise {r['noise']:.3f} (true 0.09)")
    return out


if __name__ == "__main__":
    main()
