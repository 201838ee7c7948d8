"""
The whitened sibling with the Softmax likelihood on the CPU: the M-step gradients of tests/white_grad_oracle.py, which takes g and h
of any likelihood on [N, L] moments, against central differences of the unchanged OracleTSVGPWhite.elbo with the Monte-Carlo draws
fixed (`epsilon`), for 3 and 5 classes, ARD and isotropic lengthscales, the SE and the Matern-5/2 kernel.  The sites are trained by
a few natural-gradient steps first, so that Q = A^-1 - R^-1 is far from zero.  And the binding: t_SVGP_white accepts Softmax and
still refuses the heteroskedastic likelihood.
"""
import numpy as np
import pytest

from oracle import tsvgp_oracle as orc
from tests import white_grad_oracle as wgo

KINDS = {"se": orc.SquaredExponential, "matern52": orc.Matern52}


def _model(kind, C, ard, N=40, M=7, D=3, S=20, seed=0):
    rng = np.random.default_rng(seed)
    protos = rng.standard_normal((C, D))
    y = rng.integers(0, C, size=N)
    X = protos[y] + 0.5 * rng.standard_normal((N, D))
    Z = rng.standard_normal((M, D))
    ls = np.array([0.9, 1.4, 1.1]) if ard else 1.2
    kernel = KINDS[kind](variance=1.4, lengthscales=ls)
    lik = orc.Softmax(C, num_monte_carlo_points=S, epsilon=rng.standard_normal((S, N, C)))
    m = orc.OracleTSVGPWhite(kernel, lik, orc.InducingPoints(Z), num_latent_gps=C, num_data=3 * N)
    Y = y.astype(float)[:, None]
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


@pytest.mark.parametrize("kind,C,ard", [("se", 3, True), ("se", 5, False), ("matern52", 3, False), ("matern52", 5, True)])
def test_white_softmax_gradients_against_central_differences(kind, C, ard):
    m, data = _model(kind, C, ard)
    A = m.kernel.K(np.asarray(m.inducing_variable.Z)) + orc.DEFAULT_JITTER * np.eye(m.num_inducing)
    assert np.max(np.abs(m.lambda_2)) > 1e-2 * np.max(np.abs(A))
    e, g = wgo.elbo_gradients(m, data)
    assert abs(e - m.elbo(data)) <= 1e-12 * abs(e)
    assert g["likelihood"] is None
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


def test_white_model_accepts_softmax_and_refuses_heteroskedastic():
    import tsvgp_b200 as tb
    from tsvgp_b200 import standins as st
    try:
        m = tb.t_SVGP_white(st.SquaredExponential(), st.Softmax(3), np.zeros((4, 2)), num_latent_gps=3)
    except tb.TsvgpError as e:   # no GPU here: the constructor got past the binding's checks and reached the library
        assert e.code == -2 and "no CPU fallback" in str(e)   # TSVGP_ERR_CUDA
    else:
        m.close()
    with pytest.raises(NotImplementedError):
        tb.t_SVGP_white(st.SquaredExponential(), st.HeteroskedasticTFPConditional(), np.zeros((4, 2)), num_latent_gps=2)
