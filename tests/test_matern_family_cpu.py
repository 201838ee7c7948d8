"""
The Matern-1/2 and Matern-3/2 kernels on the host side: the oracle's covariances and derivatives against their closed forms and
central differences, the M-step gradients against central differences of the ELBO, the mapping of GPflow's class names onto the
library's kernel kinds, and the dyadic inputs that the GPU parity tests (tests/test_gpu_matern_family.py) run on.

Dyadic inputs: coordinates are multiples of 2^-k in a small box and lengthscales are powers of two, so every scaled coordinate,
square, product and sum of the squared distance r2 = |x|^2 + |z|^2 - 2 x.z is exact in any order.  The oracle and the device then
see the same r2, exact zeros at coincident points included.  That matters for Matern-1/2, whose value depends on sqrt(r2): at a
generic coincident point the expansion form leaves r2 ~ 1e-16 |x|^2, i.e. a relative error ~1e-8 in k that differs between any
two implementations.
"""
import numpy as np
import pytest

from oracle import tsvgp_oracle as orc
from tests import matern_oracle as mo

KINDS = {"matern12": mo.Matern12, "matern32": mo.Matern32}


def dyadic(rng, n, D, k=3, box=2):
    """n points of D coordinates j 2^-k, |j| <= box 2^k"""
    return rng.integers(-box * 2 ** k, box * 2 ** k + 1, size=(n, D)) * 2.0 ** -k


def dyadic_lengthscales(rng, D, lo=-1, hi=2):
    """ARD lengthscales 2^e, e in [lo, hi]"""
    return 2.0 ** rng.integers(lo, hi + 1, size=D)


def exact_r2(X, Z, ls, k=3):
    """r2 between scaled points as Python integers in units of 4^-(k + e_max): [len(Z)][len(X)]"""
    e = np.round(np.log2(np.broadcast_to(np.asarray(ls, dtype=np.float64).reshape(-1), (X.shape[1],)))).astype(int)
    w = [2 ** int(e.max() - ed) for ed in e]
    IX, IZ = np.round(X * 2 ** k).astype(np.int64), np.round(Z * 2 ** k).astype(np.int64)
    r2 = [[sum((w[d] * int(IZ[i, d] - IX[j, d])) ** 2 for d in range(X.shape[1])) for j in range(len(X))] for i in range(len(Z))]
    return r2, 4 ** int(k + e.max())


# ---- dyadic inputs ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("D,ard", [(1, False), (4, True), (16, True), (16, False)])
def test_dyadic_inputs_give_exact_squared_distances(D, ard):
    rng = np.random.default_rng(D)
    X = dyadic(rng, 60, D)
    Z = np.concatenate([X[:20], dyadic(rng, 20, D)])    # coincident points and generic ones
    ls = dyadic_lengthscales(rng, D) if ard else np.array([2.0])
    r2_int, unit = exact_r2(X, Z, ls)
    got = orc.square_distance(orc.scale(Z, ls), orc.scale(X, ls))
    want = np.array([[v / unit for v in row] for row in r2_int])
    assert max(max(row) for row in r2_int) < 2 ** 53     # so every exact value, over a power of two, is a double
    np.testing.assert_array_equal(got, want)
    assert np.all(np.diagonal(got[:20, :20]) == 0.0)
    # in a different order (row-wise dots in reverse feature order): the same bits
    Zs, Xs = orc.scale(Z, ls)[:, ::-1], orc.scale(X, ls)[:, ::-1]
    alt = np.array([[float(np.sum(z * z)) + float(np.sum(x * x)) - 2.0 * float(np.dot(z, x)) for x in Xs] for z in Zs])
    np.testing.assert_array_equal(alt, want)


# ---- covariances and derivatives --------------------------------------------------------------------------------------------------
def test_covariances_against_closed_forms():
    rng = np.random.default_rng(1)
    X, Z = rng.standard_normal((30, 3)), rng.standard_normal((7, 3))
    ls = np.array([0.7, 1.3, 2.0])
    r = np.sqrt(np.sum(np.square((Z[:, None, :] - X[None, :, :]) / ls), axis=-1))
    np.testing.assert_allclose(mo.Matern12(1.7, ls).K(Z, X), 1.7 * np.exp(-r), rtol=1e-12)
    s3 = np.sqrt(3.0)
    np.testing.assert_allclose(mo.Matern32(0.6, ls).K(Z, X), 0.6 * (1.0 + s3 * r) * np.exp(-s3 * r), rtol=1e-12)
    for cls in KINDS.values():
        k = cls(2.5, 0.9)
        np.testing.assert_array_equal(k.K_diag(X), np.full(30, 2.5))
        assert np.all(np.diagonal(k.K(X)) <= 2.5) and np.allclose(np.diagonal(k.K(X)), 2.5, rtol=1e-7)
        # at r2 = 0 exactly (the clamp): variance exp(-1e-18) = variance
        assert k.K_r2(np.array([0.0, -1e-20]))[0] == 2.5 and k.K_r2(np.array([0.0, -1e-20]))[1] == 2.5


@pytest.mark.parametrize("kind", sorted(KINDS))
def test_kernel_dr2_against_central_differences(kind):
    k = KINDS[kind](1.3, 1.0)
    r2 = np.array([1e-4, 1e-3, 0.04, 0.5, 1.0, 3.7, 20.0])
    h = 1e-5 * r2
    cd = (k.K_r2(r2 + h) - k.K_r2(r2 - h)) / (2.0 * h)
    np.testing.assert_allclose(mo.kernel_dr2(k, r2), cd, rtol=1e-6)


def test_kernel_dr2_below_the_clamp():
    r2 = np.array([0.0, -3e-17, 1e-40, 9.99e-37, 1e-36, 4e-36])
    m12 = mo.kernel_dr2(mo.Matern12(2.0, 1.0), r2)
    np.testing.assert_array_equal(m12[:4], 0.0)
    # at and above the clamp: -variance exp(-r) / (2 r), r = sqrt(r2)
    np.testing.assert_allclose(m12[4:], -2.0 * np.exp(-np.sqrt(r2[4:])) / (2.0 * np.sqrt(r2[4:])), rtol=1e-15)
    assert m12[4] == pytest.approx(-1e18)
    # Matern-3/2's derivative is finite at 0: -(3/2) variance
    np.testing.assert_allclose(mo.kernel_dr2(mo.Matern32(2.0, 1.0), r2), -3.0 * np.exp(-np.sqrt(3.0 * np.maximum(r2, 1e-36))),
                               rtol=1e-15)
    assert mo.kernel_dr2(mo.Matern32(2.0, 1.0), np.array([0.0]))[0] == -3.0


# ---- M-step gradients against central differences of the ELBO (tests/test_elbo_gradients_cpu.py's method) -----------------------
class _ExactDiagonal:
    """K(Z) with its diagonal at exactly the variance.  The expansion form leaves r2 ~ 1e-16 |z|^2 on the diagonal, which moves
    Matern-1/2's K_ii by ~1e-8 relative whenever Z or the lengthscales move, and a central difference with h = 1e-6 would read that
    rounding as a slope.  elbo_gradients differentiates this function: it takes no Z or lengthscale gradient from the diagonal."""

    def K(self, X, X2=None):
        K = super().K(X, X2)
        if X2 is None:
            np.fill_diagonal(K, float(self.variance))
        return K


MIXED = {name: type(name, (_ExactDiagonal, cls), {}) for name, cls in KINDS.items()}


def _model(kind, lik_name, ard, N=40, M=7, D=3, seed=0):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((N, D))
    Z = rng.standard_normal((M, D))      # off the data: the Matern-1/2 ELBO is not differentiable where z = x
    ls = np.array([0.9, 1.4, 1.1]) if ard else 1.2
    kernel = MIXED[kind](variance=1.4, lengthscales=ls)
    assert isinstance(kernel, KINDS[kind])
    f = np.sin(X.sum(1, keepdims=True))
    if lik_name == "gaussian":
        lik, Y = orc.Gaussian(variance=0.3), f + 0.2 * rng.standard_normal((N, 1))
    elif lik_name == "bernoulli":
        lik, Y = orc.Bernoulli(), (f > 0).astype(float)
    else:
        lik, Y = orc.StudentT(scale=0.5, df=4.0), f + 0.2 * rng.standard_normal((N, 1))
    m = orc.OracleTSVGP(kernel, lik, orc.InducingPoints(Z), num_data=3 * N)
    for _ in range(2):
        m.natgrad_step((X, Y), lr=0.6)
    return m, (X, Y)


def _cd(m, data, set_value, x0, h):
    set_value(x0 + h)
    ep = m.elbo(data)
    set_value(x0 - h)
    em = m.elbo(data)
    set_value(x0)
    return (ep - em) / (2.0 * h)


@pytest.mark.parametrize("kind,lik_name,ard", [("matern12", "gaussian", True), ("matern12", "student_t", False),
                                               ("matern32", "gaussian", False), ("matern32", "bernoulli", True),
                                               ("matern32", "student_t", True), ("matern12", "bernoulli", False)])
def test_elbo_gradients_against_central_differences(kind, lik_name, ard):
    m, data = _model(kind, lik_name, ard)
    e, g = mo.elbo_gradients(m, data)
    assert abs(e - m.elbo(data)) <= 1e-12 * abs(e)
    k = m.kernel
    v0 = float(k.variance)
    cd = _cd(m, data, lambda v: setattr(k, "variance", orc._param(v)), v0, 1e-6)
    assert g["variance"] == pytest.approx(cd, rel=1e-6, abs=1e-8)
    ls0 = np.array(k.lengthscales, dtype=np.float64).reshape(-1)
    for d in range(ls0.size):
        def set_ls(v, d=d):
            a = ls0.copy()
            a[d] = v
            k.lengthscales = orc._param(a if ls0.size > 1 else a[0])
        cd = _cd(m, data, set_ls, ls0[d], 1e-6)
        assert g["lengthscales"][d] == pytest.approx(cd, rel=1e-6, abs=1e-8)
    Z0 = np.array(m.inducing_variable.Z)
    for i, d in [(0, 0), (3, 1), (6, 2)]:
        def set_z(v, i=i, d=d):
            Z = Z0.copy()
            Z[i, d] = v
            m.inducing_variable = orc.InducingPoints(Z)
        cd = _cd(m, data, set_z, Z0[i, d], 1e-6)
        assert g["Z"][i, d] == pytest.approx(cd, rel=1e-6, abs=1e-8)
    if g["likelihood"] is not None:
        lik = m.likelihood
        name = "variance" if lik_name == "gaussian" else "scale"
        p0 = float(getattr(lik, name))
        cd = _cd(m, data, lambda v: setattr(lik, name, v), p0, 1e-6)
        assert g["likelihood"] == pytest.approx(cd, rel=1e-6, abs=1e-8)


# ---- host mapping ------------------------------------------------------------------------------------------------------------------
def test_gpflow_names_map_onto_the_new_kinds():
    from tsvgp_b200 import _lib, model
    from tsvgp_b200 import standins as st
    assert (_lib.KERNEL_MATERN12, _lib.KERNEL_MATERN32) == (2, 3)
    assert _lib.ABI_VERSION == 1
    for cls, kind in [(st.Matern12, _lib.KERNEL_MATERN12), (st.Matern32, _lib.KERNEL_MATERN32),
                      (mo.Matern12, _lib.KERNEL_MATERN12), (mo.Matern32, _lib.KERNEL_MATERN32)]:
        for ls, want in [(0.5, [0.5]), ([1.0, 2.0, 4.0], [1.0, 2.0, 4.0]), ([[1.0, 2.0]], [1.0, 2.0])]:   # isotropic, ARD, [1, D]
            k, var, got = model._kernel_spec(cls(variance=1.5, lengthscales=ls))
            assert (k, var, got.tolist()) == (kind, 1.5, want)
    kind, var, ls = model._kernel_spec(st.SharedIndependent(st.Matern12(0.7, [1.0, 2.0]), 3), 3)
    assert (kind, var, ls.tolist()) == (_lib.KERNEL_MATERN12, 0.7, [1.0, 2.0])
    specs = model._kernel_spec(st.SeparateIndependent([st.Matern12(1.0, 0.5), st.SquaredExponential(0.3, 2.0),
                                                       st.Matern32(0.8, [1.0, 4.0]), st.Matern52(1.1, 1.0)]), 4)
    assert [s[0] for s in specs] == [_lib.KERNEL_MATERN12, _lib.KERNEL_SE, _lib.KERNEL_MATERN32, _lib.KERNEL_MATERN52]
    assert [s[1] for s in specs] == [1.0, 0.3, 0.8, 1.1] and specs[2][2].tolist() == [1.0, 4.0]


def test_header_and_binding_agree_on_the_kinds():
    import os
    import re
    from tsvgp_b200 import _lib
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with open(os.path.join(root, "include", "tsvgp.h")) as f:
        h = f.read()
    kinds = dict((n, int(v)) for n, v in re.findall(r"TSVGP_KERNEL_(\w+) = (\d+)", h))
    assert kinds == {"SE": _lib.KERNEL_SE, "MATERN52": _lib.KERNEL_MATERN52, "MATERN12": _lib.KERNEL_MATERN12,
                     "MATERN32": _lib.KERNEL_MATERN32}


@pytest.mark.parametrize("name", ["RationalQuadratic", "Exponential", "Periodic"])
def test_other_kernels_are_still_refused(name):
    from tsvgp_b200 import model
    k = type(name, (), {})()
    k.variance, k.lengthscales = 1.0, 1.0
    with pytest.raises(NotImplementedError):
        model._kernel_spec(k)
