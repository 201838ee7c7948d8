"""
GPU: the Matern-1/2 and Matern-3/2 kernels on every path, against the oracle at 1e-9 on dyadic inputs (tests/test_matern_family_cpu.py:
coordinates j 2^-3 and power-of-two lengthscales, so the oracle and the device form bit-identical squared distances, exact zeros at
Z = X[:M] included).  The covariance slab kernel itself runs through a shim (tests/kernels/kuf_shim.cu) and is compared with NumPy
entry by entry.  One case runs Matern-1/2 on generic inputs, where the oracle's r2 at a coincident point is a rounding residue and
no 1e-9 agreement exists (see test_matern12_on_generic_inputs).
"""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

from oracle import tsvgp_oracle as orc
from tests import matern_oracle as mo
from tests import full_cov_oracle as fco
from tests import separate_oracle as so
from tests.test_gpu_gaussian_step import _elbo_and_sites_errors
from tests.test_gpu_int8_syrk import _int8_products
from tests.test_gpu_multilatent import _pair_errors
from tests.test_gpu_parity import check, relerr
from tests.test_gpu_softmax_grad import _errs, _trained
from tests.test_matern_family_cpu import dyadic

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHIM = os.path.join(ROOT, "tests", "kernels", "kuf_shim.cu")
NVCC_FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC", "-shared"]   # csrc/Makefile
EPS = np.finfo(np.float64).eps

# cond(Kuu + 1e-9 I) at Z = X[:160] of _case: 43, 2.5e2, 1.0e3
KERNELS = {"matern12": mo.Matern12(variance=1.3, lengthscales=[1.0, 2.0, 1.0, 0.5]), "matern32": mo.Matern32(variance=0.8, lengthscales=1.0),
           "matern32_ard": mo.Matern32(variance=1.3, lengthscales=[1.0, 2.0, 1.0, 2.0])}


def _case(lik_name, N=1700, M=160, D=4, L=1, seed=21):
    rng = np.random.default_rng(seed)
    X = dyadic(rng, N, D)
    F = np.stack([np.sin(X.sum(1) * (0.5 + 0.3 * l)) for l in range(L)], axis=1)
    if lik_name == "gaussian":
        lik, Y = orc.Gaussian(variance=0.1), F + 0.3 * rng.standard_normal((N, L))
    elif lik_name == "bernoulli":
        lik, Y = orc.Bernoulli(), (F + 0.3 * rng.standard_normal((N, L)) > 0).astype(float)
    else:
        lik, Y = orc.StudentT(scale=0.3, df=3.0), F + 0.3 * rng.standard_t(3.0, size=(N, L))
    return X, Y, X[:M].copy(), lik


def _cond(kernel, Z):
    ev = np.linalg.eigvalsh(kernel.K(Z) + 1e-9 * np.eye(len(Z)))
    return ev[-1] / ev[0]


# ---- the covariance slab through the shim ------------------------------------------------------------------------------------------
@pytest.fixture(scope="session")
def shim(tmp_path_factory):
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    if not os.path.exists(nvcc):
        nvcc = shutil.which("nvcc") or nvcc
    out = str(tmp_path_factory.mktemp("kuf_shim") / "libkufshim.so")
    r = subprocess.run([nvcc, *NVCC_FLAGS, "-o", out, SHIM], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    lib = ctypes.CDLL(out)
    vp, i, l, d = ctypes.c_void_p, ctypes.c_int, ctypes.c_long, ctypes.c_double
    lib.kuf_launch.argtypes = [i, d, vp, l, vp, l, l, i, vp, vp, i, i, i, vp, vp, l, vp, l, i, vp, vp]
    lib.kuf_launch.restype = i
    return lib


SHIM_KINDS = {0: orc.SquaredExponential, 1: orc.Matern52, 2: mo.Matern12, 3: mo.Matern32}


def _slab(shim, kind, variance, ls, X, Z, ncols, Mp, n0=0, n_valid=None, deriv=True):
    """K [Mp][ncols] (and dk/dr2) for the points X[n0:n0+ncols] against the inducing inputs Z, from the scaled inputs formed here"""
    import torch
    D, M = X.shape[1], Z.shape[0]
    Xs, Zs = orc.scale(X, ls), orc.scale(Z, ls)
    ldx = max(n0 + ncols, len(X))
    XsT = np.zeros((D, ldx))
    XsT[:, :len(X)] = Xs.T
    x2 = np.zeros(ldx)
    x2[:len(X)] = np.sum(Xs * Xs, axis=1)
    Zp = np.zeros((Mp, D))
    Zp[:M] = Zs
    z2 = np.sum(Zp * Zp, axis=1)
    dev = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in dict(XsT=XsT, x2=x2, Zs=Zp, z2=z2).items()}
    K = torch.full((Mp, ncols), np.nan, dtype=torch.float64, device="cuda")
    Kp = torch.full((Mp, ncols), np.nan, dtype=torch.float64, device="cuda") if deriv else None
    rc = shim.kuf_launch(kind, variance, dev["XsT"].data_ptr(), ldx, dev["x2"].data_ptr(), n0, len(X) if n_valid is None else n_valid,
                         ncols, dev["Zs"].data_ptr(), dev["z2"].data_ptr(), M, Mp, D, None, K.data_ptr(), ncols, None, 0, 0,
                         torch.cuda.current_stream().cuda_stream, Kp.data_ptr() if deriv else None)
    assert rc == 0, rc
    torch.cuda.synchronize()
    return K.cpu().numpy(), (Kp.cpu().numpy() if deriv else None)


@pytest.mark.parametrize("deriv", [False, True])
@pytest.mark.parametrize("D,ard", [(16, True), (3, False)], ids=["D16_ard_bulk_copies", "D3_iso_plain_loads"])
@pytest.mark.parametrize("kind", [0, 1, 2, 3], ids=["se", "matern52", "matern12", "matern32"])
def test_kuf_slab_against_numpy(shim, kind, D, ard, deriv):
    rng = np.random.default_rng(10 + kind)
    n, ncols, M, Mp = 300, 384, 100, 128          # ragged: columns >= 300 and rows >= 100 are padding
    X = dyadic(rng, n, D)
    Z = np.concatenate([X[:40], dyadic(rng, M - 40, D)])
    ls = 2.0 ** rng.integers(-1, 3, size=D) if ard else np.array([2.0])
    kern = SHIM_KINDS[kind](variance=1.7, lengthscales=ls)
    K, Kp = _slab(shim, kind, 1.7, ls, X, Z, ncols, Mp, deriv=deriv)
    r2 = orc.square_distance(orc.scale(Z, ls), orc.scale(X, ls))      # exact on these inputs
    want = kern.K_r2(r2)
    # a few ulp, scaled by the size of the exponent's argument (its rounding enters exp's result relatively)
    tol = 8.0 * EPS * (2.0 + r2 + 3.0 * np.sqrt(r2))
    assert np.all(np.abs(K[:M, :n] - want) <= tol * np.abs(want)), np.max(np.abs(K[:M, :n] - want) / np.abs(want) / tol)
    assert np.all(K[M:] == 0.0) and np.all(K[:, n:] == 0.0)
    np.testing.assert_array_equal(K[np.arange(40), np.arange(40)], 1.7)          # coincident points: k = variance exactly
    if deriv:
        dwant = mo.kernel_dr2(kern, r2)
        assert np.all(np.abs(Kp[:M, :n] - dwant) <= tol * np.abs(dwant)), np.max(np.abs(Kp[:M, :n] - dwant) / np.abs(dwant) / tol)
        assert np.all(Kp[M:] == 0.0) and np.all(Kp[:, n:] == 0.0)
        if kind == 2:
            assert np.all(Kp[np.arange(40), np.arange(40)] == 0.0)     # below the clamp: the autodiff rule, not -variance / (2 r)
            assert np.count_nonzero(Kp[:M, :n] == 0.0) == np.count_nonzero(r2 == 0.0)


def test_kuf_slab_offset_chunk_and_coincident_rows(shim):
    # a chunk that starts at n0 = 256 of the resident points, with inducing inputs taken from inside it
    rng = np.random.default_rng(3)
    X = dyadic(rng, 700, 8)
    Z = X[300:364].copy()
    ls = np.array([0.5, 1.0, 2.0, 4.0, 0.5, 1.0, 2.0, 4.0])
    K, Kp = _slab(shim, 2, 0.9, ls, X, Z, 384, 64, n0=256)
    rows = np.arange(64)
    assert np.all(K[rows, rows + 44] == 0.9) and np.all(Kp[rows, rows + 44] == 0.0)
    assert np.all(np.isfinite(Kp)) and np.all(K[:, :444] > 0.0)


def test_unknown_kind_is_refused(shim):
    import torch
    buf = torch.zeros(1024, dtype=torch.float64, device="cuda")
    p = buf.data_ptr()
    assert shim.kuf_launch(4, 1.0, p, 128, p, 0, 128, 128, p, p, 64, 64, 1, None, p, 128, None, 0, 0, None, None) == -1


# ---- natgrad_step, elbo and predictions against the oracle ---------------------------------------------------------------------------
@pytest.mark.parametrize("route", [1, 2, 3])
@pytest.mark.parametrize("lik_name", ["gaussian", "bernoulli", "student_t"])
@pytest.mark.parametrize("kind", ["matern12", "matern32"])
def test_natgrad_step_matches_the_oracle(kind, lik_name, route):
    import tsvgp_b200 as tb
    X, Y, Z, lik = _case(lik_name)
    kernel = KERNELS[kind]
    assert _cond(kernel, Z) < 1e4
    ref = orc.OracleTSVGP(kernel, lik, orc.InducingPoints(Z.copy()), num_data=4 * len(X))
    dev = tb.t_SVGP(kernel, lik, Z.copy(), num_data=4 * len(X))
    for k, v in {"chunk": 512, "route": route}.items():
        dev.set_option(k, v)
    errs = _pair_errors(dev, ref, (X, Y), X[:77] + 0.0625, steps=2, lr=0.6)
    assert dev.timings()["route"] == route and dev.timings()["slabs"] >= 4
    check(errs)
    dev.close()


@pytest.mark.parametrize("kind", ["matern12", "matern32"])
def test_full_cov_and_samples(kind):
    import tsvgp_b200 as tb
    X, Y, Z, lik = _case("gaussian", L=2)
    kernel = KERNELS[kind]
    ref = orc.OracleTSVGP(kernel, lik, orc.InducingPoints(Z.copy()), num_latent_gps=2, num_data=4 * len(X))
    dev = tb.t_SVGP(kernel, lik, Z.copy(), num_latent_gps=2, num_data=4 * len(X))
    for _ in range(2):
        dev.natgrad_step((X, Y), lr=0.6)
        ref.natgrad_step((X, Y), lr=0.6)
    Xt = np.concatenate([X[:20], dyadic(np.random.default_rng(5), 44, X.shape[1])])    # 20 query points on inducing inputs
    mu_d, cov_d = dev.predict_f(Xt, full_cov=True)
    mu_r, cov_r = fco.predict_f_full_cov(ref, Xt)
    errs = {"elbo": abs(dev.elbo((X, Y)) - ref.elbo((X, Y))) / abs(ref.elbo((X, Y))), "mean": relerr(mu_d, mu_r), "cov": relerr(cov_d, cov_r)}
    eps = np.random.default_rng(1).standard_normal((5, 64, 2))
    assert max(np.linalg.cond(cov_r[l] + 1e-6 * np.eye(64)) for l in range(2)) <= 1e4
    for fc in (True, False):
        errs[f"samples_full_cov_{fc}"] = relerr(dev.predict_f_samples(Xt, 5, full_cov=fc, epsilon=eps),
                                                fco.predict_f_samples(ref, Xt, 5, full_cov=fc, epsilon=eps))
    check(errs)
    dev.close()


@pytest.mark.parametrize("kind,lik_name", [("matern12", "gaussian"), ("matern32", "gaussian"), ("matern32_ard", "gaussian"),
                                           ("matern12", "student_t"), ("matern32_ard", "bernoulli")])
def test_elbo_and_grad_matches_the_oracle(kind, lik_name):
    # Z = X[:M]: for Matern-1/2 the coincident entries of Kuf take dk/dr2 = 0 on both sides (r2 = 0 exactly on these inputs)
    import tsvgp_b200 as tb
    X, Y, Z, lik = _case(lik_name, N=2500)
    kernel = KERNELS[kind]
    ref = orc.OracleTSVGP(kernel, lik, orc.InducingPoints(Z.copy()), num_data=10_000)
    for _ in range(2):
        ref.natgrad_step((X, Y), lr=0.6)
    dev = tb.t_SVGP(kernel, lik, Z.copy(), num_data=10_000, lambda_1=ref.lambda_1, lambda_2_sqrt=ref.lambda_2_sqrt)
    dev.set_option("chunk", 1024)
    e_ref, g_ref = mo.elbo_gradients(ref, (X, Y))
    e_dev, g_dev = dev.elbo_and_grad((X, Y))
    errs = _errs(e_dev, g_dev, e_ref, g_ref)
    if g_ref["likelihood"] is None:
        assert g_dev["likelihood"] is None
    else:
        errs["likelihood"] = abs(g_dev["likelihood"] - g_ref["likelihood"]) / abs(g_ref["likelihood"])
    assert np.shape(g_dev["lengthscales"]) == np.shape(np.asarray(kernel.lengthscales))
    check(errs)
    dev.natgrad_step((X, Y), lr=0.6)     # the gradient call leaves the state alone
    ref.natgrad_step((X, Y), lr=0.6)
    check({"lambda_1": relerr(dev.lambda_1, ref.lambda_1), "lambda_2": relerr(dev.lambda_2, ref.lambda_2)})
    dev.close()


@pytest.mark.parametrize("kind", ["matern12", "matern32"])
def test_softmax_elbo_and_grad_with_fixed_draws(kind):
    rng = np.random.default_rng(4)
    N, M, D, C, S = 1200, 96, 4, 4, 30
    X = dyadic(rng, N, D)
    y = np.argmax(X[:, :C] + 0.5 * rng.standard_normal((N, C)), axis=1).astype(float)[:, None]
    Z = X[:M].copy()
    eps = rng.standard_normal((S, N, C))
    dev, ref = _trained(X, y, Z, KERNELS[kind], eps, C, 6000, {"chunk": 512, "streams": 2})
    e_ref, g_ref = mo.softmax_elbo_gradients(ref, (X, y))
    e_dev, g_dev = dev.elbo_and_grad((X, y))
    check(_errs(e_dev, g_dev, e_ref, g_ref))
    dev.close()


SEPARATE = {"matern12_se": lambda: so.SeparateIndependent([mo.Matern12(1.3, [1.0, 2.0, 1.0, 0.5]), orc.SquaredExponential(0.6, 1.0)]),
            "matern32_matern52": lambda: so.SeparateIndependent([mo.Matern32(1.0, [1.0, 2.0, 1.0, 2.0]), orc.Matern52(0.8, 1.0)])}


@pytest.mark.parametrize("lik_name", ["gaussian", "student_t"])
@pytest.mark.parametrize("pair", sorted(SEPARATE))
def test_separate_kernels(pair, lik_name):
    import tsvgp_b200 as tb
    X, Y, Z, lik = _case(lik_name, L=2)
    kernel = SEPARATE[pair]()
    assert max(_cond(k, Z) for k in kernel.kernels) < 1e4
    ref = so.OracleSeparateTSVGP(kernel, lik, orc.InducingPoints(Z.copy()), num_latent_gps=2, num_data=4 * len(X))
    dev = tb.t_SVGP(kernel, lik, Z.copy(), num_latent_gps=2, num_data=4 * len(X))
    dev.set_option("chunk", 512)
    check(_pair_errors(dev, ref, (X, Y), X[:77] + 0.0625, steps=2, lr=0.6))
    dev.close()


@pytest.mark.parametrize("pair", sorted(SEPARATE))
def test_separate_kernels_heteroskedastic_step(pair):
    import tsvgp_b200 as tb
    rng = np.random.default_rng(9)
    N, M = 1500, 120
    X = dyadic(rng, N, 4)
    Y = np.sin(X.sum(1, keepdims=True)) + np.exp(0.3 * X[:, :1]) * 0.2 * rng.standard_normal((N, 1))
    Z = X[:M].copy()
    kernel = SEPARATE[pair]()
    lik = so.HeteroskedasticTFPConditional(scale_transform=so.Exp())
    ref = so.OracleSeparateTSVGP(kernel, lik, orc.InducingPoints(Z.copy()), num_latent_gps=2, num_data=2 * N)
    dev = tb.t_SVGP(kernel, lik, Z.copy(), num_latent_gps=2, num_data=2 * N)
    dev.set_option("chunk", 512)
    errs = {}
    for s in range(2):
        e_ref = ref.elbo((X, Y))
        e_dev = dev.natgrad_step((X, Y), lr=0.5, return_elbo=True)
        ref.natgrad_step((X, Y), lr=0.5)
        errs[f"elbo_before_{s}"] = abs(e_dev - e_ref) / abs(e_ref)
        errs[f"lambda_1_{s}"], errs[f"lambda_2_{s}"] = relerr(dev.lambda_1, ref.lambda_1), relerr(dev.lambda_2, ref.lambda_2)
    for name, a, b in zip(("mean", "var"), dev.predict_f(X[:200]), ref.predict_f(X[:200])):
        errs[name] = relerr(a, b)
    check(errs)
    dev.close()


@pytest.mark.parametrize("kind", ["matern12", "matern32"])
def test_white_model(kind):
    import tsvgp_b200 as tb
    X, Y, Z, lik = _case("gaussian")
    kernel = KERNELS[kind]
    ref = orc.OracleTSVGPWhite(kernel, lik, orc.InducingPoints(Z.copy()), num_data=4 * len(X))
    dev = tb.t_SVGP_white(kernel, lik, Z.copy(), num_data=4 * len(X))
    dev.set_option("chunk", 512)
    errs = {}
    for s in range(2):
        e_ref = ref.elbo((X, Y))
        e_dev = dev.natgrad_step((X, Y), lr=0.6, return_elbo=True)
        ref.natgrad_step((X, Y), lr=0.6)
        errs[f"elbo_before_{s}"] = abs(e_dev - e_ref) / abs(e_ref)
        errs[f"lambda_1_{s}"], errs[f"lambda_2_{s}"] = relerr(dev.lambda_1, ref.lambda_1), relerr(dev.lambda_2, ref.lambda_2)
    for name, a, b in zip(("mean", "var"), dev.predict_f(X[:100] + 0.0625), ref.predict_f(X[:100] + 0.0625)):
        errs[name] = relerr(a, b)
    check(errs)
    dev.close()


# ---- the Gaussian step keeps the int8 Gram product ---------------------------------------------------------------------------------
@pytest.mark.parametrize("kernel", [mo.Matern12(variance=1.3, lengthscales=4.0), mo.Matern32(variance=1.3, lengthscales=2.0)],
                         ids=["matern12", "matern32"])
def test_gaussian_step_at_m2048_takes_the_int8_product(kernel):
    # cfg3's M and D; cond(K9) on these inputs: 1.3e3 (Matern-1/2), 1.5e2 (Matern-3/2)
    import tsvgp_b200 as tb
    X, Y, Z, lik = _case("gaussian", N=4600, M=2048, D=16, seed=22)
    assert _cond(kernel, Z) < 1e4
    ref = orc.OracleTSVGP(kernel, lik, orc.InducingPoints(Z.copy()), num_data=4 * len(X))
    dev = tb.t_SVGP(kernel, lik, Z.copy(), num_data=4 * len(X))
    dev.set_option("chunk", 1024)
    n_i8 = _int8_products(lambda: _elbo_and_sites_errors(dev, ref, (X, Y), steps=2))
    t = dev.timings()
    assert t["route"] == 1 and t["slabs"] == 5
    assert n_i8 == 2 * t["slabs"]
    dev.close()


# ---- generic inputs ------------------------------------------------------------------------------------------------------------------
def test_matern12_on_generic_inputs():
    # Z = X[:M] with standard normal X.  At a coincident point the device forms r2 = 0 exactly (x2, z2 and x.z come from the same
    # fma chain), the oracle a rounding residue of ~1e-16 |x|^2 from its BLAS product, so its k is off by up to ~sqrt(1e-16 |x|^2),
    # about 4 sqrt(eps) here (5.96e-8 measured on the CPU between the expansion and the difference form).  That moves the sites by
    # ~cond(Kuu) times as much at most; cond is 1.1e2.  So the bound is 100 sqrt(eps) = 1.5e-6, not 1e-9.
    import tsvgp_b200 as tb
    rng = np.random.default_rng(21)
    N, M, D = 1700, 160, 4
    X = rng.standard_normal((N, D))
    Y = np.sin(X.sum(1, keepdims=True)) + 0.3 * rng.standard_normal((N, 1))
    Z = X[:M].copy()
    kernel, lik = mo.Matern12(variance=1.3, lengthscales=[0.8, 1.2, 0.9, 1.0]), orc.Gaussian(variance=0.1)
    ref = orc.OracleTSVGP(kernel, lik, orc.InducingPoints(Z.copy()), num_data=4 * N)
    dev = tb.t_SVGP(kernel, lik, Z.copy(), num_data=4 * N)
    dev.set_option("chunk", 512)
    errs = _pair_errors(dev, ref, (X, Y), X[:77] + 0.05, steps=2, lr=0.6)
    print("Matern-1/2, generic inputs, Z = X[:M]: relative errors against the oracle", errs)
    check(errs, tol=100.0 * np.sqrt(EPS))
    e, g = dev.elbo_and_grad((X, Y))
    assert np.isfinite(e) and np.isfinite(g["variance"]) and np.isfinite(g["likelihood"])
    assert np.all(np.isfinite(g["lengthscales"])) and np.all(np.isfinite(g["Z"]))
    dev.close()


def test_vem_fit_with_matern32_raises_the_elbo():
    import tsvgp_b200 as tb
    from tsvgp_b200 import standins as st
    from tsvgp_b200 import vem
    rng = np.random.default_rng(0)
    X = rng.uniform(0.0, 10.0, (2000, 1))
    Y = np.sin(X) + 0.3 * rng.standard_normal((2000, 1))
    kernel, lik = st.Matern32(variance=1.0, lengthscales=0.3), st.Gaussian(variance=1.0)
    m = tb.t_SVGP(kernel, lik, np.linspace(0.0, 10.0, 30)[:, None], num_data=2000)
    trace = vem.fit(m, (X, Y), n_iters=4, n_e_steps=4, n_m_steps=10)
    assert np.all(np.isfinite(trace)) and trace[-1] > trace[0]
    assert lik.variance < 1.0
    m.close()
