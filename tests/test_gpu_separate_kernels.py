"""
GPU: one kernel per latent (gpflow.kernels.SeparateIndependent, tsvgp_set_kernels) and the heteroskedastic Normal likelihood
(HeteroskedasticTFPConditional, the model of the reference's docs/notebooks/heteroskedastic.py:58-76) against the per-latent
oracle of tests/separate_oracle.py.  Tolerance 1e-9 norm-wise, as tests/test_gpu_parity.py.
"""
import multiprocessing as mp
import os
import sys

import numpy as np
import pytest

from oracle import tsvgp_oracle as orc
from tests import separate_oracle as so
from tests.test_gpu_multi import _n_gpus
from tests.test_gpu_multilatent import _pair_errors
from tests.test_gpu_parity import check, relerr

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# cond(Kuu + 1e-9 I) at Z = X[:160] of _independent_case: 6e3, 8e3, 6e3 (as synth.py keeps its configs in 1e2..1e4)
KERNELS = [orc.Matern52(variance=1.3, lengthscales=[0.8, 1.2, 0.9, 1.0]), orc.SquaredExponential(variance=0.6, lengthscales=0.7),
           orc.Matern52(variance=0.8, lengthscales=1.0)]


def _pair(kernel, lik, Z, L, num_data, chunk=512, options=None):
    import tsvgp_b200 as tb
    ref = so.OracleSeparateTSVGP(kernel, lik, orc.InducingPoints(Z.copy()), num_latent_gps=L, num_data=num_data)
    dev = tb.t_SVGP(kernel, lik, Z.copy(), num_latent_gps=L, num_data=num_data)
    dev.set_option("chunk", chunk)     # several slabs over two streams
    for k, v in (options or {}).items():
        dev.set_option(k, v)
    return dev, ref


def _independent_case(lik_name, L, N=1500, M=160, D=4, seed=11):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((N, D))
    F = np.stack([np.sin(X.sum(1) * (0.5 + 0.3 * l)) for l in range(L)], axis=1)
    if lik_name == "gaussian":
        lik, Y = orc.Gaussian(variance=0.1), F + 0.3 * rng.standard_normal((N, L))
    elif lik_name == "bernoulli":
        lik, Y = orc.Bernoulli(), (F + 0.3 * rng.standard_normal((N, L)) > 0).astype(float)
    else:
        lik, Y = orc.StudentT(scale=0.3, df=3.0), F + 0.3 * rng.standard_t(3.0, size=(N, L))
    return X, Y, X[:M].copy(), lik


@pytest.mark.parametrize("lik_name,L", [("gaussian", 3), ("bernoulli", 2), ("student_t", 3), ("gaussian", 2)])
def test_separate_kernels_match_the_per_latent_oracle(lik_name, L):
    X, Y, Z, lik = _independent_case(lik_name, L)
    kernel = so.SeparateIndependent(KERNELS[:L])     # SE and Matern52, ARD and isotropic, different variances
    dev, ref = _pair(kernel, lik, Z, L, 4 * X.shape[0])
    check(_pair_errors(dev, ref, (X, Y), X[:77] + 0.05, steps=2, lr=0.6))
    dev.close()


def test_separate_with_equal_kernels_agrees_with_the_shared_kernel_context():
    import tsvgp_b200 as tb
    X, Y, Z, lik = _independent_case("gaussian", 2)
    k = KERNELS[0]
    a = tb.t_SVGP(k, lik, Z.copy(), num_latent_gps=2, num_data=3000)
    b = tb.t_SVGP(so.SeparateIndependent([k, k]), lik, Z.copy(), num_latent_gps=2, num_data=3000)
    for m in (a, b):
        m.set_option("chunk", 512)
    errs = {}
    for s in range(2):
        ea, eb = (m.natgrad_step((X, Y), lr=0.6, return_elbo=True) for m in (a, b))
        errs[f"elbo{s}"] = abs(ea - eb) / abs(ea)
    errs["lambda_1"], errs["lambda_2"] = relerr(b.lambda_1, a.lambda_1), relerr(b.lambda_2, a.lambda_2)
    for name, x, y in zip(("mean", "var"), b.predict_f(X[:60]), a.predict_f(X[:60])):
        errs[name] = relerr(x, y)
    check(errs, tol=1e-12)
    a.close(); b.close()


@pytest.mark.parametrize("route", [1, 2, 3])
def test_forced_routes(route):
    X, Y, Z, lik = _independent_case("student_t", 2, N=1200, M=100)
    dev, ref = _pair(so.SeparateIndependent(KERNELS[:2]), lik, Z, 2, 2400, options={"route": route})
    check(_pair_errors(dev, ref, (X, Y), X[:50], steps=2, lr=0.5))
    assert dev.timings()["route"] == route
    dev.close()


def test_automatic_route_follows_the_worst_conditioned_latent():
    rng = np.random.default_rng(4)
    N = 1500
    X = rng.uniform(0, 5, (N, 1))
    Y = np.stack([np.sin(2 * X[:, 0]), np.cos(X[:, 0])], 1) + 0.1 * rng.standard_normal((N, 2))
    Z = np.linspace(0, 5, 30)[:, None]
    good, bad = orc.Matern52(1.0, 0.2), orc.Matern52(1.0, 1.2)
    for k, lo, hi in ((good, 1.0, 1e3), (bad, 1e5, 1e7)):   # premises: one kernel below the fused threshold, one above
        assert lo < np.linalg.cond(k.K(Z) + 1e-9 * np.eye(30)) < hi
    dev, ref = _pair(so.SeparateIndependent([good, bad]), orc.Gaussian(variance=0.05), Z, 2, N)
    check(_pair_errors(dev, ref, (X, Y), X[:50], steps=2, lr=0.5))
    t = dev.timings()
    assert t["route"] == 2 and t["cond_est"] > 1e4
    dev.close()


def _demo_data(N=1001, seed=0):
    # docs/notebooks/heteroskedastic.py: X on [0, 4 pi], loc = sin(x), scale = exp(cos(x))
    rng = np.random.default_rng(seed)
    X = np.linspace(0, 4 * np.pi, N)[:, None]
    Y = rng.normal(np.sin(X), np.exp(np.cos(X)))
    return X, Y


@pytest.mark.parametrize("transform", ["exp", "softplus"])
def test_heteroskedastic_demo_matches_and_learns(transform):
    X, Y = _demo_data()
    Z = np.linspace(X.min(), X.max(), 20)[:, None]
    kernel = so.SeparateIndependent([orc.SquaredExponential(), orc.SquaredExponential()])
    lik = so.HeteroskedasticTFPConditional(scale_transform=so.Exp() if transform == "exp" else so.Softplus())
    dev, ref = _pair(kernel, lik, Z, 2, X.shape[0], chunk=256)
    check(_pair_errors(dev, ref, (X, Y), X[::7] + 0.01, steps=2, lr=0.5))
    for _ in range(28):
        dev.natgrad_step((X, Y), lr=0.5)
    mu, _ = dev.predict_f(X)
    scale = lik.scale_transform(mu[:, 1])    # T(mean of latent 1) against the true scale exp(cos x), on the log scale
    rms = float(np.sqrt(np.mean(np.square(np.log(scale) - np.cos(X[:, 0])))))
    assert rms < 0.3, rms
    dev.close()


def test_heteroskedastic_several_slabs_shared_and_separate():
    rng = np.random.default_rng(6)
    N, M, D = 5000, 300, 3
    X = rng.standard_normal((N, D))
    Y = (np.sin(X.sum(1)) + np.exp(0.5 * np.cos(X[:, 0])) * rng.standard_normal(N))[:, None]
    lik = so.HeteroskedasticTFPConditional(scale_transform=so.Softplus())
    kernel = so.SeparateIndependent([orc.Matern52(1.0, [0.5, 0.6, 0.4]), orc.SquaredExponential(0.7, 0.3)])
    dev, ref = _pair(kernel, lik, X[:M].copy(), 2, 2 * N, chunk=1024)
    check(_pair_errors(dev, ref, (X, Y), X[:100] + 0.03, steps=2, lr=0.5))
    dev.close()
    # one kernel shared by the two latents (plain and SharedIndependent): the same likelihood over one Kuf slab per launch
    import tsvgp_b200 as tb
    from tsvgp_b200 import standins as st
    k = orc.Matern52(1.0, [0.5, 0.6, 0.4])
    for kern in (k, st.SharedIndependent(k, 2)):
        dev = tb.t_SVGP(kern, lik, X[:M].copy(), num_latent_gps=2, num_data=2 * N)
        dev.set_option("chunk", 1024)
        r = so.OracleSeparateTSVGP(so.SeparateIndependent([k, k]), lik, orc.InducingPoints(X[:M].copy()), num_latent_gps=2, num_data=2 * N)
        check(_pair_errors(dev, r, (X, Y), X[:100] + 0.03, steps=2, lr=0.5))
        dev.close()


def test_full_size_heteroskedastic_step():
    # M = 2048 (cfg3's inducing size), 40 960 rows = 5 slabs of the default width, Matern52 and SE
    import tsvgp_b200.synth as synth
    N, M = 40960, 2048
    X, Y, Z = synth.make_minibatch(synth.describe("cfg3"), n_rows=N, M=M)     # cfg3's inputs: cond(Kuu) in 1e2..1e4
    kernel = so.SeparateIndependent([orc.Matern52(1.0, 3.0), orc.SquaredExponential(0.5, 2.0)])
    lik = so.HeteroskedasticTFPConditional(scale_transform=so.Exp())
    import tsvgp_b200 as tb
    ref = so.OracleSeparateTSVGP(kernel, lik, orc.InducingPoints(Z.copy()), num_latent_gps=2, num_data=10 * N)
    dev = tb.t_SVGP(kernel, lik, Z.copy(), num_latent_gps=2, num_data=10 * N)
    e_ref = ref.elbo((X, Y))
    e_dev = dev.natgrad_step((X, Y), lr=0.5, return_elbo=True)
    ref.natgrad_step((X, Y), lr=0.5)
    errs = {"elbo_before": abs(e_dev - e_ref) / abs(e_ref), "lambda_1": relerr(dev.lambda_1, ref.lambda_1),
            "lambda_2": relerr(dev.lambda_2, ref.lambda_2)}
    for name, x, y in zip(("mean", "var"), dev.predict_f(X[:500]), ref.predict_f(X[:500])):
        errs[name] = relerr(x, y)
    check(errs)
    dev.close()


def test_full_cov_samples_predict_y_and_log_density():
    X, Y = _demo_data(N=600, seed=3)
    Z = np.linspace(X.min(), X.max(), 25)[:, None]
    kernel = so.SeparateIndependent([orc.Matern52(1.2, 1.5), orc.SquaredExponential(0.8, 0.6)])
    lik = so.HeteroskedasticTFPConditional(scale_transform=so.Exp())
    dev, ref = _pair(kernel, lik, Z, 2, 600, chunk=256)
    for _ in range(2):
        dev.natgrad_step((X, Y), lr=0.5)
        ref.natgrad_step((X, Y), lr=0.5)
    Xt = np.linspace(0.1, 12.3, 150)[:, None]
    mu_d, cov_d = dev.predict_f(Xt, full_cov=True)
    mu_r, cov_r = ref.predict_f_full_cov(Xt)
    assert cov_d.shape == (2, 150, 150)
    errs = {"mean": relerr(mu_d, mu_r), "cov": relerr(cov_d, cov_r)}
    eps = np.random.default_rng(1).standard_normal((16, 150, 2))
    for fc in (True, False):
        errs[f"samples_full_cov_{fc}"] = relerr(dev.predict_f_samples(Xt, 16, full_cov=fc, epsilon=eps),
                                                ref.predict_f_samples(Xt, 16, full_cov=fc, epsilon=eps))
    m, v = ref.predict_f(Xt)
    Ey_r, Vy_r = lik.predict_mean_and_var(m, v)
    Ey, Vy = dev.predict_y(Xt)
    errs["Ey"], errs["Vy"] = relerr(Ey, Ey_r), relerr(Vy, Vy_r)
    Yt = np.sin(Xt) + 0.5
    errs["log_density"] = relerr(dev.predict_log_density((Xt, Yt)), lik.predict_log_density(m, v, Yt))
    check(errs)
    dev.close()


def test_softmax_with_separate_kernels_and_fixed_draws():
    import tsvgp_b200 as tb
    rng = np.random.default_rng(5)
    N, M, D, C, S = 900, 64, 4, 3, 40
    X = rng.standard_normal((N, D))
    W = rng.standard_normal((D, C))
    labels = np.argmax(X @ W + 0.5 * rng.standard_normal((N, C)), axis=1).astype(float)[:, None]
    eps = rng.standard_normal((S, N, C))
    kernel = so.SeparateIndependent(KERNELS[:C])
    lik = orc.Softmax(C, num_monte_carlo_points=S, epsilon=eps)
    ref = so.OracleSeparateTSVGP(kernel, lik, orc.InducingPoints(X[:M].copy()), num_latent_gps=C, num_data=3 * N)
    dev = tb.t_SVGP(kernel, lik, X[:M].copy(), num_latent_gps=C, num_data=3 * N)
    dev.set_option("chunk", 256)
    dev.set_mc_epsilon(eps)
    errs = {}
    for s in range(2):
        e_ref = ref.elbo((X, labels))
        e_dev = dev.natgrad_step((X, labels), lr=0.4, return_elbo=True)
        ref.natgrad_step((X, labels), lr=0.4)
        errs[f"elbo_before_step{s}"] = abs(e_dev - e_ref) / abs(e_ref)
        errs[f"lambda_1_step{s}"] = relerr(dev.lambda_1, ref.lambda_1)
        errs[f"lambda_2_step{s}"] = relerr(dev.lambda_2, ref.lambda_2)
    for name, x, y in zip(("mean", "var"), dev.predict_f(X[:50]), ref.predict_f(X[:50])):
        errs[name] = relerr(x, y)
    check(errs)
    dev.close()


def test_staged_heteroskedastic_minibatch_equals_set_data_bitwise():
    import tsvgp_b200 as tb
    X, Y = _demo_data(N=2000, seed=9)
    Z = np.linspace(X.min(), X.max(), 30)[:, None]
    kernel = so.SeparateIndependent([orc.SquaredExponential(), orc.Matern52(0.7, 2.0)])
    lik = so.HeteroskedasticTFPConditional(scale_transform=so.Exp())
    a = tb.t_SVGP(kernel, lik, Z.copy(), num_latent_gps=2, num_data=2000)
    b = tb.t_SVGP(kernel, lik, Z.copy(), num_latent_gps=2, num_data=2000)
    for lo in (0, 1000):
        a.set_data((X[lo:lo + 1000], Y[lo:lo + 1000]))
        a.natgrad_step(lr=0.5)
        b.stage_data((X[lo:lo + 1000], Y[lo:lo + 1000]))
        b.commit_staged()
        b.natgrad_step(lr=0.5)
    np.testing.assert_array_equal(a.lambda_1, b.lambda_1)
    np.testing.assert_array_equal(a.lambda_2_sqrt, b.lambda_2_sqrt)
    a.close(); b.close()


def test_refusals_and_per_latent_parameter_changes():
    import tsvgp_b200 as tb
    from tsvgp_b200 import _lib
    X, Y = _demo_data(N=500, seed=2)
    Z = np.linspace(X.min(), X.max(), 20)[:, None]
    k0, k1 = orc.SquaredExponential(1.0, 1.0), orc.SquaredExponential(1.0, 1.0)
    lik = so.HeteroskedasticTFPConditional()
    dev = tb.t_SVGP(so.SeparateIndependent([k0, k1]), lik, Z.copy(), num_latent_gps=2, num_data=500)
    dev.natgrad_step((X, Y), lr=0.5)
    before = dev.predict_f(X[:20])
    k1.lengthscales = orc._param(2.0)     # a changed lengthscale on latent 1 alone re-uploads the kernels
    after = dev.predict_f(X[:20])
    assert relerr(after[0][:, 0], before[0][:, 0]) < 1e-13 and relerr(after[1][:, 1], before[1][:, 1]) > 1e-3
    with pytest.raises(NotImplementedError):
        dev.elbo_and_grad((X, Y))
    with pytest.raises(_lib.InvalidArgumentError):   # the library refuses them too
        dev.set_option("white", 1)
        dev.natgrad_step((X, Y), lr=0.5)
    dev.close()
    three = tb.t_SVGP(orc.SquaredExponential(), lik, Z.copy(), num_latent_gps=3)
    with pytest.raises(_lib.InvalidArgumentError):   # heteroskedastic needs L = 2
        three.natgrad_step((X, np.zeros((500, 1))), lr=0.5)
    three.close()
    # the library's own refusals, below the Python ones: separate kernels with the whitened sibling (independent likelihood), and
    # tsvgp_elbo_grad with separate kernels or the heteroskedastic likelihood
    import ctypes as C
    Y2 = np.concatenate([Y, np.cos(X)], axis=1)
    gauss = tb.t_SVGP(so.SeparateIndependent([k0, orc.Matern52(0.7, 2.0)]), orc.Gaussian(0.1), Z.copy(), num_latent_gps=2)
    gauss.set_data((X, Y2))
    e, dv, dl = C.c_double(), C.c_double(), C.c_double()
    dls, dZ = np.empty(1), np.empty(Z.shape)
    rc = gauss._lib.tsvgp_elbo_grad(gauss._ctx, 1.0, C.byref(e), C.byref(dv), dls.ctypes.data, dZ.ctypes.data, C.byref(dl))
    assert rc == _lib.ERR_INVALID and b"separate" in gauss._lib.tsvgp_last_error(gauss._ctx)
    gauss.set_option("white", 1)
    with pytest.raises(_lib.InvalidArgumentError, match="separate"):
        gauss.natgrad_step(lr=0.5)
    gauss.close()
    shared = tb.t_SVGP(k0, lik, Z.copy(), num_latent_gps=2)
    shared.set_data((X, Y))
    rc = shared._lib.tsvgp_elbo_grad(shared._ctx, 1.0, C.byref(e), C.byref(dv), dls.ctypes.data, dZ.ctypes.data, C.byref(dl))
    assert rc == _lib.ERR_INVALID and b"heteroskedastic" in shared._lib.tsvgp_last_error(shared._ctx)
    shared.close()


def _free_device_bytes():
    import ctypes as C
    for name in ("libcudart.so.12", "/usr/local/cuda/lib64/libcudart.so.12", "libcudart.so"):
        try:
            rt = C.CDLL(name)
            break
        except OSError:
            continue
    else:
        pytest.skip("no CUDA runtime library to read the free device memory with")
    free, total = C.c_size_t(), C.c_size_t()
    assert rt.cudaSetDevice(0) == 0 and rt.cudaMemGetInfo(C.byref(free), C.byref(total)) == 0
    return free.value


def test_closing_a_separate_kernel_model_returns_its_device_memory():
    # every close must free the per-latent kernel buffers: at M = 2048 that is 5 M x M matrices (168 MB) per extra latent
    import tsvgp_b200 as tb
    import tsvgp_b200.synth as synth
    X, Y, Z = synth.make_minibatch(synth.describe("cfg3"), n_rows=4096, M=2048)
    kernel = so.SeparateIndependent([orc.Matern52(1.0, 3.0), orc.SquaredExponential(0.5, 2.0)])

    def cycle():
        m = tb.t_SVGP(kernel, so.HeteroskedasticTFPConditional(), Z.copy(), num_latent_gps=2, num_data=40960)
        m.natgrad_step((X, Y), lr=0.5)
        m.predict_f(X[:256])
        m.close()

    cycle()   # module loads and the library's one-time state
    before = _free_device_bytes()
    for _ in range(4):
        cycle()
    lost = before - _free_device_bytes()
    assert lost < 128 << 20, f"{lost / 2**20:.0f} MiB not returned after 4 models"   # a leak would be 4 x 168 MB


def _rank(rank, world, conn, out):
    sys.path.insert(0, ROOT)
    import tsvgp_b200 as tb
    X, Y = _demo_data(N=4001, seed=12)
    Z = np.linspace(X.min(), X.max(), 40)[:, None]
    kernel = so.SeparateIndependent([orc.SquaredExponential(), orc.Matern52(0.7, 2.0)])
    m = tb.t_SVGP(kernel, so.HeteroskedasticTFPConditional(), Z, num_latent_gps=2, num_data=4001, device=rank)
    m.set_option("chunk", 512)
    if rank == 0:
        uid = tb.comm_unique_id()
        for c in conn:
            c.send(uid)
    else:
        uid = conn.recv()
    m.init_comm(world, rank, uid)
    lo, hi = tb.shard_rows(X.shape[0], world, rank)
    elbos = [m.natgrad_step((X[lo:hi], Y[lo:hi]), lr=0.5, global_minibatch_size=X.shape[0], return_elbo=True) for _ in range(2)]
    out.put((rank, m.lambda_1, m.lambda_2, elbos, m.predict_f(X[:50])))
    m.close()


@pytest.mark.skipif(_n_gpus() < 2, reason="needs >= 2 GPUs")
def test_two_gpu_rows_sharded_heteroskedastic_separate_kernels():
    import tsvgp_b200 as tb
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    a, b = ctx.Pipe()
    procs = [ctx.Process(target=_rank, args=(0, 2, [a], out)), ctx.Process(target=_rank, args=(1, 2, b, out))]
    for p in procs:
        p.start()
    res = sorted([out.get(timeout=300) for _ in procs], key=lambda r: r[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    X, Y = _demo_data(N=4001, seed=12)
    Z = np.linspace(X.min(), X.max(), 40)[:, None]
    kernel = so.SeparateIndependent([orc.SquaredExponential(), orc.Matern52(0.7, 2.0)])
    single = tb.t_SVGP(kernel, so.HeteroskedasticTFPConditional(), Z, num_latent_gps=2, num_data=4001)
    single.set_option("chunk", 512)
    e = [single.natgrad_step((X, Y), lr=0.5, return_elbo=True) for _ in range(2)]
    mu, var = single.predict_f(X[:50])
    for rank, l1, l2, elbos, (mu_r, var_r) in res:
        assert relerr(l1, single.lambda_1) < 1e-10 and relerr(l2, single.lambda_2) < 1e-10
        assert relerr(elbos, e) < 1e-10 and relerr(mu_r, mu) < 1e-10 and relerr(var_r, var) < 1e-10
    np.testing.assert_array_equal(res[0][1], res[1][1])   # no skew between the ranks
    np.testing.assert_array_equal(res[0][2], res[1][2])
    single.close()
