"""
GPU: predict_f(full_cov=True) and predict_f_samples (tsvgp_predict_f_full_cov / tsvgp_predict_f_samples, DESIGN 13) against the
CPU restatement (tests/full_cov_oracle.py) of GPflow's base_conditional(full_cov=True) and sample_mvn [GPflow-recalled].
Parity tolerance 1e-9, norm-wise (relerr of test_gpu_parity).
"""
import multiprocessing as mp
import os
import sys

import numpy as np
import pytest

from oracle import tsvgp_oracle as orc
from tests import full_cov_oracle as fco
from tests.test_gpu_multi import _case, _n_gpus
from tests.test_gpu_parity import check, relerr

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _pair(cfg_name, n_rows, M, steps=2, num_data=None, mean_function=None, L=1):
    import tsvgp_b200 as tb
    import tsvgp_b200.synth as synth
    cfg = synth.describe(cfg_name)
    X, Y, Z = synth.make_minibatch(cfg, n_rows=n_rows, M=M)
    kernel, lik = synth.build_objects(cfg, orc)
    if L > 1:   # further latents: shifted copies of the config's own target
        Y = np.concatenate([Y] + [np.roll(Y, 17 * l, axis=0) for l in range(1, L)], axis=1)
    ref = orc.OracleTSVGP(kernel, lik, orc.InducingPoints(Z.copy()), num_latent_gps=L, num_data=num_data, mean_function=mean_function)
    dev = tb.t_SVGP(kernel, lik, Z.copy(), num_latent_gps=L, num_data=num_data, mean_function=mean_function)
    for _ in range(steps):
        dev.natgrad_step((X, Y), lr=cfg["lr"])
        ref.natgrad_step((X, Y), lr=cfg["lr"])
    return dev, ref, X, Y


def _query(X, n, seed=7):
    rng = np.random.default_rng(seed)
    idx = rng.integers(0, X.shape[0], n)
    return X[idx] + 0.05 * rng.standard_normal((n, X.shape[1]))


def _cov_errors(dev, ref, Xt):
    mu_d, cov_d = dev.predict_f(Xt, full_cov=True)
    mu_r, cov_r = fco.predict_f_full_cov(ref, Xt)
    L = dev.num_latent_gps
    assert mu_d.shape == (Xt.shape[0], L) and cov_d.shape == (L, Xt.shape[0], Xt.shape[0])
    # consistency with predict_f: the same means bit for bit, its variances on the diagonal
    mu_p, var_p = dev.predict_f(Xt)
    np.testing.assert_array_equal(mu_d, mu_p)
    return {"mean": relerr(mu_d, mu_r), "cov": relerr(cov_d, cov_r),
            "diag_vs_predict_f": relerr(np.diagonal(cov_d, axis1=1, axis2=2).T, var_p)}


def test_cfg1_full_cov():
    dev, ref, X, _ = _pair("cfg1", 10_000, 50)
    check(_cov_errors(dev, ref, _query(X, 300)))
    dev.close()


@pytest.mark.parametrize("n", [1, 128, 257])
def test_cfg2_full_cov_ragged(n):
    dev, ref, X, _ = _pair("cfg2", 3000, 500, num_data=100_000)
    check(_cov_errors(dev, ref, _query(X, n)))
    dev.close()


def test_cfg3_reduced_full_cov():
    dev, ref, X, _ = _pair("cfg3", 4096, 2048, num_data=60_000)
    check(_cov_errors(dev, ref, _query(X, 4096)))
    dev.close()


def test_three_latents_full_cov():
    dev, ref, X, _ = _pair("cfg2", 1500, 200, L=3)
    check(_cov_errors(dev, ref, _query(X, 200)))
    dev.close()


def test_mean_function_full_cov():
    dev, ref, X, _ = _pair("cfg2", 1500, 200, mean_function=lambda X: 0.3 + 0.1 * X[:, :1])
    check(_cov_errors(dev, ref, _query(X, 150)))
    dev.close()


def test_device_tensor_query_is_aliased():
    torch = pytest.importorskip("torch")
    dev, ref, X, _ = _pair("cfg2", 1500, 200)
    Xt = _query(X, 200)
    mu_h, cov_h = dev.predict_f(Xt, full_cov=True)
    mu_d, cov_d = dev.predict_f(torch.from_numpy(Xt).cuda(), full_cov=True)
    np.testing.assert_array_equal(mu_d, mu_h)
    np.testing.assert_array_equal(cov_d, cov_h)
    eps = np.random.default_rng(1).standard_normal((3, 200, 1))
    np.testing.assert_array_equal(dev.predict_f_samples(torch.from_numpy(Xt).cuda(), 3, epsilon=torch.from_numpy(eps).cuda()),
                                  dev.predict_f_samples(Xt, 3, epsilon=eps))
    dev.close()


def _spread(n, D, seed=3):
    # query points spread out against the lengthscale: cond(Sigma + 1e-6 I) stays moderate
    return np.random.default_rng(seed).standard_normal((n, D))


@pytest.mark.parametrize("L", [1, 3])
@pytest.mark.parametrize("full_cov", [True, False])
def test_samples_with_given_draws_match_the_oracle(L, full_cov):
    dev, ref, X, _ = _pair("cfg2", 1500, 200, L=L)
    Xt = _spread(64, X.shape[1])
    eps = np.random.default_rng(2).standard_normal((5, 64, L))
    f_d = dev.predict_f_samples(Xt, 5, full_cov=full_cov, epsilon=eps)
    f_r = fco.predict_f_samples(ref, Xt, 5, full_cov=full_cov, epsilon=eps)
    assert f_d.shape == (5, 64, L)
    if full_cov:
        # chol(Sigma + 1e-6 I) moves by at most ~cond times the relative error of Sigma (~1e-12 against the oracle, see
        # test_gpu_parity), so with cond <= 1e3 the 1e-9 gate keeps a wide margin
        _, cov = fco.predict_f_full_cov(ref, Xt)
        assert max(np.linalg.cond(cov[l] + 1e-6 * np.eye(64)) for l in range(L)) <= 1e3
    check({"samples": relerr(f_d, f_r)})
    assert dev.predict_f_samples(Xt, None, full_cov=full_cov, epsilon=eps[:1]).shape == (64, L)
    dev.close()


def test_philox_draws_reproduce_differ_and_have_the_right_moments():
    dev, ref, X, _ = _pair("cfg2", 1500, 200)
    Xt = _spread(32, X.shape[1], seed=5)
    dev.set_option("sample_seed", 1234)
    a = dev.predict_f_samples(Xt, 8192)
    b = dev.predict_f_samples(Xt, 8192)
    dev.set_option("sample_seed", 1234)
    np.testing.assert_array_equal(dev.predict_f_samples(Xt, 8192), a)
    assert not np.array_equal(a, b)
    mu, cov = dev.predict_f(Xt, full_cov=True)
    S, C = 8192, cov[0] + 1e-6 * np.eye(32)
    f = a[:, :, 0]
    d = np.sqrt(np.diag(C))
    # standard errors of the empirical mean (sqrt(C_ii / S)) and covariance (sqrt((C_ii C_jj + C_ij^2) / S)); 6 of them bound
    # 32 means and 1024 covariances with room to spare (a 6-sigma miss has probability ~2e-9 per entry)
    assert np.all(np.abs(f.mean(0) - mu[:, 0]) <= 6 * d / np.sqrt(S))
    emp = np.cov(f.T)
    assert np.all(np.abs(emp - C) <= 6 * np.sqrt((np.outer(d, d) ** 2 + C ** 2) / S))
    # the diagonal samples use the same generator: their marginals agree too
    g = dev.predict_f_samples(Xt, 8192, full_cov=False)[:, :, 0]
    assert np.all(np.abs(g.mean(0) - mu[:, 0]) <= 6 * d / np.sqrt(S))
    dev.close()


def test_softmax_steps_and_sites_are_untouched_by_sampling():
    import tsvgp_b200 as tb
    rng = np.random.default_rng(5)
    N, M, D, C = 600, 64, 4, 3
    X = rng.standard_normal((N, D))
    labels = np.argmax(X @ rng.standard_normal((D, C)), axis=1).astype(float)[:, None]
    kernel, lik = orc.Matern52(variance=1.0, lengthscales=1.7), orc.Softmax(C, num_monte_carlo_points=20)
    a = tb.t_SVGP(kernel, lik, X[:M].copy(), num_latent_gps=C, num_data=3 * N)
    b = tb.t_SVGP(kernel, lik, X[:M].copy(), num_latent_gps=C, num_data=3 * N)
    ea = [a.natgrad_step((X, labels), lr=0.4, return_elbo=True) for _ in range(2)]
    eb = [b.natgrad_step((X, labels), lr=0.4, return_elbo=True)]
    l1, l2 = b.lambda_1, b.lambda_2_sqrt
    b.predict_f_samples(X[:40], 6)
    b.predict_f_samples(X[:40], 6, full_cov=False)
    b.predict_f(X[:40], full_cov=True)
    np.testing.assert_array_equal(b.lambda_1, l1)
    np.testing.assert_array_equal(b.lambda_2_sqrt, l2)
    eb.append(b.natgrad_step((X, labels), lr=0.4, return_elbo=True))
    assert ea == eb
    np.testing.assert_array_equal(a.lambda_1, b.lambda_1)
    np.testing.assert_array_equal(a.lambda_2_sqrt, b.lambda_2_sqrt)
    a.close(); b.close()


def test_raising_cases():
    import tsvgp_b200 as tb
    dev, _, X, Y = _pair("cfg2", 1500, 200)
    with pytest.raises(NotImplementedError):
        dev.predict_f(X[:10], full_cov=True, full_output_cov=True)
    with pytest.raises(NotImplementedError):
        dev.predict_y(X[:10], full_cov=True)
    with pytest.raises(NotImplementedError):
        dev.predict_log_density((X[:10], Y[:10]), full_cov=True)
    with pytest.raises(NotImplementedError):
        dev.predict_f_samples(X[:10], 2, full_output_cov=True)
    # N x N buffers of 200 000 query points (320 GB) cannot fit: refused before anything is allocated, the context stays usable
    big = np.zeros((200_000, X.shape[1]))
    with pytest.raises(tb.InvalidArgumentError, match="bytes"):
        dev.predict_f_samples(big, 1, full_cov=True)
    mu, var = dev.predict_f(X[:10])
    np.testing.assert_array_equal(dev.predict_f(X[:10], full_cov=True)[0], mu)
    dev.close()
    cfg_kernel, lik = orc.SquaredExponential(variance=1.0, lengthscales=1.0), orc.Gaussian(variance=0.1)
    w = tb.t_SVGP_white(cfg_kernel, lik, X[:50].copy())
    wr = orc.OracleTSVGPWhite(cfg_kernel, lik, orc.InducingPoints(X[:50].copy()))
    Yg = np.sin(X[:, :1])
    w.natgrad_step((X, Yg), lr=0.5)
    wr.natgrad_step((X, Yg), lr=0.5)
    with pytest.raises(NotImplementedError):
        w.predict_f(X[:10], full_cov=True)
    with pytest.raises(NotImplementedError):
        w.predict_f(X[:10], full_output_cov=True)
    with pytest.raises(NotImplementedError):
        w.predict_f_samples(X[:10], 2)
    eps = np.random.default_rng(0).standard_normal((2, 10, 1))
    mu_r, var_r = wr.predict_f(X[:10])
    check({"white_diag_samples": relerr(w.predict_f_samples(X[:10], 2, full_cov=False, epsilon=eps), mu_r + np.sqrt(var_r) * eps)})
    w.close()


def _rank(rank, world, conn, out):
    sys.path.insert(0, ROOT)
    import tsvgp_b200 as tb
    cfg, X, Y, Z, kernel, lik = _case(300)
    m = tb.t_SVGP(kernel, lik, Z, num_data=50_010, device=rank)
    m.set_option("dist_min_m", 128)
    m.set_option("shard_min_m", 1 << 30)
    if rank == 0:
        uid = tb.comm_unique_id()
        for c in conn:
            c.send(uid)
    else:
        uid = conn.recv()
    m.init_comm(world, rank, uid)
    lo, hi = tb.shard_rows(X.shape[0], world, rank)
    m.natgrad_step((X[lo:hi], Y[lo:hi]), lr=cfg["lr"], global_minibatch_size=X.shape[0])
    eps = np.random.default_rng(0).standard_normal((3, 40, 1))
    solo = (m.predict_f(X[:40], full_cov=True), m.predict_f_samples(X[:40], 3, epsilon=eps)) if rank == 0 else None
    e = m.elbo((X[lo:hi], Y[lo:hi]), global_minibatch_size=X.shape[0])   # collective: rank 0's solo calls must not unbalance it
    out.put((rank, e, solo))
    m.close()


@pytest.mark.skipif(_n_gpus() < 2, reason="needs >= 2 GPUs")
def test_two_gpu_rank0_alone_predicts_full_cov():
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
    cfg, X, Y, Z, kernel, lik = _case(300)
    single = tb.t_SVGP(kernel, lik, Z, num_data=50_010)
    single.natgrad_step((X, Y), lr=cfg["lr"])
    eps = np.random.default_rng(0).standard_normal((3, 40, 1))
    (mu, cov), f = single.predict_f(X[:40], full_cov=True), single.predict_f_samples(X[:40], 3, epsilon=eps)
    e = single.elbo((X, Y))
    (mu0, cov0), f0 = res[0][2]
    tol = 1e-11   # summation order only, as in test_gpu_multi
    assert relerr(mu0, mu) < tol and relerr(cov0, cov) < tol and relerr(f0, f) < 1e-10
    for _, e_r, _ in res:
        assert abs(e_r - e) / abs(e) < tol
    single.close()
