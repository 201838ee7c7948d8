"""
GPU: the whitened sibling `t_SVGP_white` with the Softmax likelihood (DESIGN 10, "Softmax") against OracleTSVGPWhite with the
Monte-Carlo draws fixed (`set_mc_epsilon` / the oracle's `epsilon`): natgrad_step, elbo, predict_f, prior_kl, the posterior and
predict_f_extra_data, and the M-step gradients against the CPU restatement tests/white_grad_oracle.py (pinned by central
differences in tests/test_white_softmax_cpu.py).  Tolerance 1e-9 norm-wise relative, as for the rest of the path.
"""
import importlib.util
import os

import numpy as np
import pytest

from oracle import tsvgp_oracle as orc
from tests import white_grad_oracle as wgo

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def relerr(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def _example():
    spec = importlib.util.spec_from_file_location("vem_softmax", os.path.join(ROOT, "examples", "vem_softmax.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _problem(cfg_name, N, M, C, S, seed=5):
    """-> X, Y [N, 1] class labels, Z, kernel, eps [S, N, C].  "mnist": examples/vem_softmax.py's data at D = 784 with ARD
    Matern-5/2 lengthscales; otherwise a synthetic config's inputs (cond(Kuu) in 1e2..1e4, which the difference of inverses
    Q = A^-1 - R^-1 needs at 1e-9) labelled by the largest of C random projections."""
    rng = np.random.default_rng(seed)
    if cfg_name == "mnist":
        X, Y = _example().make_data(N, C=C)
        Z = X[:M].copy()
        kernel = orc.Matern52(variance=1.0, lengthscales=20.0 * np.linspace(0.9, 1.1, X.shape[1]))
    else:
        import tsvgp_b200.synth as synth
        cfg = synth.describe(cfg_name)
        X, _, Z = synth.make_minibatch(cfg, n_rows=N, M=M)
        Y = np.argmax(X @ rng.standard_normal((X.shape[1], C)), axis=1).astype(float)[:, None]
        kernel, _ = synth.build_objects(cfg, orc)
    return X, Y, Z, kernel, rng.standard_normal((S, N, C))


def _models(X, Y, Z, kernel, eps, num_data, opts=None, sites=None):
    """the device model (draws fixed to eps) and the oracle on the same likelihood and sites"""
    import tsvgp_b200 as tb
    S, _, C = eps.shape
    lik = orc.Softmax(C, num_monte_carlo_points=S, epsilon=eps)
    l1, l2 = sites if sites is not None else (None, None)
    dev = tb.t_SVGP_white(kernel, lik, Z.copy(), num_latent_gps=C, num_data=num_data, lambda_1=l1, lambda_2=l2)
    for k, v in (opts or {}).items():
        dev.set_option(k, v)
    dev.set_mc_epsilon(eps)
    dev.set_data((X, Y))
    ref = orc.OracleTSVGPWhite(kernel, lik, orc.InducingPoints(Z.copy()), num_latent_gps=C, num_data=num_data,
                               lambda_1=l1, lambda_2=l2)
    return dev, ref


def _grad_errs(e_dev, g_dev, e_ref, g_ref):
    assert g_dev["likelihood"] is None and g_ref["likelihood"] is None
    return {"grad_elbo": abs(e_dev - e_ref) / abs(e_ref), "d_variance": abs(g_dev["variance"] - g_ref["variance"]) / abs(g_ref["variance"]),
            "d_lengthscales": relerr(np.ravel(g_dev["lengthscales"]), g_ref["lengthscales"]), "d_Z": relerr(g_dev["Z"], g_ref["Z"])}


CASES = [  # config, rows, M, classes C, Monte-Carlo points S, num_data, library options (route 1 fused, 2 whitened, 3 exact), lr
    # (the whitened update takes h unclipped, tsvgp_white.py:183-212: with few draws or a large num_data / rows a step of the
    # reference itself can leave Lambda_2 + Kuu indefinite; lr and S are chosen so that the oracle's steps succeed)
    ("cfg2", 1000, 50, 3, 40, None, {}, 0.5),
    ("cfg2", 1500, 200, 10, 40, 15_000, {"route": 1}, 0.5),
    ("cfg2", 1500, 200, 3, 20, None, {"route": 2}, 0.5),
    ("cfg3", 3000, 384, 3, 20, 30_000, {"chunk": 1024, "route": 3}, 0.5),   # three slabs on two streams
    ("cfg3", 4096, 2048, 3, 20, 40_000, {"chunk": 1024}, 0.3),               # four slabs
    ("mnist", 200, 100, 10, 100, 60_000, {}, 0.1),                           # docs/notebooks/mnist.py's minibatch
]


@pytest.mark.parametrize("cfg_name,n,M,C,S,num_data,opts,lr", CASES)
def test_white_softmax_matches_oracle(cfg_name, n, M, C, S, num_data, opts, lr):
    X, Y, Z, kernel, eps = _problem(cfg_name, n, M, C, S)
    dev, ref = _models(X, Y, Z, kernel, eps, num_data, opts)
    errs = {}
    for s in range(3 if M <= 200 else 2):
        e_ref = ref.elbo((X, Y))
        e_dev = dev.natgrad_step(lr=lr, return_elbo=True)
        ref.natgrad_step((X, Y), lr=lr)
        errs[f"elbo_before{s}"] = abs(e_dev - e_ref) / abs(e_ref)
        errs[f"lambda_1_{s}"] = relerr(dev.lambda_1, ref.lambda_1)
        errs[f"lambda_2_{s}"] = relerr(dev.lambda_2, ref.lambda_2)
    assert dev.lambda_1.shape == (M, C) and dev.lambda_2.shape == (C, M, M)
    errs["elbo"] = abs(dev.elbo() - ref.elbo((X, Y))) / abs(ref.elbo((X, Y)))
    Xq = X[:200] + 0.05
    mu_d, var_d = dev.predict_f(Xq)
    mu_r, var_r = ref.predict_f(Xq)
    assert mu_d.shape == (200, C)
    errs["mean"], errs["var"] = relerr(mu_d, mu_r), relerr(var_d, var_r)
    errs["prior_kl"] = abs(dev.prior_kl() - ref.prior_kl()) / abs(ref.prior_kl())
    m_d, cs_d = dev.get_mean_chol_cov_inducing_posterior()
    m_r, cs_r = ref.get_mean_chol_cov_inducing_posterior()
    errs["m_q"] = relerr(m_d, m_r)
    errs["S_q"] = max(relerr(cs_d[l] @ cs_d[l].T, cs_r[l] @ cs_r[l].T) for l in range(C))
    # the diagonal samples are mean + sqrt(var) eps, predict_f's moments
    e_s = np.random.default_rng(1).standard_normal((2, 200, C))
    errs["samples"] = relerr(dev.predict_f_samples(Xq, 2, full_cov=False, epsilon=e_s), mu_r + np.sqrt(var_r) * e_s)
    # M-step gradients at the device's sites; the call leaves the state untouched
    rg = orc.OracleTSVGPWhite(kernel, ref.likelihood, orc.InducingPoints(Z.copy()), num_latent_gps=C, num_data=num_data,
                              lambda_1=dev.lambda_1, lambda_2=dev.lambda_2)
    e_ref, g_ref = wgo.elbo_gradients(rg, (X, Y))
    e_before = dev.elbo()
    e_dev, g_dev = dev.elbo_and_grad()
    assert np.shape(g_dev["lengthscales"]) == np.shape(np.asarray(kernel.lengthscales))
    errs.update(_grad_errs(e_dev, g_dev, e_ref, g_ref))
    bad = {k: v for k, v in errs.items() if not v <= 1e-9}
    assert not bad, (bad, errs)
    assert dev.elbo() == e_before
    dev.close()


@pytest.mark.parametrize("jitter", [1e-6, 0.0])
def test_predict_f_extra_data(jitter):
    # tsvgp_white.py:134-158 with Softmax: the extra data's g and h under the current sites, then the conditional with the combined
    # sites; the sites are left bitwise as they were
    X, Y, Z, kernel, eps = _problem("cfg2", 2100, 160, 5, 20)
    Xt, Yt, Xe, Ye = X[:1500], Y[:1500], X[1500:], Y[1500:]
    dev, ref = _models(Xt, Yt, Z, kernel, eps[:, :1500], 6000)
    dev.natgrad_step(lr=0.6)
    ref.natgrad_step((Xt, Yt), lr=0.6)
    l1, l2 = dev.lambda_1, dev.lambda_2
    dev.set_mc_epsilon(eps[:, 1500:])
    ref.likelihood.epsilon = eps[:, 1500:]
    Xq = X[:300] + 0.1
    mu_r, var_r = ref.predict_f_extra_data(Xq, (Xe, Ye), jitter=jitter)
    mu_d, var_d = dev.predict_f_extra_data(Xq, (Xe, Ye), jitter=jitter)
    assert relerr(mu_d, mu_r) < 1e-9 and relerr(var_d, var_r) < 1e-9
    np.testing.assert_array_equal(dev.lambda_1, l1)
    np.testing.assert_array_equal(dev.lambda_2, l2)
    mu0_d, var0_d = dev.predict_f(Xq)
    mu0_r, var0_r = ref.predict_f(Xq)
    assert relerr(mu0_d, mu0_r) < 1e-9 and relerr(var0_d, var0_r) < 1e-9
    dev.close()


def test_gradients_for_inputs_far_from_the_origin():
    # as tests/test_gpu_white_grad.py: the kernel matrices themselves lose ~ eps (|x| / l)^2 = 1e-10 relative in r^2
    rng = np.random.default_rng(9)
    N, M, D, C, S = 1500, 32, 3, 3, 20
    ls = np.array([0.9, 1.3, 1.7])
    shift = 1.0e3 * ls
    X = rng.standard_normal((N, D)) + shift
    Z = X[:M].copy()
    Y = np.argmax((X - shift) @ rng.standard_normal((D, C)), axis=1).astype(float)[:, None]
    eps = rng.standard_normal((S, N, C))
    kernel = orc.Matern52(variance=1.1, lengthscales=ls)
    lik = orc.Softmax(C, num_monte_carlo_points=S, epsilon=eps)
    ref = orc.OracleTSVGPWhite(kernel, lik, orc.InducingPoints(Z.copy()), num_latent_gps=C)
    ref.natgrad_step((X, Y), lr=0.6)
    dev, ref = _models(X, Y, Z, kernel, eps, None, sites=(ref.lambda_1, ref.lambda_2))
    e_ref, g_ref = wgo.elbo_gradients(ref, (X, Y))
    e_dev, g_dev = dev.elbo_and_grad()
    errs = _grad_errs(e_dev, g_dev, e_ref, g_ref)
    bad = {k: v for k, v in errs.items() if not v <= 1e-6}
    assert not bad, (bad, errs)
    dev.close()


def test_one_draw_per_call():
    # no explicit draws: elbo_and_grad and predict_f_extra_data each take one draw, as natgrad_step and elbo do
    import tsvgp_b200 as tb
    X, Y, Z, kernel, eps = _problem("cfg2", 1500, 64, 5, 40)
    lik = orc.Softmax(5, num_monte_carlo_points=40)
    a, b = (tb.t_SVGP_white(kernel, lik, Z.copy(), num_latent_gps=5, num_data=4000) for _ in range(2))
    for m in (a, b):
        m.set_option("mc_seed", 1234)
        m.set_data((X, Y))
        m.set_mc_epsilon(eps)           # the same sites on both: two steps with fixed draws, then back to the generator
        m.natgrad_step(lr=0.5)
        m.natgrad_step(lr=0.5)
        m.set_mc_epsilon(None)
    e_grad, _ = a.elbo_and_grad()
    e1 = b.elbo()
    assert abs(e_grad - e1) <= 1e-12 * abs(e1), (e_grad, e1)
    e2 = b.elbo()
    assert e2 != e1
    assert a.elbo() == e2
    a.predict_f_extra_data(X[:10], (X, Y))   # draw 2 on a (its data stay the same), elbo's draw 2 on b
    b.elbo()
    assert a.elbo() == b.elbo()
    a.close()
    b.close()


def test_non_finite_inputs_raise_with_the_sites_unchanged():
    import tsvgp_b200 as tb
    X, Y, Z, kernel, eps = _problem("cfg2", 1200, 80, 5, 20)
    dev, _ = _models(X, Y, Z, kernel, eps, 5000, {"chunk": 512})
    dev.natgrad_step(lr=0.5)
    l1, l2 = dev.lambda_1, dev.lambda_2
    for bad_value in (np.nan, np.inf):
        Xbad = X.copy()
        Xbad[777, 2] = bad_value
        with pytest.raises(tb.NonPositiveVarianceError):
            dev.natgrad_step((Xbad, Y), lr=0.5)
        np.testing.assert_array_equal(dev.lambda_1, l1)
        np.testing.assert_array_equal(dev.lambda_2, l2)
        with pytest.raises(tb.NonPositiveVarianceError):
            dev.elbo_and_grad((Xbad, Y))
    dev.close()


def test_vem_fit_raises_the_elbo_at_the_mnist_shape():
    # the MNIST notebook's model as examples/vem_softmax.py runs it (M = 100, D = 784, Softmax(10), S = 100, minibatches of 200,
    # train_Z), on the whitened sibling: draws fixed per minibatch, three epochs of three minibatches
    import tsvgp_b200 as tb
    from tsvgp_b200 import standins as st, vem
    mod = _example()
    n, batch, S, C = 600, 200, 100, 10
    X, y = mod.make_data(n)
    kernel = st.Matern52(variance=1.0, lengthscales=np.full(X.shape[1], 20.0))
    model = tb.t_SVGP_white(kernel, st.Softmax(C, num_monte_carlo_points=S), X[:100].copy(), num_latent_gps=C, num_data=n)
    rng, eps_rng = np.random.RandomState(7), np.random.RandomState(8)
    trace = []
    for _ in range(3):
        order = rng.permutation(n)
        for k in range(n // batch):
            idx = order[k * batch:(k + 1) * batch]
            model.set_mc_epsilon(eps_rng.randn(S, batch, C))
            trace += vem.fit(model, (X[idx], y[idx]), n_iters=1, n_e_steps=2, n_m_steps=2, lr_natgrad=0.5, lr_adam=0.01, train_Z=True)
    model.close()
    assert np.all(np.isfinite(trace))
    assert np.mean(trace[-4:]) > np.mean(trace[:4]), trace


# ---- two ranks ---------------------------------------------------------------------------------------------------------
def _rank_worker(rank, world, conn, X, Y, Z, ls, eps, l1, l2, q):
    # each rank holds its rows of the minibatch and the same rows of the explicit draws
    import sys
    sys.path.insert(0, ROOT)
    try:
        import tsvgp_b200 as tb
        from tsvgp_b200 import standins as st
        C, S = eps.shape[2], eps.shape[0]
        m = tb.t_SVGP_white(st.Matern52(variance=1.0, lengthscales=ls), st.Softmax(C, num_monte_carlo_points=S), Z.copy(),
                            num_latent_gps=C, num_data=20_000, lambda_1=l1, lambda_2=l2, device=rank)
        if rank == 0:
            uid = tb.comm_unique_id()
            for c in conn:
                c.send(uid)
        else:
            uid = conn.recv()
        m.init_comm(world, rank, uid)
        lo, hi = tb.shard_rows(X.shape[0], world, rank)
        m.set_mc_epsilon(np.ascontiguousarray(eps[:, lo:hi]))
        e, g = m.elbo_and_grad((X[lo:hi], Y[lo:hi]), global_minibatch_size=X.shape[0])
        q.put((rank, e, g["variance"], np.asarray(g["lengthscales"]), g["Z"]))
        m.close()
    except Exception as ex:   # reported to the parent, which fails the test
        q.put((rank, repr(ex), None, None, None))


def test_two_ranks_match_one():
    import multiprocessing as mp
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import tsvgp_b200 as tb
    from tsvgp_b200 import standins as st
    X, Y, Z, kernel, eps = _problem("cfg2", 3000, 128, 10, 40)
    ls = np.asarray(kernel.lengthscales)
    one = tb.t_SVGP_white(st.Matern52(variance=1.0, lengthscales=ls), st.Softmax(10, num_monte_carlo_points=40), Z.copy(),
                          num_latent_gps=10, num_data=20_000)
    one.set_mc_epsilon(eps)
    one.natgrad_step((X, Y), lr=0.5)
    l1, l2 = one.lambda_1, one.lambda_2
    e1, g1 = one.elbo_and_grad((X, Y))
    one.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    a, b = ctx.Pipe()
    procs = [ctx.Process(target=_rank_worker, args=(r, 2, [a] if r == 0 else b, X, Y, Z, ls, eps, l1, l2, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted((q.get(timeout=600) for _ in procs), key=lambda r: r[0])
    for p in procs:
        p.join(timeout=120)
    for rank, e, dv, dls, dZ in res:
        assert dv is not None, e
        assert abs(e - e1) <= 1e-11 * abs(e1)
        assert abs(dv - g1["variance"]) <= 1e-11 * abs(g1["variance"])
        assert relerr(dls, g1["lengthscales"]) <= 1e-11 and relerr(dZ, g1["Z"]) <= 1e-11
