"""
GPU: M-step gradients with the Softmax likelihood (one pass over all latents, h unclipped) and at any input dimension, against
tests/softmax_grad_oracle.py (itself pinned by central differences and by the one-latent oracle on the CPU) with fixed
Monte-Carlo draws.  Tolerance 1e-9 norm-wise relative, as for the rest of the path.
"""
import os

import numpy as np
import pytest

from oracle import tsvgp_oracle as orc
from tests import softmax_grad_oracle as sgo

pytestmark = pytest.mark.gpu


def relerr(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def _softmax_problem(N, M, D, C, S, kind, ard, seed=3):
    rng = np.random.default_rng(seed)
    protos = (rng.random((C, D)) < 0.3).astype(float)
    y = rng.integers(0, C, size=N)
    X = protos[y] + 0.4 * rng.standard_normal((N, D))
    Z = X[:M] + 0.05 * rng.standard_normal((M, D))
    ls0 = 0.6 * np.sqrt(D)
    ls = ls0 * np.linspace(0.8, 1.25, D) if ard else ls0
    kernel = (orc.Matern52 if kind == "matern52" else orc.SquaredExponential)(variance=1.3, lengthscales=ls)
    eps = rng.standard_normal((S, N, C))
    return X, y.astype(float)[:, None], Z, kernel, eps


def _trained(X, Y, Z, kernel, eps, C, num_data, opts, steps=2):
    """device model after `steps` natgrad steps with the draws fixed, and the oracle model on the device's sites"""
    import tsvgp_b200 as tb
    S = eps.shape[0]
    lik = orc.Softmax(C, num_monte_carlo_points=S, epsilon=eps)
    dev = tb.t_SVGP(kernel, lik, Z.copy(), num_latent_gps=C, num_data=num_data)
    for k, v in opts.items():
        dev.set_option(k, v)
    dev.set_mc_epsilon(eps)
    for _ in range(steps):
        dev.natgrad_step((X, Y), lr=0.5)
    l1, l2s = dev.lambda_1, dev.lambda_2_sqrt
    ref = orc.OracleTSVGP(kernel, lik, orc.InducingPoints(Z.copy()), num_latent_gps=C, num_data=num_data,
                          lambda_1=l1, lambda_2_sqrt=l2s)
    return dev, ref


def _errs(e_dev, g_dev, e_ref, g_ref):
    return {"elbo": abs(e_dev - e_ref) / abs(e_ref), "variance": abs(g_dev["variance"] - g_ref["variance"]) / abs(g_ref["variance"]),
            "lengthscales": relerr(np.ravel(g_dev["lengthscales"]), g_ref["lengthscales"]), "Z": relerr(g_dev["Z"], g_ref["Z"])}


SOFTMAX_CASES = [  # N, M, D, C, S, kernel, ARD, num_data, library options
    (1000, 64, 4, 2, 1, "matern52", True, None, {"chunk": 256, "streams": 2}),
    (1537, 100, 6, 5, 40, "se", False, 6000, {"chunk": 512, "streams": 1}),
    (2000, 128, 5, 10, 100, "matern52", True, 10_000, {"streams": 2}),
    (3001, 200, 8, 10, 40, "se", False, 30_000, {"chunk": 1024, "streams": 2}),
    (901, 72, 3, 5, 100, "matern52", False, None, {"chunk": 384, "streams": 1}),
    (200, 100, 784, 10, 100, "matern52", True, 60_000, {}),                    # docs/notebooks/mnist.py's shape
    (16384, 1024, 784, 10, 100, "matern52", True, 60_000, {}),                 # larger: M = 1024, one 16 384-point slab per stream
]


@pytest.mark.parametrize("N,M,D,C,S,kind,ard,num_data,opts", SOFTMAX_CASES)
def test_softmax_gradients_match_helper(N, M, D, C, S, kind, ard, num_data, opts):
    X, Y, Z, kernel, eps = _softmax_problem(N, M, D, C, S, kind, ard)
    dev, ref = _trained(X, Y, Z, kernel, eps, C, num_data, opts)
    e_ref, g_ref = sgo.elbo_gradients(ref, (X, Y))
    e_dev, g_dev = dev.elbo_and_grad((X, Y))
    assert g_dev["likelihood"] is None
    assert np.shape(g_dev["lengthscales"]) == np.shape(np.asarray(kernel.lengthscales))
    errs = _errs(e_dev, g_dev, e_ref, g_ref)
    bad = {k: v for k, v in errs.items() if not v <= 1e-9}
    assert not bad, (bad, errs)
    dev.close()


def test_softmax_gradient_leaves_the_state_untouched():
    # a natgrad step after elbo_and_grad still matches the oracle (test_gpu_gradients.py checks the same for one latent)
    X, Y, Z, kernel, eps = _softmax_problem(1200, 80, 5, 5, 40, "matern52", True)
    dev, ref = _trained(X, Y, Z, kernel, eps, 5, 5000, {"chunk": 512})
    dev.elbo_and_grad((X, Y))
    dev.natgrad_step((X, Y), lr=0.5)
    ref.natgrad_step((X, Y), lr=0.5)
    assert relerr(dev.lambda_1, ref.lambda_1) < 1e-9 and relerr(dev.lambda_2, ref.lambda_2) < 1e-9
    dev.close()


@pytest.mark.parametrize("lik_name", ["gaussian", "student_t"])
def test_independent_likelihood_above_63_inputs(lik_name):
    # D = 100: the augmented block [xs | 1 | xs^2] is 256 columns wide; the one-latent path against the unchanged oracle
    import tsvgp_b200 as tb
    rng = np.random.default_rng(21)
    N, M, D = 2500, 96, 100
    X = rng.standard_normal((N, D))
    Z = X[:M] + 0.05 * rng.standard_normal((M, D))
    f = np.sin(X[:, :5].sum(1, keepdims=True))
    kernel = orc.Matern52(variance=1.2, lengthscales=8.0 * np.linspace(0.9, 1.1, D))
    if lik_name == "gaussian":
        lik, Y = orc.Gaussian(variance=0.1), f + 0.3 * rng.standard_normal((N, 1))
    else:
        lik, Y = orc.StudentT(scale=0.4, df=3.0), f + 0.3 * rng.standard_t(3.0, size=(N, 1))
    ref = orc.OracleTSVGP(kernel, lik, orc.InducingPoints(Z.copy()), num_data=10_000)
    for _ in range(2):
        ref.natgrad_step((X, Y), lr=0.6)
    dev = tb.t_SVGP(kernel, lik, Z.copy(), num_data=10_000, lambda_1=ref.lambda_1, lambda_2_sqrt=ref.lambda_2_sqrt)
    dev.set_option("chunk", 1024)
    e_ref, g_ref = orc.elbo_gradients(ref, (X, Y))
    e_dev, g_dev = dev.elbo_and_grad((X, Y))
    errs = _errs(e_dev, g_dev, e_ref, g_ref)
    errs["likelihood"] = abs(g_dev["likelihood"] - g_ref["likelihood"]) / abs(g_ref["likelihood"])
    bad = {k: v for k, v in errs.items() if not v <= 1e-9}
    assert not bad, (bad, errs)
    dev.close()


def test_one_draw_per_call():
    # no explicit draws: elbo_and_grad at draw k returns the ELBO elbo returns at draw k, and advances the draw once
    import tsvgp_b200 as tb
    X, Y, Z, kernel, eps = _softmax_problem(1500, 64, 4, 5, 40, "se", False)
    lik = orc.Softmax(5, num_monte_carlo_points=40)
    a, b = (tb.t_SVGP(kernel, lik, Z.copy(), num_latent_gps=5, num_data=4000) for _ in range(2))
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
    a.close()
    b.close()


def test_vem_fit_softmax_example():
    # examples/vem_softmax.py at a reduced size (600 training rows, 3 minibatches per epoch), draws fixed: the ELBO rises and the
    # 10-class training accuracy (chance 0.1) is above 0.9 — the synthetic classes are well separated
    import importlib.util
    path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "examples", "vem_softmax.py")
    spec = importlib.util.spec_from_file_location("vem_softmax", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    trace, acc_train, acc_test = mod.main(n_train=600, n_test=300, n_epochs=3, fixed_draws=True, verbose=False)
    assert np.all(np.isfinite(trace))
    assert np.mean(trace[-4:]) > np.mean(trace[:4]), trace
    assert acc_train > 0.9 and acc_test > 0.8, (acc_train, acc_test)


# ---- two ranks ---------------------------------------------------------------------------------------------------------
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _rank_worker(rank, world, conn, X, Y, Z, ls, eps, l1, l2s, q):
    # each rank holds its rows of the minibatch and the same rows of the explicit draws
    import sys
    sys.path.insert(0, ROOT)
    try:
        import tsvgp_b200 as tb
        from tsvgp_b200 import standins as st
        C, S = eps.shape[2], eps.shape[0]
        m = tb.t_SVGP(st.Matern52(variance=1.3, lengthscales=ls), st.Softmax(C, num_monte_carlo_points=S), Z.copy(),
                      num_latent_gps=C, num_data=20_000, lambda_1=l1, lambda_2_sqrt=l2s, device=rank)
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
    X, Y, Z, kernel, eps = _softmax_problem(3000, 128, 6, 10, 40, "matern52", True)
    ls = np.asarray(kernel.lengthscales)
    one = tb.t_SVGP(st.Matern52(variance=1.3, lengthscales=ls), st.Softmax(10, num_monte_carlo_points=40), Z.copy(),
                    num_latent_gps=10, num_data=20_000)
    one.set_mc_epsilon(eps)
    one.natgrad_step((X, Y), lr=0.5)
    l1, l2s = one.lambda_1, one.lambda_2_sqrt
    e1, g1 = one.elbo_and_grad((X, Y))
    one.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    a, b = ctx.Pipe()
    procs = [ctx.Process(target=_rank_worker, args=(r, 2, [a] if r == 0 else b, X, Y, Z, ls, eps, l1, l2s, q)) for r in range(2)]
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
