"""
GPU: M-step gradients of the whitened sibling (tsvgp_elbo_grad with option "white", through t_SVGP_white.elbo_and_grad) against
the CPU restatement tests/white_grad_oracle.py, itself pinned by central differences of OracleTSVGPWhite.elbo
(tests/test_white_grad_cpu.py).  Tolerance 1e-9 norm-wise relative, as tests/test_gpu_gradients.py holds the plain model.
"""
import os

import numpy as np
import pytest

from oracle import tsvgp_oracle as orc
from tests import matern_oracle as mo
from tests import white_grad_oracle as wgo

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def relerr(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def _errs(e_dev, g_dev, e_ref, g_ref):
    errs = {"elbo": abs(e_dev - e_ref) / abs(e_ref), "variance": abs(g_dev["variance"] - g_ref["variance"]) / abs(g_ref["variance"]),
            "lengthscales": relerr(np.ravel(g_dev["lengthscales"]), g_ref["lengthscales"]), "Z": relerr(g_dev["Z"], g_ref["Z"])}
    if g_ref["likelihood"] is None:
        assert g_dev["likelihood"] is None
    else:
        errs["likelihood"] = abs(g_dev["likelihood"] - g_ref["likelihood"]) / abs(g_ref["likelihood"])
    return errs


def _trained(kernel, lik, X, Y, Z, num_data, L=1, steps=2, lr=0.5):
    ref = orc.OracleTSVGPWhite(kernel, lik, orc.InducingPoints(Z.copy()), num_latent_gps=L, num_data=num_data)
    for _ in range(steps):
        ref.natgrad_step((X, Y), lr=lr)
    return ref


CASES = [  # config, rows, M, num_data, ARD lengthscales?, library options
    ("cfg1", 3000, 50, None, False, {}),
    ("cfg2", 2500, 200, 25_000, True, {}),
    ("cfg3", 3000, 384, 30_000, False, {"chunk": 1024}),          # three slabs on two streams
    ("cfg3", 8192, 2048, 1_000_000, False, {"chunk": 2048}),     # four slabs
]


@pytest.mark.parametrize("name,n,M,num_data,ard,opts", CASES)
def test_white_gradients_match_restatement(name, n, M, num_data, ard, opts):
    import tsvgp_b200 as tb
    import tsvgp_b200.synth as synth
    cfg = synth.describe(name)
    X, Y, Z = synth.make_minibatch(cfg, n_rows=n, M=M)
    kernel, lik = synth.build_objects(cfg, orc)
    if ard:
        kernel.lengthscales = orc._param(cfg["ls"] * np.linspace(0.9, 1.2, cfg["D"]))
    ref = _trained(kernel, lik, X, Y, Z, num_data, lr=cfg["lr"])
    dev = tb.t_SVGP_white(kernel, lik, Z.copy(), num_data=num_data, lambda_1=ref.lambda_1, lambda_2=ref.lambda_2)
    for k, v in opts.items():
        dev.set_option(k, v)
    e_ref, g_ref = wgo.elbo_gradients(ref, (X, Y))
    e_before = dev.elbo((X, Y))
    e_dev, g_dev = dev.elbo_and_grad()
    errs = _errs(e_dev, g_dev, e_ref, g_ref)
    assert np.shape(g_dev["lengthscales"]) == np.shape(np.asarray(kernel.lengthscales))
    bad = {k: v for k, v in errs.items() if not v <= 1e-9}
    assert not bad, (bad, errs)
    # the call leaves the state untouched: elbo() is bitwise the same before and after, it equals the returned ELBO, and a
    # natgrad step afterwards still matches the oracle
    assert dev.elbo() == e_before
    assert abs(e_before - e_dev) <= 1e-12 * abs(e_dev)
    dev.natgrad_step((X, Y), lr=cfg["lr"])
    ref.natgrad_step((X, Y), lr=cfg["lr"])
    assert relerr(dev.lambda_1, ref.lambda_1) < 1e-9 and relerr(dev.lambda_2, ref.lambda_2) < 1e-9
    dev.close()


def _problem(lik_name, L, N=1500, M=32, D=3, seed=3, dyadic=False):
    """M = 32 keeps cond(Kuu + 1e-6 I) below 1e4, the range the synthetic configs are built for: Q = A^-1 - R^-1 is a difference of
    two inverses, and at M = 96 (cond 2.5e6 for the SE kernel here) device and restatement round it apart by 2e-8 in the Z gradient.
    dyadic: coordinates on a 2^-3 grid (with power-of-two lengthscales every r2 is exact in any order, so the device and the
    oracle see the same r2, exact zeros on the diagonal of Kuu included; Matern-1/2's k depends on sqrt(r2), and the rounding
    residue ~1e-16 |z|^2 that the expansion form leaves there generically would move k by ~1e-8, see tests/test_gpu_matern_family.py)"""
    rng = np.random.default_rng(seed)
    if dyadic:
        X, Z = (rng.integers(-16, 17, size=(n, D)) * 0.125 for n in (N, M))
    else:
        X, Z = rng.standard_normal((N, D)), rng.standard_normal((M, D))
    f = np.stack([np.sin(X.sum(1) + 0.7 * l) for l in range(L)], 1)
    if lik_name == "bernoulli":
        return X, (f + 0.3 * rng.standard_normal((N, L)) > 0).astype(float), Z, orc.Bernoulli()
    if lik_name == "student_t":
        return X, f + 0.3 * rng.standard_t(3.0, size=(N, L)), Z, orc.StudentT(scale=0.4, df=3.0)
    return X, f + 0.3 * rng.standard_normal((N, L)), Z, orc.Gaussian(variance=0.1)


@pytest.mark.parametrize("kind,lik_name,L", [("se", "bernoulli", 2), ("matern52", "student_t", 3), ("matern32", "gaussian", 1),
                                             ("matern12", "student_t", 2)])
def test_latents_likelihoods_and_kernels(kind, lik_name, L):
    import tsvgp_b200 as tb
    X, Y, Z, lik = _problem(lik_name, L, dyadic=kind == "matern12")
    cls = {"se": orc.SquaredExponential, "matern52": orc.Matern52, "matern32": mo.Matern32, "matern12": mo.Matern12}[kind]
    kernel = cls(variance=1.3, lengthscales=np.array([0.5, 1.0, 2.0]) if kind == "matern12" else np.array([0.9, 1.4, 1.1]))
    ref = _trained(kernel, lik, X, Y, Z, 10_000, L=L, lr=0.6)
    dev = tb.t_SVGP_white(kernel, lik, Z.copy(), num_data=10_000, lambda_1=ref.lambda_1, lambda_2=ref.lambda_2)
    e_ref, g_ref = wgo.elbo_gradients(ref, (X, Y))
    e_dev, g_dev = dev.elbo_and_grad((X, Y))
    errs = _errs(e_dev, g_dev, e_ref, g_ref)
    bad = {k: v for k, v in errs.items() if not v <= 1e-9}
    assert not bad, (bad, errs)
    assert abs(dev.elbo() - e_dev) <= 1e-12 * abs(e_dev)
    dev.close()


def test_gradients_for_inputs_far_from_the_origin():
    # coordinates taken relative to the centroid of the inducing inputs (tests/test_gpu_gradients.py holds the plain model to the
    # same bar): the kernel matrices themselves lose ~ eps (|x| / l)^2 = 1e-10 relative in r^2 through GPflow's expansion form
    import tsvgp_b200 as tb
    rng = np.random.default_rng(9)
    N, M, D = 1500, 32, 3
    ls = np.array([0.9, 1.3, 1.7])
    shift = 1.0e3 * ls
    X = rng.standard_normal((N, D)) + shift
    Z = X[:M].copy()
    Y = np.sin((X - shift).sum(1, keepdims=True)) + 0.2 * rng.standard_normal((N, 1))
    kernel, lik = orc.Matern52(variance=1.1, lengthscales=ls), orc.Gaussian(variance=0.1)
    ref = _trained(kernel, lik, X, Y, Z, None, steps=1, lr=0.6)
    dev = tb.t_SVGP_white(kernel, lik, Z.copy(), lambda_1=ref.lambda_1, lambda_2=ref.lambda_2)
    e_ref, g_ref = wgo.elbo_gradients(ref, (X, Y))
    e_dev, g_dev = dev.elbo_and_grad((X, Y))
    errs = _errs(e_dev, g_dev, e_ref, g_ref)
    bad = {k: v for k, v in errs.items() if not v <= 1e-6}
    assert not bad, (bad, errs)
    dev.close()


def test_mean_function_is_still_refused():
    import tsvgp_b200 as tb
    X, Y, Z, lik = _problem("gaussian", 1, N=300, M=16)
    dev = tb.t_SVGP_white(orc.SquaredExponential(variance=1.0, lengthscales=1.0), lik, Z.copy(),
                          mean_function=lambda x: np.ones((x.shape[0], 1)))
    with pytest.raises(NotImplementedError):
        dev.elbo_and_grad((X, Y))
    dev.close()


def test_variational_em_raises_both_elbos():
    import importlib.util
    spec = importlib.util.spec_from_file_location("vem_white_vs_dense", os.path.join(ROOT, "examples", "vem_white_vs_dense.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    out = mod.main(n_iters=15, verbose=False)
    for name, r in out.items():
        assert np.all(np.isfinite(r["trace"])), name
        assert r["elbo_end"] > r["elbo_start"] + 50.0, (name, r["elbo_start"], r["elbo_end"])
        assert r["trace"][-1] > r["trace"][0], name


# ---- two ranks ---------------------------------------------------------------------------------------------------------
def _rank_worker(rank, world, conn, X, Y, Z, l1, l2, q):
    import sys
    sys.path.insert(0, ROOT)
    try:
        import tsvgp_b200 as tb
        from tsvgp_b200 import standins as st
        m = tb.t_SVGP_white(st.Matern52(variance=1.3, lengthscales=np.array([0.9, 1.4, 1.1])), st.StudentT(scale=0.4, df=3.0),
                            Z.copy(), num_data=20_000, lambda_1=l1, lambda_2=l2, device=rank)
        if rank == 0:
            uid = tb.comm_unique_id()
            for c in conn:
                c.send(uid)
        else:
            uid = conn.recv()
        m.init_comm(world, rank, uid)
        lo, hi = tb.shard_rows(X.shape[0], world, rank)
        e, g = m.elbo_and_grad((X[lo:hi], Y[lo:hi]), global_minibatch_size=X.shape[0])
        q.put((rank, e, g["variance"], np.asarray(g["lengthscales"]), g["Z"], g["likelihood"]))
        m.close()
    except Exception as ex:   # reported to the parent, which fails the test
        q.put((rank, repr(ex), None, None, None, None))


def test_two_ranks_match_one():
    import multiprocessing as mp
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import tsvgp_b200 as tb
    from tsvgp_b200 import standins as st
    X, Y, Z, _ = _problem("student_t", 1, N=3000)
    one = tb.t_SVGP_white(st.Matern52(variance=1.3, lengthscales=np.array([0.9, 1.4, 1.1])), st.StudentT(scale=0.4, df=3.0),
                          Z.copy(), num_data=20_000)
    one.natgrad_step((X, Y), lr=0.5)
    l1, l2 = one.lambda_1, one.lambda_2
    e1, g1 = one.elbo_and_grad((X, Y))
    one.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    a, b = ctx.Pipe()
    procs = [ctx.Process(target=_rank_worker, args=(r, 2, [a] if r == 0 else b, X, Y, Z, l1, l2, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted((q.get(timeout=600) for _ in procs), key=lambda r: r[0])
    for p in procs:
        p.join(timeout=120)
    for rank, e, dv, dls, dZ, dl in res:
        assert dv is not None, e
        assert abs(e - e1) <= 1e-11 * abs(e1)
        assert abs(dv - g1["variance"]) <= 1e-11 * abs(g1["variance"])
        assert abs(dl - g1["likelihood"]) <= 1e-11 * abs(g1["likelihood"])
        assert relerr(dls, g1["lengthscales"]) <= 1e-11 and relerr(dZ, g1["Z"]) <= 1e-11
