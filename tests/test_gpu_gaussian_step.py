"""
The Gaussian natgrad_step without the per-point variance product.  For the Gaussian likelihood g_n and h_n do not read v_n, so the
pass skips |T^T k_n|^2 and the ELBO's variance term comes from the weighted statistics instead:
    sum_n |T^T k_n|^2 = tr(P^T B P) / c,   B = c R^-1 (sum_n k_n k_n^T) R^-T,  P = R^T T,  R = I / C9 / K9  (fused / whitened / exact).
The CPU test pins that identity; the GPU tests check the ELBO and the sites against the oracle, the device's own elbo(), the
launches the step no longer makes, and the guard on non-finite data.
"""
import multiprocessing as mp
import os
import sys

import numpy as np
import pytest
import scipy.linalg as sla

from oracle import tsvgp_oracle as orc
from tests import algo_model as am
from tests import separate_oracle as so
from tests.test_gpu_multi import _n_gpus
from tests.test_gpu_parity import relerr

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

KERNELS = [orc.Matern52(variance=1.3, lengthscales=[0.8, 1.2, 0.9, 1.0]), orc.SquaredExponential(variance=0.6, lengthscales=0.7),
           orc.Matern52(variance=0.8, lengthscales=1.0)]


def _case(L, N=1700, M=160, D=4, seed=21, noise=0.1):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((N, D))
    F = np.stack([np.sin(X.sum(1) * (0.5 + 0.3 * l)) for l in range(L)], axis=1)
    return X, F + 0.3 * rng.standard_normal((N, L)), X[:M].copy(), orc.Gaussian(variance=noise)


# ---- CPU: the identity the step relies on ---------------------------------------------------------------------------------
@pytest.mark.parametrize("route", [1, 2, 3])
@pytest.mark.parametrize("s2", [0.1, 1e8])
def test_variance_sum_from_the_statistics_cpu(route, s2):
    rng = np.random.default_rng(5)
    N, M, D, jitter = 700, 60, 3, 1e-9
    X = rng.standard_normal((N, D))
    kern = orc.Matern52(variance=1.1, lengthscales=1.3)
    Z = X[:M].copy()
    K, Kuf, kdiag = kern.K(Z), kern.K(Z, X), 1.1
    L2 = np.tril(0.3 * rng.standard_normal((M, M)), -1) - np.diag(1.0 + rng.uniform(size=M))
    p = am.prepare(K, np.zeros((M, 1)), L2)
    _, var = am.marginals(Kuf, kdiag, p["T"], p["alpha"])
    c = min(-0.5 / s2, -1e-8)
    K9 = K + jitter * np.eye(M)
    C9 = sla.cholesky(K9, lower=True)
    if route == 1:
        S, P = Kuf, p["T"]
    elif route == 2:
        S, P = sla.solve_triangular(C9, Kuf, lower=True), C9.T @ p["T"]
    else:
        S, P = sla.cho_solve((C9, True), Kuf), K9 @ p["T"]
    B = c * (S @ S.T)
    got = N * kdiag - np.trace(P.T @ B @ P) / c
    assert abs(got - var.sum()) <= 1e-12 * abs(var.sum())


# ---- GPU --------------------------------------------------------------------------------------------------------------------
def _pair(L, separate, route, streams, chunk=512, noise=0.1):
    import tsvgp_b200 as tb
    X, Y, Z, lik = _case(L, noise=noise)
    if separate:
        kernel = so.SeparateIndependent(KERNELS[:L])
        ref = so.OracleSeparateTSVGP(kernel, lik, orc.InducingPoints(Z.copy()), num_latent_gps=L, num_data=4 * len(X))
    else:
        kernel = KERNELS[0]
        ref = orc.OracleTSVGP(kernel, lik, orc.InducingPoints(Z.copy()), num_latent_gps=L, num_data=4 * len(X))
    dev = tb.t_SVGP(kernel, lik, Z.copy(), num_latent_gps=L, num_data=4 * len(X))
    for k, v in {"chunk": chunk, "route": route, "streams": streams}.items():
        dev.set_option(k, v)
    return dev, ref, (X, Y)


def _elbo_and_sites_errors(dev, ref, data, steps=3, lr=0.6):
    errs = {}
    for s in range(steps):
        e_own = dev.elbo(data)           # the device's per-point variances, on the state the step starts from
        e_ref = ref.elbo(data)
        e_dev = dev.natgrad_step(data, lr=lr, return_elbo=True)
        ref.natgrad_step(data, lr=lr)
        errs[f"elbo_vs_oracle_{s}"] = (abs(e_dev - e_ref) / abs(e_ref), 1e-9)
        errs[f"elbo_vs_device_elbo_{s}"] = (abs(e_dev - e_own) / abs(e_own), 1e-11)
        errs[f"lambda_1_{s}"] = (relerr(dev.lambda_1, ref.lambda_1), 1e-9)
        errs[f"lambda_2_{s}"] = (relerr(dev.lambda_2, ref.lambda_2), 1e-9)
    bad = {k: v for k, v in errs.items() if not (v[0] <= v[1])}
    assert not bad, f"above tolerance: {bad}"


@pytest.mark.gpu
@pytest.mark.parametrize("streams", [1, 2])
@pytest.mark.parametrize("L,separate", [(1, False), (3, False), (3, True)], ids=["L1", "L3_shared", "L3_separate"])
@pytest.mark.parametrize("route", [1, 2, 3])
def test_elbo_and_sites_match_the_oracle(route, L, separate, streams):
    dev, ref, data = _pair(L, separate, route, streams)
    _elbo_and_sites_errors(dev, ref, data)
    assert dev.timings()["route"] == route
    assert dev.timings()["slabs"] >= 3
    dev.close()


@pytest.mark.gpu
def test_clipped_weight():
    # s2 = 1e8: h = min(-1/(2 s2), -1e-8) = -1e-8 is clipped, the SYRK's weight is not -1/(2 s2)
    dev, ref, data = _pair(1, False, 1, 2, noise=1e8)
    _elbo_and_sites_errors(dev, ref, data, steps=2)
    dev.close()


def _profile(lik):
    import tsvgp_b200 as tb
    X, Y, Z, _ = _case(1, N=3000)
    if lik == "bernoulli":
        lik_obj, Y = orc.Bernoulli(), (Y > 0).astype(float)
    else:
        lik_obj = orc.Gaussian(variance=0.1)
    dev = tb.t_SVGP(KERNELS[0], lik_obj, Z, num_data=len(X))
    dev.set_option("chunk", 1024)
    dev.set_option("profile", 1)
    dev.natgrad_step((X, Y), lr=0.5)
    kp = dev.kernel_profile()
    dev.close()
    return kp


@pytest.mark.gpu
def test_gaussian_step_launches_no_variance_product():
    kp = _profile("gaussian")
    assert set(kp) == {"kuf", "variance_gemm", "point_stats", "whiten_gemm", "syrk", "kuf_g"}
    assert kp["variance_gemm"] == (0.0, 0) and kp["syrk"][1] == 3
    assert _profile("bernoulli")["variance_gemm"][1] == 3


def _launches_per_slab(L, M=256, chunk=1024):
    # two slab counts, everything else equal: the difference of the step's launches is per-slab work only
    import tsvgp_b200 as tb
    counts = []
    for n_slabs in (3, 5):
        X, Y, Z, lik = _case(L, N=n_slabs * chunk - 100, M=M)
        dev = tb.t_SVGP(KERNELS[0], lik, Z, num_latent_gps=L, num_data=len(X))
        for k, v in {"chunk": chunk, "streams": 1, "early_slabs": 0, "route": 1}.items():
            dev.set_option(k, v)
        dev.natgrad_step((X, Y), lr=0.5)
        assert dev.timings()["slabs"] == n_slabs
        counts.append(dev.timings()["launches"])
        dev.close()
    return (counts[1] - counts[0]) / 2


@pytest.mark.gpu
def test_shared_kernel_latents_share_one_syrk():
    # At M = 256 the SYRK splits its contraction over the idle SMs: a split-K product, its reduction and b += K g as a mat-vec
    # (3 launches).  A latent that reuses latent 0's B adds only its partial means, its point statistics and its b (3 launches),
    # beyond the one partial-mean pass that the single latent folds into the Kuf kernel; one SYRK per latent would add 5.
    p1, p3 = _launches_per_slab(1), _launches_per_slab(3)
    assert p3 - p1 == 1 + 2 * 3


@pytest.mark.gpu
def test_non_finite_data_skips_the_commit():
    import tsvgp_b200 as tb
    X, Y, Z, lik = _case(1)
    dev = tb.t_SVGP(KERNELS[0], lik, Z.copy(), num_data=4 * len(X))
    dev.set_option("chunk", 512)
    dev.natgrad_step((X, Y), lr=0.5)
    l1, l2 = dev.lambda_1.copy(), dev.lambda_2_sqrt.copy()
    Xbad = X.copy()
    Xbad[777, 2] = np.nan
    for return_elbo in (False, True):
        with pytest.raises(tb.InvalidArgumentError) as ei:
            dev.natgrad_step((Xbad, Y), lr=0.5, return_elbo=return_elbo)
        assert ei.value.code == tb._lib.ERR_NONPOS_VAR
        np.testing.assert_array_equal(dev.lambda_1, l1)
        np.testing.assert_array_equal(dev.lambda_2_sqrt, l2)
    # the context is still usable: the same steps as a fresh oracle from the same sites
    ref = orc.OracleTSVGP(KERNELS[0], lik, orc.InducingPoints(Z.copy()), num_data=4 * len(X))
    ref.lambda_1, ref.lambda_2_sqrt = l1.copy(), l2.copy()
    e_ref = ref.elbo((X, Y))
    e_dev = dev.natgrad_step((X, Y), lr=0.5, return_elbo=True)
    ref.natgrad_step((X, Y), lr=0.5)
    assert abs(e_dev - e_ref) <= 1e-9 * abs(e_ref)
    assert relerr(dev.lambda_1, ref.lambda_1) <= 1e-9 and relerr(dev.lambda_2, ref.lambda_2) <= 1e-9
    dev.close()


def _two_rank_case():
    X, Y, Z, lik = _case(1, N=6000, M=2048, D=6, seed=8)
    return X, Y, Z, lik, orc.Matern52(variance=1.0, lengthscales=2.0)


def _rank(rank, world, conn, out):
    sys.path.insert(0, ROOT)
    import tsvgp_b200 as tb
    X, Y, Z, lik, kernel = _two_rank_case()
    m = tb.t_SVGP(kernel, lik, Z, num_data=10 * len(X), device=rank)
    m.set_option("route", 1)
    if rank == 0:
        uid = tb.comm_unique_id()
        for c in conn:
            c.send(uid)
    else:
        uid = conn.recv()
    m.init_comm(world, rank, uid)
    lo, hi = tb.shard_rows(X.shape[0], world, rank)
    elbos = [m.natgrad_step((X[lo:hi], Y[lo:hi]), lr=0.5, global_minibatch_size=len(X), return_elbo=True) for _ in range(2)]
    out.put((rank, elbos, m.lambda_1))
    m.close()


@pytest.mark.gpu
@pytest.mark.skipif(_n_gpus() < 2, reason="needs >= 2 GPUs")
def test_two_rank_sharded_update_elbo():
    # M = 2048 (16 tile rows): the statistics are reduce-scattered by tile rows and the update formed on each rank's rows
    import tsvgp_b200 as tb
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    a, b = ctx.Pipe()
    procs = [ctx.Process(target=_rank, args=(0, 2, [a], out)), ctx.Process(target=_rank, args=(1, 2, b, out))]
    for p in procs:
        p.start()
    res = sorted([out.get(timeout=600) for _ in procs], key=lambda r: r[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    X, Y, Z, lik, kernel = _two_rank_case()
    single = tb.t_SVGP(kernel, lik, Z, num_data=10 * len(X))
    single.set_option("route", 1)
    e = [single.natgrad_step((X, Y), lr=0.5, return_elbo=True) for _ in range(2)]
    for rank, elbos, l1 in res:
        assert relerr(elbos, e) < 1e-10
        assert relerr(l1, single.lambda_1) < 1e-10
    single.close()
