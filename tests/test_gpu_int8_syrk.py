"""
The Gaussian step's constant-weight SYRK as the exact int8 Gram product (DESIGN §2).  It is taken when the weight is constant,
the operand is the raw covariance slab (fused route) and the product does not split its contraction, i.e. from M = 1536 up;
every case here runs there.  The int8 product is exact up to the fixed-point grid of 2^-52 v, so the step matches the oracle
as the FP64 product did.  The data are 16-dimensional, like the benchmark's, so that cond(K9) stays in the fused route's range
(below 1e4) at this M.
"""
import numpy as np
import pytest

from oracle import tsvgp_oracle as orc
from tests import separate_oracle as so
from tests.test_gpu_gaussian_step import _elbo_and_sites_errors
from tests.test_gpu_parity import relerr

pytestmark = pytest.mark.gpu
M = 1536
# cond(K9) at M = 1536 on these points: 5.4e3, 1.3e3, 1.9e3
KERNELS = [orc.Matern52(variance=1.3, lengthscales=3.0), orc.SquaredExponential(variance=0.6, lengthscales=2.0),
           orc.Matern52(variance=0.8, lengthscales=2.5)]
# the smallest variance first: a kernel variance left over from an earlier latent would put this latent's entries off the grid
# (above 2 v), where the residue kernel maps them to 0.  cond(K9) at M = 1536: 1.3e3, 5.4e3, 1.9e3
KERNELS_SMALL_FIRST = [orc.SquaredExponential(variance=0.3, lengthscales=2.0), orc.Matern52(variance=1.3, lengthscales=3.0),
                       orc.Matern52(variance=0.8, lengthscales=2.5)]


def _case(L, N, M, D=16, seed=21, noise=0.1):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((N, D))
    F = np.stack([np.sin(X.sum(1) * (0.3 + 0.2 * l)) for l in range(L)], axis=1)
    return X, F + 0.3 * rng.standard_normal((N, L)), X[:M].copy(), orc.Gaussian(variance=noise)


def _pair(L=1, separate=False, streams=2, early=1, N=4600, chunk=1024, M=M, kernels=KERNELS):
    import tsvgp_b200 as tb
    X, Y, Z, lik = _case(L, N=N, M=M)
    if separate:
        kernel = so.SeparateIndependent(kernels[:L])   # Matern-5/2, SE, Matern-5/2 by default
        ref = so.OracleSeparateTSVGP(kernel, lik, orc.InducingPoints(Z.copy()), num_latent_gps=L, num_data=4 * N)
    else:
        kernel = KERNELS[0]
        ref = orc.OracleTSVGP(kernel, lik, orc.InducingPoints(Z.copy()), num_latent_gps=L, num_data=4 * N)
    dev = tb.t_SVGP(kernel, lik, Z.copy(), num_latent_gps=L, num_data=4 * N)
    for k, v in {"chunk": chunk, "streams": streams, "early_slabs": early}.items():
        dev.set_option(k, v)
    return dev, ref, (X, Y)


@pytest.mark.parametrize("streams", [1, 2])
@pytest.mark.parametrize("early", [0, 1])
def test_single_latent_matches_the_oracle(streams, early):
    dev, ref, data = _pair(streams=streams, early=early)
    _elbo_and_sites_errors(dev, ref, data, steps=2)
    assert dev.timings()["slabs"] >= 4 and dev.timings()["route"] == 1
    dev.close()


def _int8_products(fn):
    """Run fn() and count the int8 products (i8_gram_kernel launches) it ran, from the CUDA kernels the profiler records."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
    return sum(1 for e in prof.events() if "i8_gram_kernel" in e.name)


@pytest.mark.parametrize("separate,m,kernels", [(False, M, KERNELS), (True, M, KERNELS), (True, M, KERNELS_SMALL_FIRST),
                                                (False, 1600, KERNELS), (False, 2048, KERNELS)],
                         ids=["L3_shared", "L3_separate_se_matern52", "L3_separate_smallest_variance_first",
                              "L3_shared_M1600_odd_tile_count", "L3_shared_M2048"])
def test_three_latents_match_the_oracle(separate, m, kernels):
    # M = 1600 pads to Mp = 1664: 13 tile rows (the planes' padding row block) and padding rows in the slab; M = 2048 is cfg3's
    dev, ref, data = _pair(L=3, separate=separate, M=m, kernels=kernels)
    Z = data[0][:m]
    for k in (kernels if separate else kernels[:1]):   # the fused route, which takes the int8 product, needs cond(K9) < 1e4
        ev = np.linalg.eigvalsh(k.K(Z))
        assert ev[-1] / ev[0] < 1e4
    n_i8 = _int8_products(lambda: _elbo_and_sites_errors(dev, ref, data, steps=2))
    t = dev.timings()
    assert t["route"] == 1
    assert n_i8 == 2 * t["slabs"] * (3 if separate else 1)   # every SYRK of both steps: one per slab and latent (one if shared)
    dev.close()


def test_ragged_last_slab():
    dev, ref, data = _pair(N=4 * 1024 - 300, streams=2)
    _elbo_and_sites_errors(dev, ref, data, steps=2)
    dev.close()


def _launches_one_slab(N, chunk):
    import tsvgp_b200 as tb
    X, Y, Z, lik = _case(1, N=N, M=M, seed=4)
    dev = tb.t_SVGP(KERNELS[1], lik, Z, num_data=N)
    for k, v in {"chunk": chunk, "streams": 1, "early_slabs": 0}.items():
        dev.set_option(k, v)
    dev.natgrad_step((X, Y), lr=0.5)
    t = dev.timings()
    out = (t["slabs"], t["launches"], dev.lambda_1.copy(), dev.lambda_2_sqrt.copy())
    dev.close()
    return out


def test_slab_width_bound():
    # int32 accumulation is exact below 2^17 points per slab.  With the "chunk" option at 130 944 (the widest multiple of 128
    # below) the slab takes the int8 product (residues, products, reconstruction, then b += K g: 4 launches); at 131 072 the
    # FP64 SYRK with b += K g fused into it (1 launch).  Both give the same step.
    s_a, l_a, a1, a2 = _launches_one_slab(130_944, 130_944)
    s_b, l_b, b1, b2 = _launches_one_slab(130_944, 131_072)
    assert s_a == s_b == 1
    assert l_a - l_b == 3
    assert relerr(a1, b1) <= 1e-10 and relerr(a2, b2) <= 1e-10


def test_profile_syrk_slot_times_the_int8_product():
    import tsvgp_b200 as tb
    X, Y, Z, lik = _case(1, N=3000, M=M)
    dev = tb.t_SVGP(KERNELS[0], lik, Z, num_data=len(X))
    dev.set_option("chunk", 1024)
    dev.set_option("profile", 1)
    dev.natgrad_step((X, Y), lr=0.5)
    kp = dev.kernel_profile()
    dev.close()
    assert set(kp) == {"kuf", "variance_gemm", "point_stats", "whiten_gemm", "syrk", "kuf_g"}
    assert kp["syrk"][1] == 3 and kp["syrk"][0] > 0.0


def test_non_finite_data_skips_the_commit():
    import tsvgp_b200 as tb
    X, Y, Z, lik = _case(1, N=4600, M=M)
    dev = tb.t_SVGP(KERNELS[0], lik, Z.copy(), num_data=4 * len(X))
    dev.set_option("chunk", 1024)
    dev.natgrad_step((X, Y), lr=0.5)
    l1, l2 = dev.lambda_1.copy(), dev.lambda_2_sqrt.copy()
    Xbad = X.copy()
    Xbad[2777, 1] = np.inf
    for return_elbo in (False, True):
        with pytest.raises(tb.InvalidArgumentError) as ei:
            dev.natgrad_step((Xbad, Y), lr=0.5, return_elbo=return_elbo)
        assert ei.value.code == tb._lib.ERR_NONPOS_VAR
        np.testing.assert_array_equal(dev.lambda_1, l1)
        np.testing.assert_array_equal(dev.lambda_2_sqrt, l2)
    dev.close()
