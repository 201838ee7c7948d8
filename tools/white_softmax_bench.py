"""Times the whitened sibling with the Softmax likelihood (t_SVGP_white.natgrad_step and .elbo_and_grad, one pass over all latents)
next to the plain model (t_SVGP) on the same data (DESIGN 10, "Softmax").

usage: python tools/white_softmax_bench.py [--reps R] [--out FILE]     (the project keeps its runs under profiles/)

Two shapes with Softmax(10) and S = 100 Monte-Carlo points drawn by the library's generator, Matern-5/2 with ARD lengthscales:
docs/notebooks/mnist.py's minibatch (M = 100, D = 784, 200 rows; latency-bound) and a throughput shape (M = 2048, D = 16,
131 072 rows).  Both models start from the same hyperparameters and take one natgrad_step before timing, so that their sites are
trained.  The data are resident on the GPU (set_data once); after one warm-up call of each entry point, each is called R times
between tsvgp_timer_start / tsvgp_timer_stop (CUDA events on the context's stream; every call ends in a synchronisation) and the
median call is reported with the range.  The work of the streaming pass is counted from the shapes (Mp = ceil(M/128) 128,
W = ceil((2D+1)/128) 128, n = ceil(N/128) 128; a triangular product counts Mp^2 per point, the SYRK's lower half Mp^2):
    white elbo_grad  n (2 Mp D + (2 + 3 L) Mp^2 + 2 Mp W)   (Kuf; LA^-1 K and LA^-T (.); per latent LR^-1 K, LR^-T (.), the SYRK; F)
    plain elbo_grad  n (2 Mp D + 3 L Mp^2 + 2 Mp W)         (Kuf; per latent T^T Kuf, T V and the SYRK; F = E Xaug)
    white natgrad    n (2 Mp D + (1 + 2 L) Mp^2 + 40 S L)   (Kuf; LA^-1 K; per latent LR^-1 K and the SYRK; the Softmax kernel)
    plain natgrad    n (2 Mp D + 2 L Mp^2 + 40 S L)         (Kuf; per latent T^T Kuf and the SYRK; the Softmax kernel)
— the dense M x M epilogues are not counted — and set against 37.1 TFLOP/s, the FP64 DMMA rate measured in DESIGN 4.  The
card's name and power limit are read in the same run (nvidia-smi --query-gpu, read-only).  Needs a GPU.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

import tsvgp_b200 as tb  # noqa: E402
from tsvgp_b200 import standins as st  # noqa: E402

SHAPES = [("mnist_minibatch", 100, 784, 200), ("throughput", 2048, 16, 131_072)]   # name, M, D, N
L, S = 10, 100
SCALE = 10.0   # num_data / rows: the whitened update takes h unclipped, and at the notebook's 300 a step can leave Lambda_2 + Kuu indefinite
PEAK_TFLOPS = 37.1


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = (f.strip() for f in out.split(","))
        return {"gpu": name, "power_limit": power}
    except Exception as e:   # the numbers below are still measured; say that the card could not be read
        return {"gpu": None, "power_limit": None, "card_error": str(e)}


def rup(x, k=128):
    return -(-x // k) * k


def flops(M, D, N):
    Mp, W, n = rup(M), rup(2 * D + 1), rup(N)
    return {"white_elbo_grad": float(n) * (2 * Mp * D + (2 + 3 * L) * Mp * Mp + 2 * Mp * W),
            "plain_elbo_grad": float(n) * (2 * Mp * D + 3 * L * Mp * Mp + 2 * Mp * W),
            "white_natgrad": float(n) * (2 * Mp * D + (1 + 2 * L) * Mp * Mp + 40 * S * L),
            "plain_natgrad": float(n) * (2 * Mp * D + 2 * L * Mp * Mp + 40 * S * L)}


def data(N, M, D, seed=0):
    """class prototypes (sparse "images" in [0, 1]^D) plus Gaussian noise, as examples/vem_softmax.py"""
    rng = np.random.RandomState(seed)
    protos = (rng.rand(L, D) < 0.2).astype(float)
    y = rng.randint(L, size=N)
    X = protos[y] + 0.3 * rng.randn(N, D)
    return X, y.astype(float)[:, None], X[:M].copy()


def run(name, M, D, N, reps):
    X, Y, Z = data(N, M, D)
    ls = np.sqrt(D) * np.linspace(0.6, 0.8, D)
    scale = SCALE
    models = {}
    for key, cls in (("white", tb.t_SVGP_white), ("plain", tb.t_SVGP)):
        m = cls(st.Matern52(variance=1.0, lengthscales=ls), st.Softmax(L, num_monte_carlo_points=S), Z.copy(), num_latent_gps=L,
                num_data=int(SCALE * N))
        xd, yd = m.device_array(X), m.device_array(Y)
        m.set_data((xd, yd))
        m.natgrad_step(lr=0.1)
        # every timed call starts from these sites (put back outside the timed window): repeated steps with fresh draws could
        # otherwise walk the whitened sites into an indefinite Lambda_2 + Kuu
        sites = (m.lambda_1, m.lambda_2 if key == "white" else m.lambda_2_sqrt)
        models[key] = (m, xd, yd, sites)
    e, dv, dl = C.c_double(), C.c_double(), C.c_double()
    dls, dZ = np.empty(D), np.empty((M, D))

    def grad(m):
        return lambda: m._check(m._lib.tsvgp_elbo_grad(m._ctx, scale, C.byref(e), C.byref(dv), dls.ctypes.data, dZ.ctypes.data,
                                                       C.byref(dl)))

    def natgrad(m):
        return lambda: m._check(m._lib.tsvgp_natgrad_step(m._ctx, 0.1, 1e-9, scale, None))
    calls = {}
    for key in ("white", "plain"):
        m, sites = models[key][0], models[key][3]
        calls[f"{key}_natgrad"] = (m, sites, natgrad(m))
        calls[f"{key}_elbo_grad"] = (m, None, grad(m))   # (leaves the sites as they are)
    fl = flops(M, D, N)
    res = {"shape": name, "M": M, "N": N, "D": D, "L": L, "S": S, "reps": reps, "flops": fl}
    for key, (m, sites, f) in calls.items():
        reset = (lambda: m.assign_sites(*sites)) if sites is not None else (lambda: None)
        reset()
        f()   # warm-up: module loads, workspace sizes
        times = []
        for _ in range(reps):
            reset()
            m.sync()
            m.timer_start()
            f()
            times.append(m.timer_stop())
        ms = float(np.median(times))   # the GPU is shared: the median call, with the range beside it
        res[f"{key}_ms"] = ms
        res[f"{key}_ms_min_max"] = [min(times), max(times)]
        res[f"{key}_pass_tflops"] = fl[key] / (ms * 1e-3) / 1e12
        res[f"{key}_fraction_of_peak"] = res[f"{key}_pass_tflops"] / PEAK_TFLOPS
    res["white_over_plain_elbo_grad"] = res["white_elbo_grad_ms"] / res["plain_elbo_grad_ms"]
    res["white_over_plain_natgrad"] = res["white_natgrad_ms"] / res["plain_natgrad_ms"]
    for m, xd, yd, _ in models.values():
        xd.free()
        yd.free()
        m.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=11)
    ap.add_argument("--out", default=None, help="also write the JSON lines here")
    a = ap.parse_args()
    lines = [json.dumps({"card": card(), "peak_tflops": PEAK_TFLOPS})]
    print(lines[0], flush=True)
    for name, M, D, N in SHAPES:
        lines.append(json.dumps(run(name, M, D, N, a.reps)))
        print(lines[-1], flush=True)
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
