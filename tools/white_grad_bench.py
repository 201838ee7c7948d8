"""Times the whitened sibling's M-step gradient (t_SVGP_white.elbo_and_grad) next to the plain model's (t_SVGP.elbo_and_grad)
and the whitened natgrad_step on the same data (DESIGN 10, "M-step gradients").

usage: python tools/white_grad_bench.py [--reps R] [--out FILE]     (the project keeps its runs under profiles/)

Shapes: cfg3's inducing set and dimension (M = 2048, D = 16, Gaussian likelihood, one latent) over 131 072 resident rows, with the
SE and the Matern-5/2 kernel, and one latency-bound shape (M = 100, 2 000 rows).  Both models start from the same hyperparameters
and take one natgrad_step before timing, so that their sites are trained.  The data are resident on the GPU (set_data once); after
one warm-up call of each entry point, each is called R times between tsvgp_timer_start / tsvgp_timer_stop (CUDA events on the
context's stream; every call ends in a synchronisation) and the median call is reported with the range.  The work of the
streaming pass is counted from the shapes (Mp = ceil(M/128) 128, W = ceil((2D+1)/128) 128, n = ceil(N/128) 128; the triangular
products count Mp^2 per point, the SYRK's lower half Mp^2):
    white elbo_grad  n (2 Mp D + 2 Mp^2 + 3 L Mp^2 + 2 Mp W)   (Kuf; LA^-1 K and LA^-T (.); per latent LR^-1 K, LR^-T (.) and the SYRK; F)
    dense elbo_grad  n (2 Mp D + 3 L Mp^2 + 2 Mp W)           (Kuf; per latent T^T Kuf, T V and the SYRK; F = E Xaug)
    white natgrad    n (2 Mp D + Mp^2 + 2 L Mp^2)             (Kuf; LA^-1 K; per latent LR^-1 K and the SYRK)
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
import tsvgp_b200.synth as synth  # noqa: E402
from tsvgp_b200 import standins as st  # noqa: E402

SHAPES = [("cfg3_se", "SquaredExponential", 2048, 131_072), ("cfg3_matern52", "Matern52", 2048, 131_072),
          ("latency", "Matern52", 100, 2_000)]   # name, kernel, M, N
D, L, NUM_DATA = 16, 1, 10_000_000
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


def flops(M, N):
    Mp, W, n = rup(M), rup(2 * D + 1), rup(N)
    return {"white_elbo_grad": float(n) * (2 * Mp * D + 2 * Mp * Mp + 3 * L * Mp * Mp + 2 * Mp * W),
            "dense_elbo_grad": float(n) * (2 * Mp * D + 3 * L * Mp * Mp + 2 * Mp * W),
            "white_natgrad": float(n) * (2 * Mp * D + Mp * Mp + 2 * L * Mp * Mp)}


def run(name, kernel, M, N, reps):
    cfg = synth.describe("cfg3")
    X, Y, Z = synth.make_minibatch(cfg, n_rows=N, M=M)
    scale = NUM_DATA / N
    models = {}
    for key, cls in (("white", tb.t_SVGP_white), ("dense", tb.t_SVGP)):
        m = cls(getattr(st, kernel)(variance=1.0, lengthscales=cfg["ls"]), st.Gaussian(variance=0.1), Z.copy(), num_data=NUM_DATA)
        xd, yd = m.device_array(X), m.device_array(Y)
        m.set_data((xd, yd))
        m.natgrad_step(lr=0.5)
        models[key] = (m, xd, yd)
    e, dv, dl = C.c_double(), C.c_double(), C.c_double()
    dls, dZ = np.empty(1), np.empty((M, D))

    def grad(m):
        return lambda: m._check(m._lib.tsvgp_elbo_grad(m._ctx, scale, C.byref(e), C.byref(dv), dls.ctypes.data, dZ.ctypes.data,
                                                       C.byref(dl)))
    mw, md = models["white"][0], models["dense"][0]
    calls = {
        "white_elbo_grad": (mw, grad(mw)),
        "dense_elbo_grad": (md, grad(md)),
        "white_natgrad": (mw, lambda: mw._check(mw._lib.tsvgp_natgrad_step(mw._ctx, 0.1, 1e-9, scale, None))),
    }
    fl = flops(M, N)
    res = {"shape": name, "kernel": kernel, "M": M, "N": N, "D": D, "L": L, "reps": reps, "flops": fl}
    for key, (m, f) in calls.items():
        f()   # warm-up: module loads, workspace sizes
        times = []
        for _ in range(reps):
            m.timer_start()
            f()
            times.append(m.timer_stop())
        ms = float(np.median(times))   # the GPU is shared: the median call, with the range beside it
        res[f"{key}_ms"] = ms
        res[f"{key}_ms_min_max"] = [min(times), max(times)]
        res[f"{key}_pass_tflops"] = fl[key] / (ms * 1e-3) / 1e12
        res[f"{key}_fraction_of_peak"] = res[f"{key}_pass_tflops"] / PEAK_TFLOPS
    res["white_over_dense_elbo_grad"] = res["white_elbo_grad_ms"] / res["dense_elbo_grad_ms"]
    for m, xd, yd in models.values():
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
    for name, kernel, M, N in SHAPES:
        lines.append(json.dumps(run(name, kernel, M, N, a.reps)))
        print(lines[-1], flush=True)
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
