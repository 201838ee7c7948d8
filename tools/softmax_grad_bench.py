"""Times the Softmax M-step gradient (tsvgp_elbo_grad, one pass over all latents) next to natgrad_step on the same data
(DESIGN 9, "Coupled likelihood").

usage: python tools/softmax_grad_bench.py [--reps R] [--out FILE]

Two shapes of docs/notebooks/mnist.py's model (Matern-5/2 with 784 ARD lengthscales, Softmax(10) with S = 100 Monte-Carlo
points drawn by the library's generator): the notebook's minibatch (M = 100, 200 rows; latency-bound) and a throughput shape
(M = 2048, 131 072 rows).  The data are resident on the GPU (set_data once); after one natgrad_step and one warm-up call of each
entry point, each is called R times between tsvgp_timer_start / tsvgp_timer_stop (CUDA events on the context's stream; every
call ends in a synchronisation) and the median call is reported with the range.  The work of the streaming pass is counted from
the shapes (Mp = ceil(M/128) 128, W = ceil((2D+1)/128) 128, n = ceil(N/128) 128):
    elbo_grad  n (2 Mp D + 3 L Mp^2 + 2 Mp W)    (Kuf; per latent T^T Kuf, T V and the SYRK, each Mp^2 per point; F = E Xaug)
    natgrad    n (2 Mp D + 2 L Mp^2)             (Kuf; per latent T^T Kuf and the SYRK)
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

SHAPES = [("mnist_minibatch", 100, 200), ("throughput", 2048, 131_072)]   # name, M, N
D, L, S, NUM_DATA = 784, 10, 100, 60_000
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
    return {"elbo_grad": float(n) * (2 * Mp * D + 3 * L * Mp * Mp + 2 * Mp * W), "natgrad": float(n) * (2 * Mp * D + 2 * L * Mp * Mp)}


def data(N, M, seed=0):
    rng = np.random.RandomState(seed)
    protos = (rng.rand(L, D) < 0.2).astype(float)
    y = rng.randint(L, size=N)
    X = protos[y] + 0.3 * rng.randn(N, D)
    return X, y.astype(float)[:, None], X[:M].copy()


def run(name, M, N, reps):
    X, Y, Z = data(N, M)
    m = tb.t_SVGP(st.Matern52(variance=1.0, lengthscales=np.full(D, 20.0)), st.Softmax(L, num_monte_carlo_points=S), Z,
                  num_latent_gps=L, num_data=NUM_DATA)
    xd, yd = m.device_array(X), m.device_array(Y)
    m.set_data((xd, yd))
    m.natgrad_step(lr=0.5)
    lib, ctx, scale = m._lib, m._ctx, NUM_DATA / N
    e, dv, dl = C.c_double(), C.c_double(), C.c_double()
    dls, dZ = np.empty(D), np.empty((M, D))
    calls = {
        "elbo_grad": lambda: m._check(lib.tsvgp_elbo_grad(ctx, scale, C.byref(e), C.byref(dv), dls.ctypes.data, dZ.ctypes.data,
                                                          C.byref(dl))),
        "natgrad": lambda: m._check(lib.tsvgp_natgrad_step(ctx, 0.1, 1e-9, scale, None)),
    }
    fl = flops(M, N)
    res = {"shape": name, "M": M, "N": N, "D": D, "L": L, "S": S, "reps": reps, "flops": fl}
    for key, f in calls.items():
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
    res["elbo_grad_over_natgrad"] = res["elbo_grad_ms"] / res["natgrad_ms"]
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
    for name, M, N in SHAPES:
        lines.append(json.dumps(run(name, M, N, a.reps)))
        print(lines[-1], flush=True)
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
