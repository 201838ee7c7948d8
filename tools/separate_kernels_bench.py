"""Times natgrad_step at the cfg3 shape with two latent GPs: one shared kernel against one kernel per latent (DESIGN 14).

usage: python tools/separate_kernels_bench.py [--rows N] [--steps K] [--warmup W] [--out FILE]

Models, all with M = 2048 inducing inputs, D = 16 and a resident minibatch of N rows (default 1 048 576, cfg3's):
  (a) shared      one Matern52 kernel for both latents, Gaussian likelihood, Y [N, 2]
  (b) separate    SeparateIndependent of two Matern52 kernels with different lengthscales, Gaussian, Y [N, 2]
  (c) hetero      SeparateIndependent([SE, SE]), HeteroskedasticTFPConditional(Normal, Exp), Y [N, 1]
Each model takes W warm-up steps, then K timed steps, each between tsvgp_timer_start / tsvgp_timer_stop (CUDA events on the
context's stream, ending in a synchronisation); the median step is reported with the spread beside it.  The work is counted
from the shapes (SURVEY 8d): per point L (2 M^2 + 4 M) + k M (2 D + 6), with the Kuf term counted once (k = 1) for the shared
kernel and once per latent (k = L) for separate kernels, plus L 8 M^3 for the dense phase; it is set against 37.1 TFLOP/s, the
FP64 DMMA rate measured in DESIGN 4.  The card's name and power limit are read in the same run (nvidia-smi --query-gpu,
read-only).  Needs a GPU: there is nothing to fall back to.
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

import tsvgp_b200 as tb  # noqa: E402
import tsvgp_b200.synth as synth  # noqa: E402
from tsvgp_b200 import standins as st  # noqa: E402
from tools.full_cov_bench import PEAK_TFLOPS, card  # noqa: E402

M, D, L = 2048, 16, 2


def models():
    gauss = st.Gaussian(variance=0.1)
    return [
        ("shared", st.Matern52(1.0, 3.0), gauss),
        ("separate", st.SeparateIndependent([st.Matern52(1.0, 3.0), st.Matern52(0.8, 2.5)]), gauss),
        ("hetero", st.SeparateIndependent([st.SquaredExponential(1.0, 2.0), st.SquaredExponential(0.5, 2.0)]),
         st.HeteroskedasticTFPConditional(st.Normal, st.Exp())),
    ]


def work(n, separate):
    k = L if separate else 1
    return float(n) * (L * (2.0 * M * M + 4.0 * M) + k * M * (2.0 * D + 6.0)) + L * 8.0 * M ** 3


def run(name, kernel, lik, X, Y2, Z, steps, warmup):
    m = tb.t_SVGP(kernel, lik, Z, num_latent_gps=L, num_data=10 * X.shape[0])
    Y = Y2[:, :1].copy() if name == "hetero" else Y2
    m.set_data((X, Y))
    for _ in range(warmup):
        m.natgrad_step(lr=0.5)
    times = []
    for _ in range(steps):
        m.timer_start()
        m.natgrad_step(lr=0.5)
        times.append(m.timer_stop())
    route = m.timings()["route"]
    m.close()
    ms = float(np.median(times))
    w = work(X.shape[0], name != "shared")
    return {"model": name, "M": M, "D": D, "L": L, "rows": X.shape[0], "steps": steps, "warmup": warmup, "route": route,
            "ms_per_step": ms, "ms_min_max": [min(times), max(times)], "points_per_s": X.shape[0] / (ms * 1e-3),
            "work_flop": w, "tflops": w / (ms * 1e-3) / 1e12, "fraction_of_peak": w / (ms * 1e-3) / 1e12 / PEAK_TFLOPS}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=1_048_576)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON lines here")
    a = ap.parse_args()
    if a.steps < 10 or a.warmup < 3:
        ap.error("at least 10 timed steps after 3 warm-up steps")
    X, Y, Z = synth.make_minibatch(synth.describe("cfg3"), n_rows=a.rows, M=M)
    Y2 = np.ascontiguousarray(np.concatenate([Y, np.cos(X[:, :1])], axis=1))   # a second output column for the L = 2 Gaussian models
    lines = [json.dumps({"card": card(), "peak_tflops": PEAK_TFLOPS})]
    print(lines[0], flush=True)
    for name, kernel, lik in models():
        lines.append(json.dumps(run(name, kernel, lik, X, Y2, Z, a.steps, a.warmup)))
        print(lines[-1], flush=True)
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
