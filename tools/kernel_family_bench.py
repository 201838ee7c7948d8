"""Times the four covariance functions against each other at cfg3's shape (M = 2048, D = 16) on three paths (DESIGN 12).

usage: python tools/kernel_family_bench.py [--rows N] [--grad-rows N] [--rounds R] [--steps K] [--warmup W] [--out FILE]

Paths, each with SquaredExponential, Matern12, Matern32 and Matern52 (variance 1, lengthscale 3, cfg3's):
  gaussian   natgrad_step, Gaussian likelihood, N resident rows (default 1 048 576): the int8 Gram product, no variance product
  student_t  natgrad_step, StudentT(scale 0.3, df 3), the same rows: the per-point variance product and 20-point quadrature
  grad       elbo_and_grad, Gaussian, 131 072 rows: the slab with its dk/dr2 companion
All three force the fused route (option "route" = 1), so every kernel runs the same products and only the covariance epilogue
differs: at lengthscale 3 on cfg3's inputs the automatic route would take the fused route for the Matern kernels but not for SE
(cond(K9) 1.1e3 Matern12, 3.8e3 Matern32, 8.4e3 Matern52, 1.6e5 SE).  Over R rounds the kernels alternate within each path; each
run takes W warm-up steps, then K timed steps between tsvgp_timer_start / tsvgp_timer_stop (CUDA events on the context's stream,
ending in a synchronisation).  The median and range over all timed steps of all rounds are reported.  A separate pass then runs
one Gaussian step per kernel with option "profile" = 1 and reads the Kuf slab class time (kernel_profile()["kuf"]).  The card's
name and power limit are read in the same run (nvidia-smi --query-gpu, read-only).  Needs a GPU: there is nothing to fall back to.
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
from tools.full_cov_bench import card  # noqa: E402

M, D, LS = 2048, 16, 3.0
KERNELS = {"se": st.SquaredExponential, "matern12": st.Matern12, "matern32": st.Matern32, "matern52": st.Matern52}


def _model(kind, lik, X, Y, profile=False):
    m = tb.t_SVGP(KERNELS[kind](1.0, LS), lik, _model.Z, num_data=10 * X.shape[0])
    m.set_option("route", 1)
    if profile:
        m.set_option("profile", 1)
    m.set_data((X, Y))
    return m


def time_path(path, kind, data, steps, warmup):
    X, Y = data
    lik = st.StudentT(scale=0.3, df=3.0) if path == "student_t" else st.Gaussian(variance=0.1)
    m = _model(kind, lik, X, Y)
    call = (lambda: m.elbo_and_grad()) if path == "grad" else (lambda: m.natgrad_step(lr=0.5))
    for _ in range(warmup):
        call()
    times = []
    for _ in range(steps):
        m.timer_start()
        call()
        times.append(m.timer_stop())
    route = m.timings()["route"]
    m.close()
    return times, route


def kuf_profile(kind, data):
    m = _model(kind, st.Gaussian(variance=0.1), *data, profile=True)
    m.natgrad_step(lr=0.5)          # warm-up: module loads, workspace
    m.natgrad_step(lr=0.5)
    kp = m.kernel_profile()
    slabs = m.timings()["slabs"]
    m.close()
    return {"kuf_ms": kp["kuf"][0], "kuf_launches": kp["kuf"][1], "slabs": slabs, "syrk_ms": kp["syrk"][0]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=1_048_576)
    ap.add_argument("--grad-rows", type=int, default=131_072)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON lines here")
    a = ap.parse_args()
    if a.steps < 10 or a.warmup < 3:
        ap.error("at least 10 timed steps after 3 warm-up steps")
    X, Y, Z = synth.make_minibatch(synth.describe("cfg3"), n_rows=a.rows, M=M)
    _model.Z = Z
    data = {"gaussian": (X, Y), "student_t": (X, Y), "grad": (X[:a.grad_rows].copy(), Y[:a.grad_rows].copy())}
    lines = [json.dumps({"card": card(), "M": M, "D": D, "lengthscale": LS, "rows": a.rows, "grad_rows": a.grad_rows,
                         "rounds": a.rounds, "steps": a.steps, "warmup": a.warmup, "route": 1})]
    print(lines[0], flush=True)
    for path in ("gaussian", "student_t", "grad"):
        acc = {k: [] for k in KERNELS}
        routes = {}
        for r in range(a.rounds):
            for kind in KERNELS:
                t, routes[kind] = time_path(path, kind, data[path], a.steps, a.warmup)
                acc[kind].append(t)
        for kind in KERNELS:
            all_t = [x for t in acc[kind] for x in t]
            rec = {"path": path, "kernel": kind, "route": routes[kind], "ms_median": float(np.median(all_t)),
                   "ms_min_max": [min(all_t), max(all_t)], "round_medians": [float(np.median(t)) for t in acc[kind]]}
            lines.append(json.dumps(rec))
            print(lines[-1], flush=True)
    for kind in KERNELS:
        lines.append(json.dumps({"path": "gaussian_profile", "kernel": kind, **kuf_profile(kind, data["gaussian"])}))
        print(lines[-1], flush=True)
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
