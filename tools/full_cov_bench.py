"""Times predict_f(full_cov=True) and predict_f_samples(S = 128, full_cov=True) with device-resident outputs (DESIGN 13).

usage: python tools/full_cov_bench.py [--reps R] [--out FILE]

For each (M, N) of the cfg3 shape (Matern-5/2, D = 16, after one natgrad_step on N training rows) both C entry points are called
once to warm up, then R times, each between tsvgp_timer_start / tsvgp_timer_stop (CUDA events on the context's stream; each call
ends in a synchronisation and includes its own allocation of the N x N temporaries); the median call is reported.  The work is counted from the shapes
(Np = ceil(N/128) 128, Sp = ceil(S/128) 128):  V = T^T Kuf  M^2 Np ;  Sigma lower tiles  Np^2 M ;  Cholesky  Np^3 / 3 ;
chol times E  Np^2 Sp — and set against 37.1 TFLOP/s, the FP64 DMMA rate measured in DESIGN 4.  The card's name and power
limit are read in the same run (nvidia-smi --query-gpu, read-only).  Needs a GPU: there is nothing to fall back to.
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

import tsvgp_b200 as tb  # noqa: E402
import tsvgp_b200.synth as synth  # noqa: E402
from tsvgp_b200 import standins as st  # noqa: E402

SHAPES = [(2048, 4096), (2048, 16384), (4096, 16384)]
S = 128
PEAK_TFLOPS = 37.1


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = (f.strip() for f in out.split(","))
        return {"gpu": name, "power_limit": power}
    except Exception as e:   # the numbers below are still measured; say that the card could not be read
        return {"gpu": None, "power_limit": None, "card_error": str(e)}


def flops(M, N):
    Np, Sp = -(-N // 128) * 128, -(-S // 128) * 128
    v, sig, chol, tri = float(M) * M * Np, float(Np) * Np * M, float(Np) ** 3 / 3.0, float(Np) * Np * Sp
    return {"V": v, "Sigma": sig, "cholesky": chol, "chol_times_E": tri, "full_cov": v + sig, "samples": v + sig + chol + tri}


def run(M, N, reps):
    cfg = synth.describe("cfg3")
    X, Y, Z = synth.make_minibatch(cfg, n_rows=N, M=M)
    Xq, _, _ = synth.make_minibatch(cfg, n_rows=N, M=M, seed_offset=1)
    kernel, lik = synth.build_objects(cfg, st)
    m = tb.t_SVGP(kernel, lik, Z, num_data=cfg["N"])
    m.natgrad_step((X, Y), lr=cfg["lr"])
    lib, ctx, D = m._lib, m._ctx, X.shape[1]
    xq = m.device_array(Xq)
    mean_d, cov_d, smp_d = (lib.tsvgp_device_alloc(ctx, n * 8) for n in (N, N * N, S * N))
    calls = {
        "full_cov": lambda: m._check(lib.tsvgp_predict_f_full_cov(ctx, xq.ptr, N, D, None, mean_d, cov_d)),
        "samples": lambda: m._check(lib.tsvgp_predict_f_samples(ctx, xq.ptr, N, D, None, S, 1, None, smp_d)),
    }
    fl = flops(M, N)
    res = {"M": M, "N": N, "S": S, "reps": reps, "flops": fl}
    for name, f in calls.items():
        f()   # warm-up: module loads, workspace sizes
        times = []
        for _ in range(reps):
            m.timer_start()
            f()
            times.append(m.timer_stop())
        ms = float(np.median(times))   # the GPU is shared: the median call, with the spread beside it
        res[f"{name}_ms"] = ms
        res[f"{name}_ms_min_max"] = [min(times), max(times)]
        res[f"{name}_tflops"] = fl[name] / (ms * 1e-3) / 1e12
        res[f"{name}_fraction_of_peak"] = res[f"{name}_tflops"] / PEAK_TFLOPS
    for p in (mean_d, cov_d, smp_d):
        lib.tsvgp_device_free(ctx, p)
    xq.free()
    m.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=11)
    ap.add_argument("--out", default=None, help="also write the JSON lines here")
    a = ap.parse_args()
    lines = [json.dumps({"card": card(), "peak_tflops": PEAK_TFLOPS})]
    print(lines[0], flush=True)
    for M, N in SHAPES:
        lines.append(json.dumps(run(M, N, a.reps)))
        print(lines[-1], flush=True)
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
