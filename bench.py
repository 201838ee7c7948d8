#!/usr/bin/env python
"""
bench.py — natgrad_step datapoints/s of the B200 t-SVGP path (BASELINE.json metric), one JSON line on rank 0.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--config cfg3] [--impl ours|reference] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

`--dump-outputs DIR` writes the sites the last timed step left behind (what a caller of natgrad_step reads back: lambda_1 [M, L],
lambda_2_sqrt [L, M, M]) as DIR/<name>.npy in float64, at most 64 MB in all; an array that does not fit is written as a fixed,
seeded sample of its rows (see dump_outputs).  The inputs are seeded, so two builds run with the same arguments can be compared
array for array.

Workload: BASELINE.json's metric is quoted "at 1/2/4/8 B200", which is configs[2] (cfg3: N=10M, M=2048, D=16, Matern-5/2, minibatch 1M
"sharded over 1/2/4/8 B200"); configs[1] (cfg2) is pinned to one B200 and holds 0.15 ms of FP64 work per step, so it measures launch
latency rather than the path.  cfg3 fits one GPU and is the default; the default N=1 run also measures cfg2 (configs[1]) and reports it
under `other_configs`; `--config cfgK` selects any config as the main line.

A "step" is one `t_SVGP.natgrad_step` (posterior factors + streaming statistics pass + all-reduce + dense site update) over
one minibatch of the named config, sharded by rows over the N ranks (strong scaling: the minibatch is fixed).
For N > 1 the library option "split_chains" is switched on (rank 0 builds the posterior factors, rank 1 the Kuu + jitter I chain, both
broadcast) and the row shares are balanced from 5 untimed calibration steps (`balance_rows`; `--no-balance`: equal shares, both chains on
every rank); the shares and the calibration table are reported under `config`.
  value : minibatch rows / step time with the minibatch resident in HBM when the clock starts (4 distinct minibatches rotate)
  e2e   : the same through the public API with HOST (pinned) buffers: H2D of the rank's rows every step, and the pre-step
          ELBO and lambda_1 read back, inside the timed region
  roofline     : the DMMA weighted-SYRK kernel, timed live with CUDA events (single-stream profiled pass after the timed region)
  cpu_baseline : the NumPy/SciPy restatement of the reference (oracle/) on the host cores, bounded sample, extrapolated in N
`--impl reference` times that CPU restatement alone (TensorFlow/GPflow are not installable in this image).
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except (AttributeError, OSError):
        return os.cpu_count() or 1


# stdout carries exactly ONE line (the JSON).  NCCL prints its NCCL_DEBUG=VERSION/INFO lines to stdout from inside the library, at
# communicator creation and again at the first collectives; NCCL_DEBUG is left exactly as the launcher set it (the driver reads
# those lines), and instead file descriptor 1 is pointed at stderr for the whole life of the process while the JSON line is
# written to a private duplicate of the original stdout.
_JSON_FD = os.dup(1)
os.dup2(2, 1)


def emit(line):
    os.write(_JSON_FD, (json.dumps(line) + "\n").encode())


# torchrun exports OMP_NUM_THREADS=1 to every rank.  The reference arm is a CPU measurement on ALL host cores, so the BLAS pool is
# sized before NumPy loads OpenBLAS (and again with threadpoolctl inside run_reference, whatever the environment said).
if "reference" in " ".join(sys.argv[1:]):
    for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[_v] = str(host_cores())

import numpy as np  # noqa: E402

FP64_PEAK_TFLOPS = 37.1   # measured on this pool: tools/fp64_peak (DMMA m8n8k4 issue rate), profiles/fp64_peak_r01.txt
N_RESIDENT_MINIBATCHES = 4


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", default="cfg3")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--minibatch", type=int, default=None, help="override the config's minibatch rows (debugging)")
    ap.add_argument("--M", type=int, default=None, help="override the number of inducing points (debugging)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-grad", action="store_true", help="skip the (reported, untimed-in-the-metric) M-step gradient measurement")
    ap.add_argument("--keep-cache", action="store_true", help="do not invalidate the kernel-matrix factors every step")
    ap.add_argument("--opt", action="append", default=[], help="library option name=value (tsvgp_set_option), repeatable")
    ap.add_argument("--no-balance", action="store_true", help="several GPUs: equal row shares and both preparation chains on every rank")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="write the sites of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl ours: the reference arm times bounded samples, not the whole step")
    return args


DUMP_BYTES = 63_900_000   # array data of --dump-outputs: with the .npy headers the files stay under 64 MB


def dump_outputs(out_dir, arrays):
    """Write each array as out_dir/<name>.npy in float64, DUMP_BYTES in all.  Smallest first, each array may take an even share of
    what is left; one larger than its share is viewed as rows of its last axis, and the rows
    sorted(np.random.default_rng(0).choice(n_rows, k, replace=False)) are written, k as many as fit in the share."""
    os.makedirs(out_dir, exist_ok=True)
    items = sorted(arrays.items(), key=lambda kv: kv[1].nbytes)
    left = DUMP_BYTES
    for i, (name, a) in enumerate(items):
        a = np.ascontiguousarray(a, dtype=np.float64)
        share = left // (len(items) - i)
        if a.nbytes > share:
            rows = a.reshape(-1, a.shape[-1])
            k = share // rows[0].nbytes
            a = rows[np.sort(np.random.default_rng(0).choice(rows.shape[0], k, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)
        left -= a.nbytes


# ---- clocks -------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--id={gpu_index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            pass

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.p.terminate()
        try:
            out, _ = self.p.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
            out, _ = self.p.communicate()
        sm, smax, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for n, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        busy = [s for s, p in zip(sm, power) if p > 0.5 * max(power)] or sm
        return {"sm_mhz": float(np.median(busy)), "sm_max_mhz": float(max(smax)), "power_w_max": float(max(power)),
                "samples": len(sm), "reasons": sorted(reasons)}


# ---- CPU baseline (oracle = NumPy restatement of the reference) -------------------------------------------------------
def cpu_reference_step_time(cfg, M, n_rows, repeats=1):
    """Seconds of one reference-order natgrad_step (oracle) on `n_rows` rows with the full M, from non-trivial sites."""
    import tsvgp_b200.synth as synth
    from oracle import tsvgp_oracle as orc
    X, Y, Z = synth.make_minibatch(cfg, n_rows=n_rows, M=M)
    kernel, lik = synth.build_objects(cfg, orc)
    m = orc.OracleTSVGP(kernel, lik, orc.InducingPoints(Z), num_data=cfg["N"])
    best = float("inf")
    for _ in range(repeats):
        t0 = time.perf_counter()
        m.natgrad_step((X, Y), lr=cfg["lr"])
        best = min(best, time.perf_counter() - t0)
    return best


def cpu_threads():
    try:
        from threadpoolctl import threadpool_info
        return max([p.get("num_threads", 1) for p in threadpool_info()] + [1])
    except Exception:
        return host_cores()


class all_host_cores:
    """Context manager: every BLAS / OpenMP pool in the process set to all host cores, whatever OMP_NUM_THREADS said."""

    def __enter__(self):
        self.ctl = None
        try:
            from threadpoolctl import threadpool_limits
            self.ctl = threadpool_limits(limits=host_cores())
        except Exception:
            pass
        return self

    def __exit__(self, *a):
        if self.ctl is not None:
            self.ctl.restore_original_limits()


CPU_FLOP_BUDGET = 2.5e12   # one bounded sample: ~10-30 s of host work at a few hundred GFLOP/s
STREAM_OVER_DENSE = 4.0    # the streaming sample carries >= 4x the flops of the dense part, so that b N >> a in t(N) = a + b N
DENSE_ROWS = 64            # rows of the "dense part only" timing (8 * 64 * M^2 flops: < 0.5 % of 37 M^3 from M = 512 up)


def reference_flops(n, M):
    return 8.0 * n * M * M + 37.0 * M ** 3   # SURVEY 3.1: what the reference's operation order executes


def sample_plan(M, budget):
    """(Mc, n_s): inducing points and rows of one bounded sample.  The 37 M^3 dense part is timed on its own (a), the streaming
    part on n_s rows with 8 n_s Mc^2 >= STREAM_OVER_DENSE * 37 Mc^3.  When even that exceeds `budget` at the config's M, the
    sample is taken at a smaller Mc and scaled by (M/Mc)^3 (a) and (M/Mc)^2 (b) — stated in the sample description."""
    per_m3 = 37.0 * (1.0 + STREAM_OVER_DENSE)
    Mc = M
    if per_m3 * M ** 3 > budget:
        Mc = max(256, int((budget / per_m3) ** (1.0 / 3.0)) // 256 * 256)
    n_s = int(STREAM_OVER_DENSE * 37.0 * Mc / 8.0) // 256 * 256
    n_s = max(n_s, 2048)
    return Mc, n_s


class CpuFit:
    """t(N) = a + b N of the reference-order step on the host: a = dense M x M part timed alone (best of 2 at DENSE_ROWS rows),
    b from one streaming sample of n_s rows per call of `sample()`."""

    def __init__(self, cfg, M, Nb, budget):
        self.cfg, self.M, self.Nb = cfg, M, Nb
        self.full = reference_flops(Nb, M) <= budget
        if self.full:
            cpu_reference_step_time(cfg, M, min(Nb, DENSE_ROWS))           # warm the BLAS threads and the allocator
            self.a = 0.0
            return
        self.Mc, self.n_s = sample_plan(M, budget)
        self.n_s = min(self.n_s, Nb)
        cpu_reference_step_time(cfg, self.Mc, DENSE_ROWS)
        self.a = min(cpu_reference_step_time(cfg, self.Mc, DENSE_ROWS), cpu_reference_step_time(cfg, self.Mc, DENSE_ROWS))

    def sample(self):
        """-> seconds of one full (Nb-row, M) step, from one bounded sample."""
        if self.full:
            return cpu_reference_step_time(self.cfg, self.M, self.Nb)
        t = cpu_reference_step_time(self.cfg, self.Mc, self.n_s)
        b = max((t - self.a) / (self.n_s - DENSE_ROWS), 1e-9)
        self.b = b
        r = self.M / self.Mc
        return self.a * r ** 3 + b * r ** 2 * self.Nb

    def describe(self):
        if self.full:
            return f"the full {self.Nb}-row minibatch at M={self.M}"
        s = (f"t(N)=a+bN with a = the dense M x M part timed alone ({DENSE_ROWS} rows, best of 2: {self.a:.3f} s) and b from one "
             f"{self.n_s}-row sample at M={self.Mc} ({self.b * 1e6:.2f} us/row; the sample's streaming part is "
             f"{self.b * self.n_s / max(self.a, 1e-9):.1f}x its dense part)")
        if self.Mc != self.M:
            s += (f", scaled to M={self.M} by (M/{self.Mc})^3 for a and (M/{self.Mc})^2 for b because 37 M^3 dense flops at "
                  f"M={self.M} alone exceed the sample budget")
        return s + f", extrapolated to the {self.Nb}-row minibatch"


def cpu_baseline(cfg, M, Nb):
    with all_host_cores():
        fit = CpuFit(cfg, M, Nb, CPU_FLOP_BUDGET)
        t_full = min(fit.sample(), fit.sample()) if fit.full else fit.sample()
        cores = cpu_threads()
    return {"value": Nb / t_full, "unit": "datapoints/s", "cores": cores, "kind": "port",
            "sample": "oracle (NumPy/SciPy restatement of the reference, not TensorFlow) natgrad_step: " + fit.describe(),
            "host_cpus": host_cores(), "t_full_step_s": t_full}


# ---- the reference arm -----------------------------------------------------------------------------------------------
REFERENCE_TOTAL_FLOP_BUDGET = 6e13   # the whole --impl reference run: a few minutes of host time (the driver's 25-step run keeps cfg3 at its full M)


def run_reference(args, cfg, M, Nb):
    """The reference's CPU implementation of the path (oracle port: the reference itself needs GPflow/TensorFlow, which this
    image cannot install) on ALL host cores.  The dense part is timed once; each step is one bounded streaming sample."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n_steps = max(args.warmup + args.steps, 1)
    with all_host_cores():
        fit = CpuFit(cfg, M, Nb, min(CPU_FLOP_BUDGET, REFERENCE_TOTAL_FLOP_BUDGET / (n_steps + 2)))
        ts = []
        for i in range(n_steps):
            t = fit.sample()
            if i >= args.warmup:
                ts.append(t)
        cores = cpu_threads()
    t_full = float(np.mean(ts))
    value = Nb / t_full
    vals = [Nb / t for t in ts]
    line = {
        "impl": "reference", "metric": "natgrad_step datapoints/sec", "value": value, "unit": "datapoints/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_full * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(cfg, M, Nb, args.gpus),
        "cpu_baseline": {"value": value, "unit": "datapoints/s", "cores": cores, "kind": "port",
                         "sample": "each step = oracle (NumPy/SciPy restatement; GPflow/TensorFlow not installable here) natgrad_step: " + fit.describe(),
                         "host_cpus": host_cores(), "omp_num_threads_env_at_launch": os.environ.get("OMP_NUM_THREADS"),
                         "spread": {"min": min(vals), "max": max(vals), "rel_std": float(np.std(vals) / np.mean(vals))}},
        "e2e": {"value": value, "unit": "datapoints/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def workload_config(cfg, M, Nb, n_gpus):
    Mp = (M + 127) // 128 * 128
    return {"workload": f"{cfg['name']}: {cfg['lik']} likelihood, synthetic D={cfg['D']}, N={cfg['N']}, M={M}, {cfg['kernel']} kernel, "
                        f"minibatch {Nb} sharded by rows over {n_gpus} GPU(s), lr={cfg['lr']}",
            "M": M, "D": cfg["D"], "minibatch": Nb, "num_data": cfg["N"], "kernel": cfg["kernel"], "likelihood": cfg["lik"],
            "parallelism": f"rows/{n_gpus} + 1 allreduce, dense phase replicated",
            "l2": (f"inputs larger than L2: {N_RESIDENT_MINIBATCHES} distinct resident minibatches of {Nb * (cfg['D'] + 1) * 8 / 1e6:.0f} MB "
                   f"rotate (plus {16 * Mp * Mp * 8 / 1e6:.0f} MB of M x M state touched every step); the Kuf slab of one launch "
                   f"({Mp} x 16384 x 8 B = {Mp * 16384 * 8 / 1e6:.0f} MB per stream) is written and re-read through L2/HBM")
                  if N_RESIDENT_MINIBATCHES * Nb * (cfg['D'] + 1) * 8 > 126e6 else
                  "inputs smaller than the 126 MB L2 and not flushed: this config is launch-latency-bound, not bandwidth-bound"}


# ---- our arm -------------------------------------------------------------------------------------------------------------
class Ranks:
    """torch.distributed (gloo) plumbing: rendezvous, barrier, max over ranks, gather of small host vectors.  No GPU tensors."""

    def __init__(self):
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("gloo")
            self.dist = dist

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()

    def max(self, x):
        if self.dist is None:
            return x
        import torch
        t = torch.tensor([x], dtype=torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t[0])

    def bcast_bytes(self, payload, n):
        import torch
        t = torch.tensor(list(payload), dtype=torch.uint8) if self.rank == 0 else torch.zeros(n, dtype=torch.uint8)
        self.dist.broadcast(t, 0)
        return bytes(t.tolist())

    def gather_rows(self, vec):
        """[world, len(vec)] on every rank."""
        if self.dist is None:
            return np.asarray(vec)[None]
        import torch
        mine = torch.from_numpy(np.ascontiguousarray(vec, dtype=np.float64))
        out = [torch.zeros_like(mine) for _ in range(self.world)]
        self.dist.all_gather(out, mine)
        return np.stack([o.numpy() for o in out])

    def close(self):
        if self.dist is not None:
            self.dist.destroy_process_group()


def host_minibatches(tb, synth, rk, cfg, M, Nb, weights=None):
    """This rank's rows [lo, hi) of N_RESIDENT_MINIBATCHES synthetic minibatches (host) and the inducing inputs: the same seeds on
    every rank, so the minibatch does not depend on how it is sharded."""
    lo, hi = tb.shard_rows(Nb, rk.world, rk.rank, weights)
    mbs_host, Z = [], None
    for i in range(N_RESIDENT_MINIBATCHES):
        X, Y, Zi = synth.make_minibatch(cfg, n_rows=Nb, M=M, seed_offset=100 * i)
        Z = Zi if Z is None else Z
        mbs_host.append((np.ascontiguousarray(X[lo:hi]), np.ascontiguousarray(Y[lo:hi])))
        del X, Y
    return mbs_host, Z, hi - lo


def build_model(tb, st, synth, rk, cfg, M, Nb, opts=()):
    """The rank's model, its rows of N_RESIDENT_MINIBATCHES synthetic minibatches (host), the row count."""
    kernel, lik = synth.build_objects(cfg, st)
    mbs_host, Z, n_local = host_minibatches(tb, synth, rk, cfg, M, Nb)
    model = tb.t_SVGP(kernel, lik, Z, num_data=cfg["N"], device=rk.local_rank)
    for kv in opts:
        k, v = kv.split("=")
        model.set_option(k, float(v))
    if rk.world > 1:
        uid = rk.bcast_bytes(tb.comm_unique_id() if rk.rank == 0 else b"", 128)
        model.init_comm(rk.world, rk.rank, uid)
    return model, mbs_host, n_local


def balance_rows(tb, synth, rk, model, cfg, M, Nb, mbs_dev, invalidate, cal_steps=5):
    """Several ranks with option "split_chains": the ranks do different things in front of the pass (DESIGN 5), so equal row shares
    leave rank 0 the straggler.  A few untimed calibration steps with equal shares measure every rank's prepare
    and stream phases; tsvgp_b200.balance_weights turns them into row shares that equalise the finish times, the rank's rows are
    cut again from the SAME minibatches, and the sites are reset so that the steps that follow start where a run without
    calibration starts (the `check` object stays comparable across N).  Returns (shares, host minibatches, rows, table) or None when the
    library did not split the chains (M above dist_min_m, another route, ...)."""
    prep = stream = 0.0
    role = 0.0
    for i in range(cal_steps):
        if invalidate:
            model.set_option("invalidate", 1)
        model.set_data(mbs_dev[i % N_RESIDENT_MINIBATCHES])
        model.natgrad_step(lr=cfg["lr"], global_minibatch_size=Nb)
        tm = model.timings()
        if i >= cal_steps - 3:
            prep += tm["prepare"] / 3
            stream += tm["stream"] / 3
            role = tm["chain_role"]
    n_local = mbs_dev[0][0].shape[0]
    table = rk.gather_rows(np.array([prep, stream, float(n_local), role]))
    model.assign_sites(None, None)          # back to the default sites
    if not np.any(table[:, 3] != 0):
        return None
    w = tb.balance_weights(table[:, 0], table[:, 1], table[:, 2], table[:, 3])
    mbs_host, _, n_new = host_minibatches(tb, synth, rk, cfg, M, Nb, w)
    return [float(x) for x in w], mbs_host, n_new, [[round(float(v), 3) for v in row] for row in table]


def result_check(model, rk, mb, lr, Nb):
    """What the step COMPUTED, so that the lines of different N can be compared with each other: one more (untimed) step on a
    fixed minibatch after the warm-up + timed steps, returning the pre-step ELBO and norms of the new sites, plus the largest
    difference of lambda_1 between any rank and rank 0 (the dense phase is replicated: it must be 0)."""
    model.set_data(mb)
    elbo = model.natgrad_step(lr=lr, global_minibatch_size=Nb, return_elbo=True)
    l1 = model.lambda_1[:, 0]
    l2 = model.lambda_2[0]
    rows = rk.gather_rows(l1)
    return {"elbo_before_check_step": elbo, "lambda_1_l2norm": float(np.linalg.norm(l1)), "lambda_2_fro": float(np.linalg.norm(l2)),
            "lambda_1_rank_skew_max": float(np.max(np.abs(rows - rows[0:1]))), "lambda_1_head": [float(v) for v in l1[:4]],
            "what": "after warmup+steps natgrad steps over the rotating minibatches, one more step on minibatch 0: pre-step ELBO, "
                    "|lambda_1|_2, |lambda_2|_F of the resulting sites, max_r |lambda_1(rank r) - lambda_1(rank 0)|"}


def timed_steps(model, rk, mbs_dev, lr, Nb, warmup, steps, invalidate, sample_clocks=True):
    def step(i):
        if invalidate:
            model.set_option("invalidate", 1)   # kernel matrices and their factors are rebuilt every step, as the reference does
        model.set_data(mbs_dev[i % N_RESIDENT_MINIBATCHES])
        model.natgrad_step(lr=lr, global_minibatch_size=Nb)

    for i in range(warmup):
        step(i)
    model.sync(); rk.barrier()
    sampler = ClockSampler(rk.local_rank) if (rk.rank == 0 and sample_clocks) else None
    launches = 0
    phase = {"prepare": 0.0, "stream": 0.0, "allreduce": 0.0, "dense": 0.0}
    model.timer_start()
    t0 = time.perf_counter()
    for i in range(steps):
        step(warmup + i)
        tm = model.timings()
        launches += int(tm["launches"])
        for k in phase:
            phase[k] += tm[k] / steps
    ms_dev = model.timer_stop()
    wall = time.perf_counter() - t0
    rk.barrier()
    clocks = sampler.stop() if sampler else None
    ms_per_step = rk.max(ms_dev) / steps
    return {"ms_per_step": ms_per_step, "value": Nb / (ms_per_step * 1e-3), "launches": launches, "phase": phase, "clocks": clocks,
            "wall_ms_per_step": wall * 1e3 / steps, "step": step}


def main():
    args = parse()
    import tsvgp_b200.synth as synth
    cfg = synth.describe(args.config)
    M = args.M or cfg["M"]
    Nb = args.minibatch or cfg["Nb"]
    if args.impl == "reference":
        return run_reference(args, cfg, M, Nb)

    rk = Ranks()
    rank, world, local_rank = rk.rank, rk.world, rk.local_rank
    import tsvgp_b200 as tb
    from tsvgp_b200 import standins as st

    opts = list(args.opt)
    balance = world > 1 and not args.no_balance and not any(o.startswith("split_chains=") for o in opts)
    if balance:
        opts.append("split_chains=1")
    model, mbs_host, n_local = build_model(tb, st, synth, rk, cfg, M, Nb, opts)
    mbs_dev = [(model.device_array(X), model.device_array(Y)) for X, Y in mbs_host]
    invalidate = not args.keep_cache
    row_shares = cal_table = None
    if balance:
        got = balance_rows(tb, synth, rk, model, cfg, M, Nb, mbs_dev, invalidate)
        if got is not None:
            row_shares, mbs_host, n_local, cal_table = got
            del mbs_dev
            mbs_dev = [(model.device_array(X), model.device_array(Y)) for X, Y in mbs_host]

    # ---------- value: device-resident inputs ----------
    res = timed_steps(model, rk, mbs_dev, cfg["lr"], Nb, args.warmup, args.steps, invalidate)
    if args.dump_outputs and rank == 0:   # the dense phase is replicated: every rank holds the same sites
        dump_outputs(args.dump_outputs, {"lambda_1": model.lambda_1, "lambda_2_sqrt": model.lambda_2_sqrt})
    ms_per_step, value, launches, phase, clocks = res["ms_per_step"], res["value"], res["launches"], res["phase"], res["clocks"]
    step_resident = res["step"]
    route = model.timings()
    check = result_check(model, rk, mbs_dev[0], cfg["lr"], Nb)

    # ---------- e2e: host (pinned) buffers through the public API, H2D + result read-back every step ----------
    e2e = None
    if not args.no_e2e:
        pinned = []
        for X, Y in mbs_host:
            px, py = tb.pinned_empty(X.shape), tb.pinned_empty(Y.shape)
            px[...] = X; py[...] = Y
            pinned.append((px, py))

        # the public API with host buffers: the input pipeline (tsvgp_b200.stream_minibatches pattern) copies minibatch i + 1 from
        # pinned host memory while step i computes; every step's rows cross the PCIe bus inside the timed region, and the
        # pre-step ELBO and lambda_1 are read back every step
        def run_e2e(n_steps):
            model.stage_data(pinned[0])
            for i in range(n_steps):
                model.commit_staged()
                model.stage_data(pinned[(i + 1) % N_RESIDENT_MINIBATCHES])
                if invalidate:
                    model.set_option("invalidate", 1)
                e = model.natgrad_step(lr=cfg["lr"], global_minibatch_size=Nb, return_elbo=True)
                l1 = model.lambda_1
            model.commit_staged()   # drain the last prefetch
            return e, l1

        run_e2e(min(args.warmup, 2))
        model.sync(); rk.barrier()
        model.timer_start()
        run_e2e(args.steps)
        ms_e2e = rk.max(model.timer_stop()) / args.steps
        rk.barrier()
        e2e = {"value": Nb / (ms_e2e * 1e-3), "unit": "datapoints/s", "ms_per_step": ms_e2e,
               "h2d_bytes_per_step": int(n_local * (cfg["D"] + 1) * 8), "d2h_bytes_per_step": int(8 + 8 * M),
               "api": "stage_data(next pinned (X, Y)) / commit_staged + t_SVGP.natgrad_step(return_elbo=True) + .lambda_1, per rank on its rows"}

    # ---------- M-step gradient pass (next-row feature; reported, not part of the metric) ----------
    grad_ms = None
    if world == 1 and cfg["D"] <= 63 and not args.no_grad:
        model.set_data(mbs_dev[0])
        model.elbo_and_grad(global_minibatch_size=Nb)
        model.timer_start()
        for i in range(2):
            model.elbo_and_grad(global_minibatch_size=Nb)
        grad_ms = model.timer_stop() / 2

    # ---------- roofline: per-kernel CUDA-event timing, single stream ----------
    model.set_option("profile", 1)
    step_resident(0); step_resident(1)
    kp = model.kernel_profile()
    model.set_option("profile", 0)
    syrk_ms, syrk_n = kp["syrk"]
    var_ms, var_n = kp["variance_gemm"]
    rows_per_launch = n_local / max(syrk_n, 1)
    syrk_flops = float(M) * M * rows_per_launch   # algorithmic: lower triangle of k k^T, 2 flops per entry = M^2 per point
    syrk_t = syrk_ms * 1e-3 / max(syrk_n, 1)
    achieved = syrk_flops / syrk_t / 1e12
    traffic, traffic_source = None, None
    summ = os.path.join(ROOT, "profiles", "ncu_summary.json")
    if os.path.exists(summ):
        try:
            ent = json.load(open(summ)).get(args.config, {})
            traffic, traffic_source = ent.get("syrk_dram_bytes_per_launch"), ent.get("source")
            if traffic is not None and ent.get("points_per_launch"):   # the capture's slab width may differ from this run's
                traffic = traffic * rows_per_launch / ent["points_per_launch"]
                traffic_source = f"{traffic_source}; scaled from {ent['points_per_launch']} to {rows_per_launch:.0f} points per launch"
        except Exception:
            traffic = None
    roofline = {"bound": "tensor", "kernel": "gemm_kernel_mb<kc,kc,scale> (weighted SYRK B += K diag(h) K^T, DMMA m8n8k4)",
                "achieved": achieved, "peak": FP64_PEAK_TFLOPS, "unit": "TFLOP/s", "frac": achieved / FP64_PEAK_TFLOPS,
                "traffic": traffic,
                "traffic_source": f"dram__bytes_read.sum + dram__bytes_write.sum of one committed ncu --set full capture ({traffic_source}); "
                                  "not measurable inside a timed run",
                "peak_source": "measured FP64 DMMA issue rate on this pool (tools/fp64_peak -> profiles/fp64_peak_r01.txt); "
                               "MEASURED_PEAKS.json carries no FP64 figure and the profiling guide states no FP64 fallback",
                "flops_per_launch": syrk_flops, "avg_launch_ms": syrk_t * 1e3, "launches_profiled": syrk_n}
    var_t = var_ms * 1e-3 / max(var_n, 1)
    q = lik_q(cfg)
    f_pt = synth.flops_per_point(M, cfg["D"], q)
    step_flops = Nb * f_pt + synth.dense_flops(M)
    kernels = {k: {"ms_total": v[0], "launches": v[1]} for k, v in kp.items()}
    kernels["variance_gemm"]["achieved_tflops"] = float(M) * M * rows_per_launch / var_t / 1e12 if var_t > 0 else None
    extra = {
        "step_fp64_frac": step_flops / (ms_per_step * 1e-3) / (world * FP64_PEAK_TFLOPS * 1e12),
        "step_algorithmic_flops": step_flops, "flops_per_point": f_pt,
        "hbm_stream_frac": Nb * 8 * (cfg["D"] + 1) / max(phase["stream"] * 1e-3, 1e-9) / (world * 6554.2e9),
        "phase_ms": phase, "kernels": kernels, "route": int(route["route"]), "cond_est": route["cond_est"],
        "wall_ms_per_step": res["wall_ms_per_step"],
        "elbo_and_grad_ms": grad_ms,
    }

    line = {
        "metric": "natgrad_step datapoints/sec", "value": value, "unit": "datapoints/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": workload_config(cfg, M, Nb, world), "clocks": clocks, "e2e": e2e,
        "gpu_launches": launches, "roofline": roofline, "check": check, "detail": extra,
    }
    if row_shares is not None:
        line["config"]["row_shares"] = row_shares
        line["config"]["calibration"] = cal_table
        line["config"]["parallelism"] += ("; option split_chains: rank 0 builds the posterior factors, rank 1 the Kuu + jitter I chain underneath "
                                          "early slabs, the others only early slabs, results by ncclBroadcast; row shares from "
                                          "tsvgp_b200.balance_weights after 5 untimed calibration steps with equal shares (sites reset afterwards); "
                                          "calibration = per rank [prepare ms, stream ms, rows, role]")
    model.close()
    del mbs_dev, model
    default_run = args.config == "cfg3" and args.minibatch is None and args.M is None and not args.no_e2e
    if default_run:
        # the north-star target config (M = 4096, Student-t GH-20, 2M-row minibatch) in the same driver record, at every N
        line["other_configs"] = {"cfg5": north_star_config(tb, st, synth, rk, invalidate)}
        if rank == 0 and world == 1:
            line["other_configs"]["cfg2"] = quick_config(tb, st, synth, "cfg2", local_rank)
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(cfg, M, Nb)
    if rank == 0:
        emit(line)
    rk.close()


def north_star_config(tb, st, synth, rk, invalidate, steps=4, warmup=3):
    """BASELINE.json's target config (cfg5: M=4096, D=32, SE, Student-t GH-20, 2M-row minibatch of N=50M) on the same ranks:
    device-resident natgrad_step datapoints/s, fraction of the FP64 roofline, clocks during its own timed region, result check."""
    cfg = synth.describe("cfg5")
    M, Nb = cfg["M"], cfg["Nb"]
    model, mbs_host, n_local = build_model(tb, st, synth, rk, cfg, M, Nb)
    mbs_dev = [(model.device_array(X), model.device_array(Y)) for X, Y in mbs_host]
    del mbs_host
    res = timed_steps(model, rk, mbs_dev, cfg["lr"], Nb, warmup, steps, invalidate)
    check = result_check(model, rk, mbs_dev[0], cfg["lr"], Nb)
    step_flops = Nb * synth.flops_per_point(M, cfg["D"], lik_q(cfg)) + synth.dense_flops(M)
    out = {"value": res["value"], "unit": "datapoints/s", "ms_per_step": res["ms_per_step"], "n_gpus": rk.world, "steps": steps, "warmup": warmup,
           "workload": workload_config(cfg, M, Nb, rk.world)["workload"],
           "step_fp64_frac": step_flops / (res["ms_per_step"] * 1e-3) / (rk.world * FP64_PEAK_TFLOPS * 1e12),
           "north_star_target": ">= 60 % of the FP64 tensor roofline at M=4096 on 8 x B200 (>= 5.7 M datapoints/s at 40 TFLOP/s nominal per GPU)",
           "phase_ms": res["phase"], "gpu_launches": res["launches"], "clocks": res["clocks"], "check": check}
    model.close()
    return out


def quick_config(tb, st, synth, name, device):
    """configs[1] measured in the same run: natgrad_step datapoints/s, device-resident and end to end (pinned host buffers)."""
    cfg = synth.describe(name)
    M, Nb = cfg["M"], cfg["Nb"]
    kernel, lik = synth.build_objects(cfg, st)
    X, Y, Z = synth.make_minibatch(cfg)
    m = tb.t_SVGP(kernel, lik, Z, num_data=cfg["N"], device=device)
    xd, yd = m.device_array(X), m.device_array(Y)
    px, py = tb.pinned_empty(X.shape), tb.pinned_empty(Y.shape)
    px[...] = X; py[...] = Y

    def resident():
        m.set_option("invalidate", 1)
        m.set_data((xd, yd))
        m.natgrad_step(lr=cfg["lr"])

    def e2e():
        m.set_option("invalidate", 1)
        e = m.natgrad_step((px, py), lr=cfg["lr"], return_elbo=True)
        return e, m.lambda_1

    out = {}
    for key, fn in (("value", resident), ("e2e", e2e)):
        for _ in range(5):
            fn()
        m.sync()
        m.timer_start()
        for _ in range(30):
            fn()
        ms = m.timer_stop() / 30
        out[key] = Nb / (ms * 1e-3)
        out[key + "_ms_per_step"] = ms
    q = lik_q(cfg)
    out.update(unit="datapoints/s", workload=f"{name}: {cfg['lik']} GH-20, D={cfg['D']}, M={M}, minibatch {Nb} (BASELINE configs[1])",
               step_fp64_frac=(Nb * synth.flops_per_point(M, cfg["D"], q) + synth.dense_flops(M)) / (out["value_ms_per_step"] * 1e-3) / (FP64_PEAK_TFLOPS * 1e12))
    m.close()
    return out


def lik_q(cfg):
    return 0 if cfg["lik"] == "Gaussian" else 20


if __name__ == "__main__":
    main()
