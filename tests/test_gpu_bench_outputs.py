"""
GPU: `bench.py --dump-outputs` writes what its timed path computed.  After --warmup W --steps K the dumped sites must be those of
W + K natgrad steps taken through the public API on the same seeded minibatches (and not those of one step fewer), within the
size cap, as a seeded sample of rows where an array does not fit.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def relerr(a, b):
    return float(np.max(np.abs(np.asarray(a) - np.asarray(b))) / max(np.max(np.abs(b)), 1e-300))


def _bench_dump(out, *args):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--no-cpu-baseline", "--no-e2e", "--no-grad",
           "--dump-outputs", str(out), *args]
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env)
    assert res.returncode == 0, res.stderr[-3000:]
    return {f[:-len(".npy")]: np.load(os.path.join(out, f)) for f in os.listdir(out)}, sum(os.path.getsize(os.path.join(out, f)) for f in os.listdir(out))


def _api_sites(config, M, Nb, n_steps):
    """bench.py's timed path through the public API: 4 minibatches in rotation, kernel matrices rebuilt before every step."""
    import tsvgp_b200 as tb
    import tsvgp_b200.synth as synth
    from tsvgp_b200 import standins as st
    cfg = synth.describe(config)
    kernel, lik = synth.build_objects(cfg, st)
    mbs = [synth.make_minibatch(cfg, n_rows=Nb, M=M, seed_offset=100 * i) for i in range(4)]
    m = tb.t_SVGP(kernel, lik, mbs[0][2], num_data=cfg["N"])
    for i in range(n_steps):
        m.set_option("invalidate", 1)
        m.set_data(mbs[i % 4][:2])
        m.natgrad_step(lr=cfg["lr"], global_minibatch_size=Nb)
    out = m.lambda_1, m.lambda_2_sqrt
    m.close()
    return out


@pytest.mark.parametrize("config,M,Nb", [("cfg2", 500, 10_000), ("cfg3", 3000, 4096)], ids=["whole", "row_sample"])
def test_dump_holds_the_sites_of_the_last_timed_step(tmp_path, config, M, Nb):
    warmup, steps = 2, 3
    got, nbytes = _bench_dump(tmp_path / "dump", "--config", config, "--M", str(M), "--minibatch", str(Nb),
                              "--warmup", str(warmup), "--steps", str(steps))
    assert sorted(got) == ["lambda_1", "lambda_2_sqrt"] and all(a.dtype == np.float64 for a in got.values())
    assert nbytes <= 64_000_000
    l1, l2s = _api_sites(config, M, Nb, warmup + steps)
    want = {"lambda_1": l1, "lambda_2_sqrt": l2s}
    if l2s.nbytes > 64_000_000:   # 3000 x 3000 doubles: written as the seeded row sample bench.dump_outputs documents
        k = got["lambda_2_sqrt"].shape[0]
        assert 0 < k < M
        want["lambda_2_sqrt"] = l2s.reshape(-1, M)[np.sort(np.random.default_rng(0).choice(M, k, replace=False))]
    for name, a in want.items():
        assert got[name].shape == a.shape, name
        assert relerr(got[name], a) <= 1e-9, name
    assert relerr(got["lambda_1"], _api_sites(config, M, Nb, warmup + steps - 1)[0]) > 1e-6   # --steps counts
