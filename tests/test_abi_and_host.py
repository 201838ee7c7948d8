"""
CPU-side checks of the boundary: libtsvgp.so loads, exports every entry point include/tsvgp.h declares, the ctypes table
matches the header, the library refuses to compute without a GPU (no CPU fallback), the DLPack view validates tensors, and
the host logic (object duck-typing, sharding, synthetic configs) behaves.
"""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "tsvgp.h")


def declared_functions():
    src = open(HEADER).read()
    return sorted(set(re.findall(r"TSVGP_API\s+[\w\s\*]+?\b(tsvgp_\w+)\s*\(", src)))


def have_gpu():
    try:
        return subprocess.run(["nvidia-smi", "-L"], capture_output=True, timeout=20).returncode == 0
    except Exception:
        return False


def test_library_exports_every_declared_symbol():
    import tsvgp_b200
    lib = tsvgp_b200.load()
    names = declared_functions()
    assert len(names) >= 30
    for n in names:
        assert hasattr(lib, n), f"{n} is declared in include/tsvgp.h but not exported by libtsvgp.so"
    assert sorted(tsvgp_b200.exported_names()) == names, "ctypes signature table and header disagree"
    assert lib.tsvgp_abi_version() == 1


def test_no_cpu_fallback():
    import tsvgp_b200
    from oracle import tsvgp_oracle as orc
    if have_gpu():
        pytest.skip("a GPU is present")
    with pytest.raises(tsvgp_b200.TsvgpError) as ei:
        tsvgp_b200.t_SVGP(orc.SquaredExponential(), orc.Gaussian(), np.zeros((3, 1)))
    assert ei.value.code == -2 and "no CPU fallback" in str(ei.value)


def test_product_never_imports_the_oracle_or_torch():
    pkg = os.path.join(ROOT, "t-svgp_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg, fn)).read()
            assert "oracle" not in src.replace("the oracle module", ""), fn
            assert not re.search(r"^\s*(import|from)\s+torch", src, re.M), fn


def test_dlpack_view_validates():
    import tsvgp_b200
    from tsvgp_b200 import _lib
    lib = tsvgp_b200.load()
    a = np.arange(12, dtype=np.float64).reshape(3, 4)
    t = _lib.as_tensor(a)
    assert t.ptr == a.ctypes.data and t.shape == (3, 4) and not t.on_device
    # non-contiguous / wrong dtype host arrays are copied into float64 row-major by the host side
    t2 = _lib.as_tensor(a.T)
    assert t2.shape == (4, 3)
    t3 = _lib.as_tensor(a.astype(np.float32))
    assert t3.shape == (3, 4)
    # the C side rejects a float32 DLPack tensor and a strided one
    for bad in (a.astype(np.float32), a[:, ::2]):
        cap = bad.__dlpack__()
        ptr = _lib._PyCapsule_GetPointer(cap, b"dltensor")
        assert lib.tsvgp_dlpack_view(ptr, C.byref(_lib.View())) == _lib.ERR_INVALID
    ro = a.copy(); ro.flags.writeable = False
    assert _lib.as_tensor(ro).ptr == ro.ctypes.data


def test_duck_typing_of_gpflow_objects():
    from tsvgp_b200 import model, standins as st, _lib
    kind, var, ls = model._kernel_spec(st.Matern52(variance=1.5, lengthscales=[[1.0, 2.0]]))   # [1, D] as uci_regression.py:42-44
    assert (kind, var, ls.tolist()) == (_lib.KERNEL_MATERN52, 1.5, [1.0, 2.0])
    assert model._kernel_spec(st.RBF(2.0, 0.5))[0] == _lib.KERNEL_SE

    class Param(float):   # gpflow.Parameter answers .numpy()
        def numpy(self):
            return float(self)

    k = st.SquaredExponential()
    k.variance, k.lengthscales = Param(2.25), Param(2.0)
    assert model._kernel_spec(k)[1:] == (2.25, np.array([2.0]))
    assert model._likelihood_spec(st.Gaussian(0.3)) == (_lib.LIK_GAUSSIAN, 0.3, 0.0, 0)
    assert model._likelihood_spec(st.Bernoulli()) == (_lib.LIK_BERNOULLI_PROBIT, 0.0, 0.0, 20)
    assert model._likelihood_spec(st.StudentT(0.4, 3.0)) == (_lib.LIK_STUDENT_T, 0.4, 3.0, 20)

    class Poisson:
        pass

    with pytest.raises(NotImplementedError):
        model._likelihood_spec(Poisson())


def test_shard_rows_partitions():
    from tsvgp_b200 import shard_rows
    for n in (1, 7, 8, 1000, 1_000_001):
        for w in (1, 2, 3, 8):
            spans = [shard_rows(n, w, r) for r in range(w)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(spans[i][1] == spans[i + 1][0] for i in range(w - 1))
            sizes = [hi - lo for lo, hi in spans]
            assert max(sizes) - min(sizes) <= 1


def test_synthetic_configs_have_the_survey_shapes():
    import tsvgp_b200.synth as synth
    for name, (M, D) in {"cfg1": (50, 1), "cfg2": (500, 8), "cfg3": (2048, 16), "cfg4": (8192, 8), "cfg5": (4096, 32)}.items():
        cfg = synth.describe(name)
        assert (cfg["M"], cfg["D"]) == (M, D)
        X, Y, Z = synth.make_minibatch(cfg, n_rows=300, M=40)
        assert X.shape == (300, D) and Y.shape == (300, 1) and Z.shape == (40, D)
    assert synth.flops_per_point(2048, 16) == 2 * 2048 ** 2 + 2048 * 38 + 4 * 2048


def test_header_is_plain_c_and_the_c_example_links():
    # the boundary is a C ABI: the header must compile as C, and a C client must link against the library
    import shutil
    import tempfile
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("no gcc")
    import tsvgp_b200
    tsvgp_b200.load()
    with tempfile.TemporaryDirectory() as td:
        exe = os.path.join(td, "c_api_example")
        cmd = [gcc, "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "examples", "c_api_example.c"),
               "-o", exe, "-L", os.path.join(ROOT, "t-svgp_b200"), "-ltsvgp", "-Wl,-rpath," + os.path.join(ROOT, "t-svgp_b200"), "-lm"]
        res = subprocess.run(cmd, capture_output=True, text=True, timeout=120)
        assert res.returncode == 0, res.stderr
        if not have_gpu():   # without a device the client must fail loudly in tsvgp_create (no CPU fallback)
            run = subprocess.run([exe], capture_output=True, text=True, timeout=60)
            assert run.returncode != 0 and "no CUDA device" in run.stderr


def _header_option_comment():
    # the comment block of include/tsvgp.h that documents tsvgp_set_option: (the options, its Environment paragraph)
    header = open(HEADER).read()
    start = header.index("/* options:")
    block = header[start:header.index("*/", start)]
    return block[:block.index("Environment")], block[block.index("Environment"):]


def test_every_library_option_is_documented_in_the_header():
    # tsvgp_set_option(name, value): the names the library accepts (csrc/tsvgp.cu) and the names the header's option comment
    # documents, in both directions
    src = open(os.path.join(ROOT, "t-svgp_b200", "csrc", "tsvgp.cu")).read()
    body = src[src.index("int tsvgp_set_option("):src.index("int tsvgp_set_kernel(")]
    accepted = set(re.findall(r'strcmp\(name, "([a-z_0-9]+)"\)', body))
    documented = set(re.findall(r'"([a-z_0-9]+)"', _header_option_comment()[0]))
    assert accepted, "no options found in tsvgp_set_option"
    assert documented, "no options found in the header's option comment"
    internal = {"profile"}   # measurement switch behind tsvgp_get_kernel_profile, described there
    assert accepted - internal <= documented, sorted(accepted - internal - documented)
    assert documented <= accepted, sorted(documented - accepted)


def test_every_environment_variable_is_documented_in_the_header():
    # every getenv("TSVGP_...") of the library is named in the Environment paragraph of the header's option comment, and
    # every name there is read
    csrc = os.path.join(ROOT, "t-svgp_b200", "csrc")
    read = set()
    for fn in os.listdir(csrc):
        if fn.endswith(".cu"):
            read |= set(re.findall(r'getenv\("(TSVGP_[A-Z0-9_]+)"\)', open(os.path.join(csrc, fn)).read()))
    documented = set(re.findall(r"\b(TSVGP_[A-Z0-9_]+)", _header_option_comment()[1]))
    assert read, "no getenv(\"TSVGP_...\") found in t-svgp_b200/csrc"
    assert read == documented, (sorted(read - documented), sorted(documented - read))


def test_weighted_shards_and_balance_weights():
    # host side of option "split_chains" (DESIGN 5): weighted contiguous shards on 128-row boundaries, and the shares that equalise
    # the ranks' finish times under the model  busy_r = offset_r + rows_r / rate
    from tsvgp_b200 import balance_weights, shard_rows
    N, W = 1_000_000, 8
    equal = [shard_rows(N, W, r) for r in range(W)]
    assert equal == [shard_rows(N, W, r, None) for r in range(W)]
    rows = np.array([hi - lo for lo, hi in equal], dtype=float)
    roles = np.array([1.0, 2.0] + [3.0] * (W - 2))      # rank 0 builds the posterior factors, rank 1 the K9 chain, the rest receive
    rate = N / W / 32.9                                    # rows per ms

    def phases(rows):                                      # rank 0: chain 2.5 ms in front; the others do part of the pass while they wait
        done = np.array([0.0, 1.2] + [2.2] * (W - 2))
        return np.where(np.arange(W) == 0, 2.5, 2.7), rows / rate - done

    prep, stream = phases(rows)
    assert np.ptp(prep + stream) > 1.9
    w = balance_weights(prep, stream, rows, roles)
    assert abs(w.sum() - 1.0) < 1e-12 and w[0] < w[1] < w[2] and np.allclose(w[2:], w[2])
    spans = [shard_rows(N, W, r, w) for r in range(W)]
    assert spans[0][0] == 0 and spans[-1][1] == N
    assert all(spans[r][1] == spans[r + 1][0] for r in range(W - 1)) and all(s[0] % 128 == 0 for s in spans)
    prep2, stream2 = phases(np.array([hi - lo for lo, hi in spans], dtype=float))
    assert np.ptp(prep2 + stream2) < 0.05                  # finish times equalised (128-row granularity)
    assert np.allclose(balance_weights(prep, stream, rows, np.zeros(W)), 1 / W)   # no split: equal shares
    with pytest.raises(ValueError):
        shard_rows(N, W, 0, [1.0] * (W - 1))
    assert [shard_rows(10, 3, r, [1, 1, 1]) for r in range(3)][-1][1] == 10


def test_bench_reference_arm_contract():
    # bench.py --impl reference (the driver's reference arm): ONE JSON line on stdout with the contract's keys, the oracle timed on
    # the host cores; under torchrun only rank 0 runs and prints, the other ranks exit 0 without work
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--config", "cfg1", "--steps", "2", "--warmup", "1"]
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=300, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
              "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["steps"] == 2 and d["warmup"] == 1 and d["higher_is_better"] is True
    assert d["metric"] == "natgrad_step datapoints/sec" and d["unit"] == "datapoints/s" and d["dtype"] == "f64" and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] == d["value"] and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]
    # a non-zero rank of a torchrun launch: no output, exit 0, no rendezvous attempted
    env1 = dict(env, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1", MASTER_ADDR="127.0.0.1", MASTER_PORT="29999")
    out1 = subprocess.run(cmd + ["--gpus", "2"], capture_output=True, text=True, timeout=120, env=env1)
    assert out1.returncode == 0 and out1.stdout.strip() == ""
