"""bench.py contract checks that run without a GPU: the reference arm (CPU oracle) on a tiny configuration must print exactly one
JSON line with the keys the driver reads, and the precision constants of the header and of the ctypes binding must agree."""
import json
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "1", "--warmup", "0",
           "--n-rows", "4096", "--d-in", "16", "--num-rf", "2", "--block", "64", "--classes", "5", "--cpu-rows", "256"]
    env = dict(os.environ, OMP_NUM_THREADS="1", RANK="0")   # what torchrun exports
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 1 and d["higher_is_better"] is True
    for key in ("metric", "value", "unit", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data", "config",
                "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["unit"] == "samples/s" and d["value"] > 0
    assert d["e2e"] == {"value": d["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and "sample" in cb and cb["value"] == d["value"]
    assert cb["per_row_seconds"] > 0 and cb["solve_seconds"] > 0 and cb["sample_rows"] <= 256
    assert cb["blas_threads"] == str(os.cpu_count())       # the CPU arm uses every host core even under torchrun (OMP_NUM_THREADS=1)
    assert d["config"]["workload"].startswith("C3 ")


_DUMP_CHECK = r"""
import os, sys
import numpy as np
sys.path.insert(0, sys.argv[1])
import bench

class Model:   # the host arrays of a fitted BlockLinearMapper: ragged last block
    def __init__(self, rng):
        self.xs = [np.asfortranarray(rng.standard_normal((r, 30))) for r in (400, 400, 150)]
        self.feature_means = [rng.standard_normal(w.shape[0]) for w in self.xs]
        self.b_opt = rng.standard_normal(30)

m = Model(np.random.default_rng(0))
W = np.concatenate(m.xs, 0)
bench.DUMP_BYTES = 10 ** 9
full = bench.dump_model(m, os.path.join(sys.argv[2], "full"))
assert full["W_sample"] == [950, 30], full
assert np.array_equal(np.load(os.path.join(sys.argv[2], "full", "W_sample.npy")), W)
bench.DUMP_BYTES = 100_000
for run in ("a", "b"):
    got = bench.dump_model(m, os.path.join(sys.argv[2], run))
d = {run: {f: np.load(os.path.join(sys.argv[2], run, f)) for f in os.listdir(os.path.join(sys.argv[2], run))} for run in "ab"}
assert sorted(d["a"]) == ["W_sample.npy", "W_sample_rows.npy", "feature_means.npy", "intercept.npy"]
assert sum(os.path.getsize(os.path.join(sys.argv[2], "a", f)) for f in d["a"]) <= 100_000
assert all(a.dtype == np.float64 for a in d["a"].values())
assert all(np.array_equal(d["a"][f], d["b"][f]) for f in d["a"])
rows = d["a"]["W_sample_rows.npy"].astype(np.int64)
assert 0 < len(rows) < 950 and np.all(np.diff(rows) > 0)
assert np.array_equal(d["a"]["W_sample.npy"], W[rows])
assert np.array_equal(d["a"]["feature_means.npy"], np.concatenate(m.feature_means))
assert np.array_equal(d["a"]["intercept.npy"], m.b_opt)
"""


def test_dump_outputs_writes_a_fixed_sample_of_the_model_within_budget(tmp_path):
    out = subprocess.run([sys.executable, "-c", _DUMP_CHECK, ROOT, str(tmp_path)], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]


def test_dump_outputs_and_steps_are_validated():
    for extra in (["--impl", "reference", "--dump-outputs", "x"], ["--steps", "0"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True, timeout=300)
        assert out.returncode == 2 and not out.stdout, (extra, out.stderr[-500:])


def test_precision_constants_agree_between_header_and_binding():
    from keystone_b200 import _capi
    hdr = open(os.path.join(ROOT, "include", "keystone_b200.h")).read()
    consts = dict(re.findall(r"#define\s+(KS_PRECISION_[A-Z0-9]+)\s+\(?(-?\d+)\)?", hdr))
    assert set(consts) == {"KS_PRECISION_DEFAULT", "KS_PRECISION_TF32", "KS_PRECISION_F16", "KS_PRECISION_F16X2"}
    for name, val in consts.items():
        assert getattr(_capi, name) == int(val), name
