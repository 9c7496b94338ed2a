"""bench.py's reference arm is the one leg of the bench contract that runs without a GPU: it times the oracle
port of CafRustFFTThreadpool (caf_rust/src/caf/mod.rs:391-461) on the host cores.  These tests hold its JSON line
to the contract (one line on stdout, `impl: reference`, the b200 arm's metric / unit / config keys, an `e2e`
with no copies, a `cpu_baseline` describing the run) and check that only rank 0 works under torchrun."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import FS, ROOT, rel_max
from oracle import oracle as O

REQUIRED = ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
            "scaling", "vs_baseline", "dtype", "data", "config", "e2e", "cpu_baseline")


def run_bench(extra_env=None, *args):
    env = dict(os.environ)
    env.pop("RANK", None)
    env.update(extra_env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", *args],
                          cwd=ROOT, env=env, capture_output=True, text=True, timeout=300)


def test_reference_arm_prints_one_contract_line():
    r = run_bench(None, "--steps", "2", "--warmup", "1")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout
    line = json.loads(lines[0])
    assert line["impl"] == "reference"
    for key in REQUIRED:
        assert key in line, key
    assert line["unit"] == "cells/s" and line["higher_is_better"] is True
    assert line["steps"] == 2 and line["warmup"] == 1 and line["n_gpus"] == 1
    assert line["dtype"] == "f64" and "workload" in line["config"] and "model" not in line["config"]
    # 2 surfaces of 400 x 8192 cells in ms_per_step each
    assert abs(line["value"] - 400 * 8192 / (line["ms_per_step"] * 1e-3)) <= 1e-6 * line["value"]
    assert line["e2e"] == {"value": line["value"], "unit": "cells/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"] and cb["sample"]
    assert line["gpu_launches"] == 0


def test_reference_arm_other_ranks_exit_without_work():
    r = run_bench({"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"}, "--gpus", "2", "--steps", "2", "--warmup", "1")
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.strip() == ""


def test_steps_must_be_positive():
    r = run_bench(None, "--steps", "0")
    assert r.returncode == 2 and "--steps" in r.stderr


DUMPED = ("peak", "row_peak_index", "row_peak_value", "surface")


def load_dump(path, dtype):
    assert sorted(os.listdir(path)) == [n + ".npy" for n in DUMPED]
    got = {n: np.load(os.path.join(path, n + ".npy")) for n in DUMPED}
    assert got["surface"].dtype == dtype and all(got[n].dtype == np.float64 for n in DUMPED if n != "surface")
    assert sum(a.nbytes for a in got.values()) <= 64 << 20
    assert got["surface"].shape == (400, 8192) and got["row_peak_value"].shape == got["row_peak_index"].shape == (400,)
    assert got["peak"].shape == (4,)
    return got


def test_reference_arm_dumps_its_last_step(tmp_path, chirp0):
    """--dump-outputs: the surface, the row peaks and find_peak's answer of the README pair on the 0.5 Hz grid."""
    from caf_cookoff_b200 import bench_shifts
    r = run_bench(None, "--steps", "2", "--warmup", "0", "--dump-outputs", str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    got = load_dump(tmp_path, np.float64)
    surf, pidx, pval = O.caf_surface(*chirp0, bench_shifts(), FS)
    assert rel_max(got["surface"], surf) <= 1e-12
    assert np.array_equal(got["row_peak_index"], pidx.astype(np.float64))
    assert np.array_equal(got["row_peak_value"], got["surface"][np.arange(400), pidx.astype(np.int64)])
    assert list(got["peak"][1:]) == [69.0, 338, 202] and got["peak"][0] == pval.max()


@pytest.mark.gpu
def test_b200_arm_dumps_its_last_timed_step(tmp_path):
    """The b200 arm runs exactly --steps timed launches and dumps the last one: rotation pair (warmup + steps - 1) mod 320,
    drawn ten per seed from seed 0 on rank 0, against the oracle on the same inputs."""
    from caf_cookoff_b200 import bench_shifts, generate as G
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "8", "--warmup", "3", "--no-blocks",
                        "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                       cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout)
    assert line["steps"] == 8 and line["gpu_launches"] == 8 and line["check_ok"]
    got = load_dump(tmp_path, np.float64)
    needle, hay = G.as_inputs(G.pair(0, seed=1))                  # last timed step k = 3 + 8 - 1 = 10: seed 1, pair 0
    freqs = bench_shifts()
    surf, pidx, pval = O.caf_surface(needle, hay[:needle.size], freqs, FS, threads=os.cpu_count() or 1)
    assert rel_max(got["surface"], surf) <= 1e-9
    assert np.array_equal(got["row_peak_index"], pidx.astype(np.float64))
    assert rel_max(got["row_peak_value"], pval) <= 1e-9
    freq, delay = O.find_peak(freqs, pidx, pval)
    assert (got["peak"][1], got["peak"][3]) == (freq, delay) and got["peak"][2] == int(np.argmax(pval))
