"""bench.py --dump-outputs DIR: the arrays the last timed step handed its caller, as DIR/<name>.npy in
float32 / float64.  The inputs are seeded, so the dump of a step is known in advance: the oracle's answer
for the ring entry that step used."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(out, *args):
    r = subprocess.run([sys.executable, "bench.py", "--workload", "cfg2", "--steps", "3", "--warmup", "3", "--dump-outputs",
                        str(out), *args], cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout)["steps"] == 3
    return {f[:-4]: np.load(os.path.join(out, f)) for f in sorted(os.listdir(out))}


def test_reference_arm_dumps_the_last_step(tmp_path, egpu, oracle_c):
    got = run_bench(tmp_path, "--impl", "reference")
    w = egpu.synth.workload("cfg2")
    # the reference arm cycles through four host batches: step 2 scores the third
    rc, rm = egpu.synth.requests(w["dist"], w["seed"], w["R"], first_row=2 * w["R"])
    exp, *_ = oracle_c.snapshot(w["free_core"], w["free_mem"], rc, rm)
    assert list(got) == ["indices"] and got["indices"].dtype == np.float32
    assert np.array_equal(got["indices"], exp)


def test_large_batches_dump_a_fixed_sample_of_rows():
    import bench
    idx = np.arange(bench.DUMP_ROWS + 12_345, dtype=np.int32) % 67 - 1
    a, b = bench.output_arrays(idx), bench.output_arrays(idx.copy())
    rows = a["indices_rows"].astype(np.int64)
    assert np.array_equal(rows, b["indices_rows"]) and np.all(np.diff(rows) > 0) and rows[-1] < idx.size
    assert np.array_equal(a["indices"], idx[rows]) and a["indices"].dtype == np.float32
    assert sum(x.nbytes for x in a.values()) <= 64 << 20


@pytest.mark.gpu
def test_native_arm_dumps_the_last_step(tmp_path, egpu, oracle_c):
    got = run_bench(tmp_path, "--no-sweep", "--cpu-budget", "0.1")
    w = egpu.synth.workload("cfg2")
    # the timed steps rotate through a ring of 64 device-resident batches: step 2 scores the third
    rc, rm = egpu.synth.requests(w["dist"], w["seed"], w["R"], first_row=2 * w["R"])
    idx, dc, dm, tab = oracle_c.snapshot(w["free_core"], w["free_mem"], rc, rm)
    assert list(got) == ["delta", "indices", "table_out"]
    assert got["indices"].dtype == np.float32 and got["delta"].dtype == got["table_out"].dtype == np.float64
    assert np.array_equal(got["indices"], idx)
    assert np.array_equal(got["delta"], np.concatenate([dc, dm])) and np.array_equal(got["table_out"], tab)
