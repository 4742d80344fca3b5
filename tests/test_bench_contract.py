"""bench.py prints ONE JSON line with the keys the driver reads; both arms, small sizes."""
import json
import os
import subprocess
import sys

import pytest

from conftest import ROOT

REQUIRED = ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
            "vs_baseline", "dtype", "data", "config")


def _run(args):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True,
                         timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, out.stdout[-2000:]
    return json.loads(lines[0])


def test_reference_arm_line():
    d = _run(["--impl", "reference", "--reads", "50000", "--steps", "2", "--warmup", "1"])
    for k in REQUIRED + ("impl", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"] > 0
    assert "workload" in d["config"]


@pytest.mark.gpu
def test_b200_arm_line():
    d = _run(["--reads", "400000", "--steps", "3", "--warmup", "3", "--cpu-seconds", "1", "--e2e-steps", "1"])
    for k in REQUIRED + ("roofline", "cpu_baseline", "e2e", "gpu_launches", "clocks", "phase_ms"):
        assert k in d, k
    assert d["n_gpus"] == 1 and d["steps"] == 3 and d["value"] > 0 and d["gpu_launches"] > 0
    r = d["roofline"]
    assert r["bound"] == "hbm" and 0 < r["frac"] < 1.2 and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] == 400000 * 150
    assert d["cpu_baseline"]["kind"] == "port" and "workload" in d["config"] and "model" not in d["config"]
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}


@pytest.mark.gpu
@pytest.mark.parametrize("R", [1, 8])
def test_dump_outputs_match_oracle(tmp_path, oracle_mod, R):
    """--dump-outputs: float32 / float64 arrays, 64 MB at most, and what the oracle computes on the same reads (rows in
    read order with one read group, the segmented layout with several)."""
    import numpy as np
    from conftest import DELTA_KEYS, TABLE_KEYS
    from kbbq import synth
    N, L = 100_000, 150
    d = _run(["--reads", str(N), "--read-groups", str(R), "--steps", "2", "--warmup", "1", "--no-configs", "--no-e2e",
              "--no-fastq", "--no-cpu", "--dump-outputs", str(tmp_path)])
    assert d["steps"] == 2
    names = os.listdir(tmp_path)
    got = {f[:-len(".npy")]: np.load(tmp_path / f) for f in names}
    assert set(got) == set(TABLE_KEYS + DELTA_KEYS + ("out_qual", "out_qual_reads"))
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert sum(os.path.getsize(tmp_path / f) for f in names) <= 64_000_000
    seq, qual, corr, rg, second = synth.synth_reads(d["config"]["seed"], 0, N, L, R)
    tables = oracle_mod.covariate_arrays(seq, qual, corr, rg, second, L, R)
    deltas = oracle_mod.get_delta_qs(*tables)
    for name, want in zip(TABLE_KEYS + DELTA_KEYS, tables + deltas):
        assert np.array_equal(got[name], want), name
    rows = got["out_qual_reads"].astype(np.int64)
    assert rows.size == 1 << 16 and np.all(np.diff(rows) > 0)
    want = oracle_mod.apply(seq[rows], qual[rows], rg[rows], second[rows], L, R, tables[0], *deltas)
    assert np.array_equal(got["out_qual"], want)
