"""bench.py's reference arm on a tiny configuration (CPU only): the JSON line carries the keys the driver reads, the
reference's own output is checked against the oracle port, and ranks other than 0 stay silent.  --dump-outputs: the
sampling of a long pair list (CPU) and the dumped results of the CUDA path against the oracle (GPU)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import train_oracle as to
from yacht_b200 import _lib, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra_env=None, *argv):
    env = dict(os.environ)
    env.update(extra_env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *argv], cwd=ROOT, env=env, stdout=subprocess.PIPE,
                          stderr=subprocess.PIPE, text=True, timeout=600)


@pytest.mark.skipif(not to.reference_available(), reason="oracle/_ref not present")
def test_reference_arm_json_line():
    cp = _run(None, "--impl", "reference", "--genomes", "300", "--seed", "11", "--steps", "2", "--warmup", "1", "--no-reference-cache")
    assert cp.returncode == 0, cp.stderr[-2000:]
    lines = [l for l in cp.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "pairs/s" and d["higher_is_better"] is True
    assert d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 1 and d["steps_run"] == 2
    assert d["value"] > 0 and d["ms_per_step"] > 0
    assert "300 genomes" in d["config"]["workload"] and d["config"]["genomes"] == 300
    cb = d["cpu_baseline"]
    assert cb["kind"] == "reference" and cb["cores"] >= 1 and cb["value"] == d["value"] and "ALL 300 of 300" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["vs_baseline"] is None


def test_reference_arm_other_ranks_stay_silent():
    cp = _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}, "--impl", "reference", "--gpus", "2", "--genomes", "300")
    assert cp.returncode == 0 and cp.stdout.strip() == ""


def test_dump_outputs_samples_a_long_pair_list_the_same_way_every_time(tmp_path, monkeypatch):
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 4096 + 24 * 1000)
    pairs = np.zeros(5000, dtype=_lib.PAIR_DTYPE)
    pairs["i"], pairs["j"], pairs["count"] = np.arange(5000) // 50, np.arange(5000) % 50, np.arange(5000)
    stats = {"n_distinct": 11, "n_singleton": 7, "n_index": 4}
    dumps = []
    for name in ("a", "b"):
        d = tmp_path / name
        bench.dump_outputs(str(d), stats, pairs)
        assert sum(os.path.getsize(d / f) for f in os.listdir(d)) <= bench.DUMP_BYTES
        dumps.append({f: np.load(d / f) for f in sorted(os.listdir(d))})
    a, b = dumps
    assert sorted(a) == ["index_stats.npy", "pairs_count.npy", "pairs_i.npy", "pairs_j.npy"]
    assert all(v.dtype == np.float64 for v in a.values())
    assert a["index_stats.npy"].tolist() == [11, 7, 4, 5000]
    rows = a["pairs_count.npy"].astype(np.int64)         # count = row number here: the sample is 1000 distinct rows, in order
    assert len(rows) == 1000 and np.all(np.diff(rows) > 0)
    assert np.array_equal(a["pairs_i.npy"], rows // 50) and np.array_equal(a["pairs_j.npy"], rows % 50)
    assert all(np.array_equal(a[f], b[f]) for f in a)


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_steps_results(tmp_path):
    launches, dumps = {}, {}
    for steps in (1, 3):
        out = tmp_path / f"dump{steps}"
        cp = _run(None, "--genomes", "1000", "--seed", "11", "--steps", str(steps), "--warmup", "1", "--no-cpu-baseline",
                  "--no-run-path", "--dump-outputs", str(out))
        assert cp.returncode == 0, cp.stderr[-2000:]
        lines = [l for l in cp.stdout.splitlines() if l.startswith("{")]
        assert len(lines) == 1
        launches[steps] = json.loads(lines[0])["gpu_launches"]     # the library's kernel launches over the timed resident steps
        dumps[steps] = {f[:-4]: np.load(out / f) for f in sorted(os.listdir(out))}
    assert launches[1] > 0 and launches[3] == 3 * launches[1]      # --steps sets the number of timed steps
    got = dumps[3]
    assert sorted(got) == sorted(dumps[1]) and all(np.array_equal(got[k], dumps[1][k]) for k in got)   # same inputs, same outputs
    assert sorted(got) == ["index_stats", "pairs_count", "pairs_i", "pairs_j"]
    assert all(v.dtype == np.float64 for v in got.values())
    db = synth.make_reference_db(1000, 11)
    ref = to.oracle_train(db.hashes, db.offsets, 0.95 ** 31)
    assert got["index_stats"].tolist() == [ref.n_distinct, ref.n_singleton, ref.n_index, len(ref.pairs)]
    for c in ("i", "j", "count"):
        assert np.array_equal(got[f"pairs_{c}"], ref.pairs[c].astype(np.float64)), c


def test_steps_below_one_are_refused():
    cp = _run(None, "--steps", "0")
    assert cp.returncode == 2 and "--steps must be at least 1" in cp.stderr
