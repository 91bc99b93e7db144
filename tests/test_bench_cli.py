"""bench.py's command line.  CPU: the reference arm prints one JSON line with the contract's
keys; --dump-outputs keeps to its byte budget.  -m gpu: the GPU arm at a small size dumps its
last step's outputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_contract(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference",
                          "--steps", "1", "--warmup", "0", "--genome-mb", "2", "--variants", "100",
                          "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "read_bases_kmer_probed_per_sec"
    assert d["unit"] == "bases/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "bases/s", "h2d_bytes_per_step": 0,
                        "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["vs_baseline"] is None
    assert d["config"]["step_fraction"] == 1.0  # small workloads run the whole step
    counts = np.load(tmp_path / "counts.npy")
    assert d["dumped_outputs"] == {"counts": [list(counts.shape)] * 2} and counts.shape[0] == 3
    assert counts.dtype == np.float64 and f" {int(counts.sum())} k-mer hits per step" in d["cpu_baseline"]["sample"]


def test_reference_arm_does_not_load_the_product(tmp_path):
    """The reference arm must not map libdkb.so (nor import the package that binds it): its
    numbers are the oracle's alone."""
    code = (
        "import sys, runpy\n"
        "sys.argv = ['bench.py', '--impl', 'reference', '--steps', '1', '--warmup', '0', '--genome-mb', '1', '--variants', '50']\n"
        "try:\n"
        "    runpy.run_path(%r, run_name='__main__')\n"
        "except SystemExit:\n"
        "    pass\n"
        "maps = open('/proc/self/maps').read()\n"
        "assert 'libdkb' not in maps, 'libdkb.so is mapped'\n"
        "assert 'libdnk_oracle' in maps\n"
        "assert not any(m == 'denovo_kmer_b200' or m.startswith('denovo_kmer_b200.') for m in sys.modules), 'package imported'\n"
        "sys.stderr.write('CLEAN\\n')\n" % os.path.join(ROOT, "bench.py"))
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "CLEAN" in out.stderr, out.stderr[-2000:]


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference",
                          "--gpus", "2", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=120, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_dump_outputs_budget_and_sample(tmp_path):
    """--dump-outputs: a group that fits is written whole; a later group that does not keeps the
    same seeded, ordered sample of its entries / variants in every array, within the byte budget."""
    import bench

    def outputs(prefix, n_entries, n_var):
        counts = np.arange(3 * n_entries, dtype=np.uint32).reshape(3, n_entries)
        per_var = [np.arange(n_var * m, dtype=np.uint32).reshape((n_var,) + s)
                   for m, s in ((6, (2, 3)), (6, (2, 3)), (2, (2,)))]
        return bench.job_outputs(prefix, counts, per_var + [(np.arange(n_var) % 251).astype(np.uint8)])

    groups = [outputs("", 1000, 40), outputs("wgs_shard_", 50_000, 2000)]
    budget = 80_000
    shapes = bench.dump_outputs(str(tmp_path / "a"), groups, budget=budget)
    bench.dump_outputs(str(tmp_path / "b"), groups, budget=budget)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == sorted(n + ".npy" for g in groups for n in g)
    total = 0
    for f in files:
        x = np.load(tmp_path / "a" / f)
        assert x.dtype == np.float64 and np.array_equal(x, np.load(tmp_path / "b" / f))
        total += os.path.getsize(tmp_path / "a" / f)
    assert total <= budget
    for name, (arr, _) in groups[0].items():  # first group: whole
        assert np.array_equal(np.load(tmp_path / "a" / (name + ".npy")), arr)
    c = np.load(tmp_path / "a" / "wgs_shard_counts.npy")
    assert 0 < c.shape[1] < 50_000 and shapes["wgs_shard_counts"] == [[3, 50_000], list(c.shape)]
    idx = c[0].astype(np.int64)  # row 0 of the arange counters holds the kept entry indices
    assert np.all(np.diff(idx) > 0) and np.array_equal(c[2], idx + 2 * 50_000)
    v = np.load(tmp_path / "a" / "wgs_shard_hits.npy")[:, 0, 0].astype(np.int64) // 6  # kept variants
    assert 0 < len(v) < 2000 and np.all(np.diff(v) > 0)
    assert np.array_equal(np.load(tmp_path / "a" / "wgs_shard_distinct.npy")[:, 0, 0], 6 * v)
    assert np.array_equal(np.load(tmp_path / "a" / "wgs_shard_n_kmers.npy")[:, 0], 2 * v)
    assert np.array_equal(np.load(tmp_path / "a" / "wgs_shard_calls.npy"), v % 251)


@pytest.mark.gpu
def test_gpu_arm_dumps_last_step_outputs(tmp_path):
    """The GPU arm at a small size: --dump-outputs writes the last step's counters and per-variant
    results, and those counters are the ones the CPU oracle matched."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1",
                          "--genome-mb", "2", "--variants", "100", "--no-e2e", "--no-wgs",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads(out.stdout)
    assert d["steps"] == 2 and d["checks"]["cpu_oracle_matches_gpu"] is True
    assert d["cpu_baseline"]["sample"].startswith("the whole step")
    counts = np.load(tmp_path / "counts.npy")
    assert counts.dtype == np.float64 and counts.shape == (3, d["config"]["table_entries"])
    assert counts.sum() == d["cpu_baseline"]["kmer_hits"] > 0
    calls = np.load(tmp_path / "calls.npy")
    assert calls.shape == (100,) and int((calls.astype(np.int64) & 1).sum()) == d["config"]["denovo_calls"]
    for name, shape in (("hits", (100, 2, 3)), ("distinct", (100, 2, 3)), ("n_kmers", (100, 2))):
        assert np.load(tmp_path / (name + ".npy")).shape == shape
