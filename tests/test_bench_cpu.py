"""CPU suite: the parts of bench.py that need no GPU — the reference arm's JSON line (bench contract)
and the helpers around it."""
import json
import os
import subprocess
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    r = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                        "--reads", "40000"], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600, cwd=REPO)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "bases/s sketched" and d["unit"] == "bases/s"
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["n_gpus"] == 1
    assert d["value"] > 0 and d["steps"] == 1 and d["warmup"] == 1 and d["ms_per_step"] > 0
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def test_reference_arm_profile_workload():
    r = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--workload", "profile", "--steps", "1",
                        "--warmup", "1", "--reads", "20000", "--genomes", "3"], stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                       text=True, timeout=600, cwd=REPO)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.strip()][-1])
    assert d["impl"] == "reference" and d["unit"] == "pairs/s" and d["value"] > 0
    assert d["config"]["genomes_per_gpu"] == 3 and d["cpu_baseline"]["value"] == d["value"]


def test_both_arms_share_the_config_object():
    sys.path.insert(0, REPO)
    import bench

    class A:
        reads, genomes, samples = 1000, 7, None
    assert bench.sketch_config(A) == bench.sketch_config(A) and set(bench.sketch_config(A)) >= {"workload", "reads_per_gpu", "k", "c"}
    assert bench.profile_config(A, 1)["samples"] == 1 and bench.profile_config(A, 8)["samples"] == 16


def test_dump_table_is_exact_seeded_and_bounded(tmp_path):
    """--dump-outputs' writer: float64 files only, uint64 values kept exactly (above 2^53), a table longer than its
    row limit cut to the same seeded sample in every run, and the row count recorded."""
    sys.path.insert(0, REPO)
    import numpy as np
    import bench
    n = bench.DUMP_ROWS["sketch"] + 5000
    i = np.arange(n, dtype=np.uint64)
    h = np.uint64(1 << 63) | (i << np.uint64(33)) | np.uint64(0x2345_6789)   # the row index sits in bits 33..62
    c = (i % np.uint64(7)).astype(np.uint32)
    bench._dumped[0] = 0
    for d in ("a", "b"):
        bench.dump_table(str(tmp_path / d), "sketch", {"hash": h, "count": c})
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == sorted(os.listdir(tmp_path / "b")) == ["sketch_count.npy", "sketch_hash_hi.npy", "sketch_hash_lo.npy",
                                                            "sketch_rows.npy"]
    for f in files:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype == np.float64 and np.array_equal(a, b), f
    load = lambda f: np.load(tmp_path / "a" / ("sketch_%s.npy" % f))  # noqa: E731
    got = (load("hash_hi").astype(np.uint64) << np.uint64(32)) | load("hash_lo").astype(np.uint64)
    rows = (got >> np.uint64(33)) & np.uint64((1 << 30) - 1)
    assert len(got) == bench.DUMP_ROWS["sketch"] and load("rows").tolist() == [n]
    assert np.all(rows[1:] > rows[:-1]) and int(rows[-1]) < n              # distinct rows, in table order
    assert np.array_equal(got, h[rows.astype(np.int64)]) and np.array_equal(load("count"), c[rows.astype(np.int64)])
    bench._dumped[0] = 0


def test_clock_sampler_degrades_without_a_gpu():
    sys.path.insert(0, REPO)
    import bench
    c = bench.ClockSampler(0)   # no NVML device and no nvidia-smi in this container: both fallbacks are taken
    c.start()
    out = c.stop()
    assert set(out) >= {"sm_mhz", "sm_max_mhz", "reasons"}
    assert out["sm_mhz"] is None or out["sm_mhz"] > 0
    off = bench.ClockSampler(None)
    off.start()
    assert off.stop() == {}
