"""GPU: bench.py at a small size — --steps sets every timed loop, and --dump-outputs writes what the timed paths
returned in their last step: float64 only, within 64 MiB, the same in two runs, and equal to the oracle's sketches of
the same synthetic inputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from tests.util import REPO

pytestmark = pytest.mark.gpu

STEPS = 3
SMALL = ["--steps", str(STEPS), "--warmup", "1", "--reads", "100000", "--genomes", "40", "--batch-genomes", "6", "--no-cpu"]


def run_bench(out):
    r = subprocess.run([sys.executable, os.path.join(REPO, "bench.py")] + SMALL + ["--dump-outputs", str(out)],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900, cwd=REPO)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    return json.loads(lines[0]), {f[:-4]: np.load(os.path.join(out, f)) for f in sorted(os.listdir(out))}


def u64(d, name):
    return (d[name + "_hi"].astype(np.uint64) << np.uint64(32)) | d[name + "_lo"].astype(np.uint64)


def test_steps_and_dumped_outputs(tmp_path):
    from oracle import oracle as O
    from sylph_b200 import synth
    line, a = run_bench(tmp_path / "a")
    assert line["steps"] == line["e2e"]["steps"] == line["pairs"]["steps"] == line["genomes"]["steps"] == STEPS
    assert all(v.dtype == np.float64 for v in a.values())
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= 64 << 20
    _, b = run_bench(tmp_path / "b")
    assert sorted(a) == sorted(b) and all(np.array_equal(a[k], b[k]) for k in a)

    # the sample sketch of the timed step == the oracle's sketch of the same reads (all rows: below the sampling limit)
    rb, ro = synth.reads(100000)
    h, c, mean, nd = O.sketch_reads(rb.numpy(), ro.numpy().astype(np.uint64), nthreads=os.cpu_count() or 1)
    assert a["sketch_rows"].tolist() == [len(h)] and np.array_equal(u64(a, "sketch_hash"), h)
    assert np.array_equal(a["sketch_count"], c)
    assert a["sketch_stats_num_dup_removed"].tolist() == [nd] and abs(a["sketch_stats_mean_read_length"][0] - mean) < 1e-9

    # the genome batch of the timed step == the oracle's per-genome sketches
    L = 4_000_000
    ends = [0] + u64(a, "genomes_kmer_end").astype(np.int64).tolist()
    tends = [0] + u64(a, "genomes_tracked_end").astype(np.int64).tolist()
    kmers, tracked = u64(a, "genome_kmers_hash"), u64(a, "genome_tracked_hash")
    assert a["genomes_rows"].tolist() == [6] and len(kmers) == ends[-1] and len(tracked) == tends[-1]
    for g in range(6):
        gb, _ = synth.db_chunk(g, g + 1, L)
        km, tr, gs = O.sketch_genome(gb.numpy(), np.array([0, L], np.uint64))
        assert np.array_equal(kmers[ends[g]:ends[g + 1]], km) and np.array_equal(tracked[tends[g]:tends[g + 1]], tr), g
        assert u64(a, "genomes_gn_size")[g] == gs

    # the profile rows of the timed step: the sample's community is genomes 0..63, of which the db holds 0..39
    n = int(a["profile_rows"][0])
    assert 0 < n <= 40 and len(a["profile_genome"]) == n and a["profile_ci"].shape == (n, 4)
    assert set(a["profile_sample"].tolist()) == {0} and a["profile_genome"].max() < 40
