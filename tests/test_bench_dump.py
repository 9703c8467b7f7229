"""bench.py --dump-outputs at a small size: the files hold what the timed path computed (the CPU oracle's spectrum,
totals and table rows on the bench's seeded reads), they do not depend on the number of steps, and --steps sets the
number of timed steps (the kernel launches of the timed region scale with it)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
READS, GENOME = 200_000, 400_000   # 15.2 M instances, a few million distinct k-mers: the table is sampled
NAMES = ("spectrum", "totals", "table_rows", "table_kmers", "table_counts")


def _bench(out_dir, steps):
    env = dict(os.environ, APGK_BENCH_READS=str(READS), APGK_BENCH_GENOME=str(GENOME), APGK_BENCH_CPU_READS="20000",
               APGK_BENCH_LOOKUPS="0", APGK_BENCH_RECORDS="0", APGK_BENCH_PARITY="0")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps),
                        "--warmup", "3", "--dump-outputs", str(out_dir)], capture_output=True, text=True, env=env,
                       timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps
    return line, {n: np.load(os.path.join(str(out_dir), n + ".npy")) for n in NAMES}


def test_dump_outputs_match_the_oracle_and_steps_scale_the_work(oracle, tmp_path):
    line1, d1 = _bench(tmp_path / "one", 1)
    line3, d3 = _bench(tmp_path / "three", 3)
    assert line3["gpu_launches"] == 3 * line1["gpu_launches"] > 0
    assert sorted(os.listdir(str(tmp_path / "one"))) == sorted(n + ".npy" for n in NAMES)
    assert sum(a.nbytes for a in d1.values()) <= 64 << 20
    for n in NAMES:
        assert d1[n].dtype == np.float64 and (d1[n] == d3[n]).all(), n
    sp = oracle.synth_params(GENOME, 100)
    p, o = oracle.synth_reads(sp, 0, READS)
    ek, ec, en = oracle.count(p, o, 25)
    assert d1["totals"].tolist() == [en, len(ek)]
    assert (d1["spectrum"] == oracle.spectrum(ec).astype(np.float64)).all()
    rows = d1["table_rows"].astype(np.int64)
    assert 0 < len(rows) < len(ek) and len(np.unique(rows)) == len(rows)
    assert (d1["table_kmers"] == ek[rows, 0].astype(np.float64)).all()
    assert (d1["table_counts"] == ec[rows].astype(np.float64)).all()
