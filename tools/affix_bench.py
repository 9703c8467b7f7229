"""Measure the affix build (apgk_build_affixes) on the benchmark store, beside the occurrence records and the bulk
frequency lookups on the same store.

    python tools/affix_bench.py [--reads 60000000] [--reps 5] [--warmup 1] [--out FILE]

One GPU, bench.py's workload: synthetic 100 Mb genome, --reads x 100 bp reads (same generator and seeds), K = 25.
After the count: --warmup + --reps affix builds, then the same for apgk_build_occurrences and apgk_read_freqs_device.
Prints one JSON line (and writes it to --out): card name and power limit (read in the same run), the device-event phase
times of every repetition, their medians, and G windows/s over the median total.  Nothing here is a pass/fail
threshold."""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

K, READ_LEN, GENOME = 25, 100, 100_000_000


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=60).stdout.strip().splitlines()[0]
        name, limit = [x.strip() for x in out.split(",")]
        return name, limit
    except Exception as e:  # noqa: BLE001
        return "unknown (%s)" % e, "unknown"


def summary(runs, n_windows):
    keys = list(runs[0])
    med = {k: round(statistics.median(r[k] for r in runs), 2) for k in keys}
    total = statistics.median(sum(r.values()) for r in runs)
    return {"reps_ms": [{k: round(v, 2) for k, v in r.items()} for r in runs], "median_ms": med,
            "median_total_ms": round(total, 2), "gwindows_per_s": round(n_windows / (total * 1e-3) / 1e9, 2)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=60_000_000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out")
    args = ap.parse_args()
    import torch

    from allpathslg_b200 import KmerCounter, synth_params

    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    name, limit = card()
    sp = synth_params(GENOME, READ_LEN)
    with KmerCounter(K, device=0, want_counts=True, reserve_bases=args.reads * READ_LEN) as kc:
        kc.synth_reads(sp, 0, args.reads)
        kc.finish()
        n_windows, n_distinct = kc.totals()
        tb, _ = kc.read_store_info()
        aff = [kc.build_affixes() for _ in range(args.warmup + args.reps)][args.warmup:]
        occ = [kc.build_occurrences()["ms"] for _ in range(args.warmup + args.reps)][args.warmup:]
        buf = torch.empty(tb, dtype=torch.int32, device="cuda:0")
        freq = [kc.read_freqs_device(buf.data_ptr()) for _ in range(args.warmup + args.reps)][args.warmup:]
        a = kc.affixes()
        pop = int(np.unpackbits(a).sum())
    res = {"metric": "build_affixes", "card": name, "power_limit": limit, "K": K, "reads": args.reads, "read_len": READ_LEN,
           "genome_len": GENOME, "windows": n_windows, "distinct": n_distinct, "affix_bits_set": pop,
           "timing": "device events around each phase, %d warm-up + %d repetitions, median" % (args.warmup, args.reps),
           "build_affixes": summary(aff, n_windows), "build_occurrences": summary(occ, n_windows),
           "read_freqs_device": summary(freq, n_windows)}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
