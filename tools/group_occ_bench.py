"""Measure the occurrence records on the sharded table (apgk_group_build_occurrences) against the single-GPU build
(apgk_build_occurrences).

    python tools/group_occ_bench.py [--ranks N] [--reads 60000000] [--steps 3] [--warmup 1] [--out FILE]

N ranks in ONE process (KmerGroup.local), spread over the visible GPUs round-robin; each holds --reads synthetic 100 bp
reads (K = 25), the slices of one read set, as bench.py gives every GPU.  First, on rank 0's store alone, one plain
context's apgk_build_occurrences (the single-GPU reference, same store), whose device records are translated to the
group encoding ((read id << 32) | ((position - 1) << 1) | rc: reads are uniform, so read id = q / 100) and digested in
chunks; then the group count and --warmup + --steps group builds.  With one rank the shard's device records must give
the same digests (asserted): the records are identical.
Prints one JSON line (and writes it to --out): card name and power limit (read in the same run), the group call's stage
times (device events, first rank, median), remote bytes, and the single-context phase times.  Nothing here is a
pass/fail threshold."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

K, READ_LEN, GENOME_PER_RANK = 25, 100, 100_000_000
CHUNK = 1 << 27


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=60).stdout.strip().splitlines()[0]
        name, limit = [x.strip() for x in out.split(",")]
        return name, limit
    except Exception as e:  # noqa: BLE001
        return "unknown (%s)" % e, "unknown"


class _CudaView:
    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<i8", "data": (ptr, False), "version": 3}


def digests(ptr, n, single):
    """position-sensitive 64-bit digests of n device records, one per CHUNK; single: translate the single-GPU encoding
    (q << 1 | rc) to the group encoding first"""
    import torch

    out = []
    for a in range(0, n, CHUNK):
        m = min(CHUNK, n - a)
        v = torch.as_tensor(_CudaView(ptr + 8 * a, m), device="cuda")
        if single:
            q = v >> 1
            v = ((q // READ_LEN) << 32) | ((q % READ_LEN) << 1) | (v & 1)
        i = torch.arange(a, a + m, dtype=torch.int64, device="cuda")
        x = v * -7046029254386353131 + i * -4417276706812531889   # 0x9E3779B97F4A7C15, 0xC2B2AE3D27D4EB4F (wrapping)
        x = x ^ (x >> 29)
        out.append(int(x.sum()))
        del v, i, x
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ranks", type=int, default=1)
    ap.add_argument("--reads", type=int, default=60_000_000, help="reads per rank")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out")
    args = ap.parse_args()
    import torch

    from allpathslg_b200 import KmerCounter, KmerGroup, synth_params

    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    name, limit = card()
    n_dev = torch.cuda.device_count()
    sp = synth_params(GENOME_PER_RANK * args.ranks, READ_LEN)
    R = args.reads

    # single-GPU reference on rank 0's store
    with KmerCounter(K, device=0, want_counts=True, reserve_bases=R * READ_LEN) as one:
        one.synth_reads(sp, 0, R)
        one.finish()
        single = [one.build_occurrences()["ms"] for _ in range(args.warmup + args.steps)][args.warmup:]
        ref = None
        if args.ranks == 1:
            _, d_occ, n_occ = one.occurrences_device()
            ref = digests(d_occ, n_occ, True)

    kcs = []
    for r in range(args.ranks):
        kc = KmerCounter(K, device=r % n_dev, want_counts=True, reserve_bases=R * READ_LEN)
        kc.synth_reads(sp, r * R, R)
        kcs.append(kc)
    with KmerGroup.local(kcs) as grp:
        grp.count()
        runs = [grp.build_occurrences() for _ in range(args.warmup + args.steps)][args.warmup:]
        match = None
        if args.ranks == 1:   # more ranks: a larger global table
            _, d_occ, n_occ = kcs[0].occurrences_device()
            match = digests(d_occ, n_occ, False) == ref
            assert match, "the one-rank group's records differ from apgk_build_occurrences's"
    for kc in kcs:
        kc.close()

    def med(rs, k):
        return round(statistics.median(r[k] for r in rs), 2)

    st = runs[-1]
    single_total = round(statistics.median(sum(r.values()) for r in single), 2)
    res = {
        "metric": "group_build_occurrences", "card": name, "power_limit": limit, "ranks": args.ranks,
        "gpus": min(args.ranks, n_dev), "reads_per_rank": R, "read_len": READ_LEN, "K": K, "steps": args.steps,
        "timing": "device events, %d warm-up + %d repetitions, median" % (args.warmup, args.steps),
        "rank0": {"total_ms": med(runs, "total_ms"), "sweep_ms": med(runs, "sweep_ms"), "exchange_ms": med(runs, "exchange_ms"),
                  "sort_ms": med(runs, "sort_ms"), "n_batches": st["n_batches"], "n_windows": st["n_windows"],
                  "n_occ": st["n_occ"], "n_big_runs": st["n_big_runs"], "remote_bytes": st["remote_bytes"],
                  "reps_total_ms": [round(r["total_ms"], 2) for r in runs]},
        "single_context_build_occurrences_ms": {k: med(single, k) for k in single[0]},
        "single_context_total_ms": single_total,
        "group_over_single": round(med(runs, "total_ms") / single_total, 3) if single_total > 0 else None,
        "rank0_equals_single_context": match,
    }
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
