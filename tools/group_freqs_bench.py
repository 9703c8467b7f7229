"""Measure the frequency lookups on the sharded table (apgk_group_read_freqs_device) against the single-GPU bulk form.

    python tools/group_freqs_bench.py [--ranks N] [--reads 60000000] [--steps 3] [--warmup 1]

N ranks in ONE process (KmerGroup.local), spread over the visible GPUs round-robin; each holds --reads synthetic
100 bp reads (K=25), the slices of one read set, as bench.py gives every GPU.  First, on rank 0's store alone, one
plain context's apgk_read_freqs_device (the single-GPU reference, same store); then the group count and --steps
timed group lookups over every rank's whole store.  With one rank its answers must equal the reference at every
base.
Prints one JSON line: card name and power limit (read in the same run), the group call's stage times (device events,
first rank), remote bytes and the rate they imply over the exchange stage, and the single-context stage times.
Nothing here is a pass/fail threshold."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

K, READ_LEN, GENOME_PER_RANK = 25, 100, 100_000_000


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=60).stdout.strip().splitlines()[0]
        name, limit = [x.strip() for x in out.split(",")]
        return name, limit
    except Exception as e:  # noqa: BLE001
        return "unknown (%s)" % e, "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ranks", type=int, default=1)
    ap.add_argument("--reads", type=int, default=60_000_000, help="reads per rank")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
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
    with KmerCounter(K, device=0) as one:
        one.synth_reads(sp, 0, R)
        one.finish()
        tb, _ = one.read_store_info()
        ref = torch.empty(tb, dtype=torch.int32, device="cuda:0")
        one.read_freqs_device(ref.data_ptr())
        single = one.read_freqs_device(ref.data_ptr())
    single["total"] = sum(single.values())
    windows = int((ref != -1).sum())

    kcs = []
    for r in range(args.ranks):
        kc = KmerCounter(K, device=r % n_dev)
        kc.synth_reads(sp, r * R, R)
        kcs.append(kc)
    outs = [torch.empty(kc.read_store_info()[0], dtype=torch.int32, device="cuda:%d" % kc.device) for kc in kcs]
    with KmerGroup.local(kcs) as grp:
        grp.count()
        for _ in range(args.warmup):
            grp.read_freqs_device([o.data_ptr() for o in outs])
        runs = [grp.read_freqs_device([o.data_ptr() for o in outs]) for _ in range(args.steps)]
        match = bool(torch.equal(outs[0], ref)) if args.ranks == 1 else None   # more ranks: a larger global table
    for kc in kcs:
        kc.close()

    def med(k):
        v = sorted(r[k] for r in runs)
        return v[len(v) // 2]

    st = runs[-1]
    res = {
        "metric": "group_read_freqs", "card": name, "power_limit": limit, "ranks": args.ranks, "gpus": min(args.ranks, n_dev),
        "reads_per_rank": R, "read_len": READ_LEN, "K": K, "steps": args.steps,
        "rank0": {"total_ms": med("total_ms"), "sweep_ms": med("sweep_ms"), "exchange_ms": med("exchange_ms"),
                  "scatter_ms": med("scatter_ms"), "n_batches": st["n_batches"], "n_queries": st["n_queries"],
                  "remote_bytes": st["remote_bytes"],
                  "remote_GBps": st["remote_bytes"] / (med("exchange_ms") * 1e-3) / 1e9 if st["remote_bytes"] else 0.0},
        "single_context_read_freqs_device_ms": single, "single_context_windows": windows,
        "rank0_equals_single_context": match,
    }
    print(json.dumps(res))


if __name__ == "__main__":
    main()
