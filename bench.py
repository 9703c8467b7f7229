#!/usr/bin/env python
"""bench.py -- headline benchmark: Gk-mers/s counted for a K=25 spectrum (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one pass of the hot path (extract -> canonicalise -> partition -> sort -> count ->
spectrum + sorted (k-mer, count) table) over the whole synthetic read set.  --steps K timed steps follow the
warm-up; --dump-outputs DIR writes what the last of them computed as float64 .npy files (see dump_outputs).

Workload (config.workload): BASELINE.json configs[2], the largest single-GPU configuration --
synthetic 100 Mb genome, 60 M x 100 bp reads (60x), K=25, 4.56 G k-mer instances per GPU.
At N > 1 (torchrun) per-GPU work is fixed (weak scaling): rank r generates reads
[r*60M, (r+1)*60M) of an N x 100 Mb genome; every rank partitions its reads by the leading bits of the
canonical k-mer, the ranks cut the bucket space into balanced contiguous ranges, each rank gathers the
ranges it owns straight from the peers' partition buffers over NVLink (the exchange is fused into the
gather kernel; APGK_SHARD_EXCHANGE=nccl selects an all-to-all instead) and sorts/counts its shard;
the spectra are all-reduced.

  value  whole-job Gk-mers/s with the reads already resident in HBM (device-timed region)
  e2e    the same through the public API with HOST (pinned) buffers: H2D of the packed reads and
         D2H of the spectrum inside the timed region
  roofline      the dominant kernel's algorithmic bytes / its CUDA-event duration vs measured HBM peak
  records       (N=1) the occurrence records of the same reads: (read id, signed position) per instance
  lookups       (N=1) the frequency of every window of the reads into a device buffer (error-correction lookups)
  cpu_baseline  the CPU oracle port (oracle/kmer_oracle.c, OpenMP, all host cores) on a bounded
                sample of the same workload.  It is a spec-derived restatement, NOT the reference's
                code: the reference source was not available (parity unpinned).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

K = 25
READ_LEN = 100
READS_PER_GPU = int(os.environ.get("APGK_BENCH_READS", 60_000_000))
GENOME_PER_GPU = int(os.environ.get("APGK_BENCH_GENOME", 100_000_000))
CPU_SAMPLE_READS = int(os.environ.get("APGK_BENCH_CPU_READS", 10_000_000))
# the CPU arm's sample keeps the workload's coverage (60x): 10 M reads of a 16.7 Mb genome, the same at every N
CPU_SAMPLE_GENOME = max(READ_LEN, GENOME_PER_GPU * CPU_SAMPLE_READS // READS_PER_GPU)
PARITY_PBITS, PARITY_PARTS = 8, (5, 77, 130, 201)   # sampled-partition oracle check: 4 of 256 leading-bit partitions
WORKLOAD = "celegans"
B_ALG_K25 = 136.0  # SURVEY.md section 8(d): 8 * (2*7 + 3) bytes per instance for the 7-pass LSD model


def traffic_file():
    for name in ("r02_traffic.json", "r01_traffic.json"):
        if os.path.exists(os.path.join(ROOT, "profiles", name)):
            return name
    return None


def ncu_traffic(stage=None):
    """DRAM bytes per launch of a stage's kernel from the committed full-size ncu capture (profiles/rNN_traffic.json:
    same workload as the N=1 bench), or None.  stage=None: the sum over the step's kernels that were captured."""
    try:
        with open(os.path.join(ROOT, "profiles", traffic_file())) as f:
            ks = json.load(f)["kernels"]
        if stage is not None:
            ks = {stage: ks[stage]}
        t = 0.0
        for k in ks.values():
            if k.get("dram_read_GB") is not None and k.get("dram_write_GB") is not None:
                t += (k["dram_read_GB"] + k["dram_write_GB"]) * 1e9
        return t if t > 0 else None
    except Exception:
        return None


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []
        self.first = 0

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def mark(self):
        """forget the samples taken so far (warm-up)"""
        self.first = len(self.lines)

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines[self.first:] or self.lines[-1:]:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_baseline(reads, genome_len, threads=0):
    """Oracle port timed on the host cores over `reads` reads of a `genome_len` genome (same generator, same
    coverage as the workload)."""
    from oracle import oracle_a as A

    A.build()
    sp = A.synth_params(genome_len, READ_LEN)
    packed, off = A.synth_reads(sp, 0, reads)
    threads = threads or (os.cpu_count() or 1)  # torchrun sets OMP_NUM_THREADS=1: ask for all host cores explicitly
    t0 = time.perf_counter()
    _, cnt, n_inst = A.count(packed, off, K, n_threads=threads)
    A.spectrum(cnt)
    dt = time.perf_counter() - t0
    return n_inst, dt, threads


def run_reference(args):
    """--impl reference: the CPU implementation of the path on the host cores.  The real reference
    could not be built (no source in /root/reference), so this times the oracle port."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    n_gpus = args.gpus
    times, n_inst, cores = [], 0, 1
    for i in range(args.warmup + args.steps):
        n_inst, dt, cores = cpu_baseline(CPU_SAMPLE_READS, CPU_SAMPLE_GENOME)
        if i >= args.warmup:
            times.append(dt)
    ms = 1e3 * sum(times) / len(times)
    val = n_inst / (ms * 1e-3) / 1e9
    sample = cpu_sample_text(n_inst) + ", per step"
    line = {
        "impl": "reference", "metric": "k-mer spectrum throughput (K=25), k-mer instances counted per second",
        "value": val, "unit": "Gk-mers/s", "n_gpus": n_gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64",
        "data": "synthetic", "config": workload_config(n_gpus),
        "cpu_baseline": {"value": val, "unit": "Gk-mers/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "Gk-mers/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "oracle port (spec-derived restatement); the reference source was not available: parity unpinned",
    }
    emit(line)
    return 0


def cpu_sample_text(n_inst):
    return ("%d reads of a %.1f Mb genome (%dx, the workload's coverage and generator; %d k-mer instances)"
            % (CPU_SAMPLE_READS, CPU_SAMPLE_GENOME / 1e6, CPU_SAMPLE_READS * READ_LEN // max(CPU_SAMPLE_GENOME, 1), n_inst))


def workload_config(n_gpus):
    if WORKLOAD == "human":
        what = ("BASELINE configs[3]: synthetic human-size %.1f Gb genome at %dx, %d M x %d bp reads split over %d GPUs, K=%d"
                % (GENOME_PER_GPU * n_gpus / 1e9, READS_PER_GPU * READ_LEN // GENOME_PER_GPU, READS_PER_GPU * n_gpus // 1_000_000,
                   READ_LEN, n_gpus, K))
    else:
        what = ("synthetic %d Mb genome, %d M x %d bp reads (%dx) per GPU, K=%d"
                % (GENOME_PER_GPU // 1_000_000, READS_PER_GPU // 1_000_000, READ_LEN, READS_PER_GPU * READ_LEN // GENOME_PER_GPU, K))
    return {"workload": what + ": spectrum to the host + sorted (k-mer, count) table resident on the device "
                        "(what the frequency-table lookups read)",
            "K": K, "reads_per_gpu": READS_PER_GPU, "read_len": READ_LEN, "genome_len": GENOME_PER_GPU * n_gpus,
            "sharding": ("canonical k-mer prefix ranges over %d ranks (balanced splitters), one exchange fused into "
                         "the gather kernel over NVLink peer memory" % n_gpus) if n_gpus > 1 else "single GPU",
            "l2_policy": "inputs (1.5 GB packed reads, 36 GB keys) exceed the 126 MB L2; no flush needed"}


def measure_lookups(kc, torch, total_bases):
    """k-mer frequency of every window of the reads (FindErrors table lookups), bulk form, device output."""
    out = torch.empty(total_bases, dtype=torch.int32, device="cuda")
    kc.read_freqs_device(out.data_ptr())
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    lms = kc.read_freqs_device(out.data_ptr())
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    n_valid = int(kc.totals()[0])  # one lookup per window that lies inside a read = per k-mer instance
    del out
    torch.cuda.empty_cache()
    return {"what": "k-mer frequency of every window of the reads (FindErrors table lookups), bulk form, device output",
            "ms": round(dt * 1e3, 2), "value": round(n_valid / dt / 1e9, 3), "unit": "G lookups/s",
            "stage_ms": {k_: round(v, 2) for k_, v in lms.items()}, "n_lookups": n_valid,
            "direct_form": "per-window table search (APGK_FREQ_DIRECT=1): see profiles/r01_occ.txt"}


def measure_records(kc, torch):
    """(read id, signed position) of every k-mer instance grouped by k-mer: second sweep over the reads."""
    kc.build_occurrences()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    info = kc.build_occurrences()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    return {"what": "(read id, signed position) of every k-mer instance grouped by k-mer: bucket scatter + per-bucket placement + per-run sort",
            "ms": round(dt * 1e3, 2), "value": round(info["n_occ"] / dt / 1e9, 3), "unit": "G records/s",
            "stage_ms": {k_: round(v, 2) for k_, v in info["ms"].items()}, "n_big_runs": info["n_big_runs"],
            "bytes_out": int(info["n_occ"]) * 8}


def sampled_parity(kc, host, n_reads):
    """SURVEY.md section 8(c)(ii): oracle over ALL reads restricted to a few leading-bit partitions vs the table."""
    from oracle import oracle_a as A

    t0 = time.perf_counter()
    keys, n_win = A.sample_prefix(host.data_ptr(), None, K, PARITY_PBITS, PARITY_PARTS, n_reads=n_reads, read_len=READ_LEN,
                                  n_threads=os.cpu_count() or 1)
    ok_, oc_ = A.count_keys(keys, K, n_threads=os.cpu_count() or 1)
    top = 2 * K
    pre = (ok_[:, 0] >> np.uint64(top - PARITY_PBITS)).astype(np.int64)
    ok = n_win == kc.totals()[0]
    n_rec = 0
    for part in PARITY_PARTS:
        first, n = kc.prefix_range(PARITY_PBITS, part)
        gk, gc = kc.counts(first, n)
        m = pre == part
        ok = ok and len(gk) == int(m.sum()) and bool((gk == ok_[m]).all()) and bool((gc.astype(np.uint64) == oc_[m]).all())
        n_rec += n
    return {"what": "CPU oracle over all reads restricted to %d of %d leading-bit partitions vs the device table, record by record"
                    % (len(PARITY_PARTS), 1 << PARITY_PBITS),
            "ok": bool(ok), "records_compared": int(n_rec), "instances_in_sample": int(len(keys)),
            "windows_scanned": int(n_win), "seconds": round(time.perf_counter() - t0, 2)}


DUMP_BLOCKS, DUMP_BLOCK_ROWS, DUMP_SEED = 256, 2048, 2025   # table sample: 256 blocks of 2048 consecutive rows
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, kc, spec, n_instances, n_distinct):
    """What a caller of the timed path receives, as float64 .npy files in out_dir, so that two builds can be compared
    output for output on the same seeded reads:
      spectrum.npy      dense spectrum, index = frequency
      totals.npy        [k-mer instances, distinct k-mers]
      table_rows.npy    row numbers of the sampled records of the sorted (k-mer, count) table
      table_kmers.npy   their k-mers (one word each: 2K = 50 bits, exact in float64)
      table_counts.npy  their counts
    The table (617 M records at the default size) is sampled: DUMP_BLOCKS runs of DUMP_BLOCK_ROWS consecutive rows at
    seeded offsets, one run per equal slice of the table; a table of at most that many rows is written whole.
    With several ranks, the spectrum and totals are global and the table is this rank's shard."""
    assert 2 * K <= 53 and kc.W == 1
    n_rows = kc.totals()[1]
    if n_rows <= DUMP_BLOCKS * DUMP_BLOCK_ROWS:
        starts, size = [0], n_rows
    else:
        rng = np.random.default_rng(DUMP_SEED)
        edges = [n_rows * b // DUMP_BLOCKS for b in range(DUMP_BLOCKS + 1)]
        starts = [lo + int(rng.integers(0, hi - lo - DUMP_BLOCK_ROWS + 1)) for lo, hi in zip(edges, edges[1:])]
        size = DUMP_BLOCK_ROWS
    rows, kmers, counts = [], [], []
    for first in starts:
        k, c = kc.counts(first, size)
        rows.append(np.arange(first, first + size, dtype=np.float64))
        kmers.append(k[:, 0].astype(np.float64))
        counts.append(c.astype(np.float64))
    out = {"spectrum": np.asarray(spec, dtype=np.float64), "totals": np.array([n_instances, n_distinct], dtype=np.float64),
           "table_rows": np.concatenate(rows), "table_kmers": np.concatenate(kmers), "table_counts": np.concatenate(counts)}
    if sum(a.nbytes for a in out.values()) > DUMP_MAX_BYTES:
        raise SystemExit("--dump-outputs: the outputs exceed %d bytes" % DUMP_MAX_BYTES)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_ours(args):
    import torch

    from allpathslg_b200 import KmerCounter, synth_params

    n_gpus = args.gpus
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != n_gpus:
        if world == 1 and n_gpus > 1:
            raise SystemExit("launch with torchrun for --gpus > 1")
        n_gpus = world
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from allpathslg_b200 import dist as shard

    genome = GENOME_PER_GPU * n_gpus
    sp = synth_params(genome, READ_LEN)
    kc = KmerCounter(K, device=local_rank, want_counts=True, reserve_bases=READS_PER_GPU * READ_LEN,
                     async_ingest=True)  # e2e: the level-0 histogram follows the H2D copy slice by slice
    kc.synth_reads(sp, rank * READS_PER_GPU, READS_PER_GPU)
    total_bases, _ = kc.read_store_info()
    if WORKLOAD == "human":   # the shard table grows round by round: give it its room up front
        kc.reserve_table(int(READS_PER_GPU * (READ_LEN - K + 1) * 0.21) + (1 << 20))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def step_resident():
        if world == 1:
            kc.finish()
            return kc.totals()[0], None
        tm = {}
        _, ni, _ = shard.sharded_count(kc, rank, world, timings=tm)
        return ni, tm

    # ---------------- value: inputs resident in HBM
    # nvidia-smi starts BEFORE the warm-up (its NVML initialisation can stall the driver for tens of
    # milliseconds); only the samples taken during the timed region are used
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        step_resident()
    sampler.mark()
    kc.reset_counters()
    stage_acc = {}
    shard_acc = {}
    shard_info = {}
    barrier()
    t0 = time.perf_counter()
    n_inst_total = 0
    for _ in range(args.steps):
        n_inst_total, tm = step_resident()
        for k_, v in kc.stage_ms().items():
            stage_acc[k_] = stage_acc.get(k_, 0.0) + v
        for k_, v in (tm or {}).items():
            if isinstance(v, (int, float)) and not isinstance(v, bool):
                shard_acc[k_] = shard_acc.get(k_, 0.0) + v
            else:
                shard_info[k_] = v
    barrier()
    dt = time.perf_counter() - t0
    launches = kc.kernel_launches()
    clocks = sampler.stop() if rank == 0 else None
    if dist is not None:
        t = torch.tensor([dt], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
    if world == 1:
        n_inst_total = kc.totals()[0]
    per_rank = None
    if dist is not None:   # where the ranks differ: every rank's stage times (rank skew shows up as "reduce" on the fast ranks)
        names = ["scatter0", "scatter1", "owner", "local", "table", "plan", "reduce", "total"]
        mine = torch.tensor([stage_acc.get(n_, 0.0) / args.steps for n_ in names] + [float(kc.totals()[0]), float(kc.totals()[1])],
                            dtype=torch.float64, device="cuda")
        allr = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        per_rank = {n_: [round(float(t[i]), 2) for t in allr] for i, n_ in enumerate(names)}
        per_rank["shard_instances"] = [int(t[len(names)]) for t in allr]
        per_rank["shard_distinct"] = [int(t[len(names) + 1]) for t in allr]
    ms_step = 1e3 * dt / args.steps
    value = n_inst_total / (ms_step * 1e-3) / 1e9
    stage_ms = {k_: v / args.steps for k_, v in stage_acc.items()}
    geo = kc.geometry()
    n_local, nd_local = kc.totals()
    if args.dump_outputs and rank == 0:   # before the e2e region below recounts the same reads
        if world == 1:
            dump_outputs(args.dump_outputs, kc, kc.spectrum(), n_local, nd_local)
        else:
            dump_outputs(args.dump_outputs, kc, kc._group.spectrum(), *kc._group.totals())

    # ---------------- e2e: host buffers through the public API, H2D + D2H inside the timed region
    nbytes = ((total_bases + 31) // 32) * 8
    host = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    kc.export_reads(host.data_ptr())
    spec_bytes = 0

    def step_e2e():
        nonlocal spec_bytes
        kc.reset()
        kc.add_reads_uniform(host.data_ptr(), READS_PER_GPU, READ_LEN)
        if world == 1:
            kc.finish()
            s = kc.spectrum()
        else:
            s, _, _ = shard.sharded_count(kc, rank, world)
        spec_bytes = 65536 * 8
        return s

    step_e2e()
    barrier()
    t0 = time.perf_counter()
    e2e_steps = args.steps
    for _ in range(e2e_steps):
        spec = step_e2e()
    barrier()
    dt_e = time.perf_counter() - t0
    if dist is not None:
        t = torch.tensor([dt_e], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt_e = float(t.item())
    e2e_val = n_inst_total / (dt_e / e2e_steps) / 1e9
    # exact size-independent invariant: sum f * spectrum[f] == instances
    inv_ok = int((spec * np.arange(len(spec), dtype=np.uint64)).sum()) == n_inst_total

    # ---------------- side measurements (N=1 only, after the timed regions; a failure here must never cost the
    # headline line): the frequency of every window of the reads into a device buffer (what error correction
    # asks), then the occurrence records (SortKmers / KmerParcels payload)
    lookups = records = None
    if world == 1 and os.environ.get("APGK_BENCH_LOOKUPS", "1") != "0":
        try:
            lookups = measure_lookups(kc, torch, total_bases)
        except Exception as e:
            lookups = {"error": str(e)[:200]}
    if world == 1 and os.environ.get("APGK_BENCH_RECORDS", "1") != "0":
        try:
            records = measure_records(kc, torch)
        except Exception as e:
            records = {"error": str(e)[:200]}

    # ---------------- sampled-partition parity of THIS workload (N=1): the CPU oracle scans all the reads, keeps the
    # k-mers of 4 of 256 leading-bit partitions, counts them and is compared record by record with the device table
    parity = None
    if world == 1 and os.environ.get("APGK_BENCH_PARITY", "1") != "0":
        try:
            parity = sampled_parity(kc, host, READS_PER_GPU)
        except Exception as e:
            parity = {"error": str(e)[:200]}

    # leave the group in two steps: every rank unmaps the peers' partition buffers, then (after a barrier) frees its own
    grp = getattr(kc, "_group", None)
    if grp is not None:
        kc._group = None
        grp.close()
    if dist is not None:
        dist.barrier()
    if rank != 0:
        kc.close()
        if dist is not None:
            dist.destroy_process_group()
        return 0

    # ---------------- roofline of the dominant kernel (algorithmic bytes, DESIGN.md section 4)
    peak, peak_kind = measured_peaks()
    eb = geo["elem_bytes"]
    n_part = READS_PER_GPU * (READ_LEN - K + 1)   # instances this rank partitions (n_local: instances of the shard it counts)
    alg_bytes = {
        "hist0": total_bases * 0.375,
        "scatter0": total_bases * 0.375 + n_part * 8.0,
        "hist1": n_part * 8.0,
        "scatter1": n_part * (8.0 + eb),
        "local": n_local * float(eb) + nd_local * 12.0,
        "table": nd_local * 24.0,
    }
    kern_names = {"hist0": "k_hist_reads", "scatter0": "k_scatter_reads", "hist1": "k_hist_keys",
                  "scatter1": "k_scatter_keys", "local": "k_local3", "table": "k_compact(+scan)"}
    dom = max(alg_bytes, key=lambda s: stage_ms.get(s, 0.0))
    dom_ms = stage_ms.get(dom, 0.0)
    achieved = alg_bytes[dom] / (dom_ms * 1e-3) / 1e9 if dom_ms > 0 else 0.0
    per_stage = {s: {"ms": round(stage_ms.get(s, 0.0), 3),
                     "alg_GBps": round(alg_bytes[s] / (stage_ms[s] * 1e-3) / 1e9, 1) if stage_ms.get(s, 0) > 0 else None}
                 for s in alg_bytes}
    for s_ in ("scan0", "scan1", "big", "owner"):   # small stages without a byte model: time only
        if stage_ms.get(s_, 0.0) > 0:
            per_stage[s_] = {"ms": round(stage_ms[s_], 3), "alg_GBps": None}
    pipeline_ms = stage_ms.get("total", ms_step)
    stage_sum = sum(v for k_, v in stage_ms.items() if k_ != "total")
    step_traffic = ncu_traffic() if (n_gpus == 1 and READS_PER_GPU == 60_000_000) else None
    # measured DRAM bytes of that kernel: one ncu --set full capture of the N=1 workload, committed under profiles/
    traffic = ncu_traffic(dom) if (n_gpus == 1 and READS_PER_GPU == 60_000_000) else None
    roofline = {"bound": "hbm", "kernel": kern_names[dom], "achieved": round(achieved, 1), "peak": peak,
                "peak_source": peak_kind, "unit": "GB/s", "frac": round(achieved / peak, 4), "traffic": traffic,
                "traffic_source": ("profiles/%s (ncu, separate run)" % traffic_file()) if traffic else None,
                "algorithmic_bytes": int(alg_bytes[dom]),
                "stages": per_stage,
                # the whole step's DRAM traffic as ncu measured it (sum over its kernels) over the step's device time:
                # what the pipeline really draws from HBM -- the figure to read as "fraction of peak"
                "pipeline_actual": ({"dram_bytes_per_step": int(step_traffic),
                                     "GBps": round(step_traffic / (pipeline_ms * 1e-3) / 1e9, 1),
                                     "frac_of_peak": round(step_traffic / (pipeline_ms * 1e-3) / 1e9 / peak, 4),
                                     "source": "profiles/%s" % traffic_file()} if step_traffic else None),
                "device_idle_ms_per_step": round(pipeline_ms - stage_sum, 3) if world == 1 else None,
                # SURVEY.md section 8(d)'s contract figure: a 7-pass LSD sort would move 136 B per instance; this MSD + hash
                # pipeline moves ~40.  "lsd_model_ratio" says how fast a model-conforming sort would have to stream to keep
                # up -- it is NOT an achieved bandwidth and can exceed 1
                "pipeline_model": {"B_alg_bytes_per_kmer": B_ALG_K25,
                                   "lsd_model_equivalent_GBps": round(n_local * B_ALG_K25 / (pipeline_ms * 1e-3) / 1e9, 1),
                                   "lsd_model_ratio": round(n_local * B_ALG_K25 / (pipeline_ms * 1e-3) / 1e9 / peak, 4)}}

    cb_inst, cb_dt, cores = cpu_baseline(CPU_SAMPLE_READS, CPU_SAMPLE_GENOME)
    line = {
        "metric": "k-mer spectrum throughput (K=25), k-mer instances counted per second",
        "value": round(value, 3), "unit": "Gk-mers/s", "n_gpus": n_gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(ms_step, 3),
        "timing": "host clock between barrier + cuda synchronize on both sides (max over ranks); device_ms_per_step and "
                  "roofline.stages are CUDA-event intervals on the library's own stream",
        "device_ms_per_step": round(stage_ms.get("total", 0.0), 3) if world == 1 else None,
        "higher_is_better": True, "scaling": "strong" if WORKLOAD == "human" else "weak", "vs_baseline": None,
        "dtype": "u64", "data": "synthetic", "config": workload_config(n_gpus),
        "e2e": {"value": round(e2e_val, 3), "unit": "Gk-mers/s", "h2d_bytes_per_step": int(nbytes) * n_gpus,
                "d2h_bytes_per_step": int(spec_bytes) * n_gpus, "steps": e2e_steps,
                "d2h": "the spectrum; the sorted (k-mer, count) table stays on the device, where the lookups read it"},
        "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline,
        "cpu_baseline": {"value": round(cb_inst / cb_dt / 1e9, 4), "unit": "Gk-mers/s", "cores": cores, "kind": "port",
                         "sample": cpu_sample_text(cb_inst) + ", oracle port (not the reference's code: parity unpinned)"},
        "geometry": geo, "shard_ms": dict({k_: round(v / args.steps, 2) for k_, v in shard_acc.items()}, **{k_: (list(v) if isinstance(v, tuple) else v) for k_, v in shard_info.items()}) if shard_acc else None,
        "per_rank_ms": per_rank, "records": records, "lookups": lookups, "parity_sample": parity,
        "n_instances": int(n_inst_total), "n_distinct_rank0": int(nd_local),
        "invariant_sum_f_spectrum_eq_instances": bool(inv_ok),
    }
    emit(line)
    kc.close()
    if dist is not None:
        dist.destroy_process_group()
    return 0


_JSON_OUT = None


def _claim_stdout():
    """stdout carries exactly ONE JSON line: libraries that print from C (NCCL's version banner under
    NCCL_DEBUG) get stderr instead -- file descriptor 1 is pointed at stderr and the JSON line goes to a
    duplicate of the original stdout."""
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(line):
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    import faulthandler

    faulthandler.enable()
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="celegans", choices=["celegans", "human"],
                    help="celegans: BASELINE configs[2] per GPU (weak scaling, the default); human: configs[3], the 3 Gb x 45x "
                         "read set split over the GPUs (k-mer-space rounds; meant for --gpus 8)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step to DIR/<name>.npy (float64; see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.workload == "human":
        global READS_PER_GPU, GENOME_PER_GPU, CPU_SAMPLE_GENOME, WORKLOAD
        world = max(1, int(os.environ.get("WORLD_SIZE", args.gpus)))
        WORKLOAD = "human"
        READS_PER_GPU = (1_350_000_000 // world) // 8 * 8
        GENOME_PER_GPU = 3_000_000_000 // world
        CPU_SAMPLE_GENOME = max(READ_LEN, int(3_000_000_000 * (CPU_SAMPLE_READS / 1_350_000_000)))
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
