"""torchrun script: the sharded count behind the C ABI (apgk_group_join / apgk_group_count: NCCL for the small
collectives, CUDA IPC peer memory for the exchange) on real GPUs, against the oracle on the union of all ranks' reads.
Single-round cases and k-mer-space rounds (outer + inner), several K, a second step on the same group; after each
step every rank's frequency lookups on the sharded table (apgk_group_read_freqs_device) for every window of its reads,
against the oracle's global table applied to them, every rank's affixes (apgk_group_build_affixes) for the rows
of its shard, against the affix oracle over all ranks' reads, and every rank's occurrence records
(apgk_group_build_occurrences) for the rows of its shard, against the oracle's records over all ranks' reads (rank r
holds reads [r * n, (r + 1) * n) of one read set, so group read ids are that set's read numbers).

   python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port 29511 tools/dist_check.py
"""
import os
import sys

sys.path.insert(0, ".")
sys.path.insert(0, "tests")
import numpy as np
import torch
import torch.distributed as dist

from allpathslg_b200 import KmerCounter, synth_params
import affix_oracle as AO
from allpathslg_b200.dist import sharded_affixes, sharded_count, sharded_occurrences, sharded_read_freqs
from oracle import oracle_a as A

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))


def rows(a):
    a = np.ascontiguousarray(a, dtype=np.uint64)
    return a.view([("", a.dtype)] * a.shape[1]).reshape(-1)


ok = True
CASES = [  # K, genome, read length, reads per rank, (outer divisor, inner divisor) of a rank's instances or None
    (25, 2_000_000, 100, 400_000, None), (64, 500_000, 250, 40_000, None), (96, 500_000, 150, 60_000, None),
    (20, 300_000, 100, 100_000, None), (25, 2_000_000, 100, 400_000, (2, 5)), (48, 500_000, 150, 60_000, (1, 3)),
]
for (K, G, L, n_per, rounds) in CASES:
    kw = {}
    if rounds:
        per = n_per * (L - K + 1)
        kw = dict(max_round_keys=per // rounds[0] + 1, max_inner_keys=per // rounds[1] + 1)
    kc = KmerCounter(K, device=local, **kw)
    kc.synth_reads(synth_params(G, L), rank * n_per, n_per)
    packed, off = A.synth_reads(A.synth_params(G, L), 0, n_per * world)
    ek, ec, en = A.count(packed, off, K)
    es = A.spectrum(ec)
    er = rows(ek)
    pr, orr = A.synth_reads(A.synth_params(G, L), rank * n_per, n_per)
    erf = A.read_freqs(pr, orr, K, ek, ec)
    erf = np.where(erf == np.uint64(0xFFFFFFFFFFFFFFFF), np.uint64(0xFFFFFFFF), erf).astype(np.uint32)
    eaff = AO.affixes_a(packed, off, K, ek)
    ero, erid, epos = A.occurrences(packed, off, K, ek, en)
    for step in range(2):
        tm = {}
        spec, ni, nd = sharded_count(kc, rank, world, timings=tm)
        gk, gc = kc.counts()
        good = ni == en and nd == len(ek) and len(spec) == len(es) and bool((spec == es).all())
        good = good and (tm["n_rounds"] >= rounds[1] if rounds else tm["n_rounds"] == 1)
        hits = np.zeros(len(ek), dtype=np.int64)
        afs = {}
        gaff = sharded_affixes(kc, rank, world, stats=afs)
        aff_ok = len(gaff) == len(gk)
        ocs = {}
        gro, grid_, gpos = sharded_occurrences(kc, rank, world, stats=ocs)
        occ_ok = len(gro) == len(gk) + 1 and len(grid_) == ocs["n_occ"]
        if len(gk):
            idx = np.searchsorted(er, rows(gk))
            good = good and bool((idx < len(er)).all())
            idx = np.minimum(idx, len(er) - 1)
            good = good and bool((er[idx] == rows(gk)).all()) and bool((ec[idx] == gc.astype(np.uint64)).all()) and bool((np.diff(idx) > 0).all())
            hits[idx] += 1
            aff_ok = aff_ok and bool((gaff == eaff[idx]).all())
            lens = (ero[idx + 1] - ero[idx]).astype(np.int64)
            occ_ok = occ_ok and bool((np.diff(gro.astype(np.int64)) == lens).all())
            if occ_ok:
                sel = np.repeat(ero[idx].astype(np.int64), lens) + (np.arange(len(grid_)) - np.repeat(gro[:-1].astype(np.int64), lens))
                occ_ok = bool((grid_ == erid[sel]).all()) and bool((gpos == epos[sel]).all())
        fst = {}
        freqs_ok = bool((sharded_read_freqs(kc, rank, world, stats=fst) == erf).all())
        good = good and freqs_ok and aff_ok and occ_ok
        t = torch.from_numpy(hits).cuda()
        dist.all_reduce(t)
        good = good and bool((t == 1).all().item())   # every k-mer of the oracle sits in exactly one shard
        f = torch.tensor([1 if good else 0], device="cuda")
        dist.all_reduce(f, op=dist.ReduceOp.MIN)
        if rank == 0:
            print("K=%d world=%d step=%d instances=%d distinct=%d all-ranks-ok=%s  (%s, rounds %d/%d, P=%d+%d; rank0: shard %d, "
                  "remote %.1f MB in %.3f ms = %.1f GB/s, step %.2f ms; read-freqs rank0 %s, %.1f MB remote, %.2f ms; "
                  "affixes rank0 %s, %.1f MB remote, %.2f ms; occurrences rank0 %s, %.1f MB remote, %.2f ms)" %
                  (K, world, step, ni, nd, bool(f.item()), tm["path"], tm["n_outer_rounds"], tm["n_rounds"], tm["prefix_bits"],
                   tm["split_bits"], tm["shard_instances"], tm["remote_bytes"] / 1e6, tm["gather_ms"], tm["gather_remote_GBps"],
                   tm["step_ms"], freqs_ok, fst["remote_bytes"] / 1e6, fst["total_ms"], aff_ok, afs["remote_bytes"] / 1e6,
                   afs["total_ms"], occ_ok, ocs["remote_bytes"] / 1e6, ocs["total_ms"]), flush=True)
        ok = ok and bool(f.item())
    kc._group.close()
    dist.barrier()   # every rank has unmapped the peers' buffers before anyone frees its own
    kc.close()
dist.barrier()
dist.destroy_process_group()
if rank == 0:
    print("DIST CHECK", "OK" if ok else "FAILED")
sys.exit(0 if ok else 1)
