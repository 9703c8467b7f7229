"""GPU tests of the occurrence records on the sharded table (apgk_group_build_occurrences, csrc/gocc.cuh): after
apgk_group_count every rank holds the records (group read id, signed position) of each k-mer its shard owns, taken over
ALL ranks' reads.  The groups are formed by ONE process over N contexts on one GPU, as in
tests/test_gpu_group_affixes.py.  Oracle: oracle_a.occurrences over the concatenation of every rank's reads (group read
ids are the read numbers of that concatenation) with the full oracle table; each shard's rows are picked from it by key."""
import os

import numpy as np
import pytest

from test_affixes_cpu import ragged_reads
from test_gpu_group_affixes import _close, _concat, _err, _n_windows, _ranks, _rows

pytestmark = pytest.mark.gpu

OCC_PLACE_CAP = 2048   # table keys of one coarse bucket k_gocc_place keeps in shared memory (csrc/occ.cuh)


def _expected(oracle, reads, K):
    """the oracle's global table over all ranks' reads and the records of each of its rows"""
    p, o = _concat(reads)
    ek, ec, en = oracle.count(p, o, K)
    ro, rid, pos = oracle.occurrences(p, o, K, ek, en)
    return ek, ec, ro, rid, pos


def _check(kcs, exp):
    """every shard's rows are rows of the oracle's table with the oracle's records, and the shards together cover the
    oracle's instances exactly once.  -> per rank, the shard's (run_off, read_id, pos)"""
    ek, ec, ero, erid, epos = exp
    er = _rows(ek)
    hits = np.zeros(len(ek), dtype=np.int64)
    out = []
    for r, kc in enumerate(kcs):
        gk, gc = kc.counts()
        ro, rid, pos = kc.occurrences()
        assert len(ro) == len(gk) + 1 and int(ro[-1]) == int(gc.astype(np.int64).sum())
        assert kc.occurrences_info()["n_occ"] == len(rid) == kc.totals()[0]
        idx = np.searchsorted(er, _rows(gk)) if len(gk) else np.zeros(0, np.int64)
        assert (idx < len(ek)).all()
        assert (ek[idx] == gk).all(), "rank %d: a shard key is not in the oracle's table" % r
        lens = (ero[idx + 1] - ero[idx]).astype(np.int64)
        assert (np.diff(ro.astype(np.int64)) == lens).all(), "rank %d: run lengths differ" % r
        sel = np.repeat(ero[idx].astype(np.int64), lens) + (np.arange(len(rid)) - np.repeat(ro[:-1].astype(np.int64), lens))
        bad = np.nonzero((rid != erid[sel]) | (pos != epos[sel]))[0]
        assert len(bad) == 0, "rank %d: %d of %d records differ, first slot %d ((%d, %d) != (%d, %d))" % (
            r, len(bad), len(rid), bad[0], rid[bad[0]], pos[bad[0]], erid[sel[bad[0]]], epos[sel[bad[0]]])
        hits[idx] += 1
        out.append((ro, rid, pos))
    assert (hits == 1).all(), "the shards do not cover the oracle's table exactly once"
    return out


@pytest.mark.parametrize("K,world,n_reads,empty,pb,elem", [(20, 3, 20_000, None, 0, 4), (25, 2, 30_000, None, 0, 8),
                                                           (25, 8, 40_000, None, 0, 8), (31, 2, 12_000, None, 0, 8),
                                                           (33, 3, 12_000, None, 0, 16), (48, 3, 12_000, None, 0, 16),
                                                           (96, 2, 8_000, 0, 0, 24), (25, 1, 10_000, None, 0, 8),
                                                           (25, 3, 30_000, 1, 20, 4), (20, 2, 20_000, None, 16, 4),
                                                           (25, 1, 10_000, None, 20, 4), (26, 3, 30_000, None, 20, 4)])
def test_group_occurrences_match_the_oracle(oracle, K, world, n_reads, empty, pb, elem):
    """elem: the level-1 element the windows travel as -- a 4-byte remainder (K = 20, or prefix_bits given; REM = 32
    at K = 26, P = 20), else the one-word key (K = 25 / 31 at these sizes) or the 2- and 3-word keys of K = 33, 48 and
    96; the records travel in a u64 plane behind the elements either way."""
    from allpathslg_b200 import KmerGroup

    kcs, reads = _ranks(oracle, K, world, n_reads, empty_rank=empty, prefix_bits=pb)
    exp = _expected(oracle, reads, K)
    with KmerGroup.local(kcs) as grp:
        grp.count()
        assert kcs[0].geometry()["elem_bytes"] == elem
        st = grp.build_occurrences()
        _check(kcs, exp)
        assert st["n_batches"] == 1
        assert st["n_windows"] == _n_windows(reads[0][1], K)
        assert st["n_occ"] == kcs[0].totals()[0]
        if world == 1:
            assert st["remote_bytes"] == 0
        assert st["total_ms"] > 0
        assert sum(kc.totals()[0] for kc in kcs) == len(exp[3]) == sum(_n_windows(o, K) for _, o in reads)
    _close(kcs)


@pytest.mark.parametrize("K", [16, 24, 25, 32, 33, 64])
def test_group_occurrences_ragged_and_palindromes(oracle, K):
    """Synthetic reads on one rank, ragged ones (empty, shorter than K) on another, and the hand-made strings of the
    single-GPU tests -- poly-A, ACGT and CG repeats, palindromes at even K -- spread over the three ranks."""
    from allpathslg_b200 import KmerGroup
    from test_gpu_group_affixes import AO

    kcs, reads = _ranks(oracle, K, 3, 6_000, ragged_rank=1)
    strs = ragged_reads(K, 700 + K)
    for r, kc in enumerate(kcs):
        p, o = oracle.pack_strings(strs[r::3])
        kc.add_reads(p, o)
        reads[r] = _concat([reads[r], (p, o)])
    exp = _expected(oracle, reads, K)
    if K % 2 == 0:
        assert (AO.revcomp_keys(exp[0], K) == exp[0]).all(axis=1).any()   # palindromes are present
    with KmerGroup.local(kcs) as grp:
        grp.count()
        grp.build_occurrences()
        _check(kcs, exp)
    _close(kcs)


def test_group_occurrences_rank_without_reads_and_empty_reads(oracle):
    """Rank 1 holds no reads at all, rank 2 only empty and too-short reads between real ones: group read ids still
    count every read of every rank in rank order."""
    from allpathslg_b200 import KmerCounter, KmerGroup

    K = 25
    strs = [["ACGTTGCAAGGCTTAACCGGTTAACGTAGCTAGCTAGGATCCAT", "", "ACGTACGTAC"],
            [],
            ["", "", "TTTTGGGGCCCCAAAATTTTGGGGCCCCAAAATTTTGGGG", "ACG", "", "ACGTTGCAAGGCTTAACCGGTTAACGTAGCTAG", ""]]
    kcs, reads = [], []
    for s in strs:
        kc = KmerCounter(K)
        if s:
            p, o = oracle.pack_strings(s)
            kc.add_reads(p, o)
            reads.append((p, o))
        else:
            reads.append((np.zeros(8, np.uint8), np.zeros(1, np.uint64)))
        kcs.append(kc)
    exp = _expected(oracle, reads, K)
    with KmerGroup.local(kcs) as grp:
        grp.count()
        grp.build_occurrences()
        _check(kcs, exp)
    _close(kcs)


@pytest.mark.parametrize("world", [1, 3])
def test_group_occurrences_long_runs(oracle, world):
    """Poly-A and a short repeat: runs of more than 256 instances (k_occ_sort_big in shared memory) and more than 4096
    (in place), each filled from several ranks' pieces."""
    from allpathslg_b200 import KmerCounter, KmerGroup

    K = 25
    strs = ["A" * 3000, "A" * 2500 + "C" * 40, "ACG" * 1500, "A" * 600, "T" * 900]
    kcs, reads = [], []
    for r in range(world):
        kc = KmerCounter(K)
        p, o = oracle.pack_strings(strs[r::world])
        kc.add_reads(p, o)
        kcs.append(kc)
        reads.append((p, o))
    exp = _expected(oracle, reads, K)
    ro = exp[2].astype(np.int64)
    assert np.diff(ro).max() > 4096 and ((np.diff(ro) > 256) & (np.diff(ro) <= 4096)).any()
    with KmerGroup.local(kcs) as grp:
        grp.count()
        st = grp.build_occurrences()
        _check(kcs, exp)
        assert sum(kc.occurrences_info()["n_big_runs"] for kc in kcs) >= 2
        if world == 1:
            assert st["n_big_runs"] >= 2
    _close(kcs)


@pytest.mark.parametrize("K,world,n_reads,outer_div,inner_div", [(25, 3, 30_000, 2, 5), (48, 2, 12_000, 2, 4),
                                                                 (20, 4, 20_000, 3, 3), (96, 2, 6_000, 2, 2)])
def test_group_occurrences_after_rounds(oracle, K, world, n_reads, outer_div, inner_div):
    """A count in k-mer-space rounds leaves every rank owning one range per inner round: a window's record goes to
    whichever rank owned its bucket in its round."""
    from allpathslg_b200 import KmerGroup

    per_rank = (n_reads // world) * (100 - K + 1)
    kcs, reads = _ranks(oracle, K, world, n_reads, max_round_keys=per_rank // outer_div + 1,
                        max_inner_keys=per_rank // inner_div + 1)
    exp = _expected(oracle, reads, K)
    with KmerGroup.local(kcs) as grp:
        grp.count()
        assert grp.stats()["n_rounds"] >= inner_div
        grp.build_occurrences()
        _check(kcs, exp)
    _close(kcs)


@pytest.mark.parametrize("K,world,budget_kb,pb", [(25, 3, 1024, 0), (48, 2, 2048, 0), (25, 2, 64, 0), (20, 3, 256, 0),
                                                  (25, 3, 256, 20)])
def test_group_occurrences_in_batches(oracle, K, world, budget_kb, pb, monkeypatch):
    """A pretend device-memory budget far below one batch of the whole store: several exchange batches, whose edges
    cut reads anywhere, give byte-identical device records to one batch."""
    import torch

    from allpathslg_b200 import KmerGroup
    from test_gpu_wide_positions import _device_array

    kcs, reads = _ranks(oracle, K, world, 30_000 if K != 48 else 12_000, ragged_rank=world - 1, prefix_bits=pb)
    exp = _expected(oracle, reads, K)

    def device_records():
        out = []
        for kc in kcs:
            _, d_occ, n = kc.occurrences_device()
            out.append(_device_array(d_occ, n, "<i8").clone() if n else torch.zeros(0, dtype=torch.int64, device="cuda"))
        return out

    with KmerGroup.local(kcs) as grp:
        grp.count()
        st1 = grp.build_occurrences()
        one = device_records()
        _check(kcs, exp)
        monkeypatch.setenv("APGK_BUDGET_BYTES", str(budget_kb << 10))
        st = grp.build_occurrences()
        assert st1["n_batches"] == 1 and st["n_batches"] >= 3
        assert st["n_windows"] == st1["n_windows"]
        for a, b in zip(one, device_records()):
            assert torch.equal(a, b)
        _check(kcs, exp)
    _close(kcs)


def test_group_occurrences_large_table_slices(oracle):
    """prefix_bits = 8 with 4-byte remainders (K = 16): some owned coarse buckets hold more table keys than shared
    memory takes (placed through the table in global memory), others fewer (placed in shared memory)."""
    from allpathslg_b200 import KmerGroup

    K = 16
    kcs, reads = _ranks(oracle, K, 2, 30_000, genome=1_000_000, prefix_bits=8)
    exp = _expected(oracle, reads, K)
    sizes = np.bincount((exp[0][:, 0] >> np.uint64(2 * K - 8)).astype(np.int64))
    assert sizes.max() > OCC_PLACE_CAP and sizes.min() < OCC_PLACE_CAP   # both owner paths run
    with KmerGroup.local(kcs) as grp:
        grp.count()
        assert grp.stats()["prefix_bits"] == 8 and kcs[0].geometry()["elem_bytes"] == 4
        grp.build_occurrences()
        _check(kcs, exp)
    _close(kcs)


@pytest.mark.parametrize("world", [1, 3])
def test_group_occurrences_equal_one_context(world):
    """At a size the oracle is slow for (2 M reads): one rank's device records are byte-identical to one context's
    records decoded through apgk_occurrences_copy; with 3 ranks every shard's host copy equals one context's
    apgk_build_occurrences over the concatenated reads."""
    from allpathslg_b200 import KmerCounter, KmerGroup
    from allpathslg_b200.kmers import synth_params
    from test_gpu_wide_positions import _device_array

    K, L, total = 25, 100, 2_000_000
    sp = synth_params(20_000_000, L)
    share = [(total * r) // world for r in range(world + 1)]
    with KmerCounter(K) as one:
        one.synth_reads(sp, 0, total)
        one.finish()
        one.build_occurrences()
        rk, _ = one.counts()
        rro, rrid, rpos = one.occurrences()
    kcs = []
    for r in range(world):
        kc = KmerCounter(K)
        kc.synth_reads(sp, share[r], share[r + 1] - share[r])
        kcs.append(kc)
    with KmerGroup.local(kcs) as grp:
        grp.count()
        st = grp.build_occurrences()
        assert st["n_windows"] == (share[1] - share[0]) * (L - K + 1)
        if world == 1:
            _, d_occ, n = kcs[0].occurrences_device()
            dev = _device_array(d_occ, n, "<i8").cpu().numpy().view(np.uint64)
            p1 = np.abs(rpos).astype(np.uint64)
            enc = (rrid.astype(np.uint64) << np.uint64(32)) | ((p1 - np.uint64(1)) << np.uint64(1)) | (rpos < 0).astype(np.uint64)
            assert n == len(enc) and (dev == enc).all()
        else:
            assert st["remote_bytes"] > 0
        gk = np.concatenate([kc.counts()[0] for kc in kcs])
        assert (gk == rk).all()
        base = 0
        for kc in kcs:
            ro, rid, pos = kc.occurrences()
            n = len(ro) - 1
            assert (ro == rro[base:base + n + 1] - rro[base]).all()
            a, b = int(rro[base]), int(rro[base + n])
            assert (rid == rrid[a:b]).all() and (pos == rpos[a:b]).all()
            base += n
        assert base == len(rk)
    _close(kcs)


def test_group_occurrences_state_and_lifetime(oracle):
    """Refusals identical on every rank (before the count, after one rank's context was given reads or reset, and
    apgk_build_occurrences on a shard); the records survive the group lookups and affixes, and release_temp or a new
    count drop them."""
    from allpathslg_b200 import KmerGroup
    from allpathslg_b200._lib import E_STATE
    from test_gpu_group_affixes import _expected_freqs, _check_freqs

    K = 25
    kcs, reads = _ranks(oracle, K, 3, 9_000)
    exp = _expected(oracle, reads, K)
    exp_f = _expected_freqs(oracle, reads, K)
    with KmerGroup.local(kcs) as grp:
        assert _err(grp.build_occurrences) == E_STATE
        grp.count()
        for kc in kcs:
            assert _err(kc.occurrences) == E_STATE            # a shard has none before the group build
            assert _err(kc.build_occurrences) == E_STATE      # and cannot build its own
        grp.build_occurrences()
        _check(kcs, exp)
        for kc in kcs:
            assert _err(kc.build_occurrences) == E_STATE
        _check_freqs(grp.read_freqs(), exp_f)
        grp.build_affixes()
        _check(kcs, exp)                                      # both leave the records alone
        for kc in kcs:
            kc.release_temp()
            assert _err(kc.occurrences) == E_STATE            # release_temp drops them, as on one GPU
        grp.build_occurrences()                               # and a build after it works
        _check(kcs, exp)
        grp.count()                                           # a new count drops them
        for kc in kcs:
            assert _err(kc.occurrences) == E_STATE
        grp.build_occurrences()
        _check(kcs, exp)
        p, o = oracle.synth_reads(oracle.synth_params(200_000, 100), 50_000, 10)
        kcs[1].add_reads(p, o)                                # one rank given reads: its records go, the build refuses
        assert _err(kcs[1].occurrences) == E_STATE
        assert _err(grp.build_occurrences) == E_STATE
        grp.count()
        reads[1] = _concat([reads[1], (p, o)])
        exp = _expected(oracle, reads, K)
        grp.build_occurrences()
        _check(kcs, exp)
        kcs[2].reset()
        assert _err(grp.build_occurrences) == E_STATE
    _close(kcs)


def test_group_occurrences_refused_without_counts(oracle):
    from allpathslg_b200 import KmerCounter, KmerGroup
    from allpathslg_b200._lib import E_STATE

    kcs, reads = _ranks(oracle, 25, 2, 4_000)
    _close(kcs)
    nk = [KmerCounter(25, want_counts=False) for _ in range(2)]
    for r, kc in enumerate(nk):
        kc.add_reads(*reads[r])
    with KmerGroup.local(nk) as grp:
        grp.count()
        assert _err(grp.build_occurrences) == E_STATE
    _close(nk)


# ---------------------------------------------------------------- the benchmark store
READS, READ_LEN, GENOME = 60_000_000, 100, 100_000_000
MIN_FREE_BYTES = 120 << 30
SLOT32 = 1 << 32


def test_group_occurrences_bench_store_one_rank():
    """bench.py's store (60 M x 100 bp synthetic, K = 25, 4.56 G instances) on a one-rank group: shard slots pass
    2^32; the records of sampled leading-bit partitions -- one of them the partition holding slot 2^32 -- equal the
    sampled oracle's instances translated to read ids."""
    import torch

    from allpathslg_b200 import KmerCounter, KmerGroup, synth_params
    from oracle import oracle_a as A
    from test_gpu_wide_positions import _device_array

    free = torch.cuda.mem_get_info()[0]
    if free < MIN_FREE_BYTES:
        pytest.skip("needs %.0f GiB of free device memory, %.1f GiB free (the card is shared)" % (MIN_FREE_BYTES / 2**30, free / 2**30))
    K, pbits = 25, 10
    sp = synth_params(GENOME, READ_LEN)
    kc = KmerCounter(K, want_counts=True, reserve_bases=READS * READ_LEN)
    kc.synth_reads(sp, 0, READS)
    with KmerGroup.local([kc]) as grp:
        grp.count()
        st = grp.build_occurrences()
        ni, nd = kc.totals()
        assert st["n_occ"] == ni == READS * (READ_LEN - K + 1) and ni > SLOT32
        d_off, _, _ = kc.occurrences_device()
        run_off = _device_array(d_off, nd + 1, "<i8")
        row = int(torch.searchsorted(run_off, torch.tensor([SLOT32], dtype=torch.int64, device="cuda"), right=True)[0]) - 1
        del run_off
        torch.cuda.empty_cache()
        k, _ = kc.counts(row, 1)
        hi_part = int(k[0, 0] >> np.uint64(2 * K - pbits))
        parts = tuple(sorted({77, hi_part}))
        host = kc.export_reads()
        keys, qpos, n_win = A.sample_prefix_pos(host, None, K, pbits, parts, n_reads=READS, read_len=READ_LEN,
                                                n_threads=os.cpu_count() or 1)
        assert n_win == st["n_windows"]
        top = (keys[:, 0] >> np.uint64(2 * K - pbits)).astype(np.int64)
        for part in parts:
            first, n = kc.prefix_range(pbits, part)
            ro, rid, pos = kc.occurrences(first, n)
            sel = top == part
            pk, pq = keys[sel], qpos[sel]
            order = np.lexsort((pq, pk[:, 0]))               # by k-mer, then by position: the order of the runs
            pk, pq = pk[order], pq[order]
            q = (pq >> np.uint64(1)).astype(np.int64)
            p1 = (q % READ_LEN + 1).astype(np.int32)
            gk, gc = kc.counts(first, n)
            assert n > 0 and (np.diff(ro.astype(np.int64)) == gc.astype(np.int64)).all()
            assert len(rid) == len(pq) and (np.repeat(gk[:, 0], gc.astype(np.int64)) == pk[:, 0]).all()
            assert (rid == (q // READ_LEN).astype(np.uint32)).all()
            assert (pos == np.where(pq & np.uint64(1), -p1, p1)).all()
        a, _ = kc.prefix_range(pbits, hi_part)
        print("\n[bench store] %d records, %d batches, total %.1f ms (sweep %.1f, exchange %.1f, sort %.1f); "
              "partitions %s, the second starting at row %d" % (ni, st["n_batches"], st["total_ms"], st["sweep_ms"],
                                                                st["exchange_ms"], st["sort_ms"], parts, a))
    kc.close()
