"""GPU tests of the k-mer affixes on the sharded table (apgk_group_build_affixes, csrc/gaffix.cuh): after
apgk_group_count every rank holds the affix byte of each k-mer its shard owns, taken over ALL ranks' reads.  The groups
are formed by ONE process over N contexts on one GPU, as in tests/test_gpu_group_freqs.py.  Oracle: tests/affix_oracle.c
(oracle A) over the concatenation of every rank's reads with the full oracle table; each shard's rows are picked
from it by key (the oracle is never given a shard's key subset: the other ranks' windows would be missing)."""
import os

import numpy as np
import pytest

import affix_oracle as AO
from test_affixes_cpu import ragged_reads

pytestmark = pytest.mark.gpu

GF_CAP = 4096   # table keys of one coarse bucket k_gaff_place keeps in shared memory (csrc/gfreq.cuh)


def _unpack(p, n):
    q = np.arange(n, dtype=np.int64)
    return (p[q >> 2] >> ((q & 3) * 2).astype(np.uint8)) & np.uint8(3)


def _pack(bases):
    n = len(bases)
    b = np.zeros(((n + 31) // 32) * 32 + 32, dtype=np.uint8)
    b[:n] = bases
    b4 = b.reshape(-1, 4)
    return (b4[:, 0] | (b4[:, 1] << 2) | (b4[:, 2] << 4) | (b4[:, 3] << 6)).astype(np.uint8)


def _concat(parts):
    """[(packed, off), ...] -> one (packed, off) holding the reads of every part in order"""
    bases = [_unpack(p, int(o[-1] - o[0])) for p, o in parts]
    offs, base = [np.zeros(1, dtype=np.uint64)], 0
    for p, o in parts:
        o = np.asarray(o, dtype=np.uint64)
        offs.append(o[1:] - o[0] + np.uint64(base))
        base += int(o[-1] - o[0])
    return _pack(np.concatenate(bases) if bases else np.zeros(0, np.uint8)), np.concatenate(offs)


def _ragged(oracle, sp, r0, n, seed):
    """reads of random lengths 0..180 (some shorter than K) cut from the synthetic reads [r0, r0 + n)"""
    p, o = oracle.synth_reads(sp, r0, n)
    total = int(o[-1])
    rng = np.random.default_rng(seed)
    cuts = np.cumsum(rng.integers(0, 181, size=total // 40 + 2))
    cuts = cuts[cuts < total]
    return p, np.concatenate([[0], cuts, [total]]).astype(np.uint64)


def _ranks(oracle, K, world, n_reads, L=100, genome=200_000, empty_rank=None, ragged_rank=None, **kw):
    """-> (counters, per-rank (packed, off)); rank r holds synthetic reads [share[r], share[r+1])"""
    from allpathslg_b200 import KmerCounter

    sp = oracle.synth_params(genome, L)
    share = [(n_reads * r) // world for r in range(world + 1)]
    if empty_rank is not None:
        share[empty_rank + 1] = share[empty_rank]
    kcs, reads = [], []
    for r in range(world):
        kc = KmerCounter(K, **kw)
        n = share[r + 1] - share[r]
        parts = []
        if n:
            pr, orr = oracle.synth_reads(sp, share[r], n)
            kc.add_reads_uniform(pr, n, L)
            parts.append((pr, orr))
        if r == ragged_rank:
            pg, og = _ragged(oracle, sp, n_reads + 1000, 3000, seed=r)
            kc.add_reads(pg, og)
            parts.append((pg, og))
        kcs.append(kc)
        reads.append(_concat(parts) if parts else (np.zeros(8, np.uint8), np.zeros(1, np.uint64)))
    return kcs, reads


def _rows(a):
    a = np.ascontiguousarray(a, dtype=np.uint64)
    return a.view([("w%d" % i, np.uint64) for i in range(a.shape[1])]).reshape(-1)


def _expected(oracle, reads, K):
    """the oracle's global table over all ranks' reads and the affix byte of each of its rows"""
    p, o = _concat(reads)
    ek, ec, _ = oracle.count(p, o, K)
    return ek, ec, AO.affixes_a(p, o, K, ek)


def _check(kcs, ek, aff):
    """every shard's rows are rows of the oracle's table, the shards together cover it once, and every shard's
    affix bytes equal the oracle's rows.  -> per rank, the shard's row indices in the oracle's table"""
    er = _rows(ek)
    hits = np.zeros(len(ek), dtype=np.int64)
    out = []
    for r, kc in enumerate(kcs):
        gk, _ = kc.counts()
        got = kc.affixes()
        assert len(got) == len(gk)
        idx = np.searchsorted(er, _rows(gk)) if len(gk) else np.zeros(0, np.int64)
        assert (idx < len(ek)).all()
        assert (ek[idx] == gk).all(), "rank %d: a shard key is not in the oracle's table" % r
        bad = np.nonzero(got != aff[idx])[0]
        assert len(bad) == 0, "rank %d: %d of %d rows differ, first row %d (%#x != %#x)" % (
            r, len(bad), len(gk), bad[0], got[bad[0]], aff[idx[bad[0]]])
        hits[idx] += 1
        out.append(idx)
    assert (hits == 1).all(), "the shards do not cover the oracle's table exactly once"
    return out


def _expected_freqs(oracle, reads, K):
    """per rank: the global table (the union of all ranks' reads) applied to the rank's reads, as uint32"""
    p, o = _concat(reads)
    ek, ec, _ = oracle.count(p, o, K)
    out = []
    for pr, orr in reads:
        if int(orr[-1]) == 0:
            out.append(np.zeros(0, np.uint32))
            continue
        f = oracle.read_freqs(pr, orr, K, ek, ec)
        out.append(np.where(f == np.uint64(0xFFFFFFFFFFFFFFFF), np.uint64(0xFFFFFFFF), f).astype(np.uint32))
    return out


def _check_freqs(got, exp):
    assert len(got) == len(exp)
    for r, (g, e) in enumerate(zip(got, exp)):
        assert g.shape == e.shape, (r, g.shape, e.shape)
        bad = np.nonzero(g != e)[0]
        assert len(bad) == 0, "rank %d: %d of %d bases differ, first at %d (%d != %d)" % (
            r, len(bad), len(e), bad[0], g[bad[0]], e[bad[0]])


def _n_windows(off, K):
    lens = np.diff(np.asarray(off, dtype=np.int64))
    return int(np.maximum(lens - K + 1, 0).sum())


def _close(kcs):
    for kc in kcs:
        kc.close()


def _err(fn):
    from allpathslg_b200 import ApgkError

    with pytest.raises(ApgkError) as e:
        fn()
    return e.value.code


@pytest.mark.parametrize("K,world,n_reads,empty,pb,elem", [(25, 2, 30_000, None, 0, 8), (25, 5, 30_000, 2, 0, 8),
                                                           (20, 3, 20_000, None, 0, 4), (25, 8, 40_000, None, 0, 8),
                                                           (31, 2, 12_000, None, 0, 8), (48, 3, 12_000, None, 0, 16),
                                                           (96, 2, 8_000, 0, 0, 24), (25, 1, 10_000, None, 0, 8),
                                                           (25, 3, 30_000, None, 20, 4), (20, 2, 20_000, 1, 16, 4),
                                                           (25, 1, 10_000, None, 20, 4), (26, 3, 30_000, None, 20, 4)])
def test_group_affixes_match_the_oracle(oracle, K, world, n_reads, empty, pb, elem):
    """elem: the level-1 element the windows travel as -- a 4-byte remainder (one u64 slot with the byte) when the
    bits below the P-bit prefix fit (K = 20, or prefix_bits given; REM = 32 at K = 26, P = 20), else the one-word key
    (K = 25 / 31 at these sizes) or the 2- and 3-word keys of K = 48 / 96, with the bytes in a plane of their own."""
    from allpathslg_b200 import KmerGroup

    kcs, reads = _ranks(oracle, K, world, n_reads, empty_rank=empty, prefix_bits=pb)
    ek, _, aff = _expected(oracle, reads, K)
    with KmerGroup.local(kcs) as grp:
        grp.count()
        assert kcs[0].geometry()["elem_bytes"] == elem
        st = grp.build_affixes()
        _check(kcs, ek, aff)
        assert st["n_batches"] == 1
        assert st["n_windows"] == _n_windows(reads[0][1], K)
        if world == 1:
            assert st["remote_bytes"] == 0
        assert st["total_ms"] > 0
    _close(kcs)


@pytest.mark.parametrize("K", [16, 24, 25, 26, 32, 33, 64, 96])
def test_group_affixes_ragged_and_palindromes(oracle, K):
    """Synthetic reads on one rank, ragged ones (empty, shorter than K) on another, and the hand-made strings of the
    single-GPU tests -- poly-A, ACGT and CG repeats, whose palindromes at even K read their neighbours both ways --
    spread over the three ranks."""
    from allpathslg_b200 import KmerGroup

    kcs, reads = _ranks(oracle, K, 3, 6_000, ragged_rank=1)
    strs = ragged_reads(K, 700 + K)
    for r, kc in enumerate(kcs):
        p, o = oracle.pack_strings(strs[r::3])
        kc.add_reads(p, o)
        reads[r] = _concat([reads[r], (p, o)])
    ek, _, aff = _expected(oracle, reads, K)
    if K % 2 == 0:
        assert (AO.revcomp_keys(ek, K) == ek).all(axis=1).any()   # palindromes are present
    with KmerGroup.local(kcs) as grp:
        grp.count()
        grp.build_affixes()
        _check(kcs, ek, aff)
    _close(kcs)


@pytest.mark.parametrize("K,world,n_reads,outer_div,inner_div", [(25, 3, 30_000, 2, 5), (48, 2, 12_000, 2, 4),
                                                                 (20, 4, 20_000, 3, 3), (96, 2, 6_000, 2, 2)])
def test_group_affixes_after_rounds(oracle, K, world, n_reads, outer_div, inner_div):
    """A count in k-mer-space rounds leaves every rank owning one range per inner round (several owned segments):
    a window's byte goes to whichever rank owned its bucket in its round."""
    from allpathslg_b200 import KmerGroup

    per_rank = (n_reads // world) * (100 - K + 1)
    kcs, reads = _ranks(oracle, K, world, n_reads, max_round_keys=per_rank // outer_div + 1,
                        max_inner_keys=per_rank // inner_div + 1)
    ek, _, aff = _expected(oracle, reads, K)
    with KmerGroup.local(kcs) as grp:
        grp.count()
        assert grp.stats()["n_rounds"] >= inner_div
        grp.build_affixes()
        _check(kcs, ek, aff)
    _close(kcs)


@pytest.mark.parametrize("K,world,budget_kb,pb", [(25, 3, 1024, 0), (48, 2, 2048, 0), (25, 2, 64, 0), (20, 3, 256, 0),
                                                  (25, 3, 256, 20)])
def test_group_affixes_in_batches(oracle, K, world, budget_kb, pb, monkeypatch):
    """A pretend device-memory budget far below one batch of the whole store: several exchange batches, whose edges
    cut reads and windows anywhere, give byte-identical affixes to one batch; a rank with a smaller store (fewer
    batches of its own) keeps taking part in every batch."""
    from allpathslg_b200 import KmerGroup

    kcs, reads = _ranks(oracle, K, world, 30_000 if K != 48 else 12_000, ragged_rank=world - 1, prefix_bits=pb)
    ek, _, aff = _expected(oracle, reads, K)
    with KmerGroup.local(kcs) as grp:
        grp.count()
        st1 = grp.build_affixes()
        one = [kc.affixes() for kc in kcs]
        _check(kcs, ek, aff)
        monkeypatch.setenv("APGK_BUDGET_BYTES", str(budget_kb << 10))
        st = grp.build_affixes()
        assert st1["n_batches"] == 1 and st["n_batches"] >= 2
        assert st["n_windows"] == st1["n_windows"]
        for kc, a in zip(kcs, one):
            assert (kc.affixes() == a).all()
    _close(kcs)


def test_group_affixes_large_table_slices(oracle):
    """prefix_bits = 8 with 4-byte remainders (K = 16): some owned coarse buckets hold more table keys than shared
    memory takes (placed through the table in global memory), others fewer (placed in shared memory)."""
    from allpathslg_b200 import KmerGroup

    K = 16
    kcs, reads = _ranks(oracle, K, 2, 30_000, genome=1_000_000, prefix_bits=8)
    ek, _, aff = _expected(oracle, reads, K)
    sizes = np.bincount((ek[:, 0] >> np.uint64(2 * K - 8)).astype(np.int64))
    assert sizes.max() > GF_CAP and sizes.min() < GF_CAP   # both owner paths run
    with KmerGroup.local(kcs) as grp:
        grp.count()
        assert grp.stats()["prefix_bits"] == 8 and kcs[0].geometry()["elem_bytes"] == 4
        grp.build_affixes()
        _check(kcs, ek, aff)
    _close(kcs)


@pytest.mark.parametrize("world", [1, 3, 8])
def test_group_affixes_equal_one_context(world):
    """At a size the oracle is slow for (2 M reads): the shard tables, concatenated in owner order, equal ONE plain
    context's table over the concatenated reads, and so do their affix bytes and apgk_build_affixes's."""
    from allpathslg_b200 import KmerCounter, KmerGroup
    from allpathslg_b200.kmers import synth_params

    K, L, total = 25, 100, 2_000_000
    sp = synth_params(20_000_000, L)
    share = [(total * r) // world for r in range(world + 1)]
    with KmerCounter(K) as one:
        one.synth_reads(sp, 0, total)
        one.finish()
        one.build_affixes()
        rk, _ = one.counts()
        ra = one.affixes()
    kcs = []
    for r in range(world):
        kc = KmerCounter(K)
        kc.synth_reads(sp, share[r], share[r + 1] - share[r])
        kcs.append(kc)
    with KmerGroup.local(kcs) as grp:
        grp.count()
        assert grp.stats()["n_rounds"] == 1
        sts = grp.build_affixes()
        gk = np.concatenate([kc.counts()[0] for kc in kcs])
        ga = np.concatenate([kc.affixes() for kc in kcs])
        assert (gk == rk).all()
        assert (ga == ra).all()
        assert sts["n_windows"] == (share[1] - share[0]) * (L - K + 1)   # rank 0's windows
        if world > 1:
            assert sts["remote_bytes"] > 0
    _close(kcs)


def test_group_affixes_windows_sent_sum_to_the_instances(oracle):
    """n_windows of each rank (read with that rank as the group's first local context) sums to the group's
    n_instances."""
    from allpathslg_b200 import KmerGroup

    K = 25
    kcs, reads = _ranks(oracle, K, 3, 12_000, ragged_rank=2)
    sent = []
    for r in range(3):
        order = kcs[r:] + kcs[:r]
        with KmerGroup.local(order) as grp:
            grp.count()
            sent.append(grp.build_affixes()["n_windows"])
            ni, _ = grp.totals()
    assert sum(sent) == ni
    _close(kcs)


def test_group_affixes_lookups_on_a_shard(oracle):
    """lookup_affixes on a shard: owned k-mers in both orientations give the byte in the query's orientation; k-mers
    that other ranks own give (0, 0), as absent ones do."""
    from allpathslg_b200 import KmerGroup

    K = 25
    kcs, reads = _ranks(oracle, K, 3, 15_000)
    ek, ec, aff = _expected(oracle, reads, K)
    with KmerGroup.local(kcs) as grp:
        grp.count()
        grp.build_affixes()
        idx = _check(kcs, ek, aff)
        for r, kc in enumerate(kcs):
            mine = idx[r][:: max(1, len(idx[r]) // 2000)]
            ga, gc = kc.lookup_affixes(ek[mine])
            assert (ga == aff[mine]).all() and (gc.astype(np.uint64) == ec[mine]).all()
            ga, gc = kc.lookup_affixes(AO.revcomp_keys(ek[mine], K))
            assert (ga == AO.affix_revcomp(aff[mine])).all() and (gc.astype(np.uint64) == ec[mine]).all()
            other = idx[(r + 1) % 3][:500]
            ga, gc = kc.lookup_affixes(ek[other])
            assert (ga == 0).all() and (gc == 0).all()
            ptr, n = kc.affixes_device()
            assert ptr and n == len(idx[r])
    _close(kcs)


def test_group_affixes_state_and_lifetime(oracle):
    """Refusals identical on every rank (before the count, after one rank's context was given reads or reset, and
    apgk_build_affixes on a shard); the affixes survive release_temp and read_freqs (which stays exact: both calls
    use the partition buffers), a build after read_freqs gives the same bytes, and count() or add_reads drop them."""
    from allpathslg_b200 import KmerGroup
    from allpathslg_b200._lib import E_STATE

    K = 25
    kcs, reads = _ranks(oracle, K, 3, 9_000)
    ek, _, aff = _expected(oracle, reads, K)
    exp_f = _expected_freqs(oracle, reads, K)
    with KmerGroup.local(kcs) as grp:
        assert _err(grp.build_affixes) == E_STATE
        grp.count()
        for kc in kcs:
            assert _err(kc.affixes) == E_STATE             # a shard has none before the group build
            assert _err(kc.build_affixes) == E_STATE       # and cannot build its own
        grp.build_affixes()
        _check(kcs, ek, aff)
        for kc in kcs:
            assert _err(kc.build_affixes) == E_STATE
            kc.release_temp()
        _check(kcs, ek, aff)
        _check_freqs(grp.read_freqs(), exp_f)
        _check(kcs, ek, aff)
        grp.build_affixes()
        _check(kcs, ek, aff)
        _check_freqs(grp.read_freqs(), exp_f)
        grp.count()                                        # a new count drops them
        for kc in kcs:
            assert _err(kc.affixes) == E_STATE
        grp.build_affixes()
        _check(kcs, ek, aff)
        p, o = oracle.synth_reads(oracle.synth_params(200_000, 100), 50_000, 10)
        kcs[1].add_reads(p, o)                             # one rank given reads: its affixes go, the build refuses
        assert _err(kcs[1].affixes) == E_STATE
        assert _err(grp.build_affixes) == E_STATE
        grp.count()
        reads[1] = _concat([reads[1], (p, o)])
        ek, _, aff = _expected(oracle, reads, K)
        grp.build_affixes()
        _check(kcs, ek, aff)
        kcs[2].reset()
        assert _err(grp.build_affixes) == E_STATE
    _close(kcs)


def test_group_affixes_refused_without_counts(oracle):
    from allpathslg_b200 import KmerCounter, KmerGroup
    from allpathslg_b200._lib import E_STATE

    kcs, reads = _ranks(oracle, 25, 2, 4_000)
    _close(kcs)
    nk = [KmerCounter(25, want_counts=False) for _ in range(2)]
    for r, kc in enumerate(nk):
        kc.add_reads(*reads[r])
    with KmerGroup.local(nk) as grp:
        grp.count()
        assert _err(grp.build_affixes) == E_STATE
    _close(nk)


# ---------------------------------------------------------------- the benchmark store
READS, READ_LEN, GENOME = 60_000_000, 100, 100_000_000
MIN_FREE_BYTES = 120 << 30


def test_group_affixes_bench_store_one_rank():
    """bench.py's store (60 M x 100 bp synthetic, K = 25) on a one-rank group: the shard's bytes equal
    apgk_build_affixes's on one plain context, and two sampled leading-bit partitions equal the sampled oracle."""
    import torch

    from allpathslg_b200 import KmerCounter, KmerGroup, synth_params
    from oracle import oracle_a as A

    free = torch.cuda.mem_get_info()[0]
    if free < MIN_FREE_BYTES:
        pytest.skip("needs %.0f GiB of free device memory, %.1f GiB free (the card is shared)" % (MIN_FREE_BYTES / 2**30, free / 2**30))
    K = 25
    sp = synth_params(GENOME, READ_LEN)
    with KmerCounter(K, want_counts=True, reserve_bases=READS * READ_LEN) as one:
        one.synth_reads(sp, 0, READS)
        one.finish()
        one.build_affixes()
        ref = one.affixes()
    kc = KmerCounter(K, want_counts=True, reserve_bases=READS * READ_LEN)
    kc.synth_reads(sp, 0, READS)
    with KmerGroup.local([kc]) as grp:
        grp.count()
        st = grp.build_affixes()
        aff = kc.affixes()
        assert st["n_windows"] == READS * (READ_LEN - K + 1)
        assert len(aff) == len(ref) and (aff == ref).all()
        host = kc.export_reads()
        pbits, parts = 10, (77, 700)
        keys, pos, n_win = A.sample_prefix_pos(host, None, K, pbits, parts, n_reads=READS, read_len=READ_LEN,
                                               n_threads=os.cpu_count() or 1)
        assert n_win == st["n_windows"]
        uk, ua = AO.sample_affixes(host, None, K, keys, pos, read_len=READ_LEN)
        del keys, pos
        for part in parts:
            first, n = kc.prefix_range(pbits, part)
            gk, _ = kc.counts(first, n)
            sel = (uk[:, 0] >> np.uint64(2 * K - pbits)) == part
            assert n > 0 and (gk == uk[sel]).all()
            assert (aff[first:first + n] == ua[sel]).all()
    kc.close()
