"""GPU parity tests of the sharded path behind the C ABI (apgk_group_*, csrc/group.cuh): the N-rank pipeline --
partition, all-gather of the bucket histograms, balanced ranges, gather over (peer) memory with sender-side
sub-bucket counts, per-bucket counting, spectrum reduction, k-mer-space rounds -- driven by ONE process over N
contexts on one GPU (the single-process form of the group; the same phase machine serves the NCCL form, which
tools/dist_check.py runs on real GPUs).  Everything is compared with the CPU oracle on the union of the reads.

Parity is UNPINNED in the sense of SURVEY.md section 8(c) (spec-derived oracle; no reference source)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _rows(a):
    a = np.ascontiguousarray(a, dtype=np.uint64)
    return a.view([("", a.dtype)] * a.shape[1]).reshape(-1)


def _make_ranks(oracle, K, world, n_reads, L=100, genome=200_000, empty_rank=None, **kw):
    from allpathslg_b200 import KmerCounter

    sp = oracle.synth_params(genome, L)
    share = [(n_reads * r) // world for r in range(world + 1)]
    if empty_rank is not None:
        share[empty_rank + 1] = share[empty_rank]
    kcs = []
    for r in range(world):
        kc = KmerCounter(K, **kw)
        n = share[r + 1] - share[r]
        if n:
            pr, _ = oracle.synth_reads(sp, share[r], n)
            kc.add_reads_uniform(pr, n, L)
        kcs.append(kc)
    p, o = oracle.synth_reads(sp, 0, share[-1])
    return kcs, p, o


def _check_against_oracle(oracle, grp, kcs, p, o, K, sorted_by_rank):
    ek, ec, en = oracle.count(p, o, K)
    es = oracle.spectrum(ec)
    ni, nd = grp.totals()
    assert (ni, nd) == (en, len(ek))
    gs = grp.spectrum()
    assert len(gs) == len(es) and (gs == es).all()
    # every oracle k-mer sits in exactly one shard table, with the oracle's count; shard tables are sorted
    hits = np.zeros(len(ek), dtype=np.int64)
    er = _rows(ek)
    tabs = []
    for kc in kcs:
        gk, gc = kc.counts()
        tabs.append((gk, gc))
        if len(gk) == 0:
            continue
        gr = _rows(gk)
        idx = np.searchsorted(er, gr)   # structured comparison is lexicographic by word: the table's order
        assert (idx < len(er)).all() and (er[idx] == gr).all()
        assert (ec[idx] == gc.astype(np.uint64)).all()
        assert (np.diff(idx) > 0).all()
        hits[idx] += 1
        assert kc.totals() == (int(gc.astype(np.uint64).sum()), len(gk))
    assert (hits == 1).all()
    if sorted_by_rank:   # one round: rank r owns the r-th contiguous range of k-mer space
        gk = np.concatenate([t[0] for t in tabs])
        assert (gk == ek).all()
    # shard tables answer lookups for their own k-mers only
    pick = ek[:: max(1, len(ek) // 400)]
    exp = ec[:: max(1, len(ek) // 400)]
    tot = np.zeros(len(pick), dtype=np.uint64)
    for kc in kcs:
        tot += kc.lookup(pick, canonicalise=False).astype(np.uint64)
    assert (tot == exp).all()
    return ek, ec, en


@pytest.mark.parametrize("bucket_cost", [None, 0])
@pytest.mark.parametrize("K,world,n_reads,empty", [(25, 2, 30_000, None), (25, 5, 30_000, 2), (20, 3, 20_000, None),
                                                   (25, 8, 40_000, None), (31, 2, 12_000, None), (48, 3, 12_000, None),
                                                   (96, 2, 8_000, 0), (25, 1, 10_000, None)])
def test_group_single_round(oracle, K, world, n_reads, empty, bucket_cost, monkeypatch):
    """bucket_cost None: the default balance of the owned ranges (by cost: keys + a charge per bucket); 0: by
    instance count alone, which must then be even up to the bucket granularity."""
    from allpathslg_b200 import KmerGroup

    if bucket_cost is not None:
        monkeypatch.setenv("APGK_BUCKET_COST", str(bucket_cost))
    kcs, p, o = _make_ranks(oracle, K, world, n_reads, empty_rank=empty)
    with KmerGroup.local(kcs) as grp:
        grp.count()
        st = grp.stats()
        assert st["world"] == world and st["n_rounds"] == 1
        ek, ec, en = _check_against_oracle(oracle, grp, kcs, p, o, K, sorted_by_rank=True)
        per_rank = [kc.totals()[0] for kc in kcs]
        if world > 1 and en > 10 * world and bucket_cost == 0:
            assert max(per_rank) < 1.25 * en / world + (en >> st["prefix_bits"]) * 64   # balanced up to bucket granularity
        # a second step over the same stores (steady state: buffers, mappings and the table's capacity are reused)
        grp.count()
        _check_against_oracle(oracle, grp, kcs, p, o, K, sorted_by_rank=True)
    for kc in kcs:
        kc.close()


@pytest.mark.parametrize("K,prefix_bits,world,n_reads", [(26, 20, 1, 10_000), (26, 20, 3, 30_000)])
def test_group_32bit_remainders_using_every_bit(oracle, K, prefix_bits, world, n_reads):
    """prefix_bits = 2K - 32: the ranks exchange 4-byte remainders that use all 32 bits.  With several ranks the
    gather splits them by their top split bits and the shards count the rest; one rank counts all 32 bits itself
    (k_local2, not k_local3, which stops at REM = 31)."""
    from allpathslg_b200 import KmerGroup

    kcs, p, o = _make_ranks(oracle, K, world, n_reads, prefix_bits=prefix_bits)
    with KmerGroup.local(kcs) as grp:
        grp.count()
        g, st = kcs[0].geometry(), grp.stats()
        assert st["prefix_bits"] == prefix_bits and g["elem_bytes"] == 4
        assert g["REM"] == 2 * K - prefix_bits - st["split_bits"]
        _check_against_oracle(oracle, grp, kcs, p, o, K, sorted_by_rank=True)
    for kc in kcs:
        kc.close()


@pytest.mark.parametrize("gather", ["direct", "pipelined"])
@pytest.mark.parametrize("K,world,n_reads,outer_div,inner_div", [(25, 3, 30_000, 2, 5), (25, 2, 30_000, 1, 3), (48, 2, 12_000, 2, 4),
                                                                 (20, 4, 20_000, 3, 3), (96, 2, 6_000, 2, 2)])
def test_group_rounds(oracle, K, world, n_reads, outer_div, inner_div, gather, monkeypatch):
    """K-mer-space rounds of the sharded form: outer rounds (one filtered extraction each) cut into inner rounds
    (level 1 + exchange + counting); every round's shard table is appended, so the contexts end up with all the
    k-mers they own.  Both gather kernels (direct peer loads; cp.async-pipelined through shared memory)."""
    from allpathslg_b200 import KmerGroup

    monkeypatch.setenv("APGK_GATHER", gather)

    L = 100
    per_rank = (n_reads // world) * (L - K + 1)
    kcs, p, o = _make_ranks(oracle, K, world, n_reads, L=L, max_round_keys=per_rank // outer_div + 1,
                            max_inner_keys=per_rank // inner_div + 1)
    with KmerGroup.local(kcs) as grp:
        grp.count()
        st = grp.stats()
        assert st["n_rounds"] >= inner_div and st["n_outer_rounds"] >= outer_div
        _check_against_oracle(oracle, grp, kcs, p, o, K, sorted_by_rank=False)
        # the appended table keeps its prefix index: parcels of k-mer space can be read off every shard
        ek, ec, _ = oracle.count(p, o, K)
        if K == 25:
            top = 2 * K
            pre = (ek[:, 0] >> np.uint64(top - 6)).astype(np.int64)
            for part in (0, 7, 33, 63):
                got = []
                for kc in kcs:
                    first, n = kc.prefix_range(6, part)
                    got.append(kc.counts(first, n))
                gk = np.concatenate([g[0] for g in got]); gc = np.concatenate([g[1] for g in got])
                order = np.argsort(gk[:, 0], kind="stable")
                assert (gk[order] == ek[pre == part]).all() and (gc[order].astype(np.uint64) == ec[pre == part]).all()
    for kc in kcs:
        kc.close()


@pytest.mark.parametrize("K,world,n_reads,budget_mb", [(25, 3, 60_000, 40), (25, 2, 60_000, 24), (48, 2, 20_000, 10)])
def test_group_rounds_sized_from_the_memory_budget(oracle, K, world, n_reads, budget_mb, monkeypatch):
    """No round sizes given: the group cuts outer and inner rounds from the device-memory budget of its tightest rank
    (here a pretend budget, far below what the k-mers need at once)."""
    from allpathslg_b200 import KmerGroup

    monkeypatch.setenv("APGK_BUDGET_BYTES", str(budget_mb << 20))
    kcs, p, o = _make_ranks(oracle, K, world, n_reads)
    with KmerGroup.local(kcs) as grp:
        grp.count()
        st = grp.stats()
        assert st["n_rounds"] >= 2
        _check_against_oracle(oracle, grp, kcs, p, o, K, sorted_by_rank=False)
    for kc in kcs:
        kc.close()


def test_group_counts_beyond_the_dense_spectrum(oracle):
    """A k-mer seen more than 65535 times lives in one rank's overflow list: the group's spectrum must carry it on
    every rank's behalf (sum f * spectrum[f] == instances)."""
    from allpathslg_b200 import KmerCounter, KmerGroup

    K = 25
    reads = ["A" * 2000] * 40 + ["ACGTTGCATGCATGCATTTGACGATCGACTAGCTAGCATCGACTACGACTAGCAT" * 3] * 30
    p, o = oracle.pack_strings(reads)
    ek, ec, en = oracle.count(p, o, K)
    assert int(ec.max()) > 65535
    world = 3
    kcs = []
    for r in range(world):
        kc = KmerCounter(K)
        lo, hi = len(reads) * r // world, len(reads) * (r + 1) // world
        pr, orr = oracle.pack_strings(reads[lo:hi])
        kc.add_reads(pr, orr)
        kcs.append(kc)
    with KmerGroup.local(kcs) as grp:
        grp.count()
        f, m = grp.spectrum_sparse()
        assert int((f * m).sum()) == en and int(m.sum()) == len(ek)
        es = oracle.spectrum(ec)
        assert (f == np.nonzero(es)[0]).all() and (m == es[np.nonzero(es)[0]]).all()
        assert grp.totals() == (en, len(ek))
    for kc in kcs:
        kc.close()


def test_group_follows_new_reads(oracle):
    """Reset + new (larger) read sets between steps: geometry, buffers and exported mappings follow."""
    from allpathslg_b200 import KmerCounter, KmerGroup

    K, L, world = 25, 100, 2
    sp = oracle.synth_params(300_000, L)
    kcs = [KmerCounter(K) for _ in range(world)]
    with KmerGroup.local(kcs) as grp:
        for n_reads in (4_000, 60_000, 9_000):
            for r, kc in enumerate(kcs):
                kc.reset()
                pr, _ = oracle.synth_reads(sp, r * n_reads, n_reads)
                kc.add_reads_uniform(pr, n_reads, L)
            grp.count()
            p, o = oracle.synth_reads(sp, 0, world * n_reads)
            _check_against_oracle(oracle, grp, kcs, p, o, K, sorted_by_rank=True)
        # a context of a group still works on its own
        kcs[0].finish()
        p0, o0 = oracle.synth_reads(sp, 0, 9_000)
        ek, ec, en = oracle.count(p0, o0, K)
        gk, gc = kcs[0].counts()
        assert (gk == ek).all() and (gc.astype(np.uint64) == ec).all()
        grp.count()
        _check_against_oracle(oracle, grp, kcs, p, o, K, sorted_by_rank=True)
    for kc in kcs:
        kc.close()
