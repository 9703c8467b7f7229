"""GPU parity tests of the frequency lookups on the sharded table (apgk_group_read_freqs_device, csrc/gfreq.cuh):
after apgk_group_count every rank asks, for every window of its own reads, the GLOBAL count of the window's canonical
k-mer, held by whichever rank owns it.  The groups are formed by ONE process over N contexts on one GPU, as in
tests/test_gpu_group.py.  The expected answer of rank r is the oracle's global table (all ranks' reads) applied to
rank r's reads, compared at every base."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

NONE32 = np.uint32(0xFFFFFFFF)


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


def _expected(oracle, reads, K):
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
    return out, ek, ec


def _close(kcs):
    for kc in kcs:
        kc.close()


def _check(got, exp):
    assert len(got) == len(exp)
    for r, (g, e) in enumerate(zip(got, exp)):
        assert g.shape == e.shape, (r, g.shape, e.shape)
        bad = np.nonzero(g != e)[0]
        assert len(bad) == 0, "rank %d: %d of %d bases differ, first at %d (%d != %d)" % (
            r, len(bad), len(e), bad[0], g[bad[0]], e[bad[0]])


@pytest.mark.parametrize("K,world,n_reads,empty,pb,elem", [(25, 2, 30_000, None, 0, 8), (25, 5, 30_000, 2, 0, 8),
                                                           (20, 3, 20_000, None, 0, 4), (25, 8, 40_000, None, 0, 8),
                                                           (31, 2, 12_000, None, 0, 8), (48, 3, 12_000, None, 0, 16),
                                                           (96, 2, 8_000, 0, 0, 24), (25, 1, 10_000, None, 0, 8),
                                                           (25, 3, 30_000, None, 20, 4), (20, 2, 20_000, 1, 16, 4),
                                                           (25, 1, 10_000, None, 20, 4)])
def test_group_read_freqs_match_the_oracle(oracle, K, world, n_reads, empty, pb, elem):
    """elem: the level-1 element the queries travel as -- a 4-byte remainder when the bits below the P-bit prefix
    fit (K = 20, or prefix_bits given: the table slices are searched in shared memory), else the one-word key (8
    bytes for K = 25 / 31 at these small sizes) or the 2- and 3-word keys of K = 48 / 96."""
    from allpathslg_b200 import KmerGroup

    kcs, reads = _ranks(oracle, K, world, n_reads, empty_rank=empty, prefix_bits=pb)
    exp, _, _ = _expected(oracle, reads, K)
    with KmerGroup.local(kcs) as grp:
        grp.count()
        assert kcs[0].geometry()["elem_bytes"] == elem
        st = {}
        got = grp.read_freqs(stats=st)
        _check(got, exp)
        assert st["n_batches"] == (1 if any(len(e) for e in exp) else 0)
        assert st["n_queries"] == int((exp[0] != NONE32).sum())
        if world == 1:
            assert st["remote_bytes"] == 0
        assert st["total_ms"] > 0
    _close(kcs)


def test_group_read_freqs_ragged_reads(oracle):
    """Reads of every length, some shorter than K, some empty, added with apgk_add_reads after uniform ones."""
    from allpathslg_b200 import KmerGroup

    K = 25
    kcs, reads = _ranks(oracle, K, 3, 30_000, ragged_rank=1)
    exp, _, _ = _expected(oracle, reads, K)
    with KmerGroup.local(kcs) as grp:
        grp.count()
        _check(grp.read_freqs(), exp)
    _close(kcs)


@pytest.mark.parametrize("K,world,n_reads,outer_div,inner_div", [(25, 3, 30_000, 2, 5), (48, 2, 12_000, 2, 4),
                                                                 (20, 4, 20_000, 3, 3), (96, 2, 6_000, 2, 2)])
def test_group_read_freqs_after_rounds(oracle, K, world, n_reads, outer_div, inner_div):
    """A count in k-mer-space rounds leaves every rank owning one range per inner round: the queries of a bucket
    go to whichever rank owned it in its round."""
    from allpathslg_b200 import KmerGroup

    per_rank = (n_reads // world) * (100 - K + 1)
    kcs, reads = _ranks(oracle, K, world, n_reads, max_round_keys=per_rank // outer_div + 1,
                        max_inner_keys=per_rank // inner_div + 1)
    exp, _, _ = _expected(oracle, reads, K)
    with KmerGroup.local(kcs) as grp:
        grp.count()
        assert grp.stats()["n_rounds"] >= inner_div
        _check(grp.read_freqs(), exp)
    _close(kcs)


@pytest.mark.parametrize("K,world,budget_kb", [(25, 3, 1024), (48, 2, 2048), (25, 2, 64)])
def test_group_read_freqs_in_batches(oracle, K, world, budget_kb, monkeypatch):
    """A pretend device-memory budget far below one batch of the whole store: several exchange batches, same
    answers; the rank whose range ends first keeps taking part in every batch."""
    from allpathslg_b200 import KmerGroup

    kcs, reads = _ranks(oracle, K, world, 30_000 if K == 25 else 12_000)
    exp, _, _ = _expected(oracle, reads, K)
    with KmerGroup.local(kcs) as grp:
        grp.count()
        st1 = {}
        one = grp.read_freqs(stats=st1)
        _check(one, exp)
        monkeypatch.setenv("APGK_BUDGET_BYTES", str(budget_kb << 10))
        st = {}
        nb = [len(e) for e in exp]
        nb[-1] //= 3   # ragged ranges: the last rank needs fewer batches than the others
        got = grp.read_freqs(n_bases=nb, stats=st)
        assert st["n_batches"] >= 2
        _check(got, [e[:n] for e, n in zip(exp, nb)])
        assert st["remote_bytes"] <= st1["remote_bytes"]
    _close(kcs)


def test_group_read_freqs_sub_ranges(oracle):
    """Unaligned ranges, a range of 0 bases on one rank only, and a range that ends at the store's end."""
    from allpathslg_b200 import KmerGroup

    K = 25
    kcs, reads = _ranks(oracle, K, 3, 30_000, ragged_rank=2)
    exp, _, _ = _expected(oracle, reads, K)
    tot = [len(e) for e in exp]
    fb = [17, 0, 5]
    nb = [tot[0] - 30, 0, tot[2] - 5]
    with KmerGroup.local(kcs) as grp:
        grp.count()
        got = grp.read_freqs(fb, nb)
        _check(got, [e[f:f + n] for e, f, n in zip(exp, fb, nb)])
        got = grp.read_freqs([1001, 3, tot[2]], [999, 77, 0])
        _check(got, [exp[0][1001:2000], exp[1][3:80], exp[2][:0]])
    _close(kcs)


def test_group_read_freqs_large_table_slices(oracle):
    """prefix_bits = 8 with 4-byte remainders (K = 16): the owners' table slices hold more keys than shared memory
    takes, so the resolution searches the shard's table in global memory instead."""
    from allpathslg_b200 import KmerGroup

    K = 16
    kcs, reads = _ranks(oracle, K, 2, 30_000, genome=1_000_000, prefix_bits=8)
    exp, ek, _ = _expected(oracle, reads, K)
    sizes = np.bincount((ek[:, 0] >> np.uint64(2 * K - 8)).astype(np.int64))
    assert sizes.max() > 4096 and sizes.min() < 4096   # both paths run
    with KmerGroup.local(kcs) as grp:
        grp.count()
        assert grp.stats()["prefix_bits"] == 8 and kcs[0].geometry()["elem_bytes"] == 4
        _check(grp.read_freqs(), exp)
    _close(kcs)


def test_group_read_freqs_repeat_release_temp_recount(oracle):
    """apgk_release_temp between count and lookup (the tables stay; the partition buffers are re-grown and
    re-exported), two lookups in a row, and a lookup after a second count: all the same answers."""
    from allpathslg_b200 import KmerGroup

    K = 25
    kcs, reads = _ranks(oracle, K, 3, 30_000)
    exp, _, _ = _expected(oracle, reads, K)
    with KmerGroup.local(kcs) as grp:
        grp.count()
        for kc in kcs:
            kc.release_temp()
        _check(grp.read_freqs(), exp)
        _check(grp.read_freqs(), exp)
        grp.count()
        _check(grp.read_freqs(), exp)
    _close(kcs)


def test_group_read_freqs_equal_one_context(oracle):
    """At a size the oracle is slow for: the ranks' outputs, concatenated, equal apgk_read_freqs of ONE plain
    context over the concatenated reads."""
    from allpathslg_b200 import KmerCounter, KmerGroup
    from allpathslg_b200.kmers import synth_params

    K, L, world, per = 25, 100, 4, 100_000
    sp = synth_params(3_000_000, L)
    kcs = []
    for r in range(world):
        kc = KmerCounter(K)
        kc.synth_reads(sp, r * per, per)
        kcs.append(kc)
    with KmerCounter(K) as one:
        one.synth_reads(sp, 0, world * per)
        one.finish()
        ref = one.read_freqs()
    with KmerGroup.local(kcs) as grp:
        grp.count()
        st = {}
        got = np.concatenate(grp.read_freqs(stats=st))
        assert (got == ref).all()
        assert st["remote_bytes"] > 0
    _close(kcs)


@pytest.mark.parametrize("K,pb,elem", [(25, 20, 4), (25, 0, 8), (48, 0, 16)])
def test_group_read_freqs_remote_bytes(oracle, K, pb, elem):
    """remote_bytes of rank 0 = (element + 4 bytes) x the queries it resolved for the other ranks: the instances of
    its shard minus those of its own windows."""
    from allpathslg_b200 import KmerGroup

    kcs, reads = _ranks(oracle, K, 3, 24_000 if K == 25 else 12_000, prefix_bits=pb)
    with KmerGroup.local(kcs) as grp:
        grp.count()
        st = {}
        grp.read_freqs(stats=st)
        shard0 = kcs[0].totals()[0]
        k0, c0, _ = oracle.count(*reads[0], K)
        owned = kcs[0].lookup(k0, canonicalise=False) > 0
        assert kcs[0].geometry()["elem_bytes"] == elem
        assert st["remote_bytes"] == (elem + 4) * (shard0 - int(c0[owned].sum()))
    _close(kcs)


def test_group_read_freqs_refusals(oracle):
    """Every refusal is the same on every rank and returns at once: no count yet, a count without tables, a context
    given reads after the count, a range beyond a store.  The group works again after each."""
    from allpathslg_b200 import KmerCounter, KmerGroup
    from allpathslg_b200._lib import E_ARG, E_STATE
    from allpathslg_b200.kmers import ApgkError

    K = 25
    kcs, reads = _ranks(oracle, K, 3, 9_000)
    exp, _, _ = _expected(oracle, reads, K)
    with KmerGroup.local(kcs) as grp:
        with pytest.raises(ApgkError) as ei:
            grp.read_freqs()
        assert ei.value.code == E_STATE
        grp.count()
        tot = [len(e) for e in exp]
        with pytest.raises(ApgkError) as ei:
            grp.read_freqs([0, 0, 1], tot)
        assert ei.value.code == E_ARG
        with pytest.raises(ApgkError) as ei:
            grp.read_freqs_device([0, 0, 0], [0, 0, 0], [0, 10, 0])   # no output buffer for a non-empty range
        assert ei.value.code == E_ARG
        _check(grp.read_freqs(), exp)
        p, o = oracle.synth_reads(oracle.synth_params(200_000, 100), 50_000, 10)
        kcs[1].add_reads(p, o)
        with pytest.raises(ApgkError) as ei:
            grp.read_freqs()
        assert ei.value.code == E_STATE
        grp.count()
        reads[1] = _concat([reads[1], (p, o)])
        exp, _, _ = _expected(oracle, reads, K)
        _check(grp.read_freqs(), exp)
    _close(kcs)
    nk = [KmerCounter(K, want_counts=False) for _ in range(2)]
    for r, kc in enumerate(nk):
        kc.add_reads(*reads[r])
    with KmerGroup.local(nk) as grp:
        grp.count()
        with pytest.raises(ApgkError) as ei:
            grp.read_freqs()
        assert ei.value.code == E_STATE
    _close(nk)
