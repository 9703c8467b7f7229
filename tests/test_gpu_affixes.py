"""GPU tests of the k-mer AFFIXES (apgk_build_affixes / apgk_affixes_* / apgk_lookup_affixes): bit-exact against
oracle A (tests/affix_oracle.c) on hand vectors, ragged reads of every key width and synthetic reads; every placement
path, shown to have run through the context's geometry; the state rules; the orientation of lookups; two oracle-free
identities against the library's own table at K+1; and the benchmark store at K = 24.  Run with `-m gpu` on a B200."""
import os

import numpy as np
import pytest

import affix_oracle as AO
from oracle import oracle_b as B
from test_affixes_cpu import HAND, K_ALL, ragged_reads

pytestmark = pytest.mark.gpu

OCC_PLACE_CAP = 2048   # distinct k-mers of a bucket k_aff_place keeps in shared memory (csrc/occ.cuh)


def _counter(packed, off, K, uniform=None, **kw):
    from allpathslg_b200 import KmerCounter

    kc = KmerCounter(K, want_counts=True, **kw)
    if uniform:
        kc.add_reads_uniform(packed, uniform[0], uniform[1])
    else:
        kc.add_reads(packed, off)
    kc.finish()
    return kc


def _check(oracle, kc, packed, off, K):
    """table == oracle's, then the affixes == oracle A's, row for row; -> (oracle table, affixes)"""
    ek, ec, _ = oracle.count(packed, off, K)
    gk, gc = kc.counts()
    assert (gk == ek).all() and (gc.astype(np.uint64) == ec).all()
    ms = kc.build_affixes()
    assert set(ms) == {"scan", "sweep", "place"}
    got = kc.affixes()
    want = AO.affixes_a(packed, off, K, ek)
    assert len(got) == len(want)
    bad = np.nonzero(got != want)[0]
    assert len(bad) == 0, "rows %s: got %s want %s" % (bad[:5], got[bad[:5]], want[bad[:5]])
    return ek, got


def _err(fn):
    from allpathslg_b200 import ApgkError

    with pytest.raises(ApgkError) as e:
        fn()
    return e.value.code


def _int_to_words(v, W):
    return [(v >> (64 * (W - 1 - i))) & ((1 << 64) - 1) for i in range(W)]


def _words_to_int(row):
    v = 0
    for w in row:
        v = (v << 64) | int(w)
    return v


@pytest.mark.parametrize("reads,K,want", HAND, ids=["%s-K%d" % ("+".join(r), k) for r, k, _ in HAND])
def test_hand_vectors(oracle, reads, K, want):
    p, o = oracle.pack_strings(reads)
    kc = _counter(p, o, K)
    kc.build_affixes()
    gk, _ = kc.counts()
    got = {int(k[0]): int(a) for k, a in zip(gk, kc.affixes())}
    expect = {}
    for s, a in want.items():
        v = 0
        for ch in s:
            v = v * 4 + "ACGT".index(ch)
        expect[v] = a
    assert got == expect
    kc.close()


@pytest.mark.parametrize("K", K_ALL)
def test_ragged_reads(oracle, K):
    """Empty reads, reads of K-1, K and K+1 bases, poly-A, ACGT and CG repeats (palindromes at even K); sub-ranges."""
    reads = ragged_reads(K, 500 + K)
    p, o = oracle.pack_strings(reads)
    kc = _counter(p, o, K)
    ek, got = _check(oracle, kc, p, o, K)
    assert got.any()
    nd = len(ek)
    ptr, n = kc.affixes_device()
    assert ptr and n == nd
    if nd >= 3:
        a, m = nd // 3, nd // 2
        assert (kc.affixes(a, m) == got[a:a + m]).all()
        assert len(kc.affixes(nd, 0)) == 0
    kc.close()


@pytest.mark.parametrize("K,L,n", [(20, 100, 300_000), (25, 100, 300_000), (48, 150, 100_000), (96, 250, 40_000)])
def test_synthetic_uniform_reads(oracle, K, L, n):
    sp = oracle.synth_params(500_000, L)
    p, o = oracle.synth_reads(sp, 0, n)
    kc = _counter(p, o, K, uniform=(n, L))
    _, got = _check(oracle, kc, p, o, K)
    assert got.any()
    kc.close()


def _n_distinct_per_bucket_max(ek, K, P):
    W = ek.shape[1]
    tb = max(2 * K, P)
    if W == 1:
        b = (ek[:, 0] << np.uint64(tb - 2 * K)) >> np.uint64(tb - P)
        return int(np.bincount(b.astype(np.int64)).max())
    return int(np.unique([_words_to_int(r) >> (2 * K - P) for r in ek], return_counts=True)[1].max())


PATHS = [
    # id, K, counter kwargs, check of the geometry
    ("u32-shared", 25, dict(prefix_bits=20), lambda g, mx: g["elem_bytes"] == 4 and mx <= OCC_PLACE_CAP),
    ("u32-rem32", 26, dict(prefix_bits=20), lambda g, mx: g["elem_bytes"] == 4 and g["REM"] == 32),
    ("key-w1", 31, dict(prefix_bits=12), lambda g, mx: g["elem_bytes"] == 8 and g["REM"] > 32),
    ("key-w2", 40, {}, lambda g, mx: g["elem_bytes"] == 16),
    ("key-w3", 96, {}, lambda g, mx: g["elem_bytes"] == 24),
    ("u32-oversize", 16, dict(prefix_bits=4), lambda g, mx: g["elem_bytes"] == 4 and mx > OCC_PLACE_CAP),
    ("key-oversize", 31, dict(prefix_bits=6), lambda g, mx: g["elem_bytes"] == 8 and mx > OCC_PLACE_CAP),
    ("rounds", 25, dict(max_round_keys=300_000, max_inner_keys=80_000), lambda g, mx: g["n_rounds"] > 1),
    ("rounds-w2", 40, dict(max_round_keys=300_000, max_inner_keys=80_000), lambda g, mx: g["n_rounds"] > 1),
    ("async-ingest", 25, dict(async_ingest=True, prefix_bits=19), lambda g, mx: g["elem_bytes"] == 4),
]


@pytest.mark.parametrize("name,K,kw,ok", PATHS, ids=[p[0] for p in PATHS])
def test_place_paths(oracle, name, K, kw, ok):
    sp = oracle.synth_params(150_000, 100)
    n = 24_000
    p, o = oracle.synth_reads(sp, 0, n)
    kc = _counter(p, o, K, uniform=(n, 100), **kw)
    ek, _ = _check(oracle, kc, p, o, K)
    g = kc.geometry()
    mx = _n_distinct_per_bucket_max(ek, K, g["D0"] + g["D1"])
    assert ok(g, mx), (g, mx)
    kc.close()


def test_refusals(oracle):
    from allpathslg_b200 import KmerCounter, KmerGroup, _lib

    reads = ragged_reads(25, 3)
    p, o = oracle.pack_strings(reads)
    # before a finish
    kc = KmerCounter(25, want_counts=True)
    kc.add_reads(p, o)
    assert _err(kc.build_affixes) == _lib.E_STATE
    assert _err(kc.affixes) == _lib.E_STATE
    kc.finish()
    # finished, affixes not built yet
    assert _err(kc.affixes) == _lib.E_STATE
    assert _err(kc.affixes_device) == _lib.E_STATE
    assert _err(lambda: kc.lookup_affixes(np.zeros(1, np.uint64))) == _lib.E_STATE
    kc.build_affixes()
    _, nd = kc.totals()
    assert _err(lambda: kc.affixes(nd, 1)) == _lib.E_ARG
    assert _err(lambda: kc.affixes(0, nd + 1)) == _lib.E_ARG
    assert _err(lambda: kc.affixes(nd + 1, 0)) == _lib.E_ARG
    # a table counted from a key array, not from the context's reads
    import torch

    keys, _ = kc.counts()
    d = torch.from_numpy(keys.view(np.int64).copy()).cuda()
    kk = KmerCounter(25, want_counts=True)
    kk.finish_keys_device(d.data_ptr(), len(keys))
    assert kk.totals()[1] == nd
    assert _err(kk.build_affixes) == _lib.E_STATE
    assert _err(kk.affixes) == _lib.E_STATE
    kk.close()
    # without APGK_WANT_COUNTS
    kn = KmerCounter(25, want_counts=False)
    kn.add_reads(p, o)
    kn.finish()
    assert _err(kn.build_affixes) == _lib.E_STATE
    kn.close()
    # shards of a group: three contexts on this device
    kcs = [KmerCounter(25, want_counts=True) for _ in range(3)]
    for r, kr in enumerate(kcs):
        pr, orr = oracle.pack_strings(reads[r::3])
        kr.add_reads(pr, orr)
    with KmerGroup.local(kcs) as grp:
        grp.count()
        for kr in kcs:
            assert _err(kr.build_affixes) == _lib.E_STATE
            assert _err(kr.affixes) == _lib.E_STATE
    for kr in kcs:
        kr.close()
    kc.close()


def test_invalidation_rebuild_and_release_temp(oracle):
    from allpathslg_b200 import _lib

    K = 33
    r1 = ragged_reads(K, 11)
    r2 = ragged_reads(K, 12)
    p1, o1 = oracle.pack_strings(r1)
    p2, o2 = oracle.pack_strings(r2)
    kc = _counter(p1, o1, K)
    _, a1 = _check(oracle, kc, p1, o1, K)
    kc.build_affixes()                        # a repeated build gives the same bytes
    assert (kc.affixes() == a1).all()
    kc.release_temp()                         # the affixes are not scratch
    assert (kc.affixes() == a1).all()
    kc.add_reads(p2, o2)                      # new reads drop them
    assert _err(kc.affixes) == _lib.E_STATE
    kc.finish()
    assert _err(kc.affixes) == _lib.E_STATE
    pa, oa = oracle.pack_strings(r1 + r2)
    _check(oracle, kc, pa, oa, K)
    kc.finish()                               # so does a finish
    assert _err(kc.affixes_device) == _lib.E_STATE
    kc.reset()                                # and a reset
    assert _err(kc.affixes) == _lib.E_STATE
    kc.add_reads(p2, o2)
    kc.finish()
    _check(oracle, kc, p2, o2, K)
    kc.close()


@pytest.mark.parametrize("K", [25, 64])
def test_affixes_occurrences_and_read_freqs_in_either_order(oracle, K):
    import torch

    sp = oracle.synth_params(80_000, 100)
    p, o = oracle.synth_reads(sp, 0, 15_000)
    ek, ec, en = oracle.count(p, o, K)
    want_aff = AO.affixes_a(p, o, K, ek)
    ero, erid, epos = oracle.occurrences(p, o, K, ek, en)
    want_freq = oracle.read_freqs(p, o, K, ek, ec).astype(np.uint32)

    def check_occ(kc):
        ro, rid, pos = kc.occurrences()
        assert (ro == ero).all() and (rid == erid).all() and (pos == epos).all()

    def check_freq(kc):
        buf = torch.empty(len(want_freq), dtype=torch.int32, device="cuda")
        kc.read_freqs_device(buf.data_ptr())
        assert (buf.cpu().numpy().view(np.uint32) == want_freq).all()

    for order in ("aff-first", "aff-last"):
        kc = _counter(p, o, K, uniform=(15_000, 100))
        if order == "aff-first":
            kc.build_affixes()
            kc.build_occurrences()
            check_freq(kc)
            check_occ(kc)
            assert (kc.affixes() == want_aff).all()
        else:
            kc.build_occurrences()
            check_freq(kc)
            kc.build_affixes()
            assert (kc.affixes() == want_aff).all()
            check_occ(kc)
            check_freq(kc)
            assert (kc.affixes() == want_aff).all()
        kc.close()


@pytest.mark.parametrize("K", [25, 40, 64, 96])
def test_lookup_affixes(oracle, K):
    rnd = np.random.default_rng(K)
    sp = oracle.synth_params(60_000, 100)
    n = 10_000
    p, o = oracle.synth_reads(sp, 0, n)
    reads = ["CG" * 60, "ACGT" * 30] if K % 2 == 0 else []
    if reads:   # palindromes at even K
        allr = B.unpack_reads(p, o) + reads
        p, o = oracle.pack_strings(allr)
        kc = _counter(p, o, K)
    else:
        kc = _counter(p, o, K, uniform=(n, 100))
    ek, aff = _check(oracle, kc, p, o, K)
    _, cnt = kc.counts()
    W = ek.shape[1]
    # table rows, canonicalised or taken as they are
    for canon in (True, False):
        ga, gc = kc.lookup_affixes(ek, canonicalise=canon)
        assert (ga == aff).all() and (gc == cnt).all()
    # their reverse complements: the transform, palindromes unchanged
    rc = AO.revcomp_keys(ek, K)
    ga, gc = kc.lookup_affixes(rc)
    assert (gc == cnt).all()
    assert (ga == AO.affix_revcomp(aff)).all()
    pal = (rc == ek).all(axis=1)
    if K % 2 == 0:
        assert pal.any() and (ga[pal] == aff[pal]).all()
    # random k-mers, mostly absent: count 0 and affixes 0; present ones as the table says
    q = rnd.integers(0, 1 << 62, size=(5000, W), dtype=np.uint64)
    top = 2 * K - 64 * (W - 1)
    q[:, 0] &= np.uint64((1 << top) - 1)
    ga, gc = kc.lookup_affixes(q)
    view = lambda a: np.ascontiguousarray(a).view([("w%d" % i, np.uint64) for i in range(W)]).ravel()
    qr = AO.revcomp_keys(q, K)
    qc = np.where(_lex_less(qr, q)[:, None], qr, q)
    idx = np.searchsorted(view(ek), view(qc))
    idx = np.minimum(idx, len(ek) - 1)
    present = (ek[idx] == qc).all(axis=1)
    assert (gc[~present] == 0).all() and (ga[~present] == 0).all()
    if present.any():
        assert (gc[present] == cnt[idx[present]]).all()
    kc.close()


def _lex_less(a, b):
    less = np.zeros(len(a), dtype=bool)
    decided = np.zeros(len(a), dtype=bool)
    for i in range(a.shape[1]):
        less |= ~decided & (a[:, i] < b[:, i])
        decided |= a[:, i] != b[:, i]
    return less


def _kp1_checks(kc, kp, ek, aff, K, rows):
    """bit (c, suf/pre, b) of row i is set iff the (K+1)-mer c.b / b.c has a count > 0 in the K+1 context kp"""
    W1 = (2 * (K + 1) + 63) // 64
    qs = []
    for i in rows:
        c = _words_to_int(ek[i])
        for b in range(4):
            qs.append(_int_to_words((b << (2 * K)) | c, W1))   # b.c: b precedes c
        for b in range(4):
            qs.append(_int_to_words((c << 2) | b, W1))         # c.b: b follows c
    cnt = kp.lookup(np.array(qs, dtype=np.uint64).ravel())
    bits = (cnt > 0).reshape(len(rows), 8)
    want = np.array([[(int(aff[i]) >> j) & 1 for j in range(8)] for i in rows], dtype=bool)
    assert (bits == want).all()


def _palindromes(kmers, K):
    """mask of the rows that are their own reverse complement (none at odd K)"""
    if K % 2:
        return np.zeros(len(kmers), dtype=bool)
    return (AO.revcomp_keys(kmers, K) == kmers).all(axis=1)


def _pal_pairs(aff):
    """bits of palindromic k-mers' affixes come in pairs (suf b, pre comp(b)) that name ONE (K+1)-mer class"""
    pc = int(np.unpackbits(np.asarray(aff, dtype=np.uint8)).sum())
    assert pc % 2 == 0
    return pc // 2


@pytest.mark.parametrize("K", [11, 24, 25, 31, 32, 47, 63, 64, 95])
def test_identities_against_the_table_at_k_plus_1(oracle, K):
    """Sum of popcounts at K = 2 D(K+1) - P(K+1) + H(K), and sampled rows bit by bit against the (K+1)-mers' counts,
    with D, P and the counts from the library's own K+1 table (no oracle).  Every canonical (K+1)-mer sets one bit on
    the k-mer of its first K bases and one on that of its last K: two bits, except that a palindromic (K+1)-mer (odd K)
    sets the same bit twice (-P), and a palindromic k-mer (even K) reads each of its neighbours both ways, so each
    class it touches sets two bits on it where one is counted (+H = half the popcount of the palindromic rows)."""
    from allpathslg_b200 import KmerCounter

    sp = oracle.synth_params(120_000, 100)
    n = 20_000
    p, _ = oracle.synth_reads(sp, 0, n)
    pe, oe = oracle.pack_strings(["CG" * 70, "ACGT" * 40, "A" * 150, "GC" * 55, "T" * K])
    kc, kp = KmerCounter(K, want_counts=True), KmerCounter(K + 1, want_counts=True)
    for k in (kc, kp):
        k.add_reads_uniform(p, n, 100)
        k.add_reads(pe, oe)
        k.finish()
    kc.build_affixes()
    aff = kc.affixes()
    ek, _ = kc.counts()
    kk1, _ = kp.counts()
    D1 = kp.totals()[1]
    P1 = int(_palindromes(kk1, K + 1).sum())
    H = _pal_pairs(aff[_palindromes(ek, K)])
    assert (P1 > 0) if K % 2 else (H > 0)     # the reads' CG repeats give both corrections something to do
    pop = int(np.unpackbits(aff).sum())
    assert pop == 2 * D1 - P1 + H, (pop, D1, P1, H)
    rows = sorted(set(np.random.default_rng(K).integers(0, len(ek), size=3000).tolist()))
    _kp1_checks(kc, kp, ek, aff, K, rows)
    kc.close()
    kp.close()


# ---------------------------------------------------------------- the benchmark store
READS, READ_LEN, GENOME = 60_000_000, 100, 100_000_000
MIN_FREE_BYTES = 120 << 30


def test_scale_bench_store_k24():
    """bench.py's store (60 M x 100 bp synthetic, 4.56 G windows of 6.0 G bases) at K = 24: K+1 = 25 is odd, so no
    palindromes and the sum of popcounts is exactly 2 D(25) + H, H = half the popcount of the palindromic 24-mers'
    rows (found by looking up all 4^12 of them).  Plus the sampled-partition oracle on two of 1024
    leading-bit partitions, a bit-by-bit check of sampled rows against the K = 25 table, and lookups."""
    import torch

    from allpathslg_b200 import KmerCounter, synth_params
    from oracle import oracle_a as A

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    free = torch.cuda.mem_get_info()[0]
    if free < MIN_FREE_BYTES:
        pytest.skip("needs %.0f GiB of free device memory, %.1f GiB free (the card is shared)" % (MIN_FREE_BYTES / 2**30, free / 2**30))
    sp = synth_params(GENOME, READ_LEN)
    kp = KmerCounter(25, want_counts=True, reserve_bases=READS * READ_LEN)
    kp.synth_reads(sp, 0, READS)
    kp.finish()
    kp.release_temp()
    D25 = kp.totals()[1]
    kc = KmerCounter(24, want_counts=True, reserve_bases=READS * READ_LEN)
    kc.synth_reads(sp, 0, READS)
    kc.finish()
    ni, nd = kc.totals()
    assert ni == READS * (READ_LEN - 24 + 1)
    ms = kc.build_affixes()
    low = torch.cuda.mem_get_info()[0]
    aff = kc.affixes()
    pop = int(np.unpackbits(aff).sum())
    half = np.arange(1 << 24, dtype=np.uint64)    # every palindromic 24-mer: 12 bases, then their reverse complement
    pal = (half << np.uint64(24)) | AO.revcomp_keys(half[:, None], 12)[:, 0]
    pa, pc = kc.lookup_affixes(pal, canonicalise=False)
    H = _pal_pairs(pa[pc > 0])
    print("\nK=24: %d instances, %d distinct (%d palindromic); build %s ms; D(25) = %d; popcount sum %d = 2 D(25) + %d; "
          "free at start %.1f GiB, after build %.1f GiB" % (ni, nd, int((pc > 0).sum()), {k: round(v, 1) for k, v in ms.items()},
                                                          D25, pop, pop - 2 * D25, free / 2**30, low / 2**30))
    assert pop == 2 * D25 + H
    # sampled partitions: every row of the two partitions against the reads
    host = kc.export_reads()
    pbits, parts = 10, (77, 700)
    keys, pos, n_win = A.sample_prefix_pos(host, None, 24, pbits, parts, n_reads=READS, read_len=READ_LEN,
                                           n_threads=os.cpu_count() or 1)
    assert n_win == ni
    uk, ua = AO.sample_affixes(host, None, 24, keys, pos, read_len=READ_LEN)
    del keys, pos
    n_rows = 0
    for part in parts:
        first, n = kc.prefix_range(pbits, part)
        gk, _ = kc.counts(first, n)
        sel = (uk[:, 0] >> np.uint64(48 - pbits)) == part
        assert (gk == uk[sel]).all()
        assert (aff[first:first + n] == ua[sel]).all()
        n_rows += n
    assert n_rows > 100_000
    # sampled rows bit by bit against the K = 25 table, and lookups of rows and their reverse complements
    rows = np.random.default_rng(24).integers(0, nd, size=20_000)
    rows.sort()
    rk = np.stack([kc.counts(int(r), 1)[0][0] for r in rows[:2000]])
    ra = aff[rows[:2000]]
    _kp1_checks(kc, kp, rk, ra, 24, range(len(rk)))
    ga, gc = kc.lookup_affixes(AO.revcomp_keys(rk, 24))
    assert (ga == AO.affix_revcomp(ra)).all() and (gc > 0).all()
    kc.close()
    kp.close()
