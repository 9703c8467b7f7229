"""The k-mer affix oracles and the affix orientation transform, without a GPU: hand vectors of the definition in
include/apgk.h against oracles A (tests/affix_oracle.c) and B (strings), A against B on ragged reads for every key
width, reverse-complemented read sets, the sampled-partition helper against A, and the library's transform
(apgk_debug_host_affix_revcomp) against a restatement."""
import random

import numpy as np
import pytest

import affix_oracle as AO

RC = str.maketrans("ACGT", "TGCA")
K_ALL = [1, 2, 3, 4, 11, 24, 25, 26, 31, 32, 33, 63, 64, 65, 95, 96]

# (reads, K, {k-mer string: affix byte})
HAND = [
    (["ACGT"], 2, {"AC": 0x40, "CG": 0x81}),
    (["AACC"], 3, {"AAC": 0x20, "ACC": 0x01}),
    (["GGTT"], 3, {"AAC": 0x20, "ACC": 0x01}),
    (["GATTACA"], 7, {"GATTACA": 0x00}),
    (["GATTAC"], 7, {}),
]


def _kint(s):
    v = 0
    for ch in s:
        v = v * 4 + "ACGT".index(ch)
    return v


def ragged_reads(K, seed):
    rnd = random.Random(seed)
    reads = ["".join(rnd.choice("ACGT") for _ in range(rnd.choice([0, max(K - 1, 0), K, K + 1, K + 2, 40, 130])))
             for _ in range(120)]
    reads += ["", "A" * (K + 30), "ACGT" * (K // 4 + 12), "CG" * (K // 2 + 10), "", "T" * K, "GC" * (K + 3)]
    reads.append(reads[5].translate(RC)[::-1])
    return reads


def oracle_a_pairs(oracle, reads, K):
    p, o = oracle.pack_strings(reads)
    ek, _, _ = oracle.count(p, o, K)
    aff = AO.affixes_a(p, o, K, ek)
    W = ek.shape[1] if len(ek) else 1
    return [(sum(int(w) << (64 * (W - 1 - i)) for i, w in enumerate(row)), int(a)) for row, a in zip(ek, aff)]


@pytest.mark.parametrize("reads,K,want", HAND, ids=["%s-K%d" % ("+".join(r), k) for r, k, _ in HAND])
def test_hand_vectors(oracle, reads, K, want):
    expect = sorted((_kint(k), a) for k, a in want.items())
    assert AO.affixes_b(reads, K) == expect
    assert oracle_a_pairs(oracle, reads, K) == expect


@pytest.mark.parametrize("K", K_ALL)
def test_oracle_a_matches_b_on_ragged_reads(oracle, K):
    reads = ragged_reads(K, 500 + K)
    b = AO.affixes_b(reads, K)
    a = oracle_a_pairs(oracle, reads, K)
    assert a == b
    assert any(v for _, v in a)
    if K % 2 == 0:   # palindromes exist ("CG" repeats): their affix sets are closed under reverse complement
        pal = [(k, v) for k, v in b if _kint(_rc_str(k, K)) == k]
        assert pal
        assert all(int(AO.affix_revcomp(np.uint8(v))) == v for _, v in pal)


def _rc_str(kint, K):
    s = "".join("ACGT"[(kint >> (2 * (K - 1 - i))) & 3] for i in range(K))
    return s.translate(RC)[::-1]


@pytest.mark.parametrize("K", [3, 24, 25, 64, 96])
def test_reverse_complemented_reads_give_the_same_affixes(oracle, K):
    reads = ragged_reads(K, 900 + K)
    rc_reads = [r.translate(RC)[::-1] for r in reads]
    assert oracle_a_pairs(oracle, reads, K) == oracle_a_pairs(oracle, rc_reads, K)
    assert AO.affixes_b(rc_reads, K) == AO.affixes_b(reads, K)


@pytest.mark.parametrize("K", [4, 24, 25, 40])
def test_sampled_partition_helper_matches_oracle_a(oracle, K):
    """The scale test's helper on uniform synthetic reads and on ragged reads: its rows equal oracle A's rows."""
    sp = oracle.synth_params(20_000, 100)
    p, o = oracle.synth_reads(sp, 0, 3000)
    for packed, off, uniform in [(p, o, True), (*oracle.pack_strings(ragged_reads(K, 77)), False)]:
        ek, _, _ = oracle.count(packed, off, K)
        full = AO.affixes_a(packed, off, K, ek)
        parts = [0, 5, 9]
        keys, pos, _ = oracle.sample_prefix_pos(packed, None if uniform else off, K, 4, parts,
                                                n_reads=len(off) - 1, read_len=100 if uniform else 0)
        uk, ua = AO.sample_affixes(packed, None if uniform else off, K, keys, pos, read_len=100 if uniform else 0)
        view = lambda a: np.ascontiguousarray(a).view([("w%d" % i, np.uint64) for i in range(a.shape[1])]).ravel()
        idx = np.searchsorted(view(ek), view(uk))
        assert (ek[idx] == uk).all()
        assert (full[idx] == ua).all()
        assert len(uk) > 0


def test_orientation_transform_hook(apgk_lib):
    def restated(a):   # pre' = complement of each base of suf, suf' = complement of each base of pre
        pre, suf = a & 15, a >> 4
        npre = sum(1 << (3 - b) for b in range(4) if (suf >> b) & 1)
        nsuf = sum(1 << (3 - b) for b in range(4) if (pre >> b) & 1)
        return npre | (nsuf << 4)

    a = np.arange(256, dtype=np.uint8)
    out = np.zeros(256, dtype=np.uint8)
    assert apgk_lib.apgk_debug_host_affix_revcomp(a.ctypes.data, 256, out.ctypes.data) == 0
    assert [int(x) for x in out] == [restated(v) for v in range(256)]
    assert (out == AO.affix_revcomp(a)).all()
    back = np.zeros(256, dtype=np.uint8)
    assert apgk_lib.apgk_debug_host_affix_revcomp(out.ctypes.data, 256, back.ctypes.data) == 0
    assert (back == a).all()   # an involution
    # hand vectors: AC = 0x40 (followed by G) -> GT preceded by C = 0x02; CG = 0x81 is its own transform
    assert int(AO.affix_revcomp(np.uint8(0x40))) == 0x02 and int(AO.affix_revcomp(np.uint8(0x81))) == 0x81
    assert apgk_lib.apgk_debug_host_affix_revcomp(None, 1, None) == -1
