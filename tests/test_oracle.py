"""CPU tests of the oracle itself: golden vectors, A-vs-B agreement, invariants.
(Parity unpinned: no reference vectors exist -- see tests/golden/make_golden.py.)"""
import json
import os
import random

import numpy as np
import pytest

from oracle import oracle_b as B

GOLD = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "known_answers.json")))


def _to_int(row):
    W = len(row)
    return sum(int(row[j]) << (64 * (W - 1 - j)) for j in range(W))


@pytest.mark.parametrize("v", GOLD["hand"], ids=lambda v: "%s-K%d" % ("+".join(v["reads"]) or "empty", v["K"]))
def test_hand_vectors(oracle, v):
    p, o = oracle.pack_strings(v["reads"])
    k, c, n = oracle.count(p, o, v["K"])
    assert [_to_int(r) for r in k] == v["kmers"]
    assert [int(x) for x in c] == v["counts"]
    assert [int(x) for x in oracle.spectrum(c)] == v["spectrum"]
    assert n == sum(max(0, len(r) - v["K"] + 1) for r in v["reads"])


@pytest.mark.parametrize("s", GOLD["synth"], ids=lambda s: "G%d-K%d" % (s["genome_len"], s["K"]))
def test_synth_golden(oracle, s):
    sp = oracle.synth_params(s["genome_len"], s["read_len"])
    p, o = oracle.synth_reads(sp, 0, s["n_reads"])
    k, c, n = oracle.count(p, o, s["K"])
    assert n == s["n_instances"] and len(k) == s["n_distinct"]
    assert [int(x) for x in oracle.spectrum(c)] == s["spectrum"]
    M = (1 << 61) - 1
    chk = 0
    for row, cnt in zip(k, c):
        chk = (chk + (_to_int(row) % M) * int(cnt)) % M
    assert chk == s["table_checksum"]
    assert [str(_to_int(r)) for r in k[:4]] == s["first_kmers"]


@pytest.mark.parametrize("K", [1, 2, 7, 16, 25, 31, 32, 33, 47, 64, 65, 96])
def test_oracle_a_matches_b(oracle, K):
    rnd = random.Random(K)
    reads = ["".join(rnd.choice("ACGT") for _ in range(rnd.choice([0, 1, K - 1, K, K + 1, K + 9, 140]))) for _ in range(50)]
    reads += ["A" * (K + 25), "ACGT" * 30, "CG" * (K + 3)]
    rc = reads[4].translate(str.maketrans("ACGT", "TGCA"))[::-1]
    reads.append(rc)
    p, o = oracle.pack_strings(reads)
    k, c, n = oracle.count(p, o, K)
    pairs = B.count_reads(reads, K)
    assert [_to_int(r) for r in k] == [x for x, _ in pairs]
    assert [int(x) for x in c] == [y for _, y in pairs]
    spec = oracle.spectrum(c)
    assert [int(x) for x in spec] == B.spectrum(pairs)
    # invariants of SURVEY.md section 8: sum f*spectrum[f] = instances ; sum spectrum = distinct
    assert int((spec * np.arange(len(spec), dtype=np.uint64)).sum()) == n
    assert int(spec.sum()) == len(pairs)


def test_strand_symmetry(oracle):
    """A read set and its reverse complement have identical canonical counts."""
    rnd = random.Random(5)
    reads = ["".join(rnd.choice("ACGT") for _ in range(120)) for _ in range(40)]
    rcs = [r.translate(str.maketrans("ACGT", "TGCA"))[::-1] for r in reads]
    for K in (8, 25, 33):
        a = oracle.count(*oracle.pack_strings(reads), K)
        b = oracle.count(*oracle.pack_strings(rcs), K)
        assert (a[0] == b[0]).all() and (a[1] == b[1]).all()


def test_thread_count_independent(oracle):
    sp = oracle.synth_params(30000, 100)
    p, o = oracle.synth_reads(sp, 0, 5000)
    a = oracle.count(p, o, 25, n_threads=1)
    b = oracle.count(p, o, 25, n_threads=4)
    assert (a[0] == b[0]).all() and (a[1] == b[1]).all()


def test_lookup_and_read_freqs(oracle):
    sp = oracle.synth_params(5000, 80)
    p, o = oracle.synth_reads(sp, 0, 300)
    K = 21
    k, c, _ = oracle.count(p, o, K)
    assert (oracle.lookup(k, c, K, k, canonicalise=False) == c).all()
    rf = oracle.read_freqs(p, o, K, k, c)
    valid = rf != np.uint64(0xFFFFFFFFFFFFFFFF)
    assert valid.sum() == 300 * (80 - K + 1)
    assert (rf[valid] >= 1).all()


# ------------------------------------------------------------------ occurrence records (read id, signed position)
def _occ_lists(run_off, rid, pos):
    return [[[int(a), int(b)] for a, b in zip(rid[int(run_off[i]):int(run_off[i + 1])], pos[int(run_off[i]):int(run_off[i + 1])])]
            for i in range(len(run_off) - 1)]


@pytest.mark.parametrize("v", GOLD["occ_hand"], ids=lambda v: "%s-K%d" % ("+".join(v["reads"]), v["K"]))
def test_occurrence_hand_vectors(oracle, v):
    p, o = oracle.pack_strings(v["reads"])
    k, c, n = oracle.count(p, o, v["K"])
    assert [_to_int(r) for r in k] == v["kmers"]
    ro, rid, pos = oracle.occurrences(p, o, v["K"], k, n)
    assert _occ_lists(ro, rid, pos) == v["occ"]
    assert [[[r, q] for r, q in lst] for _, lst in B.occurrences(v["reads"], v["K"])] == v["occ"]


@pytest.mark.parametrize("s", GOLD["occ_synth"], ids=lambda s: "G%d-K%d" % (s["genome_len"], s["K"]))
def test_occurrence_synth_golden(oracle, s):
    import hashlib

    sp = oracle.synth_params(s["genome_len"], s["read_len"])
    p, o = oracle.synth_reads(sp, 0, s["n_reads"])
    k, c, n = oracle.count(p, o, s["K"])
    ro, rid, pos = oracle.occurrences(p, o, s["K"], k, n)
    assert n == s["n_instances"] and len(k) == s["n_distinct"]
    h = hashlib.sha256(ro.tobytes() + rid.tobytes() + pos.tobytes()).hexdigest()
    assert h == s["occ_sha256"]
    assert (np.diff(ro.astype(np.int64)) == c.astype(np.int64)).all()  # run lengths are the counts


@pytest.mark.parametrize("K", [1, 2, 7, 25, 32, 33, 64, 65, 96])
def test_occurrences_a_matches_b(oracle, K):
    rnd = random.Random(100 + K)
    reads = ["".join(rnd.choice("ACGT") for _ in range(rnd.choice([0, 1, K - 1, K, K + 1, K + 9, 140]))) for _ in range(40)]
    reads += ["", "A" * (K + 25), "ACGT" * 30, "CG" * (K + 3), ""]
    reads.append(reads[4].translate(str.maketrans("ACGT", "TGCA"))[::-1])
    p, o = oracle.pack_strings(reads)
    k, c, n = oracle.count(p, o, K)
    ro, rid, pos = oracle.occurrences(p, o, K, k, n)
    ob = B.occurrences(reads, K)
    assert [_to_int(r) for r in k] == [x for x, _ in ob]
    assert _occ_lists(ro, rid, pos) == [[[r, q] for r, q in lst] for _, lst in ob]
    # every record points at a window whose canonical form is its k-mer, on the strand its sign says
    for i, (kv, lst) in enumerate(ob):
        for r, q in lst:
            w = reads[r][abs(q) - 1:abs(q) - 1 + K]
            assert len(w) == K and B.kmer_to_int(B.canonical_str(w)) == kv
            assert (q > 0) == (B.canonical_str(w) == w)


@pytest.mark.parametrize("K", [2, 5, 20, 25, 32, 33, 48, 64, 96])
def test_sampled_partition_oracle_matches_full_count(oracle, K):
    """The sampled-partition oracle used at sizes the host cannot hold (SURVEY.md section 8c, human-scale check ii):
    scanning all reads and keeping the k-mers of a few leading-bit partitions, then counting them, must give
    exactly the full oracle's records of those partitions -- ragged reads (off[]) and uniform reads (no off[])."""
    rnd = random.Random(300 + K)
    reads = ["".join(rnd.choice("ACGT") for _ in range(rnd.choice([0, 1, K - 1, K, K + 1, K + 9, 140]))) for _ in range(200)]
    reads += ["A" * (K + 25), "ACGT" * 40, "T" * (K + 3), ""]
    p, o = oracle.pack_strings(reads)
    ek, ec, en = oracle.count(p, o, K)
    W = ek.shape[1]
    pb = min(8, 2 * K)
    top = 2 * K - 64 * (W - 1)
    parts = sorted({0, 3 % (1 << pb), (1 << pb) - 1, 77 % (1 << pb)})
    keys, nw = oracle.sample_prefix(p, o, K, pb, parts)
    assert nw == en
    sk, sc = oracle.count_keys(keys, K)
    if pb <= top:
        pre = (ek[:, 0] >> np.uint64(top - pb)).astype(np.int64)
    else:  # the prefix reaches into word 1
        pre = ((ek[:, 0] << np.uint64(pb - top)) | (ek[:, 1] >> np.uint64(64 - (pb - top)))).astype(np.int64)
    m = np.isin(pre, parts)
    assert (sk == ek[m]).all() and (sc == ec[m]).all() and int(sc.sum()) == len(keys)
    sp = oracle.synth_params(100_000, 100)
    pu, ou = oracle.synth_reads(sp, 0, 5_000)
    ku, nu = oracle.sample_prefix(pu, None, K, pb, parts, n_reads=5_000, read_len=100)
    kr, nr = oracle.sample_prefix(pu, ou, K, pb, parts)
    assert nu == nr and (oracle.count_keys(ku, K)[0] == oracle.count_keys(kr, K)[0]).all()
    assert (oracle.count_keys(ku, K)[1] == oracle.count_keys(kr, K)[1]).all()


def _prefix(kmers, K, pb):
    """leading pb bits of each canonical k-mer (uint64[n, W] rows, most significant word first)"""
    top = 2 * K - 64 * (kmers.shape[1] - 1)
    if pb <= top:
        return (kmers[:, 0] >> np.uint64(top - pb)).astype(np.int64)
    return ((kmers[:, 0] << np.uint64(pb - top)) | (kmers[:, 1] >> np.uint64(64 - (pb - top)))).astype(np.int64)


@pytest.mark.parametrize("K", [1, 16, 25, 33, 96])
def test_sampled_partition_positions_match_full_records(oracle, K):
    """oracle_sample_prefix_pos (what the wide-position GPU tests compare record by record where the full oracle cannot
    run): its instances, sorted by (k-mer, position), are exactly the full oracle's occurrence records of the same
    partitions, and every sampled window's count is the full oracle's read_freqs there -- ragged and uniform reads."""
    rnd = random.Random(700 + K)
    reads = ["".join(rnd.choice("ACGT") for _ in range(rnd.choice([0, 1, K - 1, K, K + 1, K + 9, 140]))) for _ in range(200)]
    reads += ["A" * (K + 25), "ACGT" * 40, "T" * (K + 3), "", "CG" * (K + 4)]
    reads.append(reads[5].translate(str.maketrans("ACGT", "TGCA"))[::-1])
    sp = oracle.synth_params(100_000, 100)
    pu, ou = oracle.synth_reads(sp, 0, 3_000)
    pb = min(8, 2 * K)
    parts = sorted({0, 5 % (1 << pb), 77 % (1 << pb), (1 << pb) - 1})
    for p, o, uniform in ((*oracle.pack_strings(reads), False), (pu, ou, True)):
        ek, ec, en = oracle.count(p, o, K)
        ero, erid, epos = oracle.occurrences(p, o, K, ek, en)
        if uniform:
            keys, pos, nw = oracle.sample_prefix_pos(p, None, K, pb, parts, n_reads=len(o) - 1, read_len=100)
        else:
            keys, pos, nw = oracle.sample_prefix_pos(p, o, K, pb, parts)
        assert nw == en
        assert (keys == oracle.sample_prefix(p, o, K, pb, parts)[0]).all()    # the keys-only form sees the same instances
        assert (np.diff(pos >> np.uint64(1)).astype(np.int64) > 0).all()      # ascending by position
        # sort by (k-mer, position): a stable sort by k-mer keeps the position order
        order = np.lexsort(keys.T[::-1]) if len(keys) else np.zeros(0, np.int64)
        keys, pos = keys[order], pos[order]
        m = np.isin(_prefix(ek, K, pb), parts)
        inst = np.repeat(m, ec.astype(np.int64))
        assert (keys == np.repeat(ek[m], ec[m].astype(np.int64), axis=0)).all()
        q = (pos >> np.uint64(1)).astype(np.int64)
        rid = np.searchsorted(o.astype(np.int64), q, side="right") - 1
        p1 = q - o.astype(np.int64)[rid] + 1
        assert (rid == erid[inst]).all()
        assert (np.where(pos & np.uint64(1), -p1, p1) == epos[inst]).all()
        sk, sc = oracle.count_keys(keys, K)
        assert (sk == ek[m]).all() and (sc == ec[m]).all()
        erf = oracle.read_freqs(p, o, K, ek, ec)
        assert (erf[q] == np.repeat(sc, sc.astype(np.int64))).all()
