"""GPU parity tests: the CUDA path, called through the C ABI, against the CPU oracle on the same
inputs -- bit-exact k-mers, counts, spectra and table lookups.  Run with `-m gpu` on a B200.

Parity is UNPINNED in the sense of SURVEY.md section 8(c): the oracle is a spec-derived restatement
cross-checked by a second independent oracle and hand-computed vectors; the reference source was
not available to generate golden outputs."""
import json
import os
import random

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

GOLD = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "known_answers.json")))
RC = str.maketrans("ACGT", "TGCA")


def _to_int(row):
    W = len(row)
    return sum(int(row[j]) << (64 * (W - 1 - j)) for j in range(W))


def _run(packed, off, K, prefix_bits=0, uniform=None, want_counts=True):
    from allpathslg_b200 import KmerCounter

    kc = KmerCounter(K, prefix_bits=prefix_bits, want_counts=want_counts)
    if uniform:
        kc.add_reads_uniform(packed, uniform[0], uniform[1])
    else:
        kc.add_reads(packed, off)
    kc.finish()
    return kc


def _assert_equal_to_oracle(oracle, kc, packed, off, K, check_table=True):
    ek, ec, en = oracle.count(packed, off, K)
    ni, nd = kc.totals()
    assert (ni, nd) == (en, len(ek))
    es = oracle.spectrum(ec)
    gs = kc.spectrum()
    assert len(gs) == len(es) and (gs == es).all()
    f, m = kc.spectrum_sparse()
    assert (f == np.nonzero(es)[0]).all() and (m == es[np.nonzero(es)[0]]).all()
    if check_table:
        gk, gc = kc.counts()
        assert (gk == ek).all()
        assert (gc.astype(np.uint64) == ec).all()
    return ek, ec


# ------------------------------------------------------------------ known answers
@pytest.mark.parametrize("v", GOLD["hand"], ids=lambda v: "%s-K%d" % ("+".join(v["reads"]) or "empty", v["K"]))
def test_hand_vectors(oracle, v):
    p, o = oracle.pack_strings(v["reads"])
    kc = _run(p, o, v["K"])
    gk, gc = kc.counts()
    assert [_to_int(r) for r in gk] == v["kmers"]
    assert [int(x) for x in gc] == v["counts"]
    assert [int(x) for x in kc.spectrum()] == v["spectrum"]
    kc.close()


@pytest.mark.parametrize("s", GOLD["synth"], ids=lambda s: "G%d-K%d" % (s["genome_len"], s["K"]))
def test_synth_golden(oracle, s):
    sp = oracle.synth_params(s["genome_len"], s["read_len"])
    p, o = oracle.synth_reads(sp, 0, s["n_reads"])
    kc = _run(p, o, s["K"], uniform=(s["n_reads"], s["read_len"]))
    assert kc.totals() == (s["n_instances"], s["n_distinct"])
    assert [int(x) for x in kc.spectrum()] == s["spectrum"]
    gk, gc = kc.counts()
    M = (1 << 61) - 1
    chk = 0
    for row, cnt in zip(gk, gc):
        chk = (chk + (_to_int(row) % M) * int(cnt)) % M
    assert chk == s["table_checksum"]
    kc.close()


# ------------------------------------------------------------------ ragged / edge cases, every key width
@pytest.mark.parametrize("K", [1, 2, 3, 11, 16, 20, 24, 25, 26, 27, 31, 32, 33, 48, 63, 64, 65, 96])
@pytest.mark.parametrize("prefix_bits", [0, 12])
def test_ragged_reads(oracle, K, prefix_bits):
    rnd = random.Random(1000 + K)
    reads = ["".join(rnd.choice("ACGT") for _ in range(rnd.choice([0, 1, K - 1, K, K + 1, K + 7, 150, 100])))
             for _ in range(300)]
    reads += ["A" * (K + 300), "ACGT" * 100, reads[3], "T" * (K + 20), "", "CG" * (K + 5)]
    reads.append(reads[7].translate(RC)[::-1])
    p, o = oracle.pack_strings(reads)
    kc = _run(p, o, K, prefix_bits=prefix_bits)
    ek, ec = _assert_equal_to_oracle(oracle, kc, p, o, K)
    assert kc.window_upper() == kc.totals()[0]   # the instance count kept at ingest is exact, short reads included
    # frequency-table lookups: present k-mers (both strands), absent k-mers
    if len(ek):
        idx = np.random.RandomState(K).randint(0, len(ek), size=min(len(ek), 500))
        assert (kc.lookup(ek[idx], canonicalise=False).astype(np.uint64) == ec[idx]).all()
        assert (kc.lookup(ek[idx], canonicalise=True).astype(np.uint64) == ec[idx]).all()
        W = ek.shape[1]
        q = np.random.RandomState(K + 1).randint(0, 2 ** 62, size=(300, W), dtype=np.int64).astype(np.uint64)
        if 2 * K < 64 * W:
            q[:, 0] &= np.uint64((1 << (2 * K - 64 * (W - 1))) - 1)
        assert (kc.lookup(q, canonicalise=True).astype(np.uint64) == oracle.lookup(ek, ec, K, q, True)).all()
    # per-position frequencies of the reads (what error correction asks)
    rf = kc.read_freqs()
    erf = oracle.read_freqs(p, o, K, ek, ec)
    erf32 = np.where(erf == np.uint64(0xFFFFFFFFFFFFFFFF), np.uint64(0xFFFFFFFF), erf).astype(np.uint32)
    assert (rf == erf32).all()
    # the whole store goes through the bulk form (bucket scatter + per-bucket resolution); sub-ranges through the
    # per-window table search: both must agree with the oracle
    tb = len(erf32)
    if tb > 40:
        assert (kc.read_freqs(0, tb - 1) == erf32[:tb - 1]).all()
        assert (kc.read_freqs(17, tb - 30) == erf32[17:tb - 13]).all()
    kc.close()


@pytest.mark.parametrize("K", [5, 25, 40, 96])
@pytest.mark.parametrize("prefix_bits", [0, 4])
def test_low_complexity_oversize_buckets(oracle, K, prefix_bits):
    """poly-A / tandem repeats: buckets far beyond shared-memory capacity (range splitting in k_local3 /
    k_local4; the k_big path when those kernels are switched off)."""
    rnd = random.Random(K)
    reads = ["A" * 200] * 400 + ["ACGTACGTAC" * 20] * 300 + ["".join(rnd.choice("AC") for _ in range(120)) for _ in range(500)]
    p, o = oracle.pack_strings(reads)
    kc = _run(p, o, K, prefix_bits=prefix_bits)
    g = kc.geometry()
    assert g["n_big"] > 0 or g["elem_bytes"] == 4 or K <= 32 or os.environ.get("APGK_LOCAL4") == "all"  # the hash kernels (k_local3 / k_local4) split ranges instead of using k_big
    _assert_equal_to_oracle(oracle, kc, p, o, K)
    kc.close()


def test_huge_multiplicity_single_kmer(oracle):
    """One k-mer with > 65535 instances exercises the spectrum overflow list and the digit-skipping walk."""
    reads = ["A" * 1000] * 200 + ["C" * 500] * 7
    p, o = oracle.pack_strings(reads)
    for K in (25, 33):
        kc = _run(p, o, K)
        _assert_equal_to_oracle(oracle, kc, p, o, K)
        kc.close()


@pytest.mark.parametrize("K,prefix_bits", [(16, 2), (16, 6), (13, 4), (10, 2)])
def test_range_splitting_big_distinct_buckets(oracle, K, prefix_bits):
    """32-bit-remainder path with buckets far larger than the shared-memory table and almost all keys
    distinct: k_local3 has to split key ranges repeatedly (and still emit in ascending order)."""
    rnd = np.random.RandomState(K * 31 + prefix_bits)
    n_reads, L = 6000, 150
    bases = rnd.randint(0, 4, size=n_reads * L).astype(np.uint8)
    packed = np.zeros((n_reads * L + 31) // 32 * 8 + 8, dtype=np.uint8)
    for sh in range(4):
        part = bases[sh::4]
        packed[: len(part)] |= part << (2 * sh)
    off = np.arange(n_reads + 1, dtype=np.uint64) * np.uint64(L)
    kc = _run(packed, off, K, prefix_bits=prefix_bits, uniform=(n_reads, L))
    g = kc.geometry()
    assert g["elem_bytes"] == 4 and g["n_big"] == 0
    _assert_equal_to_oracle(oracle, kc, packed, off, K)
    kc.close()


def test_huge_multiplicity_32bit_path(oracle):
    """poly-A / poly-C floods on the 32-bit-remainder path: one key holds > 65535 instances of a bucket."""
    reads = ["A" * 1000] * 300 + ["C" * 700] * 11 + ["ACGTTGCA" * 50] * 40
    p, o = oracle.pack_strings(reads)
    for K, P in ((13, 0), (12, 4), (16, 8)):
        kc = _run(p, o, K, prefix_bits=P)
        assert kc.geometry()["elem_bytes"] == 4
        _assert_equal_to_oracle(oracle, kc, p, o, K)
        kc.close()


_OCC_CHILD = (
    "import sys, hashlib; sys.path.insert(0, %r)\n"
    "import numpy as np\n"
    "from allpathslg_b200 import KmerCounter\n"
    "K, P = int(sys.argv[1]), int(sys.argv[2])\n"
    "d = np.load(sys.argv[3])\n"
    "kc = KmerCounter(K, prefix_bits=P); kc.add_reads(d['p'], d['o']); kc.finish(); kc.build_occurrences()\n"
    "ro, rid, pos = kc.occurrences()\n"
    "print(kc.geometry()['REM'], hashlib.sha256(ro.tobytes() + rid.tobytes() + pos.tobytes()).hexdigest())\n")


@pytest.mark.parametrize("K,prefix_bits,rem", [(17, 2, 32), (22, 12, 32), (26, 20, 32), (28, 24, 32), (26, 21, 31)])
def test_32bit_remainders_using_every_bit(oracle, K, prefix_bits, rem, tmp_path):
    """4-byte level-1 elements whose remainder fills all 32 bits (P = 2K - 32): counted by k_local2 / k_local / k_big,
    not k_local3, which takes REM <= 31 (its widest case, REM = 31, is the last row).  (17, 2) has 4 buckets, so
    poly-A floods them past the shared-memory table and k_big runs on 32-bit remainders.  Table, spectrum, lookups,
    read_freqs (bulk and per window) and occurrence records against the full oracle; the records both with remainder
    and position packed in one word and, in a child process with APGK_OCC_NOPACK, in two arrays."""
    import hashlib
    import subprocess
    import sys

    rnd = random.Random(1000 + K)
    reads = ["".join(rnd.choice("ACGT") for _ in range(rnd.choice([0, 1, K - 1, K, K + 1, K + 7, 150, 100])))
             for _ in range(300)]
    reads += ["A" * (K + 300), "ACGT" * 100, reads[3], "T" * (K + 20), "", "CG" * (K + 5)]
    reads.append(reads[7].translate(RC)[::-1])
    reads += ["A" * 200] * 20 + ["T" * 200] * 20 + ["ACGT" * 50] * 20
    p, o = oracle.pack_strings(reads)
    kc = _run(p, o, K, prefix_bits=prefix_bits)
    g = kc.geometry()
    assert (g["REM"], g["elem_bytes"]) == (rem, 4)
    if (K, prefix_bits) == (17, 2):
        assert g["n_big"] > 0
    ek, ec = _assert_equal_to_oracle(oracle, kc, p, o, K)
    en = int(ec.sum())
    idx = np.random.RandomState(K).randint(0, len(ek), size=min(len(ek), 2000))
    assert (kc.lookup(ek[idx], canonicalise=False).astype(np.uint64) == ec[idx]).all()
    t, rc = ek[idx, 0].copy(), np.zeros(len(idx), dtype=np.uint64)   # the other strand of each k-mer
    for _ in range(K):
        rc = (rc << np.uint64(2)) | (np.uint64(3) - (t & np.uint64(3)))
        t >>= np.uint64(2)
    assert (kc.lookup(rc[:, None], canonicalise=True).astype(np.uint64) == ec[idx]).all()
    q =np.random.RandomState(K + 1).randint(0, 2 ** 62, size=(2000, 1), dtype=np.int64).astype(np.uint64)
    q[:, 0] &= np.uint64((1 << (2 * K)) - 1)
    assert (kc.lookup(q, canonicalise=True).astype(np.uint64) == oracle.lookup(ek, ec, K, q, True)).all()
    assert (kc.lookup(q, canonicalise=False).astype(np.uint64) == oracle.lookup(ek, ec, K, q, False)).all()
    erf = oracle.read_freqs(p, o, K, ek, ec)
    erf32 = np.where(erf == np.uint64(0xFFFFFFFFFFFFFFFF), np.uint64(0xFFFFFFFF), erf).astype(np.uint32)
    tb = len(erf32)
    assert (kc.read_freqs() == erf32).all()
    assert (kc.read_freqs(0, tb - 1) == erf32[:tb - 1]).all()
    assert (kc.read_freqs(17, tb - 30) == erf32[17:tb - 13]).all()
    info = kc.build_occurrences()
    assert info["n_occ"] == en
    ero, erid, epos = oracle.occurrences(p, o, K, ek, en)
    ro, rid, pos = kc.occurrences()
    assert (ro == ero).all() and (rid == erid).all() and (pos == epos).all()
    kc.close()
    np.savez(tmp_path / "reads.npz", p=p, o=o)
    env = dict(os.environ)
    env.pop("APGK_OCC_DIRECT", None)
    env["APGK_OCC_NOPACK"] = "1"
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", _OCC_CHILD % root, str(K), str(prefix_bits), str(tmp_path / "reads.npz")],
                       capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stderr
    got_rem, got_sha = r.stdout.split()
    assert int(got_rem) == rem
    assert got_sha == hashlib.sha256(ero.tobytes() + erid.tobytes() + epos.tobytes()).hexdigest()


@pytest.mark.parametrize("K", [20, 25, 31, 48, 96])
def test_kmer_space_rounds(oracle, K):
    """A small per-round budget forces several k-mer-space rounds (the SortKmers 'passes' / KmerParcels
    'parcels' mechanism): results, table order, lookup index and spectrum must not change."""
    from allpathslg_b200 import KmerCounter

    sp = oracle.synth_params(400_000, 150)
    p, o = oracle.synth_reads(sp, 0, 20_000)
    ek, ec, en = oracle.count(p, o, K)
    # (outer budget, inner budget): one level of rounds, then outer rounds (one filtered extraction each) cut
    # into inner rounds (second partition level + counting over sub-ranges of the extracted keys)
    for budget, inner in ((en // 5 + 1, 0), (en // 2 + 1, 0), (en // 2 + 1, en // 7 + 1), (en + 1, en // 4 + 1)):
        kc = KmerCounter(K, max_round_keys=budget, max_inner_keys=inner)
        kc.add_reads_uniform(p, 20_000, 150)
        kc.finish()
        assert kc.geometry()["n_rounds"] >= (2 if not inner else 4)
        _assert_equal_to_oracle(oracle, kc, p, o, K)
        idx = np.random.RandomState(K).randint(0, len(ek), size=2000)
        assert (kc.lookup(ek[idx], canonicalise=False).astype(np.uint64) == ec[idx]).all()
        rf = kc.read_freqs(0, 30_000)
        erf = oracle.read_freqs(p, o[:201], K, ek, ec)
        erf32 = np.where(erf == np.uint64(0xFFFFFFFFFFFFFFFF), np.uint64(0xFFFFFFFF), erf).astype(np.uint32)
        assert (rf == erf32).all()
        kc.close()


@pytest.mark.parametrize("K,n_reads", [(25, 40_000), (20, 30_000), (24, 3_000)])
def test_bulk_write_out_scatter(oracle, K, n_reads, monkeypatch):
    """APGK_BULK=1: the level-1 scatter whose runs leave the shared-memory stage as TMA bulk copies
    (cp.async.bulk.global.shared::cta, per-bin carry of the incomplete 16-byte granule) -- the measured alternative
    to the default register write-out must give the same table, also over several k-mer-space rounds."""
    from allpathslg_b200 import KmerCounter

    monkeypatch.setenv("APGK_BULK", "1")
    sp = oracle.synth_params(300_000, 100)
    p, o = oracle.synth_reads(sp, 0, n_reads)
    ek, ec, en = oracle.count(p, o, K)
    for budget in (0, en // 3 + 1):
        kc = KmerCounter(K, max_round_keys=budget, prefix_bits=20)   # 32-bit remainders also for these small inputs
        kc.add_reads_uniform(p, n_reads, 100)
        kc.finish()
        assert kc.geometry()["elem_bytes"] == 4
        _assert_equal_to_oracle(oracle, kc, p, o, K)
        kc.close()


def test_empty_and_short_inputs(oracle):
    from allpathslg_b200 import KmerCounter

    kc = KmerCounter(25)
    kc.finish()  # no reads at all
    assert kc.totals() == (0, 0) and list(kc.spectrum()) == [0]
    p, o = oracle.pack_strings(["ACGT", "", "AC"])  # all shorter than K
    kc.add_reads(p, o)
    kc.finish()
    assert kc.totals() == (0, 0)
    assert len(kc.counts()[0]) == 0
    kc.close()


# ------------------------------------------------------------------ streaming ingest
@pytest.mark.parametrize("K", [25, 64])
def test_batched_add_reads_equals_one_shot(oracle, K):
    rnd = random.Random(K)
    reads = ["".join(rnd.choice("ACGT") for _ in range(rnd.choice([37, 100, 101, 150, 3, K]))) for _ in range(2000)]
    p, o = oracle.pack_strings(reads)
    from allpathslg_b200 import KmerCounter

    kc = KmerCounter(K)
    cuts = [0, 1, 7, 500, 501, 1300, 2000]
    for a, b in zip(cuts[:-1], cuts[1:]):
        kc.add_reads(p, o[a:b + 1])  # offsets index into the same packed buffer: unaligned batch starts
    kc.finish()
    _assert_equal_to_oracle(oracle, kc, p, o, K)
    assert kc.read_store_info() == (int(o[-1]), 2000)
    # the device store is the concatenation of the batches
    exp = kc.export_reads()
    nb = int(o[-1])
    assert (exp[: nb // 4] == p[: nb // 4]).all()
    # reset + reuse
    kc.reset()
    kc.add_reads(p, o[:101])
    kc.finish()
    _assert_equal_to_oracle(oracle, kc, p, o[:101], K)
    kc.close()


def test_device_generator_matches_oracle(oracle):
    from allpathslg_b200 import KmerCounter, synth_params

    for (G, L, r0, n) in [(100003, 100, 0, 4000), (7001, 36, 17, 1111), (250000, 250, 5, 900)]:
        p, _ = oracle.synth_reads(oracle.synth_params(G, L), r0, n)
        kc = KmerCounter(25)
        kc.synth_reads(synth_params(G, L), r0, n)
        got = kc.export_reads()
        assert (got[: len(p)] == p[: len(got)]).all()
        kc.close()


# ------------------------------------------------------------------ BASELINE.json configurations
def test_config1_ecoli_k25(oracle):
    """configs[0]: E. coli-size genome (4.6 Mb), 2.3 M x 100 bp reads (50x), K=25 -- full diff."""
    sp = oracle.synth_params(4_600_000, 100)
    p, o = oracle.synth_reads(sp, 0, 2_300_000)
    kc = _run(p, o, 25, uniform=(2_300_000, 100))
    _assert_equal_to_oracle(oracle, kc, p, o, 25)
    assert kc.totals()[0] == 174_800_000
    kc.close()


def test_config2_saureus_k24_find_errors_tables(oracle):
    """configs[1]: S. aureus-size genome (2.9 Mb), frag + jump libraries (2 x 1.45 M x 100 bp),
    K=24 tables + the per-position lookups a FindErrors pass makes."""
    G = 2_900_000
    frag, _ = oracle.synth_reads(oracle.synth_params(G, 100), 0, 1_450_000)
    jump, _ = oracle.synth_reads(oracle.synth_params(G, 100, seed_r=0x5EED0101, seed_e=0x5EED0102), 0, 1_450_000)
    nb = 1_450_000 * 100
    packed = np.concatenate([frag[: nb // 4], jump[: nb // 4], np.zeros(16, np.uint8)])
    off = np.arange(2_900_001, dtype=np.uint64) * np.uint64(100)
    from allpathslg_b200 import KmerCounter

    kc = KmerCounter(24)
    kc.add_reads_uniform(frag, 1_450_000, 100)
    kc.add_reads_uniform(jump, 1_450_000, 100)
    kc.finish()
    ek, ec = _assert_equal_to_oracle(oracle, kc, packed, off, 24)
    assert kc.totals()[0] == 2_900_000 * 77
    # FindErrors-style lookups on a slice of the reads (both libraries)
    for first in (0, nb - 50_000):
        n = 100_000
        rf = kc.read_freqs(first, n)
        sub_off = off[first // 100: first // 100 + n // 100 + 1]
        erf = oracle.read_freqs(packed, sub_off, 24, ek, ec)
        erf32 = np.where(erf == np.uint64(0xFFFFFFFFFFFFFFFF), np.uint64(0xFFFFFFFF), erf).astype(np.uint32)
        assert (rf == erf32).all()
    kc.close()


@pytest.mark.parametrize("K,L,n", [(25, 100, 3_000_000), (96, 100, 3_000_000), (96, 250, 600_000), (20, 250, 400_000),
                                   (48, 250, 400_000), (64, 250, 400_000)])
def test_config3_and_5_scaled(oracle, K, L, n):
    """configs[2] / configs[4] at a size the oracle finishes in seconds: K=25 and K=96 on 100 bp reads,
    and the K sweep on 250 bp reads (1-, 2- and 3-word k-mers)."""
    sp = oracle.synth_params(5_000_000, L)
    p, o = oracle.synth_reads(sp, 0, n)
    kc = _run(p, o, K, uniform=(n, L))
    _assert_equal_to_oracle(oracle, kc, p, o, K)
    kc.close()


# ------------------------------------------------------------------ size-independent properties at scale
def test_properties_at_scale():
    """20 M reads (1.52 G instances), too big for a host diff in a test: exact invariants instead.
    sum f*spectrum[f] == instances; sum spectrum == distinct; table sorted strictly ascending;
    sum counts == instances; idempotence; every count >= 1; lookups of table rows return their count."""
    from allpathslg_b200 import KmerCounter, synth_params

    n, L, K = 20_000_000, 100, 25
    kc = KmerCounter(K)
    kc.synth_reads(synth_params(30_000_000, L), 0, n)
    kc.finish()
    ni, nd = kc.totals()
    assert ni == n * (L - K + 1)
    spec = kc.spectrum()
    assert int((spec * np.arange(len(spec), dtype=np.uint64)).sum()) == ni
    assert int(spec.sum()) == nd
    step = 8_000_000
    prev_last = None
    tot = 0
    hist = np.zeros(len(spec), dtype=np.uint64)
    for first in range(0, nd, step):
        m = min(step, nd - first)
        k, c = kc.counts(first, m)
        kk = k[:, 0]
        assert (kk[1:] > kk[:-1]).all()
        if prev_last is not None:
            assert kk[0] > prev_last
        prev_last = kk[-1]
        assert c.min() >= 1
        tot += int(c.sum(dtype=np.uint64))
        hist += np.bincount(c.astype(np.int64), minlength=len(spec)).astype(np.uint64)
        if first == 0:
            assert (kc.lookup(k[:5000], canonicalise=False) == c[:5000]).all()
    assert tot == ni
    assert (hist == spec).all()
    # idempotence
    kc.finish()
    assert kc.totals() == (ni, nd) and (kc.spectrum() == spec).all()
    kc.close()


def test_strand_and_order_invariance(oracle):
    """Reverse-complementing every read, or shuffling read order, leaves the table unchanged."""
    rnd = random.Random(3)
    reads = ["".join(rnd.choice("ACGT") for _ in range(150)) for _ in range(3000)]
    rcs = [r.translate(RC)[::-1] for r in reads]
    shuf = list(reads)
    rnd.shuffle(shuf)
    for K in (25, 40):
        ref = None
        for rs in (reads, rcs, shuf):
            p, o = oracle.pack_strings(rs)
            kc = _run(p, o, K)
            cur = (kc.counts(), kc.spectrum())
            kc.close()
            if ref is None:
                ref = cur
            else:
                assert (cur[0][0] == ref[0][0]).all() and (cur[0][1] == ref[0][1]).all() and (cur[1] == ref[1]).all()


def test_streamed_ingest_matches(oracle):
    """APGK_ASYNC_INGEST: add_reads_uniform returns before its copy has landed and finish follows the copy
    slice by slice; results must be identical, also after reset + re-ingest and with a sync append behind."""
    import torch

    from allpathslg_b200 import KmerCounter

    L, n = 100, 400_000
    sp = oracle.synth_params(2_000_000, L)
    p, o = oracle.synth_reads(sp, 0, n)
    ek, ec, en = oracle.count(p, o, 25)
    host = torch.from_numpy(p.copy()).pin_memory()
    kc = KmerCounter(25, async_ingest=True)
    for _ in range(2):
        kc.reset()
        kc.add_reads_uniform(host.data_ptr(), n, L)
        kc.finish()
        gk, gc = kc.counts()
        assert kc.totals() == (en, len(ek)) and (gk == ek).all() and (gc.astype(np.uint64) == ec).all()
    # a second, synchronous append behind a pending streamed one, then read_freqs (which must wait for the copy)
    kc.reset()
    half = n // 2
    kc.add_reads_uniform(host.data_ptr(), half, L)
    p2, _ = oracle.synth_reads(sp, half, n - half)
    kc.add_reads_uniform(p2, n - half, L)
    kc.finish()
    assert kc.totals() == (en, len(ek))
    assert (kc.spectrum() == oracle.spectrum(ec)).all()
    kc.close()


# ------------------------------------------------------------------ multi-GPU building blocks on one GPU
@pytest.mark.parametrize("K,world", [(25, 2), (25, 8), (64, 4), (96, 3)])
def test_owner_partition_and_key_ingest(oracle, K, world):
    """apgk_owner_plan/scatter group this rank's k-mers by owner exactly as apgk_owner_of says;
    counting each owner's group with apgk_finish_keys_device and summing spectra reproduces the
    single-GPU result (the N-rank pipeline emulated on one GPU, rank after rank)."""
    import torch

    from allpathslg_b200 import KmerCounter, owner_of

    sp = oracle.synth_params(300_000, 100)
    p, o = oracle.synth_reads(sp, 0, 30_000)
    ek, ec, en = oracle.count(p, o, K)
    W = ek.shape[1]
    kc = KmerCounter(K)
    kc.add_reads_uniform(p, 30_000, 100)
    cnts = kc.owner_plan(world)
    assert int(cnts.sum()) == en
    own = owner_of(K, ek, world)
    exp_cnts = np.array([int(ec[own == r].sum()) for r in range(world)], dtype=np.uint64)
    assert (cnts == exp_cnts).all()
    buf = torch.empty(en * W, dtype=torch.int64, device="cuda")
    kc.owner_scatter(buf.data_ptr())
    torch.cuda.synchronize()
    host = buf.cpu().numpy().astype(np.uint64).reshape(-1, W)
    total_spec = np.zeros(1, dtype=np.uint64)
    start = 0
    n_distinct = 0
    for r in range(world):
        grp = host[start:start + int(cnts[r])]
        assert (owner_of(K, grp, world) == r).all()
        kr = KmerCounter(K, max_round_keys=(int(cnts[r]) // 3 + 1) if r == 0 else 0)  # rank 0's shard in 3+ rounds
        kr.finish_keys_device(buf.data_ptr() + start * W * 8, int(cnts[r]))
        gk, gc = kr.counts()
        sel = own == r
        assert (gk == ek[sel]).all() and (gc.astype(np.uint64) == ec[sel]).all()
        s = kr.spectrum()
        if len(s) > len(total_spec):
            total_spec = np.concatenate([total_spec, np.zeros(len(s) - len(total_spec), np.uint64)])
        total_spec[: len(s)] += s
        n_distinct += kr.totals()[1]
        kr.close()
        start += int(cnts[r])
    es = oracle.spectrum(ec)
    assert n_distinct == len(ek)
    assert len(total_spec) == len(es) and (total_spec == es).all()
    kc.close()


@pytest.mark.parametrize("exchange", ["recv", "peer"])
@pytest.mark.parametrize("K,world,n_reads", [(25, 2, 30_000), (25, 5, 30_000), (20, 3, 20_000), (48, 3, 12_000), (96, 2, 8_000)])
def test_partition_first_shards_emulated_ranks(oracle, K, world, n_reads, exchange):
    """The partition-first multi-GPU path emulated on one GPU: every "rank" partitions its share of the
    reads (apgk_partition), the exchange of bucket ranges is done here with host copies exactly as
    dist.sharded_count does it with all_to_all, every rank counts its range (apgk_count_pieces).
    The union of the shard tables and the summed spectra must equal the oracle on all the reads;
    every shard table must also answer lookups for its own k-mers (and 0 for the others)."""
    import torch

    from allpathslg_b200 import KmerCounter
    from allpathslg_b200.dist import balanced_splitters

    L = 100
    sp = oracle.synth_params(200_000, L)
    p, o = oracle.synth_reads(sp, 0, n_reads)
    ek, ec, en = oracle.count(p, o, K)
    W = ek.shape[1]
    share = [(n_reads * r) // world for r in range(world + 1)]
    if world == 5:
        share[3] = share[2]  # one rank without reads
    kcs = []
    for r in range(world):
        kc = KmerCounter(K)
        n = share[r + 1] - share[r]
        if n:
            pr, _ = oracle.synth_reads(sp, share[r], n)
            kc.add_reads_uniform(pr, n, L)
        kcs.append(kc)
    P = kcs[0].choose_prefix_bits(max(kc.window_upper() for kc in kcs))
    sizes, elems, eb, eptrs, subs = [], [], None, [], []
    for kc in kcs:
        kc.partition(P)
        sp_, nb, ep, eb_, ne = kc.partition_info()
        eptrs.append(ep)
        d2, subp = kc.partition_subsizes(max(0, (world - 1).bit_length()))
        subs.append(torch.as_tensor(_CudaView(subp, nb << d2, "<i4"), device="cuda").clone())
        eb = eb_ if eb is None else eb
        assert eb_ == eb and nb == 1 << P
        sz = torch.empty(nb, dtype=torch.int64, device="cuda")
        sz.copy_(torch.as_tensor(_CudaView(sp_, nb, "<i8"), device="cuda"))
        sizes.append(sz.cpu().numpy())
        dt = "<i4" if eb == 4 else "<i8"
        words = 1 if eb == 4 else eb // 8
        e = torch.as_tensor(_CudaView(ep, max(ne, 1) * words, dt), device="cuda")[: ne * words].cpu().numpy() if ne else \
            np.zeros(0, dtype=np.int32 if eb == 4 else np.int64)
        elems.append(e)
        assert int(sizes[-1].sum()) == ne
    assert sum(int(s.sum()) for s in sizes) == en
    all_sizes = np.stack(sizes)
    bounds = balanced_splitters(all_sizes.sum(0), world)
    assert bounds[0] == 0 and bounds[-1] == 1 << P and all(a <= b for a, b in zip(bounds, bounds[1:]))
    words = 1 if eb == 4 else eb // 8
    cum = np.concatenate([np.zeros((world, 1), np.int64), np.cumsum(all_sizes, axis=1)], axis=1)
    d_sizes = torch.from_numpy(all_sizes.astype(np.int32)).cuda().contiguous()
    total_spec = np.zeros(1, dtype=np.uint64)
    got_k, got_c = [], []
    per_rank = []
    for r in range(world):
        lo, hi = bounds[r], bounds[r + 1]
        parts = [elems[s][cum[s, lo] * words: cum[s, hi] * words] for s in range(world)]
        seg_off = np.concatenate([[0], np.cumsum([len(x) // words for x in parts])[:-1]]).astype(np.uint64)
        recv = torch.from_numpy(np.concatenate(parts) if sum(len(x) for x in parts) else np.zeros(1, parts[0].dtype)).cuda()
        if exchange == "recv":
            kcs[r].count_pieces(recv.data_ptr(), world, d_sizes.data_ptr(), seg_off, lo, hi)
        else:  # the gather reads every source's own partition buffer (here: the other contexts' buffers)
            ptrs = [None if s == r else (eptrs[s] or 0) for s in range(world)]
            if any(p == 0 for p in ptrs if p is not None):
                ptrs = [None if s == r else (eptrs[s] or recv.data_ptr()) for s in range(world)]  # empty source: any valid pointer
            sub_recv = torch.cat([subs[s][lo << d2: hi << d2] for s in range(world)] + [torch.zeros(1, dtype=torch.int32, device="cuda")])
            for s in range(world):  # the senders' sub-bucket counts add up to their bucket sizes
                assert int(subs[s].sum()) == int(all_sizes[s].sum())
            kcs[r].count_pieces_peer(ptrs, d_sizes.data_ptr(), cum[:, lo].astype(np.uint64), lo, hi, split_bits=d2,
                                     d_sub_sizes=sub_recv.data_ptr() if (r % 2 == 0) else None)  # with and without
        gk, gc = kcs[r].counts()
        got_k.append(gk); got_c.append(gc)
        per_rank.append(kcs[r].totals()[0])
        s = kcs[r].spectrum()
        if len(s) > len(total_spec):
            total_spec = np.concatenate([total_spec, np.zeros(len(s) - len(total_spec), np.uint64)])
        total_spec[: len(s)] += s
    gk = np.concatenate(got_k); gc = np.concatenate(got_c)
    assert len(gk) == len(ek) and (gk == ek).all() and (gc.astype(np.uint64) == ec).all()  # ranges ascend: union is sorted
    es = oracle.spectrum(ec)
    assert len(total_spec) == len(es) and (total_spec == es).all()
    assert sum(per_rank) == en
    if world > 1 and en > 10 * world:
        assert max(per_rank) < 1.25 * en / world + (en >> P) * 64  # balanced up to bucket granularity
    # shard tables answer lookups for their own k-mers only
    pick = ek[:: max(1, len(ek) // 500)]
    exp = ec[:: max(1, len(ek) // 500)]
    tot = np.zeros(len(pick), dtype=np.uint64)
    for r in range(world):
        tot += kcs[r].lookup(pick, canonicalise=False).astype(np.uint64)
    assert (tot == exp).all()
    for kc in kcs:
        kc.close()


@pytest.mark.parametrize("K,world,n_reads", [(25, 3, 30_000), (48, 2, 12_000), (20, 2, 20_000)])
def test_partition_first_rounds_emulated_ranks(oracle, K, world, n_reads):
    """K-mer-space rounds of the partition-first form, emulated on one GPU: the level-0 bucket space is cut into
    the same ranges on every "rank" (dist.plan_rounds on the per-bucket maximum), every round is one
    apgk_partition_range -> exchange -> apgk_count_pieces, and a round's table and spectrum are harvested before
    the next round.  Tables concatenated in (round, rank) order must be the oracle's sorted table."""
    import torch

    from allpathslg_b200 import KmerCounter
    from allpathslg_b200.dist import balanced_splitters, plan_rounds

    L = 100
    sp = oracle.synth_params(200_000, L)
    p, o = oracle.synth_reads(sp, 0, n_reads)
    ek, ec, en = oracle.count(p, o, K)
    share = [(n_reads * r) // world for r in range(world + 1)]
    kcs = []
    for r in range(world):
        kc = KmerCounter(K)
        n = share[r + 1] - share[r]
        pr, _ = oracle.synth_reads(sp, share[r], n)
        kc.add_reads_uniform(pr, n, L)
        kcs.append(kc)
    P = kcs[0].choose_prefix_bits(max(kc.window_upper() for kc in kcs))
    tots = []
    for kc in kcs:
        kc.partition(P)                      # fits here; also leaves the level-0 totals behind
        t, cap = kc.level0_totals()
        assert cap > 0 and int(t.sum()) == kc.partition_info()[4]
        tots.append(t)
    rounds = plan_rounds(np.max(np.stack(tots), axis=0), max(1, en // (3 * world)))
    assert len(rounds) >= 3 and rounds[0][0] == 0 and rounds[-1][1] == len(tots[0])
    got_k, got_c = [], []
    total_spec = np.zeros(1, dtype=np.uint64)
    n_seen = 0
    for lo0, hi0 in rounds:
        sizes, elems, eb = [], [], None
        for kc in kcs:
            kc.partition_range(P, lo0, hi0)
            sp_, nb, ep, eb, ne = kc.partition_info()
            sz = torch.as_tensor(_CudaView(sp_, nb, "<i8"), device="cuda").cpu().numpy()
            dt = "<i4" if eb == 4 else "<i8"
            words = 1 if eb == 4 else eb // 8
            e = torch.as_tensor(_CudaView(ep, max(ne, 1) * words, dt), device="cuda")[: ne * words].cpu().numpy() if ne else \
                np.zeros(0, dtype=np.int32 if eb == 4 else np.int64)
            assert int(sz.sum()) == ne
            sizes.append(sz); elems.append(e)
        all_sizes = np.stack(sizes)
        bounds = balanced_splitters(all_sizes.sum(0), world)
        words = 1 if eb == 4 else eb // 8
        cum = np.concatenate([np.zeros((world, 1), np.int64), np.cumsum(all_sizes, axis=1)], axis=1)
        d_sizes = torch.from_numpy(all_sizes.astype(np.int32)).cuda().contiguous()
        for r in range(world):
            lo, hi = bounds[r], bounds[r + 1]
            parts = [elems[s][cum[s, lo] * words: cum[s, hi] * words] for s in range(world)]
            seg_off = np.concatenate([[0], np.cumsum([len(x) // words for x in parts])[:-1]]).astype(np.uint64)
            recv = torch.from_numpy(np.concatenate(parts) if sum(len(x) for x in parts) else np.zeros(1, parts[0].dtype)).cuda()
            kcs[r].count_pieces(recv.data_ptr(), world, d_sizes.data_ptr(), seg_off, lo, hi)
            gk, gc = kcs[r].counts()
            got_k.append(gk); got_c.append(gc)
            n_seen += kcs[r].totals()[0]
            s = kcs[r].spectrum()
            if len(s) > len(total_spec):
                total_spec = np.concatenate([total_spec, np.zeros(len(s) - len(total_spec), np.uint64)])
            total_spec[: len(s)] += s
    gk = np.concatenate(got_k); gc = np.concatenate(got_c)
    assert n_seen == en
    assert len(gk) == len(ek) and (gk == ek).all() and (gc.astype(np.uint64) == ec).all()
    es = oracle.spectrum(ec)
    assert len(total_spec) == len(es) and (total_spec == es).all()
    for kc in kcs:
        kc.close()


class _CudaView:
    def __init__(self, ptr, n, typestr):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (ptr, False), "version": 2}


# ------------------------------------------------------------------ reference-named host API
def test_reference_named_entry_points(oracle, tmp_path):
    from allpathslg_b200 import KmerFreqTable, KmerParcelsBuilder, KmerSpectrum, SortKmers

    sp = oracle.synth_params(100_000, 100)
    p, o = oracle.synth_reads(sp, 0, 20_000)
    ek, ec, en = oracle.count(p, o, 25)
    es = oracle.spectrum(ec)
    s = KmerSpectrum.from_reads(p, o, 25)
    assert (s.spec == es).all() and s.n_instances() == en and s.n_distinct() == len(ek)
    s.write(tmp_path / "frag_reads.25mer.kspec")
    assert (KmerSpectrum.read(tmp_path / "frag_reads.25mer.kspec").spec == es).all()
    est = s.estimate(read_len=100)
    assert 0.8 * 100_000 < est["genome_size"] < 1.3 * 100_000
    k, c = SortKmers(p, o, 25)
    assert (k == ek).all() and (c.astype(np.uint64) == ec).all()
    b = KmerParcelsBuilder(25, p, o).Build()
    assert b.NumKmersDistinct() == len(ek) and b.NumKmerInstances() == en and (b.Spectrum().spec == es).all()
    b.close()
    t = KmerFreqTable(24, p, o)
    ek24, ec24, _ = oracle.count(p, o, 24)
    assert (t.freq(ek24[:1000], canonicalise=False).astype(np.uint64) == ec24[:1000]).all()
    t.close()


def test_error_codes():
    from allpathslg_b200 import ApgkError, KmerCounter
    from allpathslg_b200 import _lib

    kc = KmerCounter(25, want_counts=False)
    with pytest.raises(ApgkError) as e:
        kc.totals()
    assert e.value.code == _lib.E_STATE
    kc.finish()
    with pytest.raises(ApgkError) as e:
        kc.counts()  # no table was requested
    assert e.value.code == _lib.E_STATE
    with pytest.raises(ApgkError) as e:
        kc.add_reads(np.zeros(8, np.uint8), np.array([5, 3], dtype=np.uint64))
    assert e.value.code == _lib.E_ARG
    kc.close()
