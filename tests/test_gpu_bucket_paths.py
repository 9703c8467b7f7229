"""The per-bucket counting kernels' recovery paths, each shown to run by its counter and checked against the oracle:
k_local2 deferring buckets to k_local, k_big on one-word keys, k_local4's tag collisions and its range splits across
32- and 64-bit key boundaries, k_local3 at its remainder extremes with both thread counts, the sharded count on the
same inputs, and one context reused across geometries and element types.  The inputs are built (and checked without
a GPU) in test_bucket_paths_cpu.py.

APGK_NO_LOCAL4 and APGK_LOCAL4 are read once per process, so the cases that need them run in a child process that
writes its results to an .npz for this process to compare with the oracle."""
import os
import random
import subprocess
import sys

import numpy as np
import pytest

from test_bucket_paths_cpu import (COLLISION_CASES, DEFERRAL_CASES, LOCAL_MAX, collision_input, deferral_input,
                                   k_local2_plan, random_reads, revcomp, row_overflow_input, to_ints, to_words, words)

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


# ------------------------------------------------------------------ run, collect, compare
def _queries(oracle, p, o, K, n=1500):
    """table rows, their reverse complements and random k-mers (mostly absent)"""
    ek, _, _ = oracle.count(p, o, K)
    rng = np.random.RandomState(K)
    rows = ek[rng.randint(0, len(ek), size=min(n, len(ek)))]
    rc = to_words([revcomp(k, K) for k in to_ints(rows)], K)
    W = words(K)
    rnd = rng.randint(0, 1 << 62, size=(n, W), dtype=np.int64).astype(np.uint64) * np.uint64(3)
    if 2 * K < 64 * W:
        rnd[:, 0] &= np.uint64((1 << (2 * K - 64 * (W - 1))) - 1)
    return np.concatenate([rows, rc, rnd])


def _results(kc, q):
    """everything a count answers, as arrays"""
    tb, _ = kc.read_store_info()
    r = dict(totals=np.array(kc.totals(), dtype=np.uint64), spectrum=kc.spectrum())
    r["sp_f"], r["sp_m"] = kc.spectrum_sparse()
    r["kmers"], r["counts"] = kc.counts()
    r["look_c"] = kc.lookup(q, canonicalise=True)
    r["look_n"] = kc.lookup(q, canonicalise=False)
    r["rf"] = kc.read_freqs()
    r["rf_a"] = kc.read_freqs(0, max(tb - 1, 0))
    r["rf_b"] = kc.read_freqs(17, max(tb - 30, 0)) if tb > 40 else np.zeros(0, np.uint32)
    kc.build_occurrences()
    r["ro"], r["rid"], r["pos"] = kc.occurrences()
    return r


def _count(K, P, p, o, q):
    from allpathslg_b200 import KmerCounter

    kc = KmerCounter(K, prefix_bits=P)
    kc.debug_counters(reset=True)
    kc.add_reads(p, o)
    kc.finish()
    r = _results(kc, q)
    g, d = kc.geometry(), kc.debug_counters(reset=True)
    kc.close()
    r.update({"g_" + k: np.int64(v) for k, v in g.items()})
    r.update({"d_" + k: np.int64(v) for k, v in d.items()})
    return r


def _child_main(argv):
    K, P, src, dst = int(argv[0]), int(argv[1]), argv[2], argv[3]
    d = np.load(src)
    np.savez(dst, **_count(K, P, d["p"], d["o"], d["q"]))


_CHILD = "import sys; sys.path[:0] = [%r, %r]\nimport test_gpu_bucket_paths as t\nt._child_main(sys.argv[1:])\n" % (HERE, ROOT)


def _count_in_child(K, P, p, o, q, env, tmp_path):
    np.savez(tmp_path / "in.npz", p=p, o=o, q=q)
    e = dict(os.environ)
    for v in ("APGK_NO_LOCAL4", "APGK_LOCAL4"):
        e.pop(v, None)
    e.update(env)
    out = tmp_path / "out.npz"
    r = subprocess.run([sys.executable, "-c", _CHILD, str(K), str(P), str(tmp_path / "in.npz"), str(out)],
                       capture_output=True, text=True, env=e, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    d = np.load(out)
    return {k: d[k] for k in d.files}


def _same(got, exp, what):
    got, exp = np.asarray(got), np.asarray(exp)
    assert got.shape == exp.shape, "%s: shape %s, oracle %s" % (what, got.shape, exp.shape)
    bad = np.nonzero((got != exp).reshape(len(got), -1).any(axis=1))[0] if got.size else []
    assert len(bad) == 0, "%s: %d rows differ, first at %d: %s, oracle %s" % (what, len(bad), bad[0], got[bad[0]], exp[bad[0]])


def _check(oracle, r, p, o, K, q):
    ek, ec, en = oracle.count(p, o, K)
    _same(r["totals"], np.array([en, len(ek)], dtype=np.uint64), "totals")
    _same(r["kmers"], ek, "table k-mers")
    _same(r["counts"].astype(np.uint64), ec, "table counts")
    es = oracle.spectrum(ec)
    _same(r["spectrum"], es, "spectrum")
    nz = np.nonzero(es)[0]
    _same(r["sp_f"], nz.astype(np.uint64), "sparse spectrum frequencies")
    _same(r["sp_m"], es[nz], "sparse spectrum")
    _same(r["look_c"].astype(np.uint64), oracle.lookup(ek, ec, K, q, True), "lookup (canonicalise)")
    _same(r["look_n"].astype(np.uint64), oracle.lookup(ek, ec, K, q, False), "lookup (as given)")
    erf = oracle.read_freqs(p, o, K, ek, ec)
    erf32 = np.where(erf == np.uint64(0xFFFFFFFFFFFFFFFF), np.uint64(0xFFFFFFFF), erf).astype(np.uint32)
    tb = len(erf32)
    _same(r["rf"], erf32, "read_freqs")
    _same(r["rf_a"], erf32[: max(tb - 1, 0)], "read_freqs [0, end - 1)")
    if tb > 40:
        _same(r["rf_b"], erf32[17: tb - 13], "read_freqs [17, end - 13)")
    ero, erid, epos = oracle.occurrences(p, o, K, ek, en)
    _same(r["ro"], ero, "occurrence run offsets")
    _same(r["rid"], erid, "occurrence read ids")
    _same(r["pos"], epos, "occurrence positions")
    return ek, ec


def _planted_counts(r, planted):
    got = dict(zip(to_ints(r["kmers"]), r["counts"].tolist()))
    return [got.get(k) for k in planted]


# ------------------------------------------------------------------ (a) k_local2 -> k_local, (b) k_big on Key<1>
@pytest.mark.parametrize("K,P,elem", DEFERRAL_CASES, ids=lambda v: str(v))
def test_deferral_to_k_local(oracle, K, P, elem, tmp_path):
    """A sub-bucket over 512 instances and a sort bin over 48 distinct keys each defer their bucket from k_local2 to
    k_local, among ordinary keys of the same and the neighbouring buckets.  Key<1> needs APGK_NO_LOCAL4."""
    reads, planted, where = deferral_input(K, P)
    p, o = oracle.pack_strings(reads)
    q = _queries(oracle, p, o, K)
    if elem == 1:
        r = _count_in_child(K, P, p, o, q, {"APGK_NO_LOCAL4": "1"}, tmp_path)
    else:
        r = _count(K, P, p, o, q)
    assert (int(r["g_REM"]), int(r["g_elem_bytes"])) == (2 * K - P if P < 2 * K else 0, 4 if elem == 4 else 8 * elem)
    assert int(r["g_local_max"]) == LOCAL_MAX[elem]
    ek, ec = _check(oracle, r, p, o, K, q)
    plan = k_local2_plan(ek, ec, K, P, LOCAL_MAX[elem])
    n_def = sum(1 for why in plan.values() if why in ("sub", "bin"))
    assert n_def == (1 if where["cluster"] is None else 2)
    assert int(r["g_n_deferred"]) == n_def and int(r["g_n_big"]) == 0


def test_k_big_on_one_word_keys(oracle, tmp_path):
    """Without k_local4, one-word keys with remainders over 32 bits take k_local2 / k_local / k_big; poly-A and
    tandem repeats overfill buckets past local_max."""
    K, P = 30, 4
    rnd = random.Random(K)
    reads = ["A" * 200] * 400 + ["ACGTACGTAC" * 20] * 300 + ["".join(rnd.choice("AC") for _ in range(120)) for _ in range(500)]
    reads += random_reads(rnd, 300, K)
    p, o = oracle.pack_strings(reads)
    q = _queries(oracle, p, o, K)
    r = _count_in_child(K, P, p, o, q, {"APGK_NO_LOCAL4": "1"}, tmp_path)
    assert (int(r["g_REM"]), int(r["g_elem_bytes"])) == (2 * K - P, 8)
    assert int(r["g_n_big"]) > 0
    ek, ec = _check(oracle, r, p, o, K, q)
    plan = k_local2_plan(ek, ec, K, P, LOCAL_MAX[1])
    assert int(r["g_n_big"]) == sum(1 for why in plan.values() if why == "big")


# ------------------------------------------------------------------ (c) k_local4 tag collisions
@pytest.mark.parametrize("K,P", COLLISION_CASES)
def test_k_local4_tag_collision(oracle, K, P, tmp_path):
    """Two k-mers of one row with the same 32-bit tag: pass B sees them, the range is redone with the next seed, and
    both come back as their own records with their own counts (3 and 5).  W > 1 needs APGK_LOCAL4=all."""
    reads, planted, (a, b) = collision_input(K, P)
    p, o = oracle.pack_strings(reads)
    q = _queries(oracle, p, o, K)
    if words(K) == 1:
        r = _count(K, P, p, o, q)
    else:
        r = _count_in_child(K, P, p, o, q, {"APGK_LOCAL4": "all"}, tmp_path)
    assert (int(r["g_REM"]), int(r["g_elem_bytes"])) == (2 * K - P, 8 * words(K))
    assert int(r["g_n_big"]) == 0 and int(r["g_n_deferred"]) == 0
    assert int(r["d_tag_collisions"]) >= 1
    assert _planted_counts(r, {a: 3, b: 5}) == [3, 5]
    _check(oracle, r, p, o, K, q)


# ------------------------------------------------------------------ (d) k_local4 range splits across word boundaries
@pytest.mark.parametrize("K,P", [(27, 21), (30, 20), (32, 2), (40, 16), (40, 15), (56, 16), (72, 16), (72, 15), (88, 16)],
                         ids=lambda v: str(v))
def test_k_local4_row_overflow_splits(oracle, K, P, tmp_path):
    """REM = 33, 40, 62 (one word), 64, 65, 96 (two words), 128, 129, 160 (three words): a bucket of near-identical
    keys overflows its row, and the range splits walk from the top of the remainder across the 64- and 32-bit
    boundaries down to the keys' differing bits."""
    reads, planted, _ = row_overflow_input(K, P, n_background=50 if P < 6 else 300)
    p, o = oracle.pack_strings(reads)
    q = _queries(oracle, p, o, K)
    if words(K) == 1:
        r = _count(K, P, p, o, q)
    else:
        r = _count_in_child(K, P, p, o, q, {"APGK_LOCAL4": "all"}, tmp_path)
    assert (int(r["g_REM"]), int(r["g_elem_bytes"])) == (2 * K - P, 8 * words(K))
    assert int(r["g_n_big"]) == 0
    assert int(r["d_row_overflows"]) > 0
    assert _planted_counts(r, planted) == list(planted.values())
    _check(oracle, r, p, o, K, q)


# ------------------------------------------------------------------ (e) k_local3
@pytest.mark.parametrize("lm", [None, 256])
@pytest.mark.parametrize("nt", [None, 256])
@pytest.mark.parametrize("K,P", [(12, 23), (12, 22), (16, 24), (20, 9)], ids=lambda v: str(v))
def test_k_local3_remainder_extremes(oracle, K, P, nt, lm, monkeypatch):
    """REM = 1, 2, 8 and 31 with 512 and 256 threads, at the default table size and at 256 keys (many splits)."""
    for var, val in (("APGK_L3_NT", nt), ("APGK_LM", lm)):
        if val is None:
            monkeypatch.delenv(var, raising=False)
        else:
            monkeypatch.setenv(var, str(val))
    rnd = random.Random(K * 100 + P)
    reads = random_reads(rnd, 2000, K) + ["A" * 300] * 30 + ["ACGTTGCA" * 30] * 20 + ["CG" * 80] * 10
    p, o = oracle.pack_strings(reads)
    q = _queries(oracle, p, o, K)
    r = _count(K, P, p, o, q)
    assert (int(r["g_REM"]), int(r["g_elem_bytes"])) == (2 * K - P, 4)
    assert int(r["g_local_max"]) == (lm or LOCAL_MAX[4]) and int(r["g_n_big"]) == 0 and int(r["g_n_deferred"]) == 0
    _check(oracle, r, p, o, K, q)


# ------------------------------------------------------------------ (f) the sharded count
@pytest.mark.parametrize("world", [1, 3])
@pytest.mark.parametrize("case", ["defer-40", "defer-26", "collide-32"])
def test_sharded_count_on_recovery_inputs(oracle, case, world):
    """The inputs of the deferral and tag-collision tests through KmerGroup.local: the shards' tables are the oracle's."""
    from allpathslg_b200 import KmerCounter, KmerGroup
    from test_gpu_group import _check_against_oracle

    kind, K = case.split("-")
    K = int(K)
    if kind == "defer":
        P = {40: 12, 26: 20}[K]
        reads, planted, _ = deferral_input(K, P)
    else:
        P = 10
        reads, planted, (a, b) = collision_input(K, P)
    p, o = oracle.pack_strings(reads)
    kcs = []
    for r in range(world):
        kc = KmerCounter(K, prefix_bits=P)
        pr, orr = oracle.pack_strings(reads[r::world])
        kc.add_reads(pr, orr)
        kcs.append(kc)
    kcs[0].debug_counters(reset=True)
    with KmerGroup.local(kcs) as grp:
        grp.count()
        st = grp.stats()
        assert st["prefix_bits"] == P
        if kind == "collide":
            assert kcs[0].debug_counters(reset=True)["tag_collisions"] >= 1
        _check_against_oracle(oracle, grp, kcs, p, o, K, sorted_by_rank=True)
    for kc in kcs:
        kc.close()


# ------------------------------------------------------------------ 2. one context, many steps
def test_one_context_many_steps(oracle, monkeypatch):
    """One KmerCounter(25) through a stream of steps whose geometry, element type and table size change."""
    from allpathslg_b200 import KmerCounter

    K = 25
    monkeypatch.delenv("APGK_PREFIX_BITS", raising=False)
    kc = KmerCounter(K)

    def check(p, o):
        q = _queries(oracle, p, o, K, n=800)
        r = _results(kc, q)
        _check(oracle, r, p, o, K, q)
        return kc.geometry()

    # 1. ragged reads, automatic prefix: full one-word keys (k_local4)
    rnd = random.Random(1)
    reads1 = random_reads(rnd, 3000, K)
    p1, o1 = oracle.pack_strings(reads1)
    kc.add_reads(p1, o1)
    kc.finish()
    g = check(p1, o1)
    assert g["elem_bytes"] == 8 and g["REM"] > 32
    # 2. a much larger read set at 20 prefix bits: 4-byte remainders (k_local3), and a table far beyond the step-1
    #    buffers, so the optimistic compaction overflows and the table is compacted again
    monkeypatch.setenv("APGK_PREFIX_BITS", "20")
    n2, L2 = 400_000, 100
    p2, o2 = oracle.synth_reads(oracle.synth_params(2_000_000, L2), 0, n2)
    kc.reset()
    kc.add_reads_uniform(p2, n2, L2)
    kc.finish()
    g = check(p2, o2)
    assert g["elem_bytes"] == 4 and g["REM"] == 30
    assert kc.totals()[1] > 20 * len(oracle.count(p1, o1, K)[0])
    # 3. the deferral input at REM = 32 (k_local2 -> k_local)
    monkeypatch.setenv("APGK_PREFIX_BITS", "18")
    reads3, _, where = deferral_input(K, 18)
    p3, o3 = oracle.pack_strings(reads3)
    kc.reset()
    kc.add_reads(p3, o3)
    kc.finish()
    g = check(p3, o3)
    assert (g["REM"], g["elem_bytes"]) == (32, 4) and g["n_deferred"] == 2
    # 4. more reads without a reset
    kc.add_reads(p1, o1)
    kc.finish()
    p4, o4 = oracle.pack_strings(reads3 + reads1)
    g = check(p4, o4)
    assert g["n_deferred"] >= 1
    # 5. temp buffers released
    kc.release_temp()
    kc.finish()
    check(p4, o4)
    # 6. a table reservation too small, then one too large
    nd = kc.totals()[1]
    for n in (16, 8 * nd):
        kc.reserve_table(n)
        kc.finish()
        check(p4, o4)
    # 7. finish twice in a row
    kc.finish()
    kc.finish()
    check(p4, o4)
    kc.close()
