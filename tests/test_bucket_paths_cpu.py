"""Inputs that drive the per-bucket counting kernels into their recovery paths, and the checks of those inputs that
need no GPU.  tests/test_gpu_bucket_paths.py feeds them to the kernels.

- Deferral from k_local2 to k_local (csrc/local2.cuh): a sub-bucket holding more than L2_WCAP = 512 instances, or
  more than L2_MAXBIN = 48 distinct keys in one comparison-sort bin.  `k_local2_plan` replays the kernel's rules on
  the oracle's table and says which buckets defer and which go to k_big.
- Tag collisions in k_local4 (csrc/local4.cuh): two keys of one row whose 32-bit tags agree.  The tag is
  sm64(key_hash(k) + seed) >> 32, key_hash folding sm64 over the words (csrc/kmer_types.cuh); the row depends on the
  32 key bits just below the range prefix.  `collision_pair` searches ~2^18 candidates for a pair with equal tags.
- Row overflows in k_local4: many near-identical keys in one row, split bit by bit down to their differing bits.
"""
import random

import numpy as np
import pytest

M64 = (1 << 64) - 1
L2_WCAP, L2_MAXBIN, L2_TARGET_SUB = 512, 48, 160
# level-1 bucket capacity of the general kernels (k_local2 / k_local / k_big) by element: 4-byte remainders, Key<1>,
# Key<2>, Key<3> (LM_U32 and Geo<W>::LM_KEY in csrc/apgk.cu)
LOCAL_MAX = {4: 5120, 1: 4096, 2: 2048, 3: 2048}


def words(K):
    return (2 * K + 63) // 64


def rem_bits(K, P):
    return max(2 * K, P) - P


def to_words(keys, K):
    """python ints -> uint64[n, W], most significant word first"""
    W = words(K)
    return np.array([[(k >> (64 * (W - 1 - j))) & M64 for j in range(W)] for k in keys], dtype=np.uint64).reshape(-1, W)


def to_ints(rows):
    W = rows.shape[1]
    out = []
    for r in rows.tolist():
        v = 0
        for j in range(W):
            v = (v << 64) | r[j]
        out.append(v)
    return out


def key_str(k, K):
    return "".join("ACGT"[(k >> (2 * (K - 1 - i))) & 3] for i in range(K))


def revcomp(k, K):
    r = 0
    for _ in range(K):
        r = (r << 2) | (3 - (k & 3))
        k >>= 2
    return r


# ------------------------------------------------------------------ the hashes, vectorised
def sm64(z):
    z = np.asarray(z, dtype=np.uint64)
    with np.errstate(over="ignore"):
        z = z + np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def key_hash(rows):
    rows = np.asarray(rows, dtype=np.uint64)
    h = np.zeros(len(rows), dtype=np.uint64)
    for j in range(rows.shape[1]):
        h = sm64(h ^ rows[:, j])
    return h


def l4_tag(rows, seed=0):
    with np.errstate(over="ignore"):
        t = (sm64(key_hash(rows) + np.uint64(seed)) >> np.uint64(32)).astype(np.uint32)
    return np.where(t == np.uint32(0xFFFFFFFF), np.uint32(0xFFFFFFFE), t)


# ------------------------------------------------------------------ constructed keys
def rand_key(rng, K, P, prefix):
    """a canonical k-mer of the level-1 bucket `prefix` (P <= 2K, prefix below 2^(P-2): first base A) whose last base
    is not T, so it is smaller than its reverse complement"""
    low = 2 * K - P
    return (prefix << low) | (rng.getrandbits(low - 2) << 2) | rng.randrange(3)


def _bucket_prefixes(rng, P, n):
    """n level-1 bucket prefixes that start with base A, away from poly-A, no two within 3 of each other"""
    if P < 6:   # too few buckets to choose from: the first one (poly-A shares it)
        assert n == 1
        return [0]
    out = []
    while len(out) < n:
        b = rng.randrange(1 << (P - 4), (1 << (P - 2)) - 2)
        if all(abs(b - x) > 3 for x in out):
            out.append(b)
    return out


def random_reads(rng, n, K, lengths=(0, 1, 30, 100, 101, 150)):
    lens = list(lengths) + [K - 1, K, K + 1]
    return ["".join(rng.choice("ACGT") for _ in range(rng.choice(lens))) for _ in range(n)]


def reads_of(planted, K):
    """every planted k-mer as reads of exactly K bases, one read per instance"""
    out = []
    for k, m in planted.items():
        out += [key_str(k, K)] * m
    return out


HEAVY = 700     # instances of the one k-mer that overfills a sub-bucket (513..2000)
CLUSTER = 60    # distinct k-mers that share a sub-bucket and a sort bin (> 48)


def deferral_input(K, P, seed=0):
    """Reads whose level-1 buckets at prefix_bits P make k_local2 defer: bucket A holds one k-mer HEAVY times among
    ordinary keys; bucket B (when REM > 0) holds CLUSTER k-mers that differ only in their last four bases.  Both are
    surrounded by ordinary keys in their own and the neighbouring buckets, and by random reads.
    -> (reads, planted {k-mer: copies}, {"heavy": bucket, "cluster": bucket or None})"""
    rng = random.Random(seed * 1_000_003 + K * 97 + P)
    planted = {}

    def put(k, m):
        planted[k] = planted.get(k, 0) + m

    REM = rem_bits(K, P)
    if REM == 0:
        # every bucket is one key value (the key left-padded to P bits): only the instance trigger exists
        pad = P - 2 * K
        h = rng.randrange(1 << (2 * K - 4), 1 << (2 * K - 2)) & ~3 | 1   # last base C
        put(h, HEAVY)
        for i, d in enumerate((-6, -4, -2, -1, 1, 2, 4, 6)):
            if (h + d) & 3 != 3:
                put(h + d, 2 + i)
        reads = reads_of(planted, K) + random_reads(rng, 300, K)
        return reads, planted, {"heavy": h << pad, "cluster": None}
    bh, bc = _bucket_prefixes(rng, P, 2)
    h = rand_key(rng, K, P, bh)
    put(h, HEAVY)
    for i in range(120):
        put(rand_key(rng, K, P, bh), 1 + i % 4)
    base = rand_key(rng, K, P, bc) >> 8 << 8
    lows = [v for v in range(256) if v & 3 != 3]
    rng.shuffle(lows)
    for i, v in enumerate(lows[:CLUSTER]):
        put(base | v, 1 + i % 6)
    for i in range(40):
        put(rand_key(rng, K, P, bc), 1 + i % 3)
    for b in (bh - 1, bh + 1, bc - 1, bc + 1):
        for i in range(50):
            put(rand_key(rng, K, P, b), 1 + i % 5)
    reads = reads_of(planted, K) + random_reads(rng, 300, K)
    rng.shuffle(reads)
    return reads, planted, {"heavy": bh, "cluster": bc}


def row_overflow_input(K, P, n_background=300, seed=0):
    """Reads with a bucket whose keys pile into one k_local4 row: 40 k-mers that differ only in their last five
    bases, so every range above those bits overflows its row and splits on the next bit, from the top of the
    remainder down to bit 10; plus poly-A / tandem-repeat floods and random reads."""
    rng = random.Random(seed * 1_000_003 + K * 89 + P)
    planted = {}
    (b,) = _bucket_prefixes(rng, P, 1)
    base = rand_key(rng, K, P, b) >> 10 << 10
    lows = [v for v in range(1024) if v & 3 != 3]
    rng.shuffle(lows)
    for i, v in enumerate(lows[:40]):
        planted[base | v] = 1 + i % 5
    reads = reads_of(planted, K) + ["A" * 200] * 30 + ["ACGTACGTAC" * 20] * 20 + random_reads(rng, n_background, K)
    rng.shuffle(reads)
    return reads, planted, b


def collision_pair(K, P, n_cand=1 << 18, seed=0):
    """Two canonical k-mers of one bucket with equal k_local4 tags (seed 0) whose 34 bits below the P-bit prefix
    agree as well, so they share a row also when a sharded count moves up to two of those bits into the prefix.
    Both start with base A and end in a base other than T.  -> (key a, key b) as python ints, a < b"""
    rng = np.random.RandomState(seed + 7 * K + P)
    REM = 2 * K - P
    free = REM - 34          # bits below the fixed part
    assert free >= 20, "too few free bits for ~2^18 candidates"
    prefix = int(rng.randint(1 << (P - 4), 1 << (P - 2)))
    mid = int(rng.randint(0, 1 << 30)) << 4 | int(rng.randint(0, 16))
    fixed = (prefix << REM) | (mid << free)
    # candidates: the free bits, last base A, C or G
    nlow = min(free, 62)
    low = rng.randint(0, 1 << 62, size=2 * n_cand, dtype=np.int64).astype(np.uint64) & np.uint64((1 << nlow) - 1)
    low = np.unique(low & ~np.uint64(3) | (low & np.uint64(3)) % np.uint64(3))[:n_cand]
    W = words(K)
    rows = np.zeros((len(low), W), dtype=np.uint64)
    fw = to_words([fixed], K)[0]
    rows[:] = fw
    rows[:, W - 1] |= low          # the varied bits all sit in the least significant word (nlow <= 62)
    tags = l4_tag(rows)
    order = np.argsort(tags, kind="stable")
    ts = tags[order]
    hit = np.nonzero(ts[1:] == ts[:-1])[0]
    assert len(hit), "no tag collision among the candidates"
    i, j = order[hit[0]], order[hit[0] + 1]
    a, b = sorted((fixed | int(low[i]), fixed | int(low[j])))
    return a, b


def collision_input(K, P, seed=0):
    """The colliding pair (3 and 5 copies) among ordinary keys of its bucket, neighbouring buckets and random reads.
    -> (reads, planted, (a, b))"""
    a, b = collision_pair(K, P, seed=seed)
    rng = random.Random(seed * 1_000_003 + K * 83 + P)
    planted = {a: 3, b: 5}
    bucket = a >> (2 * K - P)
    for bb in (bucket - 1, bucket, bucket + 1):
        for i in range(30):
            planted.setdefault(rand_key(rng, K, P, bb), 1 + i % 4)
    reads = reads_of(planted, K) + random_reads(rng, 300, K)
    rng.shuffle(reads)
    return reads, planted, (a, b)


# ------------------------------------------------------------------ k_local2's rules on the oracle's table
def _ilog2_ceil(x):
    return 0 if x <= 1 else (x - 1).bit_length()


def k_local2_plan(ek, ec, K, P, local_max):
    """Replay k_local2 on the distinct k-mers of a count: -> dict(bucket -> "big" | "sub" | "bin" | None): k_big's
    bucket (more than local_max instances), deferred because a sub-bucket holds more than 512 instances, deferred
    because a sort bin holds more than 48 distinct keys, or counted by k_local2 itself."""
    REM = rem_bits(K, P)
    pad = max(2 * K, P) - 2 * K
    mask = (1 << REM) - 1
    by_bucket = {}
    for k, c in zip(to_ints(ek), ec.tolist()):
        v = k << pad
        by_bucket.setdefault(v >> REM, []).append((v & mask, int(c)))
    out = {}
    for b, items in by_bucket.items():
        n = sum(c for _, c in items)
        if n > local_max:
            out[b] = "big"
            continue
        sb = min(_ilog2_ceil((n + L2_TARGET_SUB - 1) // L2_TARGET_SUB), 6, REM)
        sub_shift = REM - sb
        subs = {}
        for e, c in items:
            subs.setdefault((e >> sub_shift) & ((1 << sb) - 1), []).append((e, c))
        why = None
        if max(sum(c for _, c in s) for s in subs.values()) > L2_WCAP:
            why = "sub"
        else:
            sbits = min(sub_shift, 6)
            shift2 = sub_shift - sbits
            for s in subs.values():
                if len(s) < 2:
                    continue
                bins = {}
                for e, _ in s:
                    d = (e >> shift2) & ((1 << sbits) - 1)
                    bins[d] = bins.get(d, 0) + 1
                if max(bins.values()) > L2_MAXBIN:
                    why = "bin"
                    break
        out[b] = why
    return out


# (K, prefix_bits, level-1 element: 4 = 4-byte remainders, W = Key<W>) of every deferral case
DEFERRAL_CASES = [(40, 12, 2), (64, 12, 2), (65, 12, 3), (96, 12, 3), (26, 20, 4), (25, 18, 4), (10, 22, 4), (30, 12, 1)]
COLLISION_CASES = [(32, 10), (40, 12), (96, 12)]


# ------------------------------------------------------------------ tests
@pytest.mark.parametrize("K", [5, 25, 32, 33, 40, 64, 65, 96])
def test_key_hash_replica_matches_the_library(apgk_lib, K):
    """apgk_owner_of(K, keys, n, 2^32 - 1) is (key_hash >> 32) - 1 for a non-zero top half: the numpy key_hash the
    collision search uses is the library's, over one, two and three words."""
    from allpathslg_b200 import owner_of

    rng = np.random.RandomState(K)
    W = words(K)
    rows = rng.randint(0, 1 << 62, size=(4000, W), dtype=np.int64).astype(np.uint64) * np.uint64(3)
    if 2 * K < 64 * W:
        rows[:, 0] &= np.uint64((1 << (2 * K - 64 * (W - 1))) - 1)
    top = key_hash(rows) >> np.uint64(32)
    own = owner_of(K, rows, 0xFFFFFFFF).astype(np.uint64)
    nz = top != 0
    assert nz.sum() > 3900
    assert (own[nz] + np.uint64(1) == top[nz]).all()


@pytest.mark.parametrize("K,P", COLLISION_CASES)
def test_collision_pairs(oracle, K, P):
    a, b = collision_pair(K, P)
    REM = 2 * K - P
    assert a != b
    rows = to_words([a, b], K)
    ta, tb = l4_tag(rows)
    assert ta == tb
    assert l4_tag(rows, seed=1)[0] != l4_tag(rows, seed=1)[1]      # the retry with seed + 1 separates them
    assert a >> REM == b >> REM                                    # one bucket
    assert (a >> (REM - 34)) == (b >> (REM - 34))                  # the row bits, also 2 bits further down
    for k, row in ((a, rows[0]), (b, rows[1])):
        assert (oracle.canonical(row, K) == row).all()             # counted as themselves
        assert k < revcomp(k, K)


@pytest.mark.parametrize("K,P", COLLISION_CASES)
def test_collision_input_counts(oracle, K, P):
    reads, planted, (a, b) = collision_input(K, P)
    p, o = oracle.pack_strings(reads)
    ek, ec, _ = oracle.count(p, o, K)
    got = dict(zip(to_ints(ek), ec.tolist()))
    assert got[a] == 3 and got[b] == 5


@pytest.mark.parametrize("K,P,elem", DEFERRAL_CASES)
def test_deferral_inputs(oracle, K, P, elem):
    """The planted buckets reach k_local (not k_big) for the trigger they were built for, and nothing else defers."""
    reads, planted, where = deferral_input(K, P)
    p, o = oracle.pack_strings(reads)
    ek, ec, _ = oracle.count(p, o, K)
    got = dict(zip(to_ints(ek), ec.tolist()))
    for k, m in planted.items():
        assert got[k] >= m
    plan = k_local2_plan(ek, ec, K, P, LOCAL_MAX[elem])
    assert plan[where["heavy"]] == "sub"
    if where["cluster"] is not None:
        assert plan[where["cluster"]] == "bin"
    deferred = sorted(b for b, why in plan.items() if why in ("sub", "bin"))
    assert deferred == sorted(x for x in where.values() if x is not None)
    assert not any(why == "big" for why in plan.values())


@pytest.mark.parametrize("K,P", [(27, 21), (30, 20), (32, 2), (40, 16), (40, 15), (56, 16), (72, 16), (72, 15), (88, 16)])
def test_row_overflow_inputs(oracle, K, P):
    """40 distinct k-mers of one bucket agree on every bit from bit 10 up to the top of the remainder (the row bits of
    every range down to there), with k_local4's 16 slots per row."""
    reads, planted, b = row_overflow_input(K, P, n_background=50)
    REM = 2 * K - P
    keys = list(planted)
    assert len(keys) == 40 and all(k >> REM == b for k in keys)
    assert len({k >> 10 for k in keys}) == 1
    p, o = oracle.pack_strings(reads)
    ek, ec, _ = oracle.count(p, o, K)
    got = dict(zip(to_ints(ek), ec.tolist()))
    assert all(got[k] == m for k, m in planted.items())
