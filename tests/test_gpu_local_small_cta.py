"""k_local5, the small-CTA counting kernel for 32-bit remainders, and the buckets it hands to k_local3.

A CTA's hash table holds up to 1536 distinct keys of a bucket; its keys are put in order by their top eight
remainder bits (the group) and ranked inside the group by comparison.  A bucket with more distinct keys, or with
more than 65535 instances, is deferred to k_local3.  Every case is checked against the oracle, and the deferral
count (geometry n_deferred) says which kernel took which bucket."""
import random

import pytest

from test_bucket_paths_cpu import _bucket_prefixes, rand_key, random_reads, reads_of
from test_gpu_bucket_paths import _check, _count, _planted_counts, _queries

pytestmark = pytest.mark.gpu

DMAX = 1536                 # k_local5's distinct keys per bucket (its table: 2048 slots)
NMAX = 65535                # k_local5's instances per bucket

def _group_keys(rng, K, P, prefix, n, group=None):
    """n distinct canonical k-mers of bucket `prefix`; with `group`, their remainders share their top eight bits"""
    rem = 2 * K - P
    free = rem - 8 if group is not None else rem
    keys = set()
    while len(keys) < n:
        v = rng.getrandbits(free)
        if v & 3 != 3:      # last base not T: smaller than its reverse complement
            keys.add(v if group is None else (group << free) | v)
    return [(prefix << rem) | v for v in sorted(keys)]

def _flood(K, n_instances):
    """poly-A reads carrying at least n_instances copies of A^K"""
    L = 300
    per = L - K + 1
    return ["A" * L] * (n_instances // per + 1)

@pytest.mark.parametrize("extra", [0, 1])
def test_table_limits(oracle, extra):
    """Buckets of 0 and 1 instances, a bucket whose 60 keys share one group, and a bucket with exactly 1536 distinct
    keys, the most k_local5's table takes.  extra = 1 adds one distinct key to that bucket, which sends it to
    k_local3."""
    K, P = 25, 20
    rng = random.Random(7 + extra)
    b_one, b_group, b_full = _bucket_prefixes(rng, P, 3)
    planted = {rand_key(rng, K, P, b_one): 1}
    for i, k in enumerate(_group_keys(rng, K, P, b_group, 60, group=37)):
        planted[k] = 1 + i % 3
    for i, k in enumerate(_group_keys(rng, K, P, b_full, DMAX + extra)):
        planted[k] = 1 + i % 2
    reads = reads_of(planted, K)
    rng.shuffle(reads)
    p, o = oracle.pack_strings(reads)
    q = _queries(oracle, p, o, K)
    r = _count(K, P, p, o, q)
    assert (int(r["g_REM"]), int(r["g_elem_bytes"])) == (2 * K - P, 4)
    assert int(r["g_n_deferred"]) == extra and int(r["g_n_big"]) == 0
    assert _planted_counts(r, planted) == list(planted.values())
    _check(oracle, r, p, o, K, q)

def _mixed_reads(K, P, seed):
    """random reads, a poly-A flood over the instance cap (its k-mer's count is above 2^16) and, where the remainder
    is wide enough, a bucket with one distinct key more than k_local5's table takes"""
    rng = random.Random(seed)
    reads = random_reads(rng, 1500, K) + _flood(K, NMAX + 1)
    planted = {}
    if 2 * K - P >= 16:
        (b,) = _bucket_prefixes(rng, P, 1)
        for i, k in enumerate(_group_keys(rng, K, P, b, DMAX + 1)):
            planted[k] = 1 + i % 4
        reads += reads_of(planted, K)
    rng.shuffle(reads)
    return reads, planted

def test_mixed_counted_and_deferred(oracle):
    """One run in which k_local5 counts almost every bucket and k_local3 takes the poly-A bucket (over the
    instance cap; its count takes the spectrum's overflow list) and a bucket with too many distinct keys."""
    K, P = 25, 20
    reads, planted = _mixed_reads(K, P, 3)
    p, o = oracle.pack_strings(reads)
    q = _queries(oracle, p, o, K)
    r = _count(K, P, p, o, q)
    assert (int(r["g_REM"]), int(r["g_elem_bytes"])) == (2 * K - P, 4)
    assert int(r["g_n_deferred"]) == 2 and int(r["g_n_big"]) == 0
    ek, ec = _check(oracle, r, p, o, K, q)
    assert int(ec.max()) > 1 << 16
    assert _planted_counts(r, planted) == list(planted.values())

@pytest.mark.parametrize("K,P", [(12, 23), (12, 22), (16, 24), (20, 9)], ids=lambda v: str(v))
def test_remainder_extremes_both_kernels(oracle, K, P):
    """REM = 1, 2, 8 and 31: k_local5 takes the ordinary buckets, k_local3 the poly-A bucket (and at REM = 31
    the bucket with too many distinct keys) at the same remainder width."""
    reads, planted = _mixed_reads(K, P, K * 100 + P)
    p, o = oracle.pack_strings(reads)
    q = _queries(oracle, p, o, K)
    r = _count(K, P, p, o, q)
    assert (int(r["g_REM"]), int(r["g_elem_bytes"])) == (2 * K - P, 4)
    assert int(r["g_n_deferred"]) == (2 if planted else 1) and int(r["g_n_big"]) == 0
    _check(oracle, r, p, o, K, q)
    assert _planted_counts(r, planted) == list(planted.values())

@pytest.mark.parametrize("world", [1, 3])
def test_sharded_mixed(oracle, world):
    """The mixed input through KmerGroup.local: the ranks' owned bucket ranges start inside the bucket table."""
    from allpathslg_b200 import KmerCounter, KmerGroup
    from test_gpu_group import _check_against_oracle

    K, P = 25, 20
    reads, _ = _mixed_reads(K, P, 11)
    p, o = oracle.pack_strings(reads)
    kcs = []
    for r in range(world):
        kc = KmerCounter(K, prefix_bits=P)
        pr, orr = oracle.pack_strings(reads[r::world])
        kc.add_reads(pr, orr)
        kcs.append(kc)
    with KmerGroup.local(kcs) as grp:
        grp.count()
        assert grp.stats()["prefix_bits"] == P
        _check_against_oracle(oracle, grp, kcs, p, o, K, sorted_by_rank=True)
    for kc in kcs:
        kc.close()
