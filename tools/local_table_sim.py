#!/usr/bin/env python
"""Distinct keys per level-1 bucket on reads of the bench's generator, and how they load a per-bucket table (CPU only).

  python tools/local_table_sim.py [--genome 1600000] [--prefix-bits 14]

The bench's reads (60x coverage, 0.5 % errors, planted repeats) at a 1/62 genome with 6 fewer prefix bits, so a
bucket holds about as many instances as at the bench geometry (2^20 buckets of 4.56 G).  Prints the distinct keys per
bucket, the share of buckets in which a row of R slots chosen by the top remainder bits (k_local3's order-preserving
layout, at a fixed table size) would overflow, and how many keys share their top G remainder bits (what a kernel that
orders distinct keys by a counting sort on those bits has to rank by comparison).  profiles/r04_local_warp.txt."""
import argparse
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--genome", type=int, default=1_600_000)
    ap.add_argument("--prefix-bits", type=int, default=14)
    a = ap.parse_args()
    from oracle import oracle_a as A

    A.build()
    K, L = 25, 100
    n_reads = a.genome * 60 // L
    p, o = A.synth_reads(A.synth_params(a.genome, L), 0, n_reads)
    ek, ec, en = A.count(p, o, K)
    P = a.prefix_bits
    REM = 2 * K - P
    k = ek[:, -1].astype(np.uint64)
    b = (k >> np.uint64(REM)).astype(np.int64)
    r = k & np.uint64((1 << REM) - 1)
    nb = 1 << P
    inst = np.bincount(b, weights=ec.astype(np.float64), minlength=nb)
    dist = np.bincount(b, minlength=nb)
    print("%d reads, %d instances, %d distinct; P = %d: instances per bucket mean %.0f max %.0f; distinct per bucket "
          "mean %.0f p99 %.0f max %d" % (n_reads, en, len(ek), P, inst.mean(), inst.max(), dist.mean(),
                                         np.percentile(dist, 99), dist.max()))
    top32 = (r << np.uint64(64 - REM)) >> np.uint64(32)
    for S, R in [(2048, 16), (2048, 32), (3072, 32), (4096, 16), (4096, 32), (8192, 16)]:
        nrows = S // R
        row = ((top32 * np.uint64(nrows)) >> np.uint64(32)).astype(np.int64)
        load = np.bincount(b * nrows + row, minlength=nb * nrows).reshape(nb, nrows)
        print("monotone rows: %5d slots, rows of %2d: %.4f of the buckets overflow a row (fullest row %d)"
              % (S, R, (load > R).any(axis=1).mean(), load.max()))
    for G in [6, 7, 8, 9]:
        cell = b * (1 << G) + (r >> np.uint64(REM - G)).astype(np.int64)
        sz = np.bincount(cell, minlength=nb << G)
        per_key = sz[np.sort(cell)]
        m = len(per_key) // 32 * 32
        print("groups of %d bits: a key is ranked against %.1f keys on average, %.1f for the largest of 32 "
              "consecutive keys; largest group %d" % (G, per_key.mean(), per_key[:m].reshape(-1, 32).max(axis=1).mean(),
                                                     sz.max()))


if __name__ == "__main__":
    main()
