"""Oracles of the k-mer AFFIXES (apgk_build_affixes; definition in include/apgk.h).  TEST INFRASTRUCTURE.

  affixes_a        oracle A: tests/affix_oracle.c (roll + binary search over the oracle's sorted table, OpenMP with a
                   per-thread OR-reduction), compiled on first use into a temporary directory.
  affixes_b        oracle B: strings and a dict, written from the definition; shares no code with A.
  sample_affixes   the affixes of a SAMPLED partition, from oracle_a.sample_prefix_pos output and the packed reads
                   (numpy): the check at a scale no full oracle table fits on the host.
  affix_revcomp    the orientation transform (affix byte of a k-mer -> that of its reverse complement).
"""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "affix_oracle.c")
_lib = None


def lib():
    global _lib
    if _lib is None:
        src = open(_SRC, "rb").read()
        d = os.path.join(tempfile.gettempdir(), "apgk_affix_oracle_%d_%s" % (os.getuid(), hashlib.sha256(src).hexdigest()[:16]))
        so = os.path.join(d, "libaffix_oracle.so")
        if not os.path.exists(so):
            os.makedirs(d, exist_ok=True)
            tmp = so + ".%d" % os.getpid()
            subprocess.check_call(["gcc", "-O3", "-march=x86-64-v3", "-fopenmp", "-fPIC", "-Wall", "-Wextra", "-std=c11",
                                   "-shared", "-o", tmp, _SRC])
            os.replace(tmp, so)
        L = C.CDLL(so)
        L.oracle_affixes.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_void_p, C.c_uint64, C.c_void_p]
        L.oracle_affixes.restype = C.c_int
        _lib = L
    return _lib


def affixes_a(packed, off, K, kmers):
    """-> uint8[n_distinct]: the affix byte of every k-mer of `kmers` (the oracle's sorted table, uint64[n, W])."""
    packed = np.ascontiguousarray(packed, dtype=np.uint8)
    off = np.ascontiguousarray(off, dtype=np.uint64)
    kmers = np.ascontiguousarray(kmers, dtype=np.uint64)
    nd = len(kmers)
    out = np.zeros(max(nd, 1), dtype=np.uint8)
    rc = lib().oracle_affixes(packed.ctypes.data, off.ctypes.data, len(off) - 1, K, kmers.ctypes.data, nd, out.ctypes.data)
    if rc != 0:
        raise RuntimeError("oracle_affixes failed rc=%d" % rc)
    return out[:nd]


_COMP = str.maketrans("ACGT", "TGCA")


def affixes_b(reads, K):
    """-> sorted list of (kmer_int, affix byte) from ACGT strings.  A window read forward gives its left neighbour
    as a predecessor and its right one as a successor; read as its reverse complement, the complemented right
    neighbour precedes and the complemented left one follows; a palindrome is read both ways."""
    pre, suf = {}, {}
    for s in reads:
        for p in range(len(s) - K + 1):
            w = s[p:p + K]
            rc = w.translate(_COMP)[::-1]
            left = s[p - 1] if p > 0 else ""
            right = s[p + K] if p + K < len(s) else ""
            c = min(w, rc)
            pre.setdefault(c, set())
            suf.setdefault(c, set())
            if w <= rc:
                pre[c].update(left)
                suf[c].update(right)
            if w >= rc:
                pre[c].update(right.translate(_COMP))
                suf[c].update(left.translate(_COMP))
    out = []
    for c in pre:
        v = 0
        for b in pre[c]:
            v |= 1 << "ACGT".index(b)
        for b in suf[c]:
            v |= 16 << "ACGT".index(b)
        iv = 0
        for ch in c:
            iv = iv * 4 + "ACGT".index(ch)
        out.append((iv, v))
    return sorted(out)


_REV4 = np.array([int("{:04b}".format(m)[::-1], 2) for m in range(16)], dtype=np.uint8)


def affix_revcomp(aff):
    """affix bytes of k-mers -> affix bytes of their reverse complements: pre' = comp(suf), suf' = comp(pre)."""
    a = np.asarray(aff, dtype=np.uint8)
    return (_REV4[a >> 4] | (_REV4[a & 15] << 4)).astype(np.uint8)


def revcomp_keys(keys, K):
    """reverse complements of k-mers uint64[n, W] (numpy, base by base)."""
    keys = np.ascontiguousarray(keys, dtype=np.uint64).reshape(len(keys), -1)
    W = keys.shape[1]
    out = np.zeros_like(keys)
    for i in range(K):   # base at bit 2i (from the last) -> bit 2(K-1-i), complemented
        s, d = 2 * i, 2 * (K - 1 - i)
        b = (keys[:, W - 1 - s // 64] >> np.uint64(s % 64)) & np.uint64(3)
        out[:, W - 1 - d // 64] |= (np.uint64(3) - b) << np.uint64(d % 64)
    return out


def _base_at(packed, q):
    return (packed[(q >> np.uint64(2)).astype(np.int64)] >> ((q & np.uint64(3)) * np.uint64(2)).astype(np.uint8)) & 3


def sample_affixes(packed, off, K, keys, pos, read_len=0):
    """Affixes of a sampled partition.  keys uint64[n, W] and pos ((q << 1) | canonical_is_reverse, q = the window's
    first base in `packed`) are oracle_a.sample_prefix_pos output; read boundaries come from `off` (uint64[n+1]) or,
    with off None, from uniform reads of read_len bases starting at base 0.
    -> (distinct keys uint64[d, W] ascending, affix bytes uint8[d]): what the table's rows for them must hold."""
    packed = np.asarray(packed, dtype=np.uint8)
    keys = np.ascontiguousarray(keys, dtype=np.uint64).reshape(len(keys), -1)
    pos = np.asarray(pos, dtype=np.uint64)
    q = pos >> np.uint64(1)
    rev = (pos & np.uint64(1)).astype(bool)
    if off is None:
        rl = np.uint64(read_len)
        s = (q // rl) * rl
        e = s + rl
    else:
        off = np.asarray(off, dtype=np.uint64)
        r = np.searchsorted(off, q, side="right") - 1
        s, e = off[r], off[r + 1]
    has_l = q > s
    has_r = q + np.uint64(K) < e
    L = _base_at(packed, np.where(has_l, q - np.uint64(1), q)).astype(np.int64)
    R = _base_at(packed, np.where(has_r, q + np.uint64(K), q)).astype(np.int64)
    a = (np.where(has_l, 1 << L, 0) | np.where(has_r, 16 << R, 0)).astype(np.uint8)   # the window's own orientation
    pal = np.zeros(len(keys), dtype=bool)
    if K % 2 == 0:
        pal = (keys == revcomp_keys(keys, K)).all(axis=1)
    a = np.where(rev, affix_revcomp(a), np.where(pal, a | affix_revcomp(a), a)).astype(np.uint8)
    W = keys.shape[1]
    view = keys[:, 0] if W == 1 else keys.view([("w%d" % i, np.uint64) for i in range(W)]).ravel()
    uk, inv = np.unique(view, return_inverse=True)
    out = np.zeros(len(uk), dtype=np.uint8)
    np.bitwise_or.at(out, inv.ravel(), a)
    return np.ascontiguousarray(uk).view(np.uint64).reshape(len(uk), W), out
