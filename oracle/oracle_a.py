"""ctypes wrapper around oracle/_build/liboracle.so (oracle "A", kmer_oracle.c).

TEST INFRASTRUCTURE, NOT PRODUCT.  PARITY UNPINNED (see kmer_oracle.c header).
Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / reference
arm may import this module.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "liboracle.so")


class SynthParams(C.Structure):
    _fields_ = [
        ("genome_len", C.c_uint64),
        ("seed_g", C.c_uint64),
        ("seed_p", C.c_uint64),
        ("seed_q", C.c_uint64),
        ("seed_r", C.c_uint64),
        ("seed_e", C.c_uint64),
        ("read_len", C.c_uint32),
        ("err_per_200", C.c_uint32),
    ]


# Seeds fixed by SURVEY.md section 8(d) (seed_p / seed_q added for the planted repeats).
DEFAULT_SEEDS = dict(seed_g=0xA11BA7C5, seed_p=0x5EED00A0, seed_q=0x5EED00A1, seed_r=0x5EED0001, seed_e=0x5EED0002)


def build(force=False):
    src = os.path.join(_HERE, "kmer_oracle.c")
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-s"])
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_SO)
        u64p = C.POINTER(C.c_uint64)
        L.oracle_count.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_int,
                                   C.POINTER(u64p), C.POINTER(u64p), u64p, u64p]
        L.oracle_count.restype = C.c_int
        L.oracle_spectrum.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(u64p), u64p]
        L.oracle_spectrum.restype = C.c_int
        L.oracle_free.argtypes = [C.c_void_p]
        L.oracle_synth_reads.argtypes = [C.POINTER(SynthParams), C.c_uint64, C.c_uint64, C.c_void_p]
        L.oracle_lookup.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_void_p, C.c_uint64, C.c_int,
                                    C.c_void_p]
        L.oracle_read_freqs.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_void_p, C.c_void_p,
                                        C.c_uint64, C.c_void_p]
        L.oracle_canonical.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        L.oracle_num_threads.restype = C.c_int
        L.oracle_occurrences.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_void_p, C.c_uint64,
                                         C.c_void_p, C.c_void_p, C.c_void_p]
        L.oracle_occurrences.restype = C.c_int
        L.oracle_sample_prefix.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_int, C.c_int, C.c_void_p,
                                           C.c_int, C.POINTER(u64p), u64p, u64p]
        L.oracle_sample_prefix.restype = C.c_int
        L.oracle_sample_prefix_pos.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_int, C.c_int,
                                               C.c_void_p, C.c_int, C.POINTER(u64p), C.POINTER(u64p), u64p, u64p]
        L.oracle_sample_prefix_pos.restype = C.c_int
        L.oracle_count_keys.argtypes = [C.c_void_p, C.c_uint64, C.c_int, C.c_int, C.POINTER(u64p), C.POINTER(u64p), u64p]
        L.oracle_count_keys.restype = C.c_int
        _lib = L
    return _lib


def n_words(K):
    return (2 * K + 63) // 64


def synth_params(genome_len, read_len, errors=True, **seeds):
    s = dict(DEFAULT_SEEDS)
    s.update(seeds)
    return SynthParams(genome_len=genome_len, read_len=read_len, err_per_200=1 if errors else 0, **s)


def synth_reads(params, r0, n):
    """-> (packed uint8 array padded to 8 bytes, off uint64[n+1])."""
    nb = n * params.read_len
    nbytes = ((nb + 31) // 32) * 8
    packed = np.zeros(max(nbytes, 8), dtype=np.uint8)
    lib().oracle_synth_reads(C.byref(params), r0, n, packed.ctypes.data)
    off = np.arange(n + 1, dtype=np.uint64) * np.uint64(params.read_len)
    return packed, off


def count(packed, off, K, n_threads=0):
    """-> (kmers uint64[n, W] sorted, counts uint64[n], n_instances)."""
    L = lib()
    packed = np.ascontiguousarray(packed, dtype=np.uint8)
    off = np.ascontiguousarray(off, dtype=np.uint64)
    n_reads = len(off) - 1
    kp = C.POINTER(C.c_uint64)()
    cp = C.POINTER(C.c_uint64)()
    nd = C.c_uint64()
    ni = C.c_uint64()
    rc = L.oracle_count(packed.ctypes.data, off.ctypes.data, n_reads, K, n_threads,
                        C.byref(kp), C.byref(cp), C.byref(nd), C.byref(ni))
    if rc != 0:
        raise RuntimeError("oracle_count failed rc=%d" % rc)
    W = n_words(K)
    n = nd.value
    kmers = np.ctypeslib.as_array(kp, shape=(max(n, 1) * W,))[: n * W].copy().reshape(n, W)
    counts = np.ctypeslib.as_array(cp, shape=(max(n, 1),))[:n].copy()
    L.oracle_free(kp)
    L.oracle_free(cp)
    return kmers, counts, ni.value


def _sample_args(packed, off, pbits, parts, n_reads):
    if isinstance(packed, np.ndarray):
        packed = np.ascontiguousarray(packed, dtype=np.uint8)
        paddr = packed.ctypes.data
    else:
        paddr = int(packed)
    oaddr = None
    if off is not None:
        off = np.ascontiguousarray(off, dtype=np.uint64)
        n_reads = len(off) - 1
        oaddr = off.ctypes.data
    sel = np.zeros(1 << pbits, dtype=np.uint8)
    sel[np.asarray(list(parts), dtype=np.int64)] = 1
    return (packed, off, sel), paddr, oaddr, n_reads


def sample_prefix(packed, off, K, pbits, parts, n_reads=None, read_len=0, n_threads=0):
    """Sampled-partition oracle, step 1 (SURVEY.md section 8c "human-scale check" ii): the canonical k-mer INSTANCES
    of all reads whose leading `pbits` bits are one of `parts`.  packed: uint8 array or an integer address; off:
    uint64[n+1] or None for uniform reads (n_reads x read_len).  -> (keys uint64[n, W] unsorted, n_windows_seen)."""
    L = lib()
    keep, paddr, oaddr, n_reads = _sample_args(packed, off, pbits, parts, n_reads)
    kp = C.POINTER(C.c_uint64)()
    n = C.c_uint64()
    nw = C.c_uint64()
    rc = L.oracle_sample_prefix(paddr, oaddr, n_reads, read_len, K, pbits, keep[2].ctypes.data, n_threads,
                                C.byref(kp), C.byref(n), C.byref(nw))
    if rc != 0:
        raise RuntimeError("oracle_sample_prefix failed rc=%d" % rc)
    W = n_words(K)
    keys = np.ctypeslib.as_array(kp, shape=(max(n.value, 1) * W,))[: n.value * W].copy().reshape(n.value, W)
    L.oracle_free(kp)
    return keys, nw.value


def sample_prefix_pos(packed, off, K, pbits, parts, n_reads=None, read_len=0, n_threads=0):
    """sample_prefix with where each instance sits: -> (keys uint64[n, W], pos uint64[n], n_windows_seen).
    pos = (q << 1) | canonical_is_reverse, q = the window's first base in the packed stream (a palindrome counts as
    forward): the encoding of apgk_occurrences_device.  Instances come ascending by q."""
    L = lib()
    keep, paddr, oaddr, n_reads = _sample_args(packed, off, pbits, parts, n_reads)
    kp = C.POINTER(C.c_uint64)()
    pp = C.POINTER(C.c_uint64)()
    n = C.c_uint64()
    nw = C.c_uint64()
    rc = L.oracle_sample_prefix_pos(paddr, oaddr, n_reads, read_len, K, pbits, keep[2].ctypes.data, n_threads,
                                    C.byref(kp), C.byref(pp), C.byref(n), C.byref(nw))
    if rc != 0:
        raise RuntimeError("oracle_sample_prefix_pos failed rc=%d" % rc)
    W = n_words(K)
    m = n.value
    keys = np.ctypeslib.as_array(kp, shape=(max(m, 1) * W,))[: m * W].copy().reshape(m, W)
    pos = np.ctypeslib.as_array(pp, shape=(max(m, 1),))[:m].copy()
    L.oracle_free(kp)
    L.oracle_free(pp)
    return keys, pos, nw.value


def count_keys(keys, K, n_threads=0):
    """Sampled-partition oracle, step 2: sort + count canonical k-mer instances (uint64[n, W], any order).
    -> (kmers uint64[d, W] sorted, counts uint64[d])."""
    L = lib()
    W = n_words(K)
    keys = np.ascontiguousarray(keys, dtype=np.uint64).reshape(-1, W)
    kp = C.POINTER(C.c_uint64)()
    cp = C.POINTER(C.c_uint64)()
    nd = C.c_uint64()
    rc = L.oracle_count_keys(keys.ctypes.data, len(keys), K, n_threads, C.byref(kp), C.byref(cp), C.byref(nd))
    if rc != 0:
        raise RuntimeError("oracle_count_keys failed rc=%d" % rc)
    n = nd.value
    kmers = np.ctypeslib.as_array(kp, shape=(max(n, 1) * W,))[: n * W].copy().reshape(n, W)
    counts = np.ctypeslib.as_array(cp, shape=(max(n, 1),))[:n].copy()
    L.oracle_free(kp)
    L.oracle_free(cp)
    return kmers, counts


def spectrum(counts):
    """dense uint64 spectrum, index = frequency (index 0 is 0)."""
    counts = np.ascontiguousarray(counts, dtype=np.uint64)
    if len(counts) == 0:
        return np.zeros(1, dtype=np.uint64)
    return np.bincount(counts.astype(np.int64)).astype(np.uint64)


def lookup(kmers, counts, K, queries, canonicalise=True):
    kmers = np.ascontiguousarray(kmers, dtype=np.uint64)
    counts = np.ascontiguousarray(counts, dtype=np.uint64)
    queries = np.ascontiguousarray(queries, dtype=np.uint64)
    W = n_words(K)
    nq = queries.size // W
    out = np.zeros(nq, dtype=np.uint64)
    lib().oracle_lookup(kmers.ctypes.data, counts.ctypes.data, len(counts), K, queries.ctypes.data, nq,
                        1 if canonicalise else 0, out.ctypes.data)
    return out


def read_freqs(packed, off, K, kmers, counts):
    packed = np.ascontiguousarray(packed, dtype=np.uint8)
    off = np.ascontiguousarray(off, dtype=np.uint64)
    kmers = np.ascontiguousarray(kmers, dtype=np.uint64)
    counts = np.ascontiguousarray(counts, dtype=np.uint64)
    total = int(off[-1] - off[0])
    out = np.zeros(max(total, 1), dtype=np.uint64)
    lib().oracle_read_freqs(packed.ctypes.data, off.ctypes.data, len(off) - 1, K, kmers.ctypes.data,
                            counts.ctypes.data, len(counts), out.ctypes.data)
    return out[:total]


def occurrences(packed, off, K, kmers, n_instances):
    """-> (run_off uint64[n_distinct+1], read_id uint32[n_instances], pos int32[n_instances]): the instances of
    every distinct k-mer of `kmers` (table order), ascending by (read id, position) inside a k-mer; pos is
    1-based, negative when the canonical form is the reverse complement of the read's window."""
    packed = np.ascontiguousarray(packed, dtype=np.uint8)
    off = np.ascontiguousarray(off, dtype=np.uint64)
    kmers = np.ascontiguousarray(kmers, dtype=np.uint64)
    nd = kmers.size // n_words(K)
    run_off = np.zeros(nd + 1, dtype=np.uint64)
    rid = np.zeros(max(n_instances, 1), dtype=np.uint32)
    pos = np.zeros(max(n_instances, 1), dtype=np.int32)
    rc = lib().oracle_occurrences(packed.ctypes.data, off.ctypes.data, len(off) - 1, K, kmers.ctypes.data, nd,
                                  run_off.ctypes.data, rid.ctypes.data, pos.ctypes.data)
    if rc != 0:
        raise RuntimeError("oracle_occurrences failed rc=%d" % rc)
    return run_off, rid[:n_instances], pos[:n_instances]


def canonical(kmer_words, K):
    x = np.ascontiguousarray(kmer_words, dtype=np.uint64)
    out = np.zeros_like(x)
    lib().oracle_canonical(x.ctypes.data, out.ctypes.data, K)
    return out


def num_threads():
    return lib().oracle_num_threads()


def pack_strings(reads):
    """list of ACGT strings -> (packed uint8 padded to 8 bytes, off uint64)."""
    off = np.zeros(len(reads) + 1, dtype=np.uint64)
    total = sum(len(r) for r in reads)
    packed = np.zeros(((total + 31) // 32) * 8 + 8, dtype=np.uint8)
    q = 0
    for i, r in enumerate(reads):
        for ch in r:
            packed[q >> 2] |= "ACGT".index(ch) << ((q & 3) * 2)
            q += 1
        off[i + 1] = q
    return packed, off
