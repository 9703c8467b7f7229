"""Host-side mirror of the reference's k-mer layer over the C ABI (include/apgk.h).

Names follow the reference's entry points as BASELINE.json's north_star lists
them (their signatures could not be read -- the reference tree was empty, see
SURVEY.md section 0 -- so argument lists follow the survey's recollection):

  KmerCounter      the engine context: reads in, apgk_finish, results out
  KmerSpectrum     `class KmerSpectrum` (kmers/KmerSpectra.h): vector indexed by
                   frequency, .kspec-style text I/O, genome-size estimate
  SortKmers        `SortKmers<K>(reads, ...)`: sorted canonical k-mers with counts
  KmerParcelsBuilder  builder object with Build(); parcels = prefix buckets
  KmerFreqTable    the frequency table FindErrors queries

Everything computes on the GPU through libapgk.so; there is no CPU path here.
"""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import ASYNC_INGEST, Config, SynthParams, WANT_COUNTS, WANT_SPECTRUM, N_STAGES


class ApgkError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("apgk error %d: %s" % (code, msg))
        self.code = code


def words_per_kmer(K):
    return (2 * K + 63) // 64


DEFAULT_SEEDS = dict(seed_g=0xA11BA7C5, seed_p=0x5EED00A0, seed_q=0x5EED00A1, seed_r=0x5EED0001, seed_e=0x5EED0002)


def synth_params(genome_len, read_len, errors=True, **seeds):
    """Parameters of the synthetic read generator (SURVEY.md section 8d)."""
    s = dict(DEFAULT_SEEDS)
    s.update(seeds)
    return SynthParams(genome_len=genome_len, read_len=read_len, err_per_200=1 if errors else 0, **s)


class KmerCounter:
    """One engine context on one GPU."""

    def __init__(self, K, device=0, want_counts=True, prefix_bits=0, reserve_bases=0, max_round_keys=0,
                 async_ingest=False, max_inner_keys=0):
        self._L = _lib.lib()
        self.K = int(K)
        self.W = words_per_kmer(self.K)
        self.device = int(device)
        cfg = Config(K=self.K, device=device,
                     flags=WANT_SPECTRUM | (WANT_COUNTS if want_counts else 0) | (ASYNC_INGEST if async_ingest else 0),
                     prefix_bits=prefix_bits, reserve_bases=reserve_bases, max_round_keys=max_round_keys,
                     max_inner_keys=max_inner_keys)
        h = C.c_void_p()
        rc = self._L.apgk_create(C.byref(cfg), C.byref(h))
        if rc != 0:
            raise ApgkError(rc, "apgk_create failed (no CUDA device? there is no CPU fallback)")
        self._h = h

    # -- plumbing
    def _ck(self, rc):
        if rc != 0:
            raise ApgkError(rc, self._L.apgk_last_error(self._h).decode())

    def close(self):
        grp = getattr(self, "_group", None)
        if grp is not None:          # a group made for this counter by dist.sharded_count goes first
            self._group = None
            grp.close()
        if getattr(self, "_h", None):
            self._L.apgk_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # -- reads in
    def reset(self):
        self._ck(self._L.apgk_reset(self._h))

    def add_reads(self, packed, off):
        packed = np.ascontiguousarray(packed, dtype=np.uint8)
        off = np.ascontiguousarray(off, dtype=np.uint64)
        self._keep = (packed, off)
        self._ck(self._L.apgk_add_reads(self._h, packed.ctypes.data, off.ctypes.data, len(off) - 1))

    def add_reads_uniform(self, packed, n_reads, read_len, first_base=0):
        ptr = packed if isinstance(packed, int) else np.ascontiguousarray(packed, dtype=np.uint8).ctypes.data
        self._ck(self._L.apgk_add_reads_uniform(self._h, ptr, first_base, n_reads, read_len))

    def synth_reads(self, params, r0, n_reads):
        self._ck(self._L.apgk_synth_reads(self._h, C.byref(params), r0, n_reads))

    def export_reads(self, out=None):
        tb, _ = self.read_store_info()
        nbytes = ((tb + 31) // 32) * 8
        if out is None:
            out = np.zeros(max(nbytes, 8), dtype=np.uint8)
        ptr = out if isinstance(out, int) else out.ctypes.data
        self._ck(self._L.apgk_export_reads(self._h, ptr))
        return out

    def read_store_info(self):
        a, b = C.c_uint64(), C.c_uint64()
        self._ck(self._L.apgk_read_store_info(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    # -- hot path
    def finish(self):
        self._ck(self._L.apgk_finish(self._h))

    def finish_keys_device(self, d_ptr, n):
        self._ck(self._L.apgk_finish_keys_device(self._h, d_ptr, n))

    # -- results
    def totals(self):
        a, b = C.c_uint64(), C.c_uint64()
        self._ck(self._L.apgk_totals(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def spectrum(self):
        """dense uint64 array indexed by frequency (copy)."""
        p = C.POINTER(C.c_uint64)()
        n = C.c_uint64()
        self._ck(self._L.apgk_spectrum(self._h, C.byref(p), C.byref(n)))
        return np.ctypeslib.as_array(p, shape=(n.value,)).copy()

    def spectrum_sparse(self):
        f = C.POINTER(C.c_uint64)()
        m = C.POINTER(C.c_uint64)()
        n = C.c_uint64()
        self._ck(self._L.apgk_spectrum_sparse(self._h, C.byref(f), C.byref(m), C.byref(n)))
        if n.value == 0:
            return np.zeros(0, np.uint64), np.zeros(0, np.uint64)
        return (np.ctypeslib.as_array(f, shape=(n.value,)).copy(), np.ctypeslib.as_array(m, shape=(n.value,)).copy())

    def counts(self, first=0, n=None):
        """-> (kmers uint64[n, W], counts uint32[n]) copied to the host."""
        _, nd = self.totals()
        if n is None:
            n = nd - first
        k = np.zeros((max(n, 1), self.W), dtype=np.uint64)
        c = np.zeros(max(n, 1), dtype=np.uint32)
        self._ck(self._L.apgk_counts_copy(self._h, first, n, k.ctypes.data, c.ctypes.data))
        return k[:n], c[:n]

    def release_temp(self):
        self._ck(self._L.apgk_release_temp(self._h))

    def reserve_table(self, n_records):
        self._ck(self._L.apgk_reserve_table(self._h, n_records))

    def prefix_range(self, prefix_bits, prefix):
        """(first, n): the table records whose k-mers start with the `prefix_bits`-bit value `prefix`."""
        a, b = C.c_uint64(), C.c_uint64()
        self._ck(self._L.apgk_prefix_range(self._h, prefix_bits, prefix, C.byref(a), C.byref(b)))
        return a.value, b.value

    def counts_device(self):
        a, b = C.c_void_p(), C.c_void_p()
        n = C.c_uint64()
        self._ck(self._L.apgk_counts_device(self._h, C.byref(a), C.byref(b), C.byref(n)))
        return a.value, b.value, n.value

    def lookup(self, kmers, canonicalise=True):
        q = np.ascontiguousarray(kmers, dtype=np.uint64)
        n = q.size // self.W
        out = np.zeros(max(n, 1), dtype=np.uint32)
        self._ck(self._L.apgk_lookup(self._h, q.ctypes.data, n, 1 if canonicalise else 0, out.ctypes.data))
        return out[:n]

    def read_freqs(self, first_base=0, n_bases=None):
        tb, _ = self.read_store_info()
        if n_bases is None:
            n_bases = tb - first_base
        out = np.zeros(max(n_bases, 1), dtype=np.uint32)
        self._ck(self._L.apgk_read_freqs(self._h, first_base, n_bases, out.ctypes.data))
        return out[:n_bases]

    def read_freqs_device(self, d_out):
        """Count of the canonical k-mer at every base of the store into a DEVICE buffer (uint32[total_bases],
        0xFFFFFFFF where the window leaves its read).  -> device ms {clear, sweep, place}."""
        ms = (C.c_float * 3)()
        self._ck(self._L.apgk_read_freqs_device(self._h, d_out, ms))
        return dict(zip(("clear", "sweep", "place"), [float(x) for x in ms]))

    # -- occurrence records: (read id, signed position) of every instance, grouped by k-mer
    def build_occurrences(self):
        """Second sweep over the read store: every window takes a slot in its k-mer's run (needs finish()
        with want_counts).  -> dict(n_occ, n_big_runs, ms={scan, scatter, place, sort, sort_big})."""
        self._ck(self._L.apgk_build_occurrences(self._h))
        return self.occurrences_info()

    def occurrences_info(self):
        n, nb = C.c_uint64(), C.c_uint64()
        ms = (C.c_float * 5)()
        self._ck(self._L.apgk_occurrences_info(self._h, C.byref(n), C.byref(nb), ms))
        return dict(n_occ=n.value, n_big_runs=nb.value, ms=dict(zip(("scan", "scatter", "place", "sort", "sort_big"), [float(x) for x in ms])))

    def occurrences(self, first=0, n=None):
        """-> (run_off uint64[n+1] rebased to 0, read_id uint32[m], pos int32[m]) for k-mers [first, first+n) of
        the sorted table; k-mer first+i owns slots [run_off[i], run_off[i+1]), ascending by (read id, position);
        pos is 1-based, negative when the canonical form is the reverse complement of the read's window.  On a shard
        after KmerGroup.build_occurrences() the read ids are group read ids."""
        _, nd = self.totals()
        if n is None:
            n = nd - first
        ro = np.zeros(n + 1, dtype=np.uint64)
        self._ck(self._L.apgk_occurrences_copy(self._h, first, n, ro.ctypes.data, None, None))
        m = int(ro[-1] - ro[0])
        rid = np.zeros(max(m, 1), dtype=np.uint32)
        pos = np.zeros(max(m, 1), dtype=np.int32)
        if m:
            self._ck(self._L.apgk_occurrences_copy(self._h, first, n, None, rid.ctypes.data, pos.ctypes.data))
        return ro - ro[0], rid[:m], pos[:m]

    def occurrences_device(self):
        """-> (device pointer of the run offsets, device pointer of the records, n_occ); the record encoding is
        include/apgk.h's (read-id form on a shard after KmerGroup.build_occurrences())."""
        a, b = C.c_void_p(), C.c_void_p()
        n = C.c_uint64()
        self._ck(self._L.apgk_occurrences_device(self._h, C.byref(a), C.byref(b), C.byref(n)))
        return a.value, b.value, n.value

    # -- affixes: which bases precede (bits 0-3) and follow (bits 4-7) every distinct k-mer, canonical orientation
    def build_affixes(self):
        """Sweep of the read store that ORs every window's neighbour bases into its k-mer's affix byte (needs
        finish() with want_counts).  -> device ms {scan, sweep, place}."""
        ms = (C.c_float * 3)()
        self._ck(self._L.apgk_build_affixes(self._h, ms))
        return dict(zip(("scan", "sweep", "place"), [float(x) for x in ms]))

    def affixes(self, first=0, n=None):
        """-> uint8[n]: the affix bytes of rows [first, first+n) of the sorted table."""
        _, nd = self.totals()
        if n is None:
            n = nd - first
        out = np.zeros(max(n, 1), dtype=np.uint8)
        self._ck(self._L.apgk_affixes_copy(self._h, first, n, out.ctypes.data))
        return out[:n]

    def affixes_device(self):
        """-> (device pointer of uint8[n_distinct], n_distinct)"""
        p = C.c_void_p()
        n = C.c_uint64()
        self._ck(self._L.apgk_affixes_device(self._h, C.byref(p), C.byref(n)))
        return p.value, n.value

    def lookup_affixes(self, kmers, canonicalise=True):
        """-> (affixes uint8[n] in each query's own orientation, counts uint32[n]); absent k-mers give (0, 0)."""
        q = np.ascontiguousarray(kmers, dtype=np.uint64)
        n = q.size // self.W
        aff = np.zeros(max(n, 1), dtype=np.uint8)
        cnt = np.zeros(max(n, 1), dtype=np.uint32)
        self._ck(self._L.apgk_lookup_affixes(self._h, q.ctypes.data, n, 1 if canonicalise else 0, aff.ctypes.data,
                                             cnt.ctypes.data))
        return aff[:n], cnt[:n]

    # -- multi-GPU building blocks
    def owner_plan(self, n_ranks):
        out = np.zeros(n_ranks, dtype=np.uint64)
        self._ck(self._L.apgk_owner_plan(self._h, n_ranks, out.ctypes.data))
        return out

    def owner_scatter(self, d_ptr):
        self._ck(self._L.apgk_owner_scatter(self._h, d_ptr))

    def key_buffer(self, n_keys):
        """device pointer of the library's level-0 key buffer, sized for n_keys k-mers"""
        p = C.c_void_p()
        self._ck(self._L.apgk_key_buffer(self._h, n_keys, C.byref(p)))
        return p.value

    # -- multi-GPU, partition-first form
    def window_upper(self):
        u = C.c_uint64()
        self._ck(self._L.apgk_window_upper(self._h, C.byref(u)))
        return u.value

    def choose_prefix_bits(self, upper):
        p = C.c_int32()
        self._ck(self._L.apgk_choose_prefix_bits(self._h, upper, C.byref(p)))
        return p.value

    def partition(self, prefix_bits=0):
        """levels 0+1 only; raises ApgkError (code APGK_E_RANGE) if one k-mer-space round is not enough"""
        self._ck(self._L.apgk_partition(self._h, prefix_bits))

    def partition_range(self, prefix_bits, d0_lo, d0_hi):
        """Levels 0 + 1 restricted to the level-0 buckets [d0_lo, d0_hi): one k-mer-space round of the sharded form."""
        self._ck(self._L.apgk_partition_range(self._h, prefix_bits, d0_lo, d0_hi))

    def level0_totals(self):
        """-> (uint64[2^D0] instances per level-0 bucket of the last partition call, round capacity in instances)."""
        n = C.c_uint32()
        cap = C.c_uint64()
        self._ck(self._L.apgk_level0_totals(self._h, None, 0, C.byref(n), C.byref(cap)))
        out = np.zeros(n.value, dtype=np.uint64)
        self._ck(self._L.apgk_level0_totals(self._h, out.ctypes.data, n.value, None, None))
        return out, cap.value

    def partition_info(self):
        """-> (d_bucket_sizes ptr (uint64[n_buckets]), n_buckets, d_elems ptr, elem_bytes, n_elems)"""
        a, b = C.c_void_p(), C.c_void_p()
        nb, ne = C.c_uint64(), C.c_uint64()
        eb = C.c_uint32()
        self._ck(self._L.apgk_partition_info(self._h, C.byref(a), C.byref(nb), C.byref(b), C.byref(eb), C.byref(ne)))
        return a.value, nb.value, b.value, eb.value, ne.value

    def count_pieces(self, d_recv, n_src, d_sizes_all, seg_off, bucket_lo, bucket_hi, split_bits=None):
        so = np.ascontiguousarray(seg_off, dtype=np.uint64)
        if split_bits is None:
            split_bits = max(0, (n_src - 1).bit_length())
        self._ck(self._L.apgk_count_pieces(self._h, d_recv, n_src, d_sizes_all, so.ctypes.data, bucket_lo, bucket_hi,
                                           split_bits))

    def partition_subsizes(self, split_bits):
        """-> (effective split bits, device pointer of uint32[n_buckets << bits] sub-bucket sizes)"""
        eff = C.c_int32()
        p = C.c_void_p()
        self._ck(self._L.apgk_partition_subsizes(self._h, split_bits, C.byref(eff), C.byref(p)))
        return eff.value, p.value

    def count_pieces_peer(self, src_ptrs, d_sizes_all, src_off, bucket_lo, bucket_hi, split_bits=None, d_sub_sizes=None):
        """src_ptrs: one device pointer per source rank (0 / None = this context's own partition buffer)"""
        n_src = len(src_ptrs)
        bases = (C.c_void_p * n_src)(*[C.c_void_p(int(p) if p else 0) for p in src_ptrs])
        so = np.ascontiguousarray(src_off, dtype=np.uint64)
        if split_bits is None:
            split_bits = max(0, (n_src - 1).bit_length())
        self._ck(self._L.apgk_count_pieces_peer(self._h, bases, n_src, d_sizes_all, so.ctypes.data, bucket_lo, bucket_hi,
                                                split_bits, d_sub_sizes))

    def partition_export(self):
        h = np.zeros(64, dtype=np.uint8)
        self._ck(self._L.apgk_partition_export(self._h, h.ctypes.data))
        return h

    def peer_open(self, handle):
        h = np.ascontiguousarray(handle, dtype=np.uint8)
        p = C.c_void_p()
        self._ck(self._L.apgk_peer_open(self._h, h.ctypes.data, C.byref(p)))
        return p.value

    def peer_close(self, ptr):
        self._ck(self._L.apgk_peer_close(self._h, ptr))

    def spectrum_device(self):
        p = C.c_void_p()
        n = C.c_uint64()
        self._ck(self._L.apgk_spectrum_device(self._h, C.byref(p), C.byref(n)))
        return p.value, n.value

    def spectrum_reload(self):
        self._ck(self._L.apgk_spectrum_reload(self._h))

    # -- instrumentation
    def stage_ms(self):
        arr = (C.c_float * N_STAGES)()
        self._ck(self._L.apgk_stage_ms(self._h, arr))
        return {self._L.apgk_stage_name(i).decode(): float(arr[i]) for i in range(N_STAGES)}

    def kernel_launches(self):
        return int(self._L.apgk_kernel_launches(self._h))

    def reset_counters(self):
        self._L.apgk_reset_counters(self._h)

    def debug_counters(self, reset=True):
        out = np.zeros(8, dtype=np.uint64)
        self._ck(self._L.apgk_debug_counters(self._h, out.ctypes.data, 1 if reset else 0))
        return dict(passes=int(out[0]), row_overflows=int(out[1]), tag_collisions=int(out[2]), buckets=int(out[3]))

    def geometry(self):
        g = (C.c_int32 * 8)()
        self._ck(self._L.apgk_geometry(self._h, g))
        return dict(D0=g[0], D1=g[1], REM=g[2], elem_bytes=g[3], n_big=g[4], n_deferred=g[5], local_max=g[6],
                    n_rounds=g[7])


class KmerGroup:
    """A group of ranks counting one read set sharded by canonical k-mer (include/apgk.h "a GROUP of ranks").
    `KmerGroup.local([kc0, kc1, ...])`: one process drives all the contexts; `KmerGroup.join(kc, uid, rank, world)`:
    one process per GPU, uid = KmerGroup.unique_id() made on rank 0 and handed to every rank by the caller."""

    def __init__(self, handle, counters):
        self._L = _lib.lib()
        self._h = handle
        self.counters = list(counters)

    @staticmethod
    def unique_id():
        buf = np.zeros(128, dtype=np.uint8)
        rc = _lib.lib().apgk_group_unique_id(buf.ctypes.data)
        if rc != 0:
            raise ApgkError(rc, "apgk_group_unique_id failed (libnccl.so.2 not loadable?)")
        return buf

    @classmethod
    def join(cls, kc, uid, rank, world):
        uid = np.ascontiguousarray(uid, dtype=np.uint8)
        assert uid.size == 128
        h = C.c_void_p()
        rc = _lib.lib().apgk_group_join(kc._h, uid.ctypes.data, rank, world, C.byref(h))
        if rc != 0:
            raise ApgkError(rc, kc._L.apgk_last_error(kc._h).decode())
        return cls(h, [kc])

    @classmethod
    def local(cls, counters):
        arr = (C.c_void_p * len(counters))(*[kc._h for kc in counters])
        h = C.c_void_p()
        rc = _lib.lib().apgk_group_local(arr, len(counters), C.byref(h))
        if rc != 0:
            raise ApgkError(rc, counters[0]._L.apgk_last_error(counters[0]._h).decode())
        return cls(h, counters)

    def _ck(self, rc):
        if rc != 0:
            raise ApgkError(rc, self._L.apgk_group_last_error(self._h).decode())

    def count(self):
        """The sharded hot path over the read stores the contexts hold now (collective)."""
        self._ck(self._L.apgk_group_count(self._h))
        return self

    def totals(self):
        a, b = C.c_uint64(), C.c_uint64()
        self._ck(self._L.apgk_group_totals(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def spectrum_sparse(self):
        f, m, n = C.POINTER(C.c_uint64)(), C.POINTER(C.c_uint64)(), C.c_uint64()
        self._ck(self._L.apgk_group_spectrum_sparse(self._h, C.byref(f), C.byref(m), C.byref(n)))
        k = n.value
        if not k:
            return np.zeros(0, np.uint64), np.zeros(0, np.uint64)
        return (np.ctypeslib.as_array(f, shape=(k,)).copy(), np.ctypeslib.as_array(m, shape=(k,)).copy())

    def spectrum(self):
        """dense global spectrum: index = frequency"""
        f, m = self.spectrum_sparse()
        out = np.zeros(int(f[-1]) + 1 if len(f) else 1, dtype=np.uint64)
        out[f.astype(np.int64)] = m
        return out

    def stats(self):
        st = _lib.GroupStats()
        self._ck(self._L.apgk_group_stats_get(self._h, C.byref(st)))
        return {k: getattr(st, k) for k, _ in st._fields_}

    def read_freqs_device(self, d_outs, first_base=None, n_bases=None):
        """Frequency lookups on the sharded table (collective): for every local counter j, d_outs[j] (a DEVICE pointer
        on that counter's device, n_bases[j] uint32) receives the GLOBAL count of the canonical k-mer at every base of
        [first_base[j], first_base[j] + n_bases[j]) of its read store, 0xFFFFFFFF where the window leaves its read.
        Defaults: the whole store.  -> dict(n_batches, n_queries, remote_bytes, sweep_ms, exchange_ms, scatter_ms,
        total_ms)."""
        first_base, n_bases = self._ranges(first_base, n_bases)
        n = len(self.counters)
        outs = (C.c_void_p * n)(*[int(p) if p else None for p in d_outs])
        fb = np.ascontiguousarray(first_base, dtype=np.uint64)
        nb = np.ascontiguousarray(n_bases, dtype=np.uint64)
        st = _lib.GroupFreqStats()
        self._ck(self._L.apgk_group_read_freqs_device(self._h, outs, fb.ctypes.data, nb.ctypes.data, C.byref(st)))
        return {k: getattr(st, k) for k, _ in st._fields_}

    def read_freqs(self, first_base=None, n_bases=None, stats=None):
        """The same into host arrays: a list of uint32 arrays, one per local counter (device buffers from torch on each
        counter's device).  stats: a dict to receive the call's statistics."""
        import torch

        first_base, n_bases = self._ranges(first_base, n_bases)
        bufs = [torch.empty(max(int(n), 1), dtype=torch.int32, device="cuda:%d" % kc.device)
                for kc, n in zip(self.counters, n_bases)]
        st = self.read_freqs_device([b.data_ptr() for b in bufs], first_base, n_bases)
        if stats is not None:
            stats.update(st)
        return [b.cpu().numpy().view(np.uint32)[: int(n)] for b, n in zip(bufs, n_bases)]

    def build_affixes(self):
        """K-mer affixes on the sharded table (collective): afterwards every local counter's affixes() /
        lookup_affixes() answer for the k-mers its shard owns, each byte taken over all ranks' reads.
        -> dict(n_batches, n_windows, remote_bytes, sweep_ms, exchange_ms, total_ms)."""
        st = _lib.GroupAffixStats()
        self._ck(self._L.apgk_group_build_affixes(self._h, C.byref(st)))
        return {k: getattr(st, k) for k, _ in st._fields_}

    def build_occurrences(self):
        """K-mer occurrence records on the sharded table (collective): afterwards every local counter's occurrences() /
        occurrences_device() answer for the rows of its shard, taken over all ranks' reads, with GROUP read ids (every
        rank's reads in rank order).  -> dict(n_batches, n_windows, n_occ, n_big_runs, remote_bytes, sweep_ms,
        exchange_ms, sort_ms, total_ms)."""
        st = _lib.GroupOccStats()
        self._ck(self._L.apgk_group_build_occurrences(self._h, C.byref(st)))
        return {k: getattr(st, k) for k, _ in st._fields_}

    def _ranges(self, first_base, n_bases):
        n = len(self.counters)
        if first_base is None:
            first_base = [0] * n
        if n_bases is None:
            n_bases = [kc.read_store_info()[0] - int(f) for kc, f in zip(self.counters, first_base)]
        first_base, n_bases = [int(x) for x in first_base], [int(x) for x in n_bases]
        if len(first_base) != n or len(n_bases) != n:
            raise ValueError("one first_base and one n_bases per local counter")
        return first_base, n_bases

    def close(self):
        if getattr(self, "_h", None):
            self._L.apgk_group_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def owner_of(K, kmers, n_ranks):
    q = np.ascontiguousarray(kmers, dtype=np.uint64)
    n = q.size // words_per_kmer(K)
    out = np.zeros(max(n, 1), dtype=np.uint32)
    rc = _lib.lib().apgk_owner_of(K, q.ctypes.data, n, n_ranks, out.ctypes.data)
    if rc:
        raise ApgkError(rc, "apgk_owner_of")
    return out[:n]


# ---------------------------------------------------------------------------
# Reference-named entry points
# ---------------------------------------------------------------------------
class KmerSpectrum:
    """Mirror of the reference's `class KmerSpectrum` (kmers/KmerSpectra.h, unverified path):
    a vector indexed by k-mer frequency holding the number of distinct k-mers with that
    frequency, with text I/O and the genome-size / coverage estimate the pipeline reports."""

    def __init__(self, K, spec=None):
        self.K = int(K)
        self.spec = np.zeros(1, dtype=np.uint64) if spec is None else np.asarray(spec, dtype=np.uint64).copy()

    def __len__(self):
        return len(self.spec)

    def __getitem__(self, f):
        return int(self.spec[f]) if 0 <= f < len(self.spec) else 0

    def n_distinct(self):
        return int(self.spec.sum())

    def n_instances(self):
        return int((self.spec * np.arange(len(self.spec), dtype=np.uint64)).sum())

    @classmethod
    def from_reads(cls, packed, off, K, device=0):
        with KmerCounter(K, device=device, want_counts=False) as kc:
            kc.add_reads(packed, off)
            kc.finish()
            return cls(K, kc.spectrum())

    def write(self, path):
        """Text form: a header line, then `frequency n_kmers` per non-zero entry."""
        with open(path, "w") as f:
            f.write("# kmer spectrum K=%d\n" % self.K)
            for fr in np.nonzero(self.spec)[0]:
                f.write("%d %d\n" % (fr, int(self.spec[fr])))

    @classmethod
    def read(cls, path):
        K, pairs = 0, []
        with open(path) as f:
            for line in f:
                if line.startswith("#"):
                    if "K=" in line:
                        K = int(line.split("K=")[1].split()[0])
                    continue
                a, b = line.split()
                pairs.append((int(a), int(b)))
        spec = np.zeros((max(a for a, _ in pairs) + 1) if pairs else 1, dtype=np.uint64)
        for a, b in pairs:
            spec[a] = b
        return cls(K, spec)

    def estimate(self, read_len=None):
        """Coverage peak and genome size from the spectrum: the first local minimum separates
        error k-mers from genomic ones; the mode above it is the k-mer coverage; genome size is
        (instances above the minimum) / coverage.  (The estimators are floating point and are not
        part of the bit-exact parity contract -- SURVEY.md section 8a.)"""
        s = self.spec.astype(np.float64)
        if len(s) < 4:
            return dict(f_min=0, kmer_coverage=0.0, genome_size=0.0, coverage=0.0)
        f_min = 1
        while f_min + 1 < len(s) and s[f_min + 1] < s[f_min]:
            f_min += 1
        f_peak = f_min + int(np.argmax(s[f_min:]))
        inst = float((s[f_min:] * np.arange(f_min, len(s))).sum())
        g = inst / f_peak if f_peak else 0.0
        cov = f_peak * read_len / (read_len - self.K + 1) if read_len else 0.0
        return dict(f_min=f_min, kmer_coverage=float(f_peak), genome_size=g, coverage=cov)


def SortKmers(packed, off, K, device=0, records=False):
    """Mirror of the reference's SortKmers builder: all canonical k-mers of the reads, sorted ascending.
    records=False (the counting contract) -> (kmers uint64[n, W], counts uint32[n]).
    records=True (the full kmer-record vector: one record per INSTANCE, sorted by k-mer, ties by
    (read id, position)) -> (kmers uint64[N, W], read_id uint32[N], pos int32[N]); pos is 1-based and
    negative when the canonical k-mer is the reverse complement of the read's window."""
    with KmerCounter(K, device=device, want_counts=True) as kc:
        kc.add_reads(packed, off)
        kc.finish()
        k, c = kc.counts()
        if not records:
            return k, c
        kc.build_occurrences()
        _, rid, pos = kc.occurrences()
        return np.repeat(k, c.astype(np.int64), axis=0), rid, pos


class KmerParcelsBuilder:
    """Mirror of the reference's KmerParcelsBuilder: construct with the reads, call Build(),
    then read parcels.  A parcel here is one level-0 bucket of k-mer space (the leading D0 bits);
    within a parcel the batches of identical k-mers are the (k-mer, count) records."""

    def __init__(self, K, packed, off, device=0):
        self.K = K
        self._kc = KmerCounter(K, device=device, want_counts=True)
        self._kc.add_reads(packed, off)
        self._built = False
        self._occ = False

    def Build(self):
        self._kc.finish()
        self._built = True
        return self

    def NumKmersDistinct(self):
        return self._kc.totals()[1]

    def NumKmerInstances(self):
        return self._kc.totals()[0]

    def Spectrum(self):
        return KmerSpectrum(self.K, self._kc.spectrum())

    def Records(self, first=0, n=None):
        return self._kc.counts(first, n)

    def Batches(self, first=0, n=None):
        """The batches of k-mers [first, first+n): (kmers, run_off, read_id, pos) -- k-mer i's instances are
        (read_id, pos)[run_off[i]:run_off[i+1]] (KmerParcels' "k-mer + list of (read id, position)")."""
        if not self._occ:
            self._kc.build_occurrences()
            self._occ = True
        k, _ = self._kc.counts(first, n)
        ro, rid, pos = self._kc.occurrences(first, n)
        return k, ro, rid, pos

    def close(self):
        self._kc.close()


class KmerFreqTable:
    """The k-mer frequency table error correction queries (FindErrors): built once from the reads,
    then asked for the frequency of arbitrary k-mers or of every window of the reads."""

    def __init__(self, K, packed, off, device=0):
        self.K = K
        self._kc = KmerCounter(K, device=device, want_counts=True)
        self._kc.add_reads(packed, off)
        self._kc.finish()

    def freq(self, kmers, canonicalise=True):
        return self._kc.lookup(kmers, canonicalise)

    def read_freqs(self, first_base=0, n_bases=None):
        return self._kc.read_freqs(first_base, n_bases)

    def spectrum(self):
        return KmerSpectrum(self.K, self._kc.spectrum())

    def close(self):
        self._kc.close()
