"""ctypes binding of libapgk.so (the C ABI in include/apgk.h).

The shared library is built in-tree by __graft_entry__.build() / `make -C allpathslg_b200/csrc`.
There is no fallback: if the library is missing, import of the symbols fails loudly.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libapgk.so")

APGK_OK = 0
E_ARG, E_CUDA, E_NOMEM, E_STATE, E_RANGE = -1, -2, -3, -4, -5
WANT_SPECTRUM, WANT_COUNTS, ASYNC_INGEST = 1, 2, 4
N_STAGES = 14
MAX_K = 96


class Config(C.Structure):
    _fields_ = [("K", C.c_int32), ("device", C.c_int32), ("flags", C.c_uint32), ("prefix_bits", C.c_int32),
                ("reserve_bases", C.c_uint64), ("max_round_keys", C.c_uint64),
                ("max_inner_keys", C.c_uint64)]


class GroupStats(C.Structure):
    _fields_ = [("world", C.c_int32), ("n_rounds", C.c_int32), ("n_outer_rounds", C.c_int32), ("prefix_bits", C.c_int32),
                ("split_bits", C.c_int32), ("peer_exchange", C.c_int32), ("shard_instances", C.c_uint64),
                ("remote_bytes", C.c_uint64), ("gather_ms", C.c_float), ("step_ms", C.c_float)]


class GroupFreqStats(C.Structure):
    _fields_ = [("n_batches", C.c_int32), ("n_queries", C.c_uint64), ("remote_bytes", C.c_uint64), ("sweep_ms", C.c_float),
                ("exchange_ms", C.c_float), ("scatter_ms", C.c_float), ("total_ms", C.c_float)]


class SynthParams(C.Structure):
    _fields_ = [("genome_len", C.c_uint64), ("seed_g", C.c_uint64), ("seed_p", C.c_uint64), ("seed_q", C.c_uint64),
                ("seed_r", C.c_uint64), ("seed_e", C.c_uint64), ("read_len", C.c_uint32), ("err_per_200", C.c_uint32)]


# every symbol include/apgk.h declares: name -> (restype, argtypes)
_u64p = C.POINTER(C.c_uint64)
_u32p = C.POINTER(C.c_uint32)
_vp = C.c_void_p
SYMBOLS = {
    "apgk_create": (C.c_int, [C.POINTER(Config), C.POINTER(_vp)]),
    "apgk_destroy": (None, [_vp]),
    "apgk_last_error": (C.c_char_p, [_vp]),
    "apgk_words_per_kmer": (C.c_int, [C.c_int]),
    "apgk_reset": (C.c_int, [_vp]),
    "apgk_add_reads": (C.c_int, [_vp, _vp, _vp, C.c_uint64]),
    "apgk_add_reads_uniform": (C.c_int, [_vp, _vp, C.c_uint64, C.c_uint64, C.c_uint32]),
    "apgk_synth_reads": (C.c_int, [_vp, C.POINTER(SynthParams), C.c_uint64, C.c_uint64]),
    "apgk_export_reads": (C.c_int, [_vp, _vp]),
    "apgk_read_store_info": (C.c_int, [_vp, _u64p, _u64p]),
    "apgk_finish": (C.c_int, [_vp]),
    "apgk_totals": (C.c_int, [_vp, _u64p, _u64p]),
    "apgk_spectrum": (C.c_int, [_vp, C.POINTER(_u64p), _u64p]),
    "apgk_spectrum_sparse": (C.c_int, [_vp, C.POINTER(_u64p), C.POINTER(_u64p), _u64p]),
    "apgk_counts_device": (C.c_int, [_vp, C.POINTER(_vp), C.POINTER(_vp), _u64p]),
    "apgk_counts_copy": (C.c_int, [_vp, C.c_uint64, C.c_uint64, _vp, _vp]),
    "apgk_reserve_table": (C.c_int, [_vp, C.c_uint64]),
    "apgk_release_temp": (C.c_int, [_vp]),
    "apgk_prefix_range": (C.c_int, [_vp, C.c_int32, C.c_uint64, _u64p, _u64p]),
    "apgk_lookup": (C.c_int, [_vp, _vp, C.c_uint64, C.c_int, _vp]),
    "apgk_read_freqs": (C.c_int, [_vp, C.c_uint64, C.c_uint64, _vp]),
    "apgk_read_freqs_device": (C.c_int, [_vp, _vp, C.POINTER(C.c_float)]),
    "apgk_build_occurrences": (C.c_int, [_vp]),
    "apgk_occurrences_info": (C.c_int, [_vp, _u64p, _u64p, C.POINTER(C.c_float)]),
    "apgk_occurrences_device": (C.c_int, [_vp, C.POINTER(_vp), C.POINTER(_vp), _u64p]),
    "apgk_occurrences_copy": (C.c_int, [_vp, C.c_uint64, C.c_uint64, _vp, _vp, _vp]),
    "apgk_owner_plan": (C.c_int, [_vp, C.c_uint32, _vp]),
    "apgk_owner_scatter": (C.c_int, [_vp, _vp]),
    "apgk_key_buffer": (C.c_int, [_vp, C.c_uint64, C.POINTER(_vp)]),
    "apgk_owner_of": (C.c_int, [C.c_int, _vp, C.c_uint64, C.c_uint32, _vp]),
    "apgk_finish_keys_device": (C.c_int, [_vp, _vp, C.c_uint64]),
    "apgk_window_upper": (C.c_int, [_vp, C.POINTER(C.c_uint64)]),
    "apgk_choose_prefix_bits": (C.c_int, [_vp, C.c_uint64, C.POINTER(C.c_int32)]),
    "apgk_partition": (C.c_int, [_vp, C.c_int32]),
    "apgk_partition_range": (C.c_int, [_vp, C.c_int32, C.c_int32, C.c_int32]),
    "apgk_level0_totals": (C.c_int, [_vp, _vp, C.c_uint32, C.POINTER(C.c_uint32), C.POINTER(C.c_uint64)]),
    "apgk_partition_info": (C.c_int, [_vp, C.POINTER(_vp), C.POINTER(C.c_uint64), C.POINTER(_vp), C.POINTER(C.c_uint32),
                                      C.POINTER(C.c_uint64)]),
    "apgk_count_pieces": (C.c_int, [_vp, _vp, C.c_uint32, _vp, _vp, C.c_uint64, C.c_uint64, C.c_int32]),
    "apgk_count_pieces_peer": (C.c_int, [_vp, _vp, C.c_uint32, _vp, _vp, C.c_uint64, C.c_uint64, C.c_int32, _vp]),
    "apgk_partition_subsizes": (C.c_int, [_vp, C.c_int32, C.POINTER(C.c_int32), C.POINTER(_vp)]),
    "apgk_partition_export": (C.c_int, [_vp, _vp]),
    "apgk_peer_open": (C.c_int, [_vp, _vp, C.POINTER(_vp)]),
    "apgk_peer_close": (C.c_int, [_vp, _vp]),
    "apgk_group_unique_id": (C.c_int, [_vp]),
    "apgk_group_join": (C.c_int, [_vp, _vp, C.c_int32, C.c_int32, C.POINTER(_vp)]),
    "apgk_group_local": (C.c_int, [C.POINTER(_vp), C.c_int32, C.POINTER(_vp)]),
    "apgk_group_destroy": (None, [_vp]),
    "apgk_group_last_error": (C.c_char_p, [_vp]),
    "apgk_group_count": (C.c_int, [_vp]),
    "apgk_group_totals": (C.c_int, [_vp, _u64p, _u64p]),
    "apgk_group_spectrum_sparse": (C.c_int, [_vp, C.POINTER(_u64p), C.POINTER(_u64p), _u64p]),
    "apgk_group_stats_get": (C.c_int, [_vp, C.POINTER(GroupStats)]),
    "apgk_group_read_freqs_device": (C.c_int, [_vp, _vp, _vp, _vp, C.POINTER(GroupFreqStats)]),
    "apgk_spectrum_device": (C.c_int, [_vp, C.POINTER(_vp), _u64p]),
    "apgk_spectrum_reload": (C.c_int, [_vp]),
    "apgk_stage_ms": (C.c_int, [_vp, C.POINTER(C.c_float)]),
    "apgk_stage_name": (C.c_char_p, [C.c_int]),
    "apgk_kernel_launches": (C.c_uint64, [_vp]),
    "apgk_reset_counters": (None, [_vp]),
    "apgk_geometry": (C.c_int, [_vp, C.POINTER(C.c_int32)]),
    "apgk_device_alloc": (C.c_int, [_vp, C.POINTER(_vp), C.c_size_t]),
    "apgk_device_free": (C.c_int, [_vp, _vp]),
    "apgk_device_copy_to_host": (C.c_int, [_vp, _vp, _vp, C.c_size_t]),
    "apgk_host_alloc": (C.c_int, [C.POINTER(_vp), C.c_size_t]),
    "apgk_host_free": (C.c_int, [_vp]),
    "apgk_debug_counters": (C.c_int, [_vp, _vp, C.c_int]),
    "apgk_debug_host_extract": (C.c_int, [_vp, _vp, C.c_uint64, C.c_int, _vp, _vp]),
    "apgk_debug_host_topdigits": (C.c_int, [_vp, _vp, C.c_uint64, C.c_int, C.c_int, _vp]),
    "apgk_debug_host_canonical": (C.c_int, [C.c_int, _vp, C.c_uint64, _vp]),
    "apgk_debug_host_table_find": (C.c_int, [C.c_int, _vp, C.c_uint64, C.c_int, _vp, C.c_uint64, _vp]),
    "apgk_debug_host_splitters": (C.c_int, [_vp, C.c_uint32, C.c_uint32, C.c_uint32, _vp]),
    "apgk_debug_host_synth": (C.c_int, [C.POINTER(SynthParams), C.c_uint64, C.c_uint64, _vp]),
}

_lib = None


def lib():
    """Load libapgk.so.  Raises (never falls back) if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "libapgk.so is missing at %s: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "or `make -C allpathslg_b200/csrc`.  There is no CPU fallback." % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            f = getattr(L, name)  # AttributeError if the symbol is not exported
            f.restype = res
            f.argtypes = args
        _lib = L
    return _lib
