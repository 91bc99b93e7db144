"""ctypes binding of libdkb.so (include/dkb.h).  The library is built in-tree by
`denovo_kmer_b200.build.build()`; importing this module never builds or falls back:
a missing library is an ImportError, a missing GPU is DKB_ENODEV at ctx_create."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("DKB_LIBRARY") or os.path.join(_HERE, "libdkb.so")  # override: A/B builds

OK, EINVAL, ECUDA, ENOMEM, ESTATE, ENODEV, ENCCL = range(7)
COMM_ID_BYTES = 128
MAX_MULTI = 4
MAX_CHILDREN = 6

u8p = C.POINTER(C.c_uint8)
u16p = C.POINTER(C.c_uint16)
u32p = C.POINTER(C.c_uint32)
u64p = C.POINTER(C.c_uint64)


class Thresholds(C.Structure):
    _fields_ = [("min_child_alt_hits", C.c_uint32), ("min_child_alt_distinct", C.c_uint32),
                ("max_parent_alt_hits", C.c_uint32), ("min_parent_ref_hits", C.c_uint32)]


class Tuning(C.Structure):
    _fields_ = [("seed_len", C.c_int), ("stride", C.c_int), ("bloom_hashes", C.c_int),
                ("filter_mode", C.c_int)]


class Stats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in (
        "n_entries", "n_live_entries", "table_slots", "n_seeds", "seed_slots", "bloom_words",
        "bloom_bits_set", "scan_launches", "positions_scanned", "bloom_hits", "seed_hits",
        "windows_probed", "window_hits", "scan_launches_timed")] + [
        ("scan_ms_total", C.c_double), ("last_scan_ms", C.c_float), ("prefilter_words", C.c_uint32),
        ("gated_lookups", C.c_uint32), ("occupied_halves", C.c_uint64), ("direct_halves", C.c_uint64)]


# every symbol include/dkb.h declares: (restype, argtypes)
SYMBOLS = {
    "dkb_abi_version": (C.c_int, []),
    "dkb_strerror": (C.c_char_p, [C.c_int]),
    "dkb_last_error": (C.c_char_p, [C.c_void_p]),
    "dkb_ctx_create": (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "dkb_ctx_create_family": (C.c_int, [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "dkb_ctx_get_children": (C.c_int, [C.c_void_p, C.POINTER(C.c_int)]),
    "dkb_ctx_destroy": (C.c_int, [C.c_void_p]),
    "dkb_ctx_set_tuning": (C.c_int, [C.c_void_p, C.POINTER(Tuning)]),
    "dkb_ctx_get_tuning": (C.c_int, [C.c_void_p, C.POINTER(Tuning)]),
    "dkb_kmer_encode": (C.c_int, [C.c_char_p, C.c_int, u64p]),
    "dkb_kmer_revcomp": (C.c_uint64, [C.c_uint64, C.c_int]),
    "dkb_kmer_canonical": (C.c_uint64, [C.c_uint64, C.c_int]),
    "dkb_stream_positions": (C.c_uint64, [u64p, C.c_size_t]),
    "dkb_stream_bases_words": (C.c_size_t, [C.c_uint64]),
    "dkb_stream_mask_words": (C.c_size_t, [C.c_uint64]),
    "dkb_pack_reads": (C.c_int, [u8p, u8p, u64p, C.c_size_t, C.c_int, u32p, u32p, u64p]),
    "dkb_pack_reads_fmt": (C.c_int, [u8p, C.c_int, u8p, u64p, C.c_size_t, C.c_int, u32p, u32p, u64p]),
    "dkb_zero_list_blocks": (C.c_size_t, [C.c_uint64]),
    "dkb_mask_to_zero_list": (C.c_int, [u32p, C.c_uint64, u32p, u8p, C.c_size_t, C.POINTER(C.c_size_t)]),
    "dkb_variant_kmers": (C.c_int, [C.POINTER(C.c_char_p)] * 4 + [C.c_size_t, C.c_int, C.c_int,
                                    u64p, u32p, u8p, u16p, u16p, C.POINTER(C.c_size_t)]),
    "dkb_table_build": (C.c_int, [C.c_void_p, u64p, u32p, u8p, u16p, u16p, C.c_size_t,
                                  C.c_uint32]),
    "dkb_batch_submit": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_int]),
    "dkb_batch_submit_sparse": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                                          C.c_uint64, C.c_int]),
    "dkb_batch_submit_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64,
                                          C.c_int]),
    "dkb_batch_submit_reads": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                         C.c_size_t, C.c_int, C.c_int]),
    "dkb_batch_submit_device_multi": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p),
                                                C.POINTER(C.c_void_p), u64p, C.POINTER(C.c_int)]),
    "dkb_table_set_regions": (C.c_int, [C.c_void_p, u64p, u64p, C.c_uint32]),
    "dkb_batch_set_loci": (C.c_int, [C.c_void_p, u64p, u64p, u64p, C.c_size_t]),
    "dkb_batch_submit_multi": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), u64p,
                                         C.POINTER(C.c_int)]),
    "dkb_batch_submit_sparse_multi": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p),
                                                C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), u64p,
                                                C.POINTER(C.c_int)]),
    "dkb_batch_submit_reads_multi": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.c_int,
                                               C.POINTER(C.c_void_p), C.POINTER(C.c_void_p),
                                               C.POINTER(C.c_size_t), C.c_int, C.POINTER(C.c_int)]),
    "dkb_batch_set_loci_multi": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(u64p), C.POINTER(u64p), C.POINTER(u64p),
                                           C.POINTER(C.c_size_t)]),
    "dkb_sync": (C.c_int, [C.c_void_p]),
    "dkb_counts_reset": (C.c_int, [C.c_void_p]),
    "dkb_entry_counts_fetch": (C.c_int, [C.c_void_p, u32p]),
    "dkb_entry_counts_device": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p),
                                          C.POINTER(C.c_size_t)]),
    "dkb_finalise": (C.c_int, [C.c_void_p, C.POINTER(Thresholds)]),
    "dkb_finalise_from": (C.c_int, [C.c_void_p, C.POINTER(Thresholds), C.c_void_p]),
    "dkb_results_fetch": (C.c_int, [C.c_void_p, u32p, u32p, u32p, u8p]),
    "dkb_table_set_locus_classes": (C.c_int, [C.c_void_p, u8p, C.c_uint32]),
    "dkb_ctx_set_child_sexes": (C.c_int, [C.c_void_p, u8p, C.c_int]),
    "dkb_host_alloc": (C.c_int, [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]),
    "dkb_host_free": (C.c_int, [C.c_void_p, C.c_void_p]),
    "dkb_thread_bind_near_gpu": (C.c_int, [C.c_void_p, C.POINTER(C.c_int)]),
    "dkb_comm_unique_id": (C.c_int, [C.c_void_p]),
    "dkb_comm_init": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int]),
    "dkb_comm_destroy": (C.c_int, [C.c_void_p]),
    "dkb_comm_info": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int),
                                C.POINTER(C.c_int)]),
    "dkb_counts_allreduce": (C.c_int, [C.c_void_p]),
    "dkb_reduce_push": (C.c_int, [C.c_void_p, C.POINTER(Thresholds)]),
    "dkb_reduce_flush": (C.c_int, [C.c_void_p, C.POINTER(Thresholds)]),
    "dkb_reduced_counts_fetch": (C.c_int, [C.c_void_p, u32p]),
    "dkb_stats_get": (C.c_int, [C.c_void_p, C.POINTER(Stats)]),
    "dkb_profile_counters": (C.c_int, [C.c_void_p, C.c_int]),
    "dkb_scan_stream": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
}

_lib = None


def lib():
    """Load libdkb.so; raise ImportError if it has not been built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise ImportError(
                f"{SO_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(denovo_kmer_b200 has no CPU or PyTorch fallback)")
        L = C.CDLL(SO_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)  # AttributeError if the ABI lost a symbol
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


class DkbError(RuntimeError):
    def __init__(self, code, detail):
        self.code = code
        super().__init__(f"dkb error {code} ({lib().dkb_strerror(code).decode()}): {detail}")


def check(code, ctx=None):
    if code != OK:
        raise DkbError(code, (lib().dkb_last_error(ctx) or b"").decode())
