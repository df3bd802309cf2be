"""ctypes declarations for libdnagpu.so (include/dnagpu.h).

The library is the product; this module only describes its C ABI to Python.
Loading fails loudly when the shared object is missing: there is no Python or
CPU implementation of any operation to fall back to.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# DNAGPU_LIB names another build of the same library, e.g. to compare two builds on the same inputs
LIB_PATH = os.environ.get("DNAGPU_LIB") or os.path.join(os.path.dirname(_HERE), "libdnagpu.so")

u64 = C.c_uint64
u64p = C.POINTER(C.c_uint64)
vp = C.c_void_p


class Where(C.Structure):
    """dnagpu_where: WHERE kmer ^@ prefix AND qkmer @> kmer."""
    _fields_ = [("prefix_bits", C.c_uint64), ("prefix_len", C.c_int32),
                ("flags", C.c_int32), ("qkmer", C.c_char_p)]


class Stats(C.Structure):
    _fields_ = [("total", C.c_uint64), ("distinct", C.c_uint64), ("unique", C.c_uint64)]


class ShufflePlan(C.Structure):
    _fields_ = [("bits1", C.c_int32), ("bits2", C.c_int32), ("n_parts", C.c_uint32), ("n_digits", C.c_uint32)]


class CountOpts(C.Structure):
    _fields_ = [("method", C.c_int32), ("flags", C.c_int32),
                ("load_factor", C.c_double), ("expected_keys", C.c_uint64),
                ("owner_parts", C.c_uint32), ("owner_part", C.c_uint32)]


# name -> (restype, argtypes); every symbol include/dnagpu.h declares
SIGNATURES = {
    "dnagpu_version": (C.c_int, []),
    "dnagpu_strerror": (C.c_char_p, [C.c_int]),
    "dnagpu_create": (C.c_int, [C.POINTER(vp), C.c_int]),
    "dnagpu_create_multi": (C.c_int, [C.POINTER(vp), C.POINTER(C.c_int), C.c_int]),
    "dnagpu_device_count": (C.c_int, [vp]),
    "dnagpu_destroy": (None, [vp]),
    "dnagpu_last_error": (C.c_char_p, [vp]),
    "dnagpu_set_stream": (C.c_int, [vp, vp]),
    "dnagpu_synchronize": (C.c_int, [vp]),
    "dnagpu_device_info": (C.c_int, [vp, C.c_char_p, C.c_size_t, C.POINTER(C.c_int), u64p, u64p]),
    "dnagpu_host_alloc": (C.c_int, [vp, C.POINTER(vp), u64]),
    "dnagpu_host_free": (None, [vp, vp]),
    "dnagpu_seq_upload": (C.c_int, [vp, vp, u64, C.POINTER(vp)]),
    "dnagpu_seq_upload_reads": (C.c_int, [vp, vp, u64, C.c_uint32, C.c_uint32, C.POINTER(vp)]),
    "dnagpu_seq_upload_ragged": (C.c_int, [vp, vp, vp, vp, u64, C.POINTER(vp)]),
    "dnagpu_seq_synth": (C.c_int, [vp, u64, u64, C.c_uint32, C.POINTER(vp)]),
    "dnagpu_seq_synth_range": (C.c_int, [vp, u64, u64, C.c_uint32, u64, u64, C.c_int, C.POINTER(vp)]),
    "dnagpu_seq_synth_reads": (C.c_int, [vp, u64, u64, C.c_uint32, C.c_uint32, u64, C.c_uint32, C.POINTER(vp)]),
    "dnagpu_seq_wrap": (C.c_int, [vp, vp, u64, u64, C.POINTER(vp)]),
    "dnagpu_seq_wrap_reads": (C.c_int, [vp, vp, u64, C.c_uint32, C.c_uint32, u64, C.POINTER(vp)]),
    "dnagpu_seq_wrap_pieces": (C.c_int, [vp, C.POINTER(vp), u64p, u64p, C.c_uint32, u64, C.POINTER(vp)]),
    "dnagpu_seq_set_start_limit": (C.c_int, [vp, u64]),
    "dnagpu_seq_download": (C.c_int, [vp, vp, vp, u64]),
    "dnagpu_seq_words": (u64, [vp]),
    "dnagpu_seq_device_words": (vp, [vp]),
    "dnagpu_seq_kmer_count": (u64, [vp, C.c_int]),
    "dnagpu_seq_free": (None, [vp]),
    "dnagpu_encode_dna": (C.c_int, [vp, C.c_char_p, u64, vp]),
    "dnagpu_seq_from_text": (C.c_int, [vp, C.c_char_p, u64, C.POINTER(vp)]),
    "dnagpu_decode_dna": (C.c_int, [vp, vp, u64, C.c_char_p]),
    "dnagpu_generate_kmers": (C.c_int, [vp, vp, u64, C.c_int, vp, u64, u64p]),
    "dnagpu_extract": (C.c_int, [vp, vp, C.c_int, vp, u64, u64p]),
    "dnagpu_filter_kmers": (C.c_int, [vp, vp, u64, C.c_int, C.POINTER(Where), vp, u64, u64p]),
    "dnagpu_filter": (C.c_int, [vp, vp, C.c_int, C.POINTER(Where), vp, u64, u64p]),
    "dnagpu_collect": (C.c_int, [vp, vp, C.c_int, C.POINTER(Where), vp, u64, u64p]),
    "dnagpu_filter_keys": (C.c_int, [vp, vp, u64, C.c_int, C.POINTER(Where), vp, u64, u64p]),
    "dnagpu_count_kmers": (C.c_int, [vp, vp, u64, C.c_int, C.POINTER(Where), C.POINTER(Stats), C.POINTER(vp)]),
    "dnagpu_count_reads": (C.c_int, [vp, vp, u64, C.c_uint32, C.c_uint32, C.c_int, C.POINTER(Where),
                                     C.POINTER(Stats), C.POINTER(vp)]),
    "dnagpu_count": (C.c_int, [vp, vp, C.c_int, C.POINTER(Where), C.POINTER(CountOpts),
                               C.POINTER(Stats), C.POINTER(vp)]),
    "dnagpu_count_keys": (C.c_int, [vp, vp, u64, C.c_int, C.POINTER(CountOpts), C.POINTER(Stats),
                                    C.POINTER(vp)]),
    "dnagpu_count_spectrum": (C.c_int, [vp, vp, C.c_int, C.POINTER(Where), C.POINTER(CountOpts), C.c_uint32,
                                        vp, C.POINTER(Stats)]),
    "dnagpu_count_kmers_spectrum": (C.c_int, [vp, vp, u64, C.c_int, C.POINTER(Where), C.c_uint32, vp,
                                              C.POINTER(Stats)]),
    "dnagpu_table_rows": (u64, [vp]),
    "dnagpu_table_k": (C.c_int, [vp]),
    "dnagpu_table_fetch": (C.c_int, [vp, vp, u64, u64, vp, vp]),
    "dnagpu_table_device": (C.c_int, [vp, C.POINTER(vp), C.POINTER(vp)]),
    "dnagpu_table_free": (None, [vp]),
    "dnagpu_owner_of": (C.c_uint32, [u64, C.c_uint32]),
    "dnagpu_partition": (C.c_int, [vp, vp, C.c_int, C.POINTER(Where), C.c_uint32, vp, u64, u64p]),
    "dnagpu_shuffle_plan_make": (C.c_int, [u64, C.c_uint32, C.POINTER(ShufflePlan)]),
    "dnagpu_shuffle_owner": (C.c_uint32, [C.POINTER(ShufflePlan), C.c_uint32]),
    "dnagpu_shuffle_send": (C.c_int, [vp, vp, C.c_int, C.POINTER(Where), C.POINTER(ShufflePlan), vp, u64, u64p,
                                      u64p, u64p]),
    "dnagpu_shuffle_count": (C.c_int, [vp, vp, u64p, C.c_uint32, C.c_uint32, C.POINTER(ShufflePlan), C.c_int,
                                       C.POINTER(Stats), C.POINTER(vp)]),
    "dnagpu_peer_alloc": (C.c_int, [vp, u64, C.POINTER(vp), C.c_char_p]),
    "dnagpu_peer_open": (C.c_int, [vp, C.c_char_p, C.POINTER(vp)]),
    "dnagpu_peer_close": (C.c_int, [vp, vp]),
    "dnagpu_peer_free": (C.c_int, [vp, vp]),
    "dnagpu_shuffle_hist": (C.c_int, [vp, vp, C.c_int, C.POINTER(Where), C.POINTER(ShufflePlan), u64p]),
    "dnagpu_shuffle_scatter_to": (C.c_int, [vp, vp, C.c_int, C.POINTER(Where), C.POINTER(ShufflePlan), u64p, u64p,
                                            u64p]),
    "dnagpu_shuffle_hist_keys": (C.c_int, [vp, vp, u64, C.POINTER(ShufflePlan), u64p]),
    "dnagpu_shuffle_scatter_keys_to": (C.c_int, [vp, vp, u64, C.POINTER(ShufflePlan), u64p, u64p]),
    "dnagpu_index_build": (C.c_int, [vp, vp, u64, C.c_int, C.POINTER(vp)]),
    "dnagpu_index_rows": (u64, [vp]),
    "dnagpu_index_k": (C.c_int, [vp]),
    "dnagpu_index_device": (C.c_int, [vp, C.POINTER(vp), C.POINTER(vp)]),
    "dnagpu_index_equal": (C.c_int, [vp, vp, u64, C.c_int, vp, u64, u64p]),
    "dnagpu_index_search": (C.c_int, [vp, vp, C.POINTER(Where), vp, u64, u64p]),
    "dnagpu_index_free": (None, [vp]),
    "dnagpu_profile_enable": (C.c_int, [vp, C.c_int]),
    "dnagpu_profile_reset": (C.c_int, [vp]),
    "dnagpu_profile_query": (C.c_int, [vp, C.c_char_p, C.POINTER(C.c_double), u64p]),
    "dnagpu_profile_dump": (C.c_int, [vp, C.c_char_p, C.c_size_t]),
}

_lib = None


def load():
    """dlopen libdnagpu.so and attach the prototypes.  Raises if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is not built (run `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C dna-sequences-pg-extension_b200/csrc`); libdnagpu has no CPU fallback")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
