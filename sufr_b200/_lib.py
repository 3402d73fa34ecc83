"""ctypes binding of libsufr_b200.so (the C ABI declared in include/sufr_b200.h).

There is no Python or CPU implementation behind this module: if the shared library has not been
built (``python -c 'import __graft_entry__ as g; g.build()'`` or ``make -C sufr_b200/csrc``) the
import of the library raises, and every compute call needs a CUDA device.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

PKG_DIR = Path(__file__).resolve().parent
LIB_PATH = PKG_DIR / "libsufr_b200.so"

MEM_HOST = 0
MEM_DEVICE = 1

OK = 0
ERR_ARGUMENT = 1
ERR_OUT_OF_MEMORY = 2
ERR_INTERNAL = 3
ERR_IO = 4
ERR_UNSUPPORTED = 5
ERR_CUDA = 100


class Args(C.Structure):
    """struct SufrB200Args"""
    _fields_ = [
        ("text", C.c_void_p),
        ("text_len", C.c_uint64),
        ("path", C.c_char_p),
        ("low_memory", C.c_uint8),
        ("has_max_query_len", C.c_uint8),
        ("is_dna", C.c_uint8),
        ("allow_ambiguity", C.c_uint8),
        ("ignore_softmask", C.c_uint8),
        ("reserved", C.c_uint8 * 3),
        ("max_query_len", C.c_uint64),
        ("sequence_starts", C.c_void_p),
        ("sequence_names", C.POINTER(C.c_char_p)),
        ("num_sequences", C.c_uint64),
        ("num_partitions", C.c_uint64),
        ("seed_mask", C.c_char_p),
        ("random_seed", C.c_uint64),
        ("rank", C.c_int32),
        ("world_size", C.c_int32),
    ]


class Timings(C.Structure):
    """struct SufrB200Timings"""
    _fields_ = [(k, C.c_double) for k in
                ("h2d_ms", "encode_ms", "keys_ms", "sort_ms", "refine_ms", "lcp_ms", "finish_ms", "d2h_ms", "total_ms",
                 "dominant_kernel_ms")] + [("dominant_kernel_launches", C.c_uint64), ("dominant_kernel_bytes", C.c_uint64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class Result(C.Structure):
    """struct SufrB200Result"""
    _fields_ = [
        ("index_bits", C.c_uint32),
        ("memory", C.c_uint32),
        ("text_len", C.c_uint64),
        ("num_suffixes", C.c_uint64),
        ("total_suffixes", C.c_uint64),
        ("shard_offset", C.c_uint64),
        ("first_suffix", C.c_uint64),
        ("last_suffix", C.c_uint64),
        ("text", C.c_void_p),
        ("sa", C.c_void_p),
        ("lcp", C.c_void_p),
        ("n_ranges", C.POINTER(C.c_uint64)),
        ("num_n_ranges", C.c_uint64),
        ("timings", Timings),
        ("kernel_launches", C.c_uint64),
        ("peak_device_bytes", C.c_uint64),
        ("alphabet_size", C.c_uint32),
        ("bits_per_symbol", C.c_uint32),
        ("refine_rounds", C.c_uint32),
        ("doubling_rounds", C.c_uint32),
        ("h2d_bytes", C.c_uint64),
        ("d2h_bytes", C.c_uint64),
        ("position_bits", C.c_uint32),
        ("reserved2", C.c_uint32),
        ("owner", C.c_void_p),
    ]


class VerifyReport(C.Structure):
    """struct SufrB200VerifyReport"""
    _fields_ = [(k, C.c_uint64) for k in
                ("pairs_checked", "order_errors", "lcp_errors", "out_of_range", "not_indexed", "duplicates",
                 "first_bad_rank", "max_lcp", "lcp_sum", "expected_suffixes", "deferred_pairs")] + \
               [("method", C.c_uint32), ("reserved", C.c_uint32), ("ms", C.c_double)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class Sequences(C.Structure):
    """struct SufrB200Sequences"""
    _fields_ = [
        ("seq", C.c_void_p),
        ("seq_len", C.c_uint64),
        ("start_positions", C.POINTER(C.c_uint64)),
        ("sequence_names", C.POINTER(C.c_char_p)),
        ("num_sequences", C.c_uint64),
    ]


class FileInfo(C.Structure):
    """struct SufrB200FileInfo"""
    _fields_ = [
        ("version", C.c_uint32),
        ("index_bits", C.c_uint32),
        ("is_dna", C.c_uint8),
        ("allow_ambiguity", C.c_uint8),
        ("ignore_softmask", C.c_uint8),
        ("reserved", C.c_uint8 * 5),
        ("text_len", C.c_uint64),
        ("num_suffixes", C.c_uint64),
        ("max_query_len", C.c_uint64),
        ("num_sequences", C.c_uint64),
        ("text_pos", C.c_uint64),
        ("sa_pos", C.c_uint64),
        ("lcp_pos", C.c_uint64),
        ("file_bytes", C.c_uint64),
        ("seed_mask", C.c_char_p),
        ("sequence_starts", C.POINTER(C.c_uint64)),
        ("sequence_names", C.POINTER(C.c_char_p)),
    ]


# every symbol include/sufr_b200.h declares (tests check that the library exports all of them)
ABI_SYMBOLS = [
    "sufr_b200_ctx_create", "sufr_b200_ctx_destroy", "sufr_b200_ctx_reserve", "sufr_b200_ctx_trim",
    "sufr_b200_build", "sufr_b200_result_free", "sufr_b200_patch_seam", "sufr_b200_verify", "sufr_b200_write",
    "sufr_b200_create", "sufr_b200_create_multi",
    "sufr_b200_index_create", "sufr_b200_index_subsample", "sufr_b200_index_search", "sufr_b200_index_suffixes",
    "sufr_b200_index_free", "sufr_b200_file_info", "sufr_b200_file_info_free", "sufr_b200_index_open",
    "sufr_b200_index_locate", "sufr_b200_index_hits", "sufr_b200_index_extract", "sufr_b200_index_list",
    "sufr_b200_index_string_at", "sufr_b200_index_matching_stats", "sufr_b200_index_mems",
    "sufr_b200_index_kmer_spectrum", "sufr_b200_index_kmers", "sufr_b200_index_kmer_multiplicity",
    "sufr_b200_index_approx", "sufr_b200_index_approx_matches", "sufr_b200_index_approx_levels",
    "sufr_b200_seed_mask", "sufr_b200_find_lcp_full_offset", "sufr_b200_read_sequence_file",
    "sufr_b200_sequences_free", "sufr_b200_synth_dna", "sufr_b200_last_error", "sufr_b200_abi_version",
    "sufr_b200_device_count",
]

_lib = None


class LibraryMissing(ImportError):
    pass


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise LibraryMissing(
            f"{LIB_PATH} is not built. Run `make -C sufr_b200/csrc` (or __graft_entry__.build()). "
            "sufr_b200 has no CPU fallback.")
    L = C.CDLL(str(LIB_PATH))
    L.sufr_b200_abi_version.restype = C.c_int
    L.sufr_b200_device_count.restype = C.c_int
    L.sufr_b200_last_error.restype = C.c_char_p
    L.sufr_b200_ctx_create.restype = C.c_int
    L.sufr_b200_ctx_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
    L.sufr_b200_ctx_destroy.restype = None
    L.sufr_b200_ctx_destroy.argtypes = [C.c_void_p]
    L.sufr_b200_ctx_reserve.restype = C.c_int
    L.sufr_b200_ctx_reserve.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32]
    L.sufr_b200_ctx_trim.restype = None
    L.sufr_b200_ctx_trim.argtypes = [C.c_void_p]
    L.sufr_b200_build.restype = C.c_int
    L.sufr_b200_build.argtypes = [C.c_void_p, C.POINTER(Args), C.c_uint32, C.c_int, C.c_int, C.POINTER(Result)]
    L.sufr_b200_result_free.restype = None
    L.sufr_b200_result_free.argtypes = [C.c_void_p, C.POINTER(Result)]
    L.sufr_b200_patch_seam.restype = C.c_int
    L.sufr_b200_patch_seam.argtypes = [C.c_void_p, C.POINTER(Args), C.POINTER(Result), C.c_uint64]
    L.sufr_b200_verify.restype = C.c_int
    L.sufr_b200_verify.argtypes = [C.c_void_p, C.POINTER(Args), C.POINTER(Result), C.c_int, C.c_uint64,
                                   C.POINTER(VerifyReport)]
    L.sufr_b200_write.restype = C.c_int
    L.sufr_b200_write.argtypes = [C.POINTER(Args), C.POINTER(Result)]
    L.sufr_b200_create.restype = C.c_int
    L.sufr_b200_create.argtypes = [C.POINTER(Args), C.c_int, C.POINTER(Result)]
    L.sufr_b200_create_multi.restype = C.c_int
    L.sufr_b200_create_multi.argtypes = [C.POINTER(Args), C.POINTER(C.c_int), C.c_int, C.c_uint32, C.POINTER(Result)]
    L.sufr_b200_index_create.restype = C.c_int
    L.sufr_b200_index_create.argtypes = [C.c_void_p, C.POINTER(Args), C.POINTER(Result), C.POINTER(C.c_void_p)]
    L.sufr_b200_index_subsample.restype = C.c_int
    L.sufr_b200_index_subsample.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
    L.sufr_b200_index_search.restype = C.c_int
    L.sufr_b200_index_search.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_uint64, C.c_int,
                                         C.c_void_p, C.c_void_p]
    L.sufr_b200_index_suffixes.restype = C.c_int
    L.sufr_b200_index_suffixes.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p]
    L.sufr_b200_index_free.restype = None
    L.sufr_b200_index_free.argtypes = [C.c_void_p]
    L.sufr_b200_file_info.restype = C.c_int
    L.sufr_b200_file_info.argtypes = [C.c_char_p, C.POINTER(FileInfo)]
    L.sufr_b200_file_info_free.restype = None
    L.sufr_b200_file_info_free.argtypes = [C.POINTER(FileInfo)]
    L.sufr_b200_index_open.restype = C.c_int
    L.sufr_b200_index_open.argtypes = [C.c_void_p, C.c_char_p, C.POINTER(C.c_void_p)]
    L.sufr_b200_index_locate.restype = C.c_int
    L.sufr_b200_index_locate.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_uint64, C.c_int,
                                         C.c_void_p, C.c_void_p, C.c_void_p]
    L.sufr_b200_index_hits.restype = C.c_int
    L.sufr_b200_index_hits.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]
    L.sufr_b200_index_extract.restype = C.c_int
    L.sufr_b200_index_extract.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64,
                                          C.POINTER(C.c_uint64), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_void_p]
    L.sufr_b200_index_list.restype = C.c_int
    L.sufr_b200_index_list.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64,
                                       C.POINTER(C.c_uint64), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.sufr_b200_index_string_at.restype = C.c_int
    L.sufr_b200_index_string_at.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p, C.POINTER(C.c_uint64)]
    L.sufr_b200_index_matching_stats.restype = C.c_int
    L.sufr_b200_index_matching_stats.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p,
                                                 C.c_void_p, C.c_void_p]
    L.sufr_b200_index_mems.restype = C.c_int
    L.sufr_b200_index_mems.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64,
                                       C.POINTER(C.c_uint64), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p]
    L.sufr_b200_index_kmer_spectrum.restype = C.c_int
    L.sufr_b200_index_kmer_spectrum.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p, C.POINTER(C.c_uint64),
                                                C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    L.sufr_b200_index_kmers.restype = C.c_int
    L.sufr_b200_index_kmers.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64,
                                        C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_void_p]
    L.sufr_b200_index_kmer_multiplicity.restype = C.c_int
    L.sufr_b200_index_kmer_multiplicity.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p]
    L.sufr_b200_index_approx.restype = C.c_int
    L.sufr_b200_index_approx.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p,
                                         C.POINTER(C.c_uint64)]
    L.sufr_b200_index_approx_matches.restype = C.c_int
    L.sufr_b200_index_approx_matches.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p,
                                                 C.c_void_p]
    L.sufr_b200_index_approx_levels.restype = C.c_int
    L.sufr_b200_index_approx_levels.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64), C.c_void_p, C.c_void_p]
    L.sufr_b200_seed_mask.restype = C.c_int64
    L.sufr_b200_seed_mask.argtypes = [C.c_char_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.sufr_b200_find_lcp_full_offset.restype = C.c_uint64
    L.sufr_b200_find_lcp_full_offset.argtypes = [C.c_uint64, C.c_char_p]
    L.sufr_b200_read_sequence_file.restype = C.c_int
    L.sufr_b200_read_sequence_file.argtypes = [C.c_char_p, C.c_uint8, C.POINTER(Sequences)]
    L.sufr_b200_sequences_free.restype = None
    L.sufr_b200_sequences_free.argtypes = [C.POINTER(Sequences)]
    L.sufr_b200_synth_dna.restype = C.c_int
    L.sufr_b200_synth_dna.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p, C.c_uint64, C.c_uint8]
    if L.sufr_b200_abi_version() != 2:
        raise LibraryMissing("libsufr_b200.so has an unexpected ABI version")
    _lib = L
    return L
