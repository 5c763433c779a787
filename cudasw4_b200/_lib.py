"""ctypes loader for libsw4b200.so (the C ABI of include/sw4b200.h). No fallback: a missing library is an error."""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SW4B200_LIB") or os.path.join(_HERE, "libsw4b200.so")  # override: kernel-variant sweeps only

EXPORTS = [
    "sw4_create", "sw4_destroy", "sw4_last_error", "sw4_set_gap_scores", "sw4_set_num_top", "sw4_set_blosum",
    "sw4_set_kernel_types", "sw4_set_mem_config", "sw4_set_shard", "sw4_set_database_files", "sw4_set_database_memory",
    "sw4_set_database_shard_memory", "sw4_set_pseudo_database", "sw4_set_pseudo_database_lengths", "sw4_upload_database", "sw4_scan", "sw4_scan_many",
    "sw4_last_scan_all_scores", "sw4_reference_header",
    "sw4_reference_length", "sw4_reference_sequence", "sw4_total_timer_start", "sw4_total_timer_stop",
    "sw4_get_db_info", "sw4_version", "sw4_alignment_coordinates",
    "sw4_alignment_traceback", "sw4_last_cigars", "sw4_scan_pssm", "sw4_scan_many_pssm", "sw4_alignment_coordinates_pssm",
    "sw4_alignment_traceback_pssm", "sw4_fit_score_statistics", "sw4_set_score_statistics", "sw4_last_score_statistics",
    "sw4_last_score_histogram", "sw4_build_pssm", "sw4_search_iterative",
]

SCORE_BINS = 4096  # SW4_SCORE_BINS: score bins of the histogram, plus one overflow bin


class MemConfig(ctypes.Structure):
    _fields_ = [("max_batch_bytes", ctypes.c_size_t), ("max_batch_sequences", ctypes.c_size_t),
                ("max_temp_bytes", ctypes.c_size_t), ("max_gpu_mem", ctypes.c_size_t)]


class Stats(ctypes.Structure):
    _fields_ = [("num_overflows", ctypes.c_int32), ("seconds", ctypes.c_double), ("gcups", ctypes.c_double),
                ("kernel_seconds", ctypes.c_double), ("cells", ctypes.c_double), ("kernel_launches", ctypes.c_int32)]


class Alignment(ctypes.Structure):
    _fields_ = [("score", ctypes.c_int32), ("query_begin", ctypes.c_int32), ("query_end", ctypes.c_int32),
                ("reference_begin", ctypes.c_int32), ("reference_end", ctypes.c_int32)]


class AlignmentSummary(ctypes.Structure):
    _fields_ = [("coordinates", Alignment), ("length", ctypes.c_int32), ("identities", ctypes.c_int32),
                ("positives", ctypes.c_int32), ("gaps", ctypes.c_int32), ("cigar_offset", ctypes.c_size_t),
                ("cigar_length", ctypes.c_size_t)]


class ScoreStatistics(ctypes.Structure):
    _fields_ = [("status", ctypes.c_int32), ("whole_database", ctypes.c_int32), ("lambda_", ctypes.c_double),
                ("K", ctypes.c_double), ("query_length", ctypes.c_int64), ("db_residues", ctypes.c_int64),
                ("num_subjects", ctypes.c_int64), ("fitted", ctypes.c_int64), ("left_censored", ctypes.c_int64),
                ("right_censored", ctypes.c_int64), ("c_lo", ctypes.c_int32), ("c_hi", ctypes.c_int32)]


class DbInfo(ctypes.Structure):
    _fields_ = [("num_sequences", ctypes.c_uint64), ("num_residues", ctypes.c_uint64), ("min_length", ctypes.c_int32),
                ("max_length", ctypes.c_int32), ("partition_counts", ctypes.c_uint64 * 36),
                ("shard_rank", ctypes.c_int32), ("shard_world", ctypes.c_int32), ("shard_sequences", ctypes.c_uint64),
                ("shard_residues", ctypes.c_uint64), ("streaming", ctypes.c_int32), ("num_batches", ctypes.c_int32)]


_lib = None


def load() -> ctypes.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: build it with `make lib` (or __graft_entry__.build()); "
                           "cudasw4_b200 has no CPU or PyTorch fallback")
    lib = ctypes.CDLL(LIB_PATH)
    vp, ci, cs = ctypes.c_void_p, ctypes.c_int, ctypes.c_size_t
    lib.sw4_create.argtypes = [vp, ci, ci, ci, ci, ci, ctypes.POINTER(MemConfig), ci, ctypes.POINTER(vp)]
    lib.sw4_destroy.argtypes = [vp]
    lib.sw4_last_error.argtypes = [vp]
    lib.sw4_last_error.restype = ctypes.c_char_p
    lib.sw4_set_gap_scores.argtypes = [vp, ci, ci]
    lib.sw4_set_num_top.argtypes = [vp, ci]
    lib.sw4_set_blosum.argtypes = [vp, ci]
    lib.sw4_set_kernel_types.argtypes = [vp, ci, ci, ci, ci]
    lib.sw4_set_mem_config.argtypes = [vp, ctypes.POINTER(MemConfig)]
    lib.sw4_set_shard.argtypes = [vp, ci, ci]
    lib.sw4_set_database_files.argtypes = [vp, ctypes.c_char_p, ci]
    lib.sw4_set_database_memory.argtypes = [vp, vp, vp, vp, vp, vp, cs]
    lib.sw4_set_database_shard_memory.argtypes = [vp, vp, vp, vp, vp, vp, cs, vp, cs]
    lib.sw4_set_pseudo_database.argtypes = [vp, cs, ci, ci]
    lib.sw4_set_pseudo_database_lengths.argtypes = [vp, vp, cs, ctypes.c_uint64, vp, ctypes.POINTER(vp), ctypes.c_int32]
    lib.sw4_upload_database.argtypes = [vp]
    lib.sw4_scan.argtypes = [vp, ctypes.c_char_p, ctypes.c_int32, vp, vp, ctypes.POINTER(ctypes.c_int32),
                             ctypes.POINTER(Stats)]
    lib.sw4_scan_many.argtypes = [vp, ctypes.POINTER(ctypes.c_char_p), ctypes.POINTER(ctypes.c_int32), ctypes.c_int32, vp, vp, vp,
                                  ctypes.POINTER(Stats), ctypes.POINTER(Stats)]
    lib.sw4_alignment_coordinates.argtypes = [vp, ctypes.c_char_p, ctypes.c_int32, vp, ctypes.c_int32, vp,
                                              ctypes.POINTER(Stats)]
    lib.sw4_alignment_traceback.argtypes = [vp, ctypes.c_char_p, ctypes.c_int32, vp, ctypes.c_int32, vp,
                                            ctypes.POINTER(Stats)]
    lib.sw4_scan_pssm.argtypes = [vp, ctypes.c_char_p, vp, ctypes.c_int32, vp, vp, ctypes.POINTER(ctypes.c_int32),
                                  ctypes.POINTER(Stats)]
    lib.sw4_scan_many_pssm.argtypes = [vp, ctypes.POINTER(ctypes.c_char_p), ctypes.POINTER(vp), ctypes.POINTER(ctypes.c_int32),
                                       ctypes.c_int32, vp, vp, vp, ctypes.POINTER(Stats), ctypes.POINTER(Stats)]
    lib.sw4_alignment_coordinates_pssm.argtypes = [vp, ctypes.c_char_p, vp, ctypes.c_int32, vp, ctypes.c_int32, vp,
                                                   ctypes.POINTER(Stats)]
    lib.sw4_alignment_traceback_pssm.argtypes = [vp, ctypes.c_char_p, vp, ctypes.c_int32, vp, ctypes.c_int32, vp,
                                                 ctypes.POINTER(Stats)]
    lib.sw4_last_cigars.argtypes = [vp, ctypes.POINTER(vp), ctypes.POINTER(cs)]
    lib.sw4_fit_score_statistics.argtypes = [vp, vp, ctypes.c_int32, ctypes.c_int64, ctypes.POINTER(ScoreStatistics)]
    lib.sw4_set_score_statistics.argtypes = [vp, ci, ctypes.c_double]
    lib.sw4_last_score_statistics.argtypes = [vp, ctypes.c_int32, ctypes.POINTER(ScoreStatistics)]
    lib.sw4_last_score_histogram.argtypes = [vp, ctypes.c_int32, vp, vp, ctypes.c_int32]
    lib.sw4_build_pssm.argtypes = [vp, ctypes.c_char_p, vp, ctypes.c_int32, vp, ctypes.c_int32, ctypes.c_double, vp,
                                   ctypes.POINTER(Stats)]
    i32p = ctypes.POINTER(ctypes.c_int32)
    lib.sw4_search_iterative.argtypes = [vp, ctypes.c_char_p, ctypes.c_int32, ctypes.c_int32, ctypes.c_double, ctypes.c_double,
                                         vp, vp, i32p, vp, i32p, i32p, ctypes.POINTER(Stats)]
    lib.sw4_last_scan_all_scores.argtypes = [vp, vp, vp, cs, ctypes.POINTER(cs)]
    lib.sw4_reference_header.argtypes = [vp, ctypes.c_int32, ctypes.POINTER(vp), ctypes.POINTER(cs)]
    lib.sw4_reference_length.argtypes = [vp, ctypes.c_int32, ctypes.POINTER(ctypes.c_int32)]
    lib.sw4_reference_sequence.argtypes = [vp, ctypes.c_int32, ctypes.c_char_p, cs, ctypes.POINTER(cs)]
    lib.sw4_total_timer_start.argtypes = [vp]
    lib.sw4_total_timer_stop.argtypes = [vp, ctypes.POINTER(Stats)]
    lib.sw4_get_db_info.argtypes = [vp, ctypes.POINTER(DbInfo)]
    lib.sw4_version.restype = ctypes.c_char_p
    _lib = lib
    return lib
