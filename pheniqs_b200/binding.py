"""binding.py — ctypes view of libpheniqs_b200.so (include/pheniqs_b200.h).

The shared library IS the product: this module only declares its entry points. If the
library has not been built the import fails loudly; there is no Python or CPU fallback
for the classification path.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIBRARY_PATH = os.path.join(HERE, "libpheniqs_b200.so")

PHQ_MAX_SEGMENTS = 8
PHQ_MAX_NUCLEOTIDES = 64
PHQ_ABSENT_QUALITY = 0xFF

PHQ_OK = 0
PHQ_INTERNAL_ERROR = 2
PHQ_CONFIGURATION_ERROR = 3
PHQ_OUT_OF_MEMORY_ERROR = 4
PHQ_SEQUENCE_ERROR = 7
PHQ_OVERFLOW_ERROR = 8

ALGORITHM_NAME = {0: "pamld", 1: "mdd", 2: "naive", 3: "passthrough"}
TOPIC_NAME = {0: "sample", 1: "molecular", 2: "cellular"}


class PheniqsError(RuntimeError):
    """Carries the reference's ErrorCode (error.h:32-44) as .code."""

    def __init__(self, code: int, message: str):
        super().__init__(message)
        self.code = code


class ConfigurationError(PheniqsError):
    pass


class DecoderInfo(C.Structure):
    _fields_ = [
        ("algorithm", C.c_int32), ("topic", C.c_int32), ("index", C.c_int32),
        ("barcode_cardinality", C.c_int32), ("segment_cardinality", C.c_int32), ("nucleotide_cardinality", C.c_int32),
        ("segment_length", C.c_int32 * PHQ_MAX_SEGMENTS),
        ("word_cardinality", C.c_int32), ("quality_word_cardinality", C.c_int32), ("has_tile", C.c_int32),
    ]


class Tile(C.Structure):
    _fields_ = [("bases", C.c_void_p), ("nmask", C.c_void_p), ("quality", C.c_void_p), ("pitch", C.c_int64),
                ("quality_bits", C.c_int32), ("quality_codebook", C.c_uint8 * 16)]


class RawSegment(C.Structure):
    _fields_ = [("sequence", C.c_void_p), ("quality", C.c_void_p), ("offset", C.c_void_p), ("length", C.c_int64)]


class CompactResult(C.Structure):
    _fields_ = [("packed", C.c_uint32), ("error_probability", C.c_float)]


class Result(C.Structure):
    _fields_ = [("index", C.c_int32), ("distance", C.c_int32), ("confidence", C.c_double)]


EXPORTS = (
    "phq_compile_job", "phq_load_job", "phq_free", "phq_last_global_error", "phq_create", "phq_destroy", "phq_last_error",
    "phq_decoder_count", "phq_decoder_describe", "phq_pack", "phq_decode_batch", "phq_decode_batch_compact",
    "phq_decode_batch_device", "phq_decode_batch_device_compact", "phq_decode_batch_raw", "phq_decode_batch_raw_compact",
    "phq_decode_batch_raw_tags", "phq_tag_record_bytes", "phq_decode_batch_bam", "phq_decode_batch_bam_compact", "phq_decode_batch_bam_tags",
    "phq_host_alloc", "phq_host_free", "phq_accumulators", "phq_totals", "phq_accumulator_buffer",
    "phq_reset_accumulators", "phq_reset_accumulators_async", "phq_collect", "phq_comm_unique_id", "phq_comm_create", "phq_comm_destroy", "phq_estimate_priors", "phq_set_priors", "phq_report", "phq_encode_report", "phq_adjust_job",
    "phq_statistics", "phq_kernel_description", "phq_reference_power",
    "phq_last_kernel_milliseconds",
)

_library = None


def library() -> C.CDLL:
    global _library
    if _library is not None:
        return _library
    if not os.path.exists(LIBRARY_PATH):
        raise ImportError(
            "pheniqs_b200: %s is missing. Build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). There is no CPU fallback for the classification path." % LIBRARY_PATH)
    lib = C.CDLL(LIBRARY_PATH)
    P = C.POINTER
    lib.phq_compile_job.argtypes = [C.c_char_p, P(C.c_void_p)]
    lib.phq_load_job.argtypes = [C.c_char_p, P(C.c_void_p)]
    lib.phq_free.argtypes = [C.c_void_p]
    lib.phq_free.restype = None
    lib.phq_last_global_error.restype = C.c_char_p
    lib.phq_create.argtypes = [C.c_char_p, C.c_int, P(C.c_void_p)]
    lib.phq_destroy.argtypes = [C.c_void_p]
    lib.phq_destroy.restype = None
    lib.phq_last_error.argtypes = [C.c_void_p]
    lib.phq_last_error.restype = C.c_char_p
    lib.phq_decoder_count.argtypes = [C.c_void_p]
    lib.phq_decoder_describe.argtypes = [C.c_void_p, C.c_int, P(DecoderInfo)]
    lib.phq_pack.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, P(Tile)]
    lib.phq_decode_batch.argtypes = [C.c_void_p, C.c_int64, P(Tile), C.c_void_p, P(C.c_void_p), C.c_void_p]
    lib.phq_decode_batch_device.argtypes = [C.c_void_p, C.c_int64, P(Tile), C.c_void_p, P(C.c_void_p), C.c_void_p]
    lib.phq_decode_batch_compact.argtypes = [C.c_void_p, C.c_int64, P(Tile), C.c_void_p, P(C.c_void_p)]
    lib.phq_decode_batch_device_compact.argtypes = [C.c_void_p, C.c_int64, P(Tile), C.c_void_p, P(C.c_void_p), C.c_void_p]
    lib.phq_decode_batch_raw.argtypes = [C.c_void_p, C.c_int64, C.c_int32, P(RawSegment), C.c_int32, C.c_void_p, P(C.c_void_p), C.c_void_p]
    lib.phq_decode_batch_raw_compact.argtypes = [C.c_void_p, C.c_int64, C.c_int32, P(RawSegment), C.c_int32, C.c_void_p, P(C.c_void_p)]
    lib.phq_decode_batch_raw_tags.argtypes = [C.c_void_p, C.c_int64, C.c_int32, P(RawSegment), C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, P(C.c_void_p)]
    lib.phq_tag_record_bytes.argtypes = [C.c_void_p, P(C.c_int32)]
    lib.phq_decode_batch_bam.argtypes = [C.c_void_p, C.c_int64, C.c_int32, P(RawSegment), C.c_void_p, P(C.c_void_p), C.c_void_p]
    lib.phq_decode_batch_bam_compact.argtypes = [C.c_void_p, C.c_int64, C.c_int32, P(RawSegment), C.c_void_p, P(C.c_void_p)]
    lib.phq_decode_batch_bam_tags.argtypes = [C.c_void_p, C.c_int64, C.c_int32, P(RawSegment), C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, P(C.c_void_p)]
    lib.phq_host_alloc.argtypes = [P(C.c_void_p), C.c_size_t]
    lib.phq_host_free.argtypes = [C.c_void_p]
    lib.phq_host_free.restype = None
    lib.phq_accumulators.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    lib.phq_totals.argtypes = [C.c_void_p, P(C.c_uint64), P(C.c_uint64)]
    lib.phq_accumulator_buffer.argtypes = [C.c_void_p, P(C.c_void_p), P(C.c_int64), P(C.c_int64)]
    lib.phq_reset_accumulators.argtypes = [C.c_void_p]
    lib.phq_reset_accumulators_async.argtypes = [C.c_void_p, C.c_void_p]
    lib.phq_collect.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    lib.phq_comm_unique_id.argtypes = [C.c_void_p]
    lib.phq_comm_create.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, P(C.c_void_p)]
    lib.phq_comm_destroy.argtypes = [C.c_void_p]
    lib.phq_estimate_priors.argtypes = [C.c_void_p, C.c_int, P(C.c_double), C.c_void_p]
    lib.phq_set_priors.argtypes = [C.c_void_p, C.c_int, C.c_double, C.c_void_p]
    lib.phq_statistics.argtypes = [C.c_void_p, P(C.c_uint64), P(C.c_uint64), P(C.c_uint64)]
    lib.phq_report.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_int, P(C.c_void_p)]
    lib.phq_encode_report.argtypes = [C.c_void_p, P(C.c_void_p), P(C.c_void_p), C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, C.c_int, P(C.c_void_p)]
    lib.phq_adjust_job.argtypes = [C.c_char_p, C.c_char_p, C.c_int, P(C.c_void_p)]
    lib.phq_reference_power.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
    lib.phq_kernel_description.argtypes = [C.c_void_p, C.c_int, C.c_char_p, C.c_size_t]
    lib.phq_last_kernel_milliseconds.argtypes = [C.c_void_p, P(C.c_float)]
    _library = lib
    return lib


def check(status: int, handle=None) -> None:
    if status == PHQ_OK:
        return
    lib = library()
    message = (lib.phq_last_error(handle) if handle else lib.phq_last_global_error()) or b""
    cls = ConfigurationError if status == PHQ_CONFIGURATION_ERROR else PheniqsError
    raise cls(status, message.decode("utf-8", "replace"))
