"""ctypes binding of the C ABI declared in include/nafgpu.h.

The product library is nafcodec_b200/csrc/libnafgpu.so (nvcc, sm_100a).  There is NO fallback: if it cannot be
loaded, or no CUDA device exists, every decode raises.  (`Library(path)` with an explicit path exists so the test
tier can point the same binding at the CPU SIMT emulator build of the identical kernel sources.)
"""
import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB_PATH = os.path.join(CSRC, "libnafgpu.so")

OK = 0
ERR_UNEXPECTED_EOF, ERR_INVALID_DATA, ERR_PARSE, ERR_UTF8, ERR_CUDA, ERR_NOMEM, ERR_ARGUMENT, ERR_NO_DEVICE, ERR_UNSUPPORTED = range(-1, -10, -1)
WANT_ID, WANT_COMMENT, WANT_SEQUENCE, WANT_QUALITY, WANT_MASK, WANT_ALL = 1, 2, 4, 8, 16, 31
N_SECTIONS = 6
NO_RECORD = 2 ** 64 - 1
TEXT_AUTO, TEXT_FASTA, TEXT_FASTQ = 0, 1, 2
LINE_LENGTH_FROM_HEADER = 2 ** 64 - 1
SEC_ID, SEC_COMMENT, SEC_LENGTH, SEC_MASK, SEC_SEQUENCE, SEC_QUALITY = range(6)
EXPORT_FLAT, EXPORT_ROWS, EXPORT_OFFSETS = 0, 1, 2


class Header(C.Structure):
    _fields_ = [("format_version", C.c_int32), ("sequence_type", C.c_int32), ("flags", C.c_uint32),
                ("name_separator", C.c_int32), ("line_length", C.c_uint64), ("number_of_sequences", C.c_uint64)]


class Section(C.Structure):
    _fields_ = [("data", C.c_void_p), ("compressed_size", C.c_uint64), ("original_size", C.c_uint64),
                ("present", C.c_int32), ("_pad", C.c_int32)]


class Archive(C.Structure):
    _fields_ = [("header", Header), ("sections", Section * N_SECTIONS)]


class Result(C.Structure):
    _fields_ = [("n_records", C.c_uint64), ("n_ids", C.c_uint64), ("n_comments", C.c_uint64), ("n_lengths", C.c_uint64),
                ("total_residues", C.c_uint64),
                ("ids", C.c_void_p), ("id_offsets", C.c_void_p), ("comments", C.c_void_p), ("comment_offsets", C.c_void_p),
                ("lengths", C.c_void_p), ("record_offsets", C.c_void_p), ("sequence", C.c_void_p), ("quality", C.c_void_p),
                ("first_bad_record", C.c_uint64), ("record_status", C.c_int32), ("status", C.c_int32)]


class Text(C.Structure):
    _fields_ = [("data", C.c_void_p), ("size", C.c_uint64), ("format", C.c_int32), ("status", C.c_int32),
                ("first_bad_record", C.c_uint64)]


class PackInput(C.Structure):
    _fields_ = [("sequence", C.c_void_p), ("lengths", C.c_void_p), ("n_records", C.c_uint64), ("n_residues", C.c_uint64),
                ("sequence_type", C.c_int32), ("extract_mask", C.c_int32)]


class PackResult(C.Structure):
    _fields_ = [("packed", C.c_void_p), ("packed_size", C.c_uint64), ("length_words", C.c_void_p), ("length_size", C.c_uint64),
                ("mask", C.c_void_p), ("mask_size", C.c_uint64), ("n_mask_runs", C.c_uint64), ("first_invalid", C.c_uint64)]


class JobStats(C.Structure):
    _fields_ = [("n_archives", C.c_uint64), ("n_frames", C.c_uint64), ("n_blocks", C.c_uint64), ("n_sequences", C.c_uint64),
                ("compressed_bytes", C.c_uint64), ("section_bytes", C.c_uint64), ("ascii_bytes", C.c_uint64),
                ("quality_bytes", C.c_uint64), ("id_bytes", C.c_uint64), ("comment_bytes", C.c_uint64),
                ("algorithmic_bytes", C.c_uint64), ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64),
                ("kernel_launches", C.c_uint32), ("n_stages", C.c_uint32), ("lz_handover", C.c_uint32),
                ("lz_rounds", C.c_uint32), ("lz_unresolved", C.c_uint32),
                ("text_kernel_ms", C.c_float), ("text_bytes", C.c_uint64), ("lz_pending", C.c_uint32 * 24),
                ("lz_flow", C.c_uint32), ("_pad", C.c_uint32)]


class Counts(C.Structure):
    _fields_ = [("n_records", C.c_uint64), ("n_ids", C.c_uint64), ("n_comments", C.c_uint64), ("n_lengths", C.c_uint64),
                ("total_residues", C.c_uint64), ("id_bytes", C.c_uint64), ("comment_bytes", C.c_uint64),
                ("first_bad_record", C.c_uint64), ("record_status", C.c_int32), ("status", C.c_int32)]


class Export(C.Structure):
    _fields_ = [("field", C.c_int32), ("layout", C.c_int32), ("table", C.c_uint8 * 256), ("pad", C.c_uint8), ("_pad", C.c_uint8 * 7),
                ("out", C.c_void_p), ("out_bytes", C.c_uint64), ("rows", C.c_void_p), ("n_rows", C.c_uint64), ("row_length", C.c_uint64)]


# every symbol include/nafgpu.h declares (tests check the library exports all of them)
SYMBOLS = ["nafgpu_parse_archive", "nafgpu_variable_u64", "nafgpu_strerror", "nafgpu_version", "nafgpu_ctx_create",
           "nafgpu_ctx_destroy", "nafgpu_last_error", "nafgpu_host_alloc", "nafgpu_host_free", "nafgpu_decode",
           "nafgpu_decode_batch", "nafgpu_job_prepare", "nafgpu_job_run", "nafgpu_job_fetch", "nafgpu_job_fetch_window", "nafgpu_job_sync",
           "nafgpu_job_get_stats", "nafgpu_job_time", "nafgpu_job_run_profiled", "nafgpu_stage_name",
           "nafgpu_job_device_result", "nafgpu_zstd_decompress", "nafgpu_job_format", "nafgpu_format_batch", "nafgpu_pack", "nafgpu_pipeline_create", "nafgpu_pipeline_destroy", "nafgpu_pipeline_submit",
           "nafgpu_pipeline_wait", "nafgpu_pipeline_release", "nafgpu_pipeline_last_error", "nafgpu_pipeline_lanes", "nafgpu_pipeline_lane_stats",
           "nafgpu_job_counts", "nafgpu_job_export", "nafgpu_pipeline_submit_device", "nafgpu_pipeline_wait_counts", "nafgpu_pipeline_export"]


class Library:
    """A loaded nafgpu shared library with typed prototypes."""

    def __init__(self, path=LIB_PATH):
        if not os.path.exists(path):
            raise ImportError(
                f"{path} is missing: build it with `make -C {CSRC}` (nvcc, sm_100a). nafcodec_b200 has no CPU fallback.")
        self.path = path
        L = self.dll = C.CDLL(path)
        L.nafgpu_parse_archive.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(Archive)]
        L.nafgpu_variable_u64.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
        L.nafgpu_strerror.restype = C.c_char_p
        L.nafgpu_strerror.argtypes = [C.c_int]
        L.nafgpu_version.restype = C.c_char_p
        L.nafgpu_ctx_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        L.nafgpu_ctx_destroy.argtypes = [C.c_void_p]
        L.nafgpu_ctx_destroy.restype = None
        L.nafgpu_last_error.restype = C.c_char_p
        L.nafgpu_last_error.argtypes = [C.c_void_p]
        L.nafgpu_host_alloc.restype = C.c_void_p
        L.nafgpu_host_alloc.argtypes = [C.c_size_t]
        L.nafgpu_host_free.argtypes = [C.c_void_p]
        L.nafgpu_host_free.restype = None
        L.nafgpu_decode.argtypes = [C.c_void_p, C.POINTER(Archive), C.c_uint32, C.POINTER(Result)]
        L.nafgpu_decode_batch.argtypes = [C.c_void_p, C.POINTER(Archive), C.c_uint32, C.c_uint32, C.POINTER(Result)]
        L.nafgpu_job_prepare.argtypes = [C.c_void_p, C.POINTER(Archive), C.c_uint32, C.c_uint32]
        L.nafgpu_job_run.argtypes = [C.c_void_p]
        L.nafgpu_job_fetch.argtypes = [C.c_void_p, C.POINTER(Result), C.c_uint32]
        L.nafgpu_job_fetch_window.argtypes = [C.c_void_p, C.c_uint32, C.c_uint64, C.c_uint64, C.c_uint64, C.POINTER(Result)]
        L.nafgpu_job_sync.argtypes = [C.c_void_p]
        L.nafgpu_job_get_stats.argtypes = [C.c_void_p, C.POINTER(JobStats)]
        L.nafgpu_job_time.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_float)]
        L.nafgpu_job_run_profiled.argtypes = [C.c_void_p, C.POINTER(C.c_float), C.c_uint32]
        L.nafgpu_stage_name.restype = C.c_char_p
        L.nafgpu_stage_name.argtypes = [C.c_uint32]
        L.nafgpu_zstd_decompress.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p]
        L.nafgpu_job_format.argtypes = [C.c_void_p, C.c_int, C.c_uint64, C.POINTER(Text), C.c_uint32]
        L.nafgpu_format_batch.argtypes = [C.c_void_p, C.POINTER(Archive), C.c_uint32, C.c_uint32, C.c_int, C.c_uint64, C.POINTER(Text)]
        L.nafgpu_pipeline_create.argtypes = [C.c_int, C.c_uint32, C.POINTER(C.c_void_p)]
        L.nafgpu_pipeline_destroy.argtypes = [C.c_void_p]
        L.nafgpu_pipeline_destroy.restype = None
        L.nafgpu_pipeline_submit.argtypes = [C.c_void_p, C.POINTER(Archive), C.c_uint32, C.c_uint32]
        L.nafgpu_pipeline_submit.restype = C.c_int64
        L.nafgpu_pipeline_wait.argtypes = [C.c_void_p, C.c_int64, C.POINTER(Result), C.c_uint32]
        L.nafgpu_pipeline_release.argtypes = [C.c_void_p, C.c_int64]
        L.nafgpu_pipeline_last_error.argtypes = [C.c_void_p]
        L.nafgpu_pipeline_last_error.restype = C.c_char_p
        L.nafgpu_pipeline_lanes.argtypes = [C.c_void_p]
        L.nafgpu_pipeline_lanes.restype = C.c_uint32
        L.nafgpu_pipeline_lane_stats.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(JobStats)]
        L.nafgpu_pack.argtypes = [C.c_void_p, C.POINTER(PackInput), C.POINTER(PackResult)]
        L.nafgpu_job_device_result.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)]
        L.nafgpu_job_counts.argtypes = [C.c_void_p, C.POINTER(Counts), C.c_uint32]
        L.nafgpu_job_export.argtypes = [C.c_void_p, C.POINTER(Export), C.c_void_p]
        L.nafgpu_pipeline_submit_device.argtypes = [C.c_void_p, C.POINTER(Archive), C.c_uint32, C.c_uint32]
        L.nafgpu_pipeline_submit_device.restype = C.c_int64
        L.nafgpu_pipeline_wait_counts.argtypes = [C.c_void_p, C.c_int64, C.POINTER(Counts), C.c_uint32]
        L.nafgpu_pipeline_export.argtypes = [C.c_void_p, C.c_int64, C.POINTER(Export), C.c_void_p]

    def strerror(self, code):
        return self.dll.nafgpu_strerror(code).decode()


_default = None


def build():
    """Compile the CUDA library in-tree (used by __graft_entry__.build)."""
    subprocess.run(["make", "-s", "-j8", "-C", CSRC], check=True)


def default_library() -> Library:
    global _default
    if _default is None:
        _default = Library(LIB_PATH)
    return _default
