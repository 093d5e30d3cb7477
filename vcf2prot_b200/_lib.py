"""ctypes binding of libv2p_engine.so (include/v2p_engine.h).  Fails loudly when the library is absent:
there is no CPU implementation behind this package."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("V2P_ENGINE_LIB") or os.path.join(HERE, "libv2p_engine.so")  # env: kernel A/B builds

V2P_OK = 0
ERR_INVALID_ARG, ERR_CUDA, ERR_BAD_ENGINE, ERR_BAD_STREAM, ERR_RES_OOB, ERR_SRC_OOB = 1, 2, 3, 4, 5, 6
ERR_NOT_CONTIGUOUS, ERR_NOT_GPU_ENGINE, ERR_TASKGEN, ERR_VCF_PARSE, ERR_BGZF = 7, 9, 10, 11, 12
ENGINE_ST, ENGINE_MT, ENGINE_GPU = 0, 1, 2
FLAG_FILL_DOT, FLAG_VALIDATE, FLAG_DEVICE_PTRS, FLAG_ASYNC, FLAG_ALIGNED_LAYOUT = 1, 2, 4, 8, 16
REF_NO_TMA = 0x200
GEN_ALIGNED, GEN_FASTA, GEN_SKIP_ABORTS = 1, 2, 4

STATUS_NAMES = {0: "OK", 1: "INVALID_ARG", 2: "CUDA", 3: "BAD_ENGINE", 4: "BAD_STREAM", 5: "RES_OOB", 6: "SRC_OOB",
                7: "NOT_CONTIGUOUS", 9: "NOT_GPU_ENGINE", 10: "TASKGEN",
                11: "VCF_PARSE", 12: "BGZF"}


class Task16(C.Structure):
    _fields_ = [("src_off", C.c_uint32), ("len", C.c_uint32), ("dst_off", C.c_uint32), ("stream", C.c_uint32)]


class Batch(C.Structure):
    _fields_ = [("task_begin", C.c_void_p), ("tasks", C.c_void_p), ("ref", C.c_void_p), ("ref_base", C.c_void_p),
                ("n_ref", C.c_uint64), ("alt", C.c_void_p), ("alt_base", C.c_void_p), ("out", C.c_void_p),
                ("out_base", C.c_void_p), ("n_hap", C.c_uint64), ("n_tasks", C.c_uint64), ("n_alt", C.c_uint64),
                ("n_out", C.c_uint64)]


class Result(C.Structure):
    _fields_ = [("status", C.c_int), ("bad_hap", C.c_uint64), ("bad_task", C.c_uint64), ("kernel_ms", C.c_float), ("copy_ms", C.c_float)]


class Generated(C.Structure):
    _fields_ = [("batch", Batch), ("n_rows", C.c_uint64), ("ann_hap", C.c_void_p), ("ann_tx", C.c_void_p),
                ("ann_start", C.c_void_p), ("ann_end", C.c_void_p), ("n_sites", C.c_uint64), ("gen_ms", C.c_float),
                ("n_skipped", C.c_uint64), ("n_aborted", C.c_uint64)]


# every symbol include/*.h declares: (restype, argtypes)
_P = C.c_void_p
class SiteLists(C.Structure):
    _fields_ = [("n_hap", C.c_uint64), ("n_sites", C.c_uint64), ("site_begin", C.c_void_p), ("sites", C.c_void_p),
                ("decode_ms", C.c_float)]


class GzipResult(C.Structure):
    _fields_ = [("in_bytes", C.c_uint64), ("out_bytes", C.c_uint64), ("n_chunks", C.c_uint64), ("n_stored_chunks", C.c_uint64),
                ("ms", C.c_float)]


class PipelineResult(C.Structure):
    _fields_ = [("n_samples", C.c_uint64), ("n_chunks", C.c_uint64), ("n_sites", C.c_uint64), ("n_tasks", C.c_uint64),
                ("n_records", C.c_uint64), ("image_bytes", C.c_uint64), ("out_bytes", C.c_uint64), ("h2d_bytes", C.c_uint64),
                ("decode_ms", C.c_float), ("gen_ms", C.c_float), ("exec_ms", C.c_float), ("gzip_ms", C.c_float),
                ("wall_s", C.c_double), ("n_skipped", C.c_uint64), ("n_aborted", C.c_uint64), ("gen_wall_s", C.c_double),
                ("exec_wall_s", C.c_double), ("gzip_wall_s", C.c_double), ("wait_wall_s", C.c_double), ("sink_wall_s", C.c_double)]


COHORT_MAX_DEVICES = 16
COHORT_CONCURRENT_SINK = 0x100
COHORT_DEVICE_MASKS = 0x200


class VcfLines(C.Structure):  # include/v2p_vcf.h: v2p_vcf_lines
    _fields_ = [("n_samples", C.c_uint64), ("header_begin", C.c_uint64), ("header_end", C.c_uint64), ("n_lines", C.c_uint64),
                ("line_begin", C.c_void_p), ("cells_begin", C.c_void_p), ("h2d_bytes", C.c_uint64), ("h2d_ms", C.c_float),
                ("index_ms", C.c_float)]


class VcfBgzf(C.Structure):  # v2p_vcf_bgzf
    _fields_ = [("n_blocks", C.c_uint64), ("text_bytes", C.c_uint64), ("text", C.c_void_p), ("head", C.c_void_p),
                ("fixed", C.c_void_p), ("fixed_begin", C.c_void_p), ("inflate_ms", C.c_float), ("fixed_ms", C.c_float)]


class VcfMasks(C.Structure):  # v2p_vcf_masks
    _fields_ = [("masks", C.c_void_p), ("n_records", C.c_uint64), ("n_samples", C.c_uint64), ("words_per_cell", C.c_uint32),
                ("parse_ms", C.c_float)]


class CohortInputs(C.Structure):  # include/v2p_cohort.h: v2p_cohort_inputs
    _fields_ = [("proteome", C.c_void_p), ("n_proteome", C.c_uint64), ("n_tx", C.c_uint64), ("tx_offsets", C.c_void_p),
                ("name_off", C.c_void_p), ("names", C.c_void_p), ("general", C.c_int), ("n_sites", C.c_uint64),
                ("site_tx", C.c_void_p), ("site_pos", C.c_void_p), ("site_cls", C.c_void_p), ("site_rlen", C.c_void_p),
                ("ins_code", C.c_void_p), ("ins_flags", C.c_void_p), ("ins_pos_ref", C.c_void_p), ("ins_pos_res", C.c_void_p),
                ("ins_len", C.c_void_p), ("site_doff", C.c_void_p), ("site_dlen", C.c_void_p), ("pool", C.c_void_p),
                ("n_pool", C.c_uint64)]


class CohortResult(C.Structure):  # v2p_cohort_result
    _fields_ = [("n_devices", C.c_uint32), ("total", PipelineResult), ("per_device", PipelineResult * COHORT_MAX_DEVICES),
                ("first_sample", C.c_uint64 * (COHORT_MAX_DEVICES + 1))]


# int sink(void* user, uint64_t first_sample, uint64_t n_samples, const uint8_t* data, const uint64_t* file_begin)
FILE_SINK = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p, C.POINTER(C.c_uint64))
PIPE_GZIP, PIPE_SKIP_ABORTS, PIPE_ALL_RECORDS = 1, 2, 4

SYMBOLS = {
    "v2p_abi_version": (C.c_int, []),
    "v2p_engine_device": (C.c_int, [_P]),
    "v2p_engine_from_str": (C.c_int, [C.c_char_p, C.POINTER(C.c_int)]),
    "v2p_engine_create": (C.c_int, [C.c_int, C.POINTER(_P)]),
    "v2p_engine_destroy": (None, [_P]),
    "v2p_last_error": (C.c_char_p, [_P]),
    "v2p_host_alloc": (C.c_int, [C.POINTER(_P), C.c_size_t]),
    "v2p_host_free": (C.c_int, [_P]),
    "v2p_execute_soa": (C.c_int, [_P, C.c_size_t, _P, _P, _P, _P, _P, C.c_size_t, _P, C.c_size_t, _P, C.c_size_t,
                                  C.c_uint32, C.POINTER(C.c_uint64)]),
    "v2p_gir_execute": (C.c_int, [_P, C.c_int, C.c_size_t, _P, _P, _P, _P, _P, C.c_size_t, _P, C.c_size_t, _P,
                                  C.c_size_t, C.c_uint32, C.POINTER(C.c_uint64)]),
    "v2p_execute_batch": (C.c_int, [_P, C.POINTER(Batch), C.c_uint32, C.POINTER(Result), C.POINTER(_P)]),
    "v2p_event_wait": (C.c_int, [_P, _P, C.POINTER(Result)]),
    "v2p_kernel_launch_count": (C.c_uint64, [_P]),
    "v2p_engine_set_tuning": (C.c_int, [_P, C.c_int, C.c_int]),
    "v2p_engine_set_stream": (C.c_int, [_P, _P]),
    "v2p_engine_profile_warps": (C.c_int, [_P, C.c_int]),
    "v2p_engine_read_warp_ns": (C.c_int, [_P, _P, C.c_uint64, C.POINTER(C.c_uint64)]),
    "v2p_engine_set_reference": (C.c_int, [_P, _P, C.c_uint64, C.c_uint32]),
    # include/v2p_taskgen.h
    "v2p_catalogue_create": (C.c_int, [C.c_int, C.c_uint64, _P, C.c_uint64, _P, _P, _P, _P, _P, _P, _P, C.c_uint64,
                                       C.POINTER(_P)]),
    "v2p_catalogue_create_ins": (C.c_int, [C.c_int, C.c_uint64, _P, C.c_uint64, _P, _P, _P, _P, _P, _P, _P, _P, _P, C.c_uint64,
                                           C.POINTER(_P)]),
    "v2p_catalogue_destroy": (None, [_P]),
    "v2p_catalogue_set_names": (C.c_int, [_P, _P, _P]),
    "v2p_catalogue_last_error": (C.c_char_p, [_P]),
    "v2p_generate_tasks": (C.c_int, [_P, C.c_uint64, _P, _P, C.c_uint32, C.POINTER(Generated)]),
    "v2p_sites_from_masks": (C.c_int, [_P, C.c_uint64, C.c_uint64, C.c_uint32, _P, _P, _P, C.c_uint32, C.POINTER(SiteLists)]),
    "v2p_generate_tasks_from_lists": (C.c_int, [_P, C.POINTER(SiteLists), C.c_uint32, C.POINTER(Generated)]),
    "v2p_device_read": (C.c_int, [_P, _P, C.c_size_t]),
    "v2p_gzip_create": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "v2p_gzip_destroy": (None, [_P]),
    "v2p_gzip_last_error": (C.c_char_p, [_P]),
    "v2p_gzip_bound": (C.c_uint64, [C.c_uint64, C.c_uint64]),
    "v2p_gzip_files": (C.c_int, [_P, _P, _P, C.c_uint64, _P, C.c_uint64, _P, C.c_uint32, C.POINTER(GzipResult)]),
    # include/v2p_pipeline.h
    "v2p_pipeline_create": (C.c_int, [_P, C.POINTER(_P), C.c_uint32, C.POINTER(_P)]),
    "v2p_pipeline_destroy": (None, [_P]),
    "v2p_pipeline_enable_all_records": (C.c_int, [_P, _P, C.c_uint64, C.c_uint64, _P, _P, _P]),
    "v2p_pipeline_last_error": (C.c_char_p, [_P]),
    "v2p_pipeline_run_lists": (C.c_int, [_P, C.c_uint64, _P, _P, C.c_uint32, C.c_uint32, _P, C.c_uint64, _P, FILE_SINK, _P,
                                         C.POINTER(PipelineResult)]),
    "v2p_dir_writer_create": (C.c_int, [C.c_char_p, C.POINTER(C.c_char_p), C.c_uint64, C.c_int, C.c_uint32, C.POINTER(_P)]),
    "v2p_dir_writer_sink": (C.c_int, [_P, C.c_uint64, C.c_uint64, _P, C.POINTER(C.c_uint64)]),
    "v2p_dir_writer_bytes": (C.c_uint64, [_P]),
    "v2p_dir_writer_files": (C.c_uint64, [_P]),
    "v2p_dir_writer_last_error": (C.c_char_p, [_P]),
    "v2p_dir_writer_destroy": (None, [_P]),
    # include/v2p_cohort.h
    "v2p_cohort_create": (C.c_int, [C.POINTER(C.c_int), C.c_uint32, C.POINTER(CohortInputs), C.c_uint32, C.POINTER(_P)]),
    "v2p_cohort_destroy": (None, [_P]),
    "v2p_cohort_last_error": (C.c_char_p, [_P]),
    "v2p_cohort_run_lists": (C.c_int, [_P, C.c_uint64, _P, _P, C.c_uint32, C.c_uint32, FILE_SINK, _P, C.POINTER(CohortResult)]),
    "v2p_cohort_launch_count": (C.c_uint64, [_P]),
    "v2p_cohort_enable_all_records": (C.c_int, [_P, C.POINTER(CohortInputs)]),
    "v2p_cohort_run_masks": (C.c_int, [_P, C.c_uint64, C.c_uint64, C.c_uint32, _P, _P, _P, C.c_uint32, C.c_uint32, FILE_SINK, _P,
                                       C.POINTER(CohortResult)]),
    "v2p_pipeline_run_masks": (C.c_int, [_P, C.c_uint64, C.c_uint64, C.c_uint32, _P, _P, _P, C.c_uint32, C.c_uint32, C.c_uint32,
                                         _P, C.c_uint64, _P, FILE_SINK, _P, C.POINTER(PipelineResult)]),
    # include/v2p_vcf.h
    "v2p_vcf_create": (C.c_int, [C.c_int, C.POINTER(_P)]),
    "v2p_vcf_destroy": (None, [_P]),
    "v2p_vcf_last_error": (C.c_char_p, [_P]),
    "v2p_vcf_load": (C.c_int, [_P, _P, C.c_uint64, C.c_uint32, C.POINTER(VcfLines)]),
    "v2p_vcf_load_bgzf": (C.c_int, [_P, _P, C.c_uint64, C.c_uint32, C.POINTER(VcfLines), C.POINTER(VcfBgzf)]),
    "v2p_vcf_parse_masks": (C.c_int, [_P, C.c_uint64, _P, C.c_uint32, C.POINTER(VcfMasks)]),
}

_lib = None


def load() -> C.CDLL:
    """dlopen the engine library and type every exported symbol.  Raises if it was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise ImportError(
            "vcf2prot_b200: %s is missing -- run `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C vcf2prot_b200/csrc`).  There is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the header and the library disagree
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
