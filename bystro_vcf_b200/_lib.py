"""ctypes binding of libbvcf.so (include/bvcf.h).  No CPU fallback: if the library or a CUDA device is
missing, calls fail loudly."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libbvcf.so")
SYNTH_LIB_PATH = os.path.join(HERE, "lib", "libbvcfsynth.so")


class BvcfError(RuntimeError):
    pass


class CConfig(C.Structure):
    _fields_ = [
        ("empty_field", C.c_char_p),
        ("field_delim", C.c_char_p),
        ("keep_id", C.c_int),
        ("keep_info", C.c_int),
        ("keep_pos", C.c_int),
        ("want_tsv", C.c_int),
        ("want_dosage", C.c_int),
        ("allow", C.POINTER(C.c_char_p)),
        ("n_allow", C.c_int),
        ("exclude", C.POINTER(C.c_char_p)),
        ("n_exclude", C.c_int),
        ("eol_width", C.c_int),
        ("normalize_dots", C.c_int),
        ("n_slots", C.c_int),
        ("max_chunk_bytes", C.c_size_t),
        ("resident_subchunk_bytes", C.c_size_t),
    ]


class CDiag(C.Structure):
    _fields_ = [("line_no", C.c_uint64), ("alt_no", C.c_int32), ("code", C.c_int32), ("line_start", C.c_uint64)]


class CDosageBatch(C.Structure):
    _fields_ = [
        ("n_rows", C.c_uint64),
        ("n_samples", C.c_uint32),
        ("dosage", C.POINTER(C.c_int8)),
        ("loci", C.POINTER(C.c_uint8)),
        ("loci_off", C.POINTER(C.c_uint64)),
    ]


class CChunkStats(C.Structure):
    _fields_ = [
        ("n_lines", C.c_uint64),
        ("n_records", C.c_uint64),
        ("n_rows", C.c_uint64),
        ("in_bytes", C.c_uint64),
        ("out_bytes", C.c_uint64),
        ("retries", C.c_uint32),
    ]


BGZF_BLOCK_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_size_t, C.c_void_p)  # (user, i, bvcf_bgzf_blk *)
BGZF_EMIT_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t, C.c_void_p, C.c_size_t)


class CKernelTimes(C.Structure):
    _fields_ = [
        ("scan_ms", C.c_float),
        ("compact_ms", C.c_float),
        ("stats_ms", C.c_float),
        ("rows_ms", C.c_float),
        ("names_ms", C.c_float),
        ("total_ms", C.c_float),
        ("launches", C.c_uint32),
        ("compose_ms", C.c_float),
        ("copyout_ms", C.c_float),
    ]


# every symbol include/bvcf.h declares
SYMBOLS = [
    "bvcf_create", "bvcf_destroy", "bvcf_header_line", "bvcf_set_header", "bvcf_host_alloc", "bvcf_host_free",
    "bvcf_submit", "bvcf_collect", "bvcf_release", "bvcf_resident_alloc", "bvcf_resident_upload",
    "bvcf_resident_run", "bvcf_resident_download", "bvcf_resident_peek", "bvcf_resident_line_index", "bvcf_strerror",
    "bvcf_last_error", "bvcf_abi_version", "bvcf_launch_count", "bvcf_resident_run_at", "bvcf_resident_inflate_bgzf",
    "bvcf_bgzf_text_bytes", "bvcf_resident_download_bgzf", "bvcf_resident_write_output", "bvcf_resident_results",
    "bvcf_submit_bgzf", "bvcf_diag_fields", "bvcf_resident_download_bgzf_level", "bvcf_set_regions", "bvcf_index_spans",
    "bvcf_bgzf_block", "bvcf_bgzf_blocks", "bvcf_bgzf_inflate", "bvcf_bgzf_plan",
]

_lib = None


def lib():
    """Load libbvcf.so.  Raises BvcfError when it has not been built (python -m bystro_vcf_b200.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise BvcfError(
            f"{LIB_PATH} is missing: build the CUDA library first (python -m bystro_vcf_b200.build). "
            "There is no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, sz, u64 = C.c_void_p, C.c_size_t, C.c_uint64
    L.bvcf_create.restype = C.c_int
    L.bvcf_create.argtypes = [C.POINTER(vp), C.c_int, C.POINTER(CConfig)]
    L.bvcf_destroy.restype = None
    L.bvcf_destroy.argtypes = [vp]
    L.bvcf_header_line.restype = C.c_int
    L.bvcf_header_line.argtypes = [C.POINTER(CConfig), C.c_char_p, sz]
    L.bvcf_set_header.restype = C.c_int
    L.bvcf_set_header.argtypes = [vp, C.c_char_p, sz]
    L.bvcf_host_alloc.restype = C.c_int
    L.bvcf_host_alloc.argtypes = [C.POINTER(vp), sz]
    L.bvcf_host_free.restype = None
    L.bvcf_host_free.argtypes = [vp]
    L.bvcf_submit.restype = C.c_int
    L.bvcf_submit.argtypes = [vp, u64, vp, sz]
    L.bvcf_collect.restype = C.c_int
    L.bvcf_collect.argtypes = [vp, u64, C.POINTER(vp), C.POINTER(sz), C.POINTER(CDosageBatch),
                               C.POINTER(C.POINTER(CDiag)), C.POINTER(sz), C.POINTER(CChunkStats)]
    L.bvcf_release.restype = C.c_int
    L.bvcf_submit_bgzf.restype = C.c_int
    L.bvcf_submit_bgzf.argtypes = [vp, u64, vp, sz, sz, vp, sz]
    L.bvcf_diag_fields.restype = C.c_int
    L.bvcf_diag_fields.argtypes = [vp, u64, C.POINTER(vp), C.POINTER(C.POINTER(u64))]
    L.bvcf_release.argtypes = [vp, u64]
    L.bvcf_resident_alloc.restype = C.c_int
    L.bvcf_resident_alloc.argtypes = [vp, sz, sz, C.POINTER(vp), C.POINTER(vp)]
    L.bvcf_resident_upload.restype = C.c_int
    L.bvcf_resident_upload.argtypes = [vp, sz, vp, sz]
    L.bvcf_resident_run.restype = C.c_int
    L.bvcf_resident_run.argtypes = [vp, sz, C.POINTER(CChunkStats), C.POINTER(CKernelTimes)]
    L.bvcf_resident_run_at.restype = C.c_int
    L.bvcf_resident_run_at.argtypes = [vp, sz, sz, C.POINTER(CChunkStats), C.POINTER(CKernelTimes)]
    L.bvcf_resident_inflate_bgzf.restype = C.c_int
    L.bvcf_resident_inflate_bgzf.argtypes = [vp, vp, sz, sz, C.POINTER(sz)]
    L.bvcf_bgzf_text_bytes.restype = C.c_int
    L.bvcf_bgzf_text_bytes.argtypes = [vp, sz, C.POINTER(u64), C.POINTER(u64)]
    L.bvcf_resident_results.restype = C.c_int
    L.bvcf_resident_results.argtypes = [vp, C.POINTER(CDosageBatch), C.POINTER(C.POINTER(CDiag)), C.POINTER(sz)]
    L.bvcf_resident_write_output.restype = C.c_int
    L.bvcf_resident_write_output.argtypes = [vp, sz, vp, sz]
    L.bvcf_resident_download_bgzf.restype = C.c_int
    L.bvcf_resident_download_bgzf.argtypes = [vp, sz, sz, vp, sz, C.POINTER(sz)]
    L.bvcf_resident_download_bgzf_level.restype = C.c_int
    L.bvcf_resident_download_bgzf_level.argtypes = [vp, sz, sz, C.c_int, vp, sz, C.POINTER(sz)]
    L.bvcf_resident_download.restype = C.c_int
    L.bvcf_resident_download.argtypes = [vp, sz, vp, sz]
    L.bvcf_resident_peek.restype = C.c_int
    L.bvcf_resident_peek.argtypes = [vp, sz, vp, sz]
    L.bvcf_resident_line_index.restype = C.c_int
    L.bvcf_resident_line_index.argtypes = [vp, C.POINTER(u64), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), sz,
                                           C.POINTER(sz)]
    L.bvcf_set_regions.restype = C.c_int
    L.bvcf_set_regions.argtypes = [vp, C.POINTER(C.c_char_p), C.POINTER(C.c_int64), C.POINTER(C.c_int64), sz]
    L.bvcf_index_spans.restype = C.c_int
    L.bvcf_index_spans.argtypes = [vp, sz, C.POINTER(C.c_char_p), C.POINTER(C.c_int64), C.POINTER(C.c_int64), sz,
                                   C.POINTER(u64), sz, C.POINTER(sz)]
    L.bvcf_bgzf_block.restype = C.c_int
    L.bvcf_bgzf_block.argtypes = [vp, sz, C.POINTER(sz), C.POINTER(C.c_uint32), C.POINTER(C.c_char_p)]
    L.bvcf_bgzf_blocks.restype = C.c_int
    L.bvcf_bgzf_blocks.argtypes = [vp, sz, vp, vp, sz, C.POINTER(sz), C.POINTER(C.c_char_p)]
    L.bvcf_bgzf_inflate.restype = C.c_int
    L.bvcf_bgzf_inflate.argtypes = [vp, sz, vp, sz, C.POINTER(C.c_char_p)]
    L.bvcf_bgzf_plan.restype = C.c_int
    L.bvcf_bgzf_plan.argtypes = [BGZF_BLOCK_FN, BGZF_EMIT_FN, vp, u64, sz, sz, C.POINTER(C.c_char_p)]
    L.bvcf_strerror.restype = C.c_char_p
    L.bvcf_strerror.argtypes = [C.c_int]
    L.bvcf_last_error.restype = C.c_char_p
    L.bvcf_last_error.argtypes = [vp]
    L.bvcf_abi_version.restype = C.c_int
    L.bvcf_launch_count.restype = u64
    L.bvcf_launch_count.argtypes = [vp]
    _lib = L
    return L


def check(rc: int, ctx=None, what: str = "") -> None:
    if rc == 0:
        return
    L = lib()
    msg = L.bvcf_strerror(rc).decode()
    if ctx is not None and rc in (-1, -2):
        detail = L.bvcf_last_error(ctx).decode()
        if detail or rc == -2:
            msg += ": " + detail
    raise BvcfError(f"{what or 'libbvcf'} failed ({rc}): {msg}")
