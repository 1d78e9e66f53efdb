"""ctypes binding of libbioseqdb_gpu.so (include/bioseqdb_gpu.h). The library is built in-tree by
``bioseqdb_b200/csrc/Makefile``; there is no CPU fallback -- if it is missing or no GPU is present the
calls fail loudly."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libbioseqdb_gpu.so")
CSRC = os.path.join(_HERE, "csrc")

# rows as the parity tests and the oracle binding see them: every mem_alnreg_t / mem_aln_t field side by side.  The library returns
# them as two records per row -- bsq_row (64 bytes, always) and bsq_row_ext (48 bytes, with BSQ_FLAG_ROWS_EXT) -- which
# BwaIndex._collect joins into this dtype (extension fields are zero when they were not requested).
ROW_DTYPE = np.dtype([
    ("rb", "<i8"), ("re", "<i8"), ("pos", "<i8"), ("hash", "<u8"),
    ("qb", "<i4"), ("qe", "<i4"), ("rid", "<i4"), ("score", "<i4"), ("truesc", "<i4"), ("sub", "<i4"),
    ("csub", "<i4"), ("sub_n", "<i4"), ("w", "<i4"), ("seedcov", "<i4"), ("secondary", "<i4"),
    ("seedlen0", "<i4"), ("n_comp", "<i4"), ("frac_rep", "<f4"),
    ("is_rev", "<i4"), ("mapq", "<i4"), ("NM", "<i4"), ("flag", "<i4"),
    ("cigar_off", "<u4"), ("n_cigar", "<u4"), ("ref_id", "<i8"),
])
assert ROW_DTYPE.itemsize == 120
PUB_ROW_DTYPE = np.dtype([   # bsq_row
    ("rb", "<i8"), ("re", "<i8"), ("pos", "<i8"), ("ref_id", "<i8"),
    ("qb", "<i4"), ("qe", "<i4"), ("rid", "<i4"), ("score", "<i4"), ("NM", "<i4"),
    ("cigar_off", "<u4"), ("n_cigar", "<u4"), ("flag", "<u2"), ("mapq", "u1"), ("is_rev", "u1"),
])
assert PUB_ROW_DTYPE.itemsize == 64
EXT_ROW_DTYPE = np.dtype([   # bsq_row_ext
    ("hash", "<u8"), ("truesc", "<i4"), ("sub", "<i4"), ("csub", "<i4"), ("sub_n", "<i4"), ("w", "<i4"), ("seedcov", "<i4"),
    ("secondary", "<i4"), ("seedlen0", "<i4"), ("n_comp", "<i4"), ("frac_rep", "<f4"),
])
assert EXT_ROW_DTYPE.itemsize == 48
FLAG_ROWS_EXT = 1
FLAG_TWO_CHUNKS = 2
HOLE_DTYPE = np.dtype([("offset", "<i8"), ("len", "<i4"), ("amb", "S1"), ("_pad", "V3")])

ARR_PAC, ARR_OCC, ARR_SA, ARR_ANN_OFFSET, ARR_ANN_LEN, ARR_ANN_ID, ARR_COUNT = range(7)


class BsqOpts(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "min_seed_len", "max_occ", "a", "b", "pen_clip3", "pen_clip5", "zdrop", "w", "o_del", "e_del", "o_ins", "e_ins")]


class BsqResult(C.Structure):
    _fields_ = [("n_reads", C.c_uint64), ("row_off", C.POINTER(C.c_uint64)), ("rows", C.c_void_p),
                ("cigar", C.POINTER(C.c_uint32)), ("n_cigar_words", C.c_uint64), ("rows_ext", C.c_void_p)]


class BsqTuples(C.Structure):
    _fields_ = [("n_rows", C.c_uint64), ("off", C.POINTER(C.c_uint64)), ("ref_match", C.POINTER(C.c_int32)), ("bytes", C.POINTER(C.c_uint8)),
                ("n_bytes", C.c_uint64), ("device_ms", C.c_float)]


class BsqNuclseqs(C.Structure):
    _fields_ = [("n", C.c_uint64), ("off", C.POINTER(C.c_uint64)), ("bytes", C.POINTER(C.c_uint8)), ("n_bytes", C.c_uint64), ("device_ms", C.c_float)]


class BsqTiming(C.Structure):
    _fields_ = [("h2d", C.c_float), ("seed", C.c_float), ("chain", C.c_float), ("extend", C.c_float), ("finalize", C.c_float),
                ("d2h", C.c_float), ("total", C.c_float), ("notes", C.c_uint32), ("launches", C.c_uint64), ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64)]


class BsqMeta(C.Structure):
    _fields_ = [("l_pac", C.c_int64), ("seq_len", C.c_uint64), ("primary", C.c_uint64), ("L2", C.c_uint64 * 5), ("n_anns", C.c_uint64),
                ("sa_bytes", C.c_uint32), ("built", C.c_uint32), ("arr_bytes", C.c_uint64 * ARR_COUNT), ("build_ms", C.c_double),
                ("build_launches", C.c_uint64), ("sort_pass_bytes", C.c_uint64), ("sa_interval", C.c_uint32), ("reserved", C.c_uint32)]


class BsqIndexCheck(C.Structure):
    _fields_ = [("rows", C.c_uint64), ("exhaustive", C.c_uint64), ("sa_permutation_ok", C.c_uint64), ("sa_out_of_range", C.c_uint64),
                ("order_checked", C.c_uint64), ("order_bad", C.c_uint64), ("order_undecided", C.c_uint64),
                ("rows_checked", C.c_uint64), ("bwt_bad", C.c_uint64), ("lf_bad", C.c_uint64),
                ("occ_blocks_checked", C.c_uint64), ("occ_bad", C.c_uint64), ("l2_ok", C.c_uint64), ("ms", C.c_double)]


class BsqLoadInfo(C.Structure):
    _fields_ = [("file_bytes", C.c_uint64), ("read_ms", C.c_float), ("checksum_ms", C.c_float), ("sa_ms", C.c_float), ("host_ms", C.c_float),
                ("total_ms", C.c_float), ("lf_steps", C.c_uint64), ("lane_slots", C.c_uint64)]


def build_library(force: bool = False) -> str:
    """Compile libbioseqdb_gpu.so for sm_100a (nvcc cross-compiles without a GPU)."""
    if force:
        subprocess.check_call(["make", "-s", "-C", CSRC, "clean"])
    subprocess.check_call(["make", "-s", "-j8", "-C", CSRC])
    return LIB_PATH


_LIB = None


def lib():
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(LIB_PATH):
        raise RuntimeError("libbioseqdb_gpu.so is not built (run __graft_entry__.build() or make -C bioseqdb_b200/csrc); "
                           "there is no CPU fallback")
    L = C.CDLL(LIB_PATH)
    vp, u64, i64, u32, i32 = C.c_void_p, C.c_uint64, C.c_int64, C.c_uint32, C.c_int32
    L.bsq_last_error.restype = C.c_char_p
    L.bsq_device_count.restype = C.c_int
    L.bsq_opts_init.argtypes = [C.POINTER(BsqOpts)]
    L.bsq_index_new.restype = vp
    L.bsq_index_new.argtypes = [C.POINTER(BsqOpts), C.c_int]
    L.bsq_index_set_opts.argtypes = [vp, C.POINTER(BsqOpts)]
    L.bsq_index_set_flags.argtypes = [vp, u32]
    L.bsq_index_add_ref.argtypes = [vp, i64, vp, u32, vp, u32]
    L.bsq_index_add_ref_datums.argtypes = [vp, u64, vp, vp, vp]
    L.bsq_index_build.argtypes = [vp]
    L.bsq_index_free.argtypes = [vp]
    L.bsq_align_batch.argtypes = [vp, vp, vp, vp, u64, C.POINTER(C.POINTER(BsqResult))]
    L.bsq_align_batch_datums.argtypes = [vp, vp, vp, vp, u64, C.POINTER(C.POINTER(BsqResult))]
    L.bsq_session_lrand48.argtypes = [vp, C.c_int, C.POINTER(C.c_uint64)]
    L.bsq_result_free.argtypes = [C.POINTER(BsqResult)]
    L.bsq_last_timing.argtypes = [vp, C.POINTER(BsqTiming)]
    L.bsq_result_tuples.argtypes = [vp, C.POINTER(BsqResult), vp, vp, u32, C.POINTER(C.POINTER(BsqTuples))]
    L.bsq_tuples_free.argtypes = [C.POINTER(BsqTuples)]
    L.bsq_nuclseq_from_text_batch.argtypes = [C.c_int, vp, vp, u64, C.POINTER(C.POINTER(BsqNuclseqs))]
    L.bsq_nuclseqs_free.argtypes = [C.POINTER(BsqNuclseqs)]
    L.bsq_reads_upload.argtypes = [vp, vp, vp, vp, u64]
    L.bsq_align_resident.argtypes = [vp]
    L.bsq_result_download.argtypes = [vp, C.POINTER(C.POINTER(BsqResult))]
    L.bsq_index_get_meta.argtypes = [vp, C.POINTER(BsqMeta)]
    L.bsq_index_device_bytes.argtypes = [vp, C.POINTER(C.c_uint64)]
    L.bsq_index_device_ptr.argtypes = [vp, C.c_int, C.POINTER(vp)]
    L.bsq_index_download.argtypes = [vp, C.c_int, vp, u64]
    L.bsq_index_alloc_replica.argtypes = [vp, C.POINTER(BsqMeta)]
    L.bsq_index_host_state_size.argtypes = [vp, C.POINTER(C.c_uint64)]
    L.bsq_index_host_state_get.argtypes = [vp, vp, u64]
    L.bsq_index_replica_finish.argtypes = [vp, vp, u64]
    L.bsq_index_prepare.argtypes = [vp, C.POINTER(C.c_float)]
    L.bsq_index_save.argtypes = [vp, C.c_char_p, vp]
    L.bsq_index_load.argtypes = [vp, C.c_char_p, vp, C.POINTER(C.c_float)]
    L.bsq_index_last_load.argtypes = [vp, C.POINTER(BsqLoadInfo)]
    L.bsq_multi_new.restype = vp
    L.bsq_multi_new.argtypes = [vp, vp, C.c_int]
    L.bsq_multi_free.argtypes = [vp]
    L.bsq_multi_devices.argtypes = [vp]
    L.bsq_multi_align_batch.argtypes = [vp, vp, vp, vp, u64, C.POINTER(C.POINTER(BsqResult))]
    L.bsq_multi_align_batch_datums.argtypes = [vp, vp, vp, vp, u64, C.POINTER(C.POINTER(BsqResult))]
    L.bsq_multi_last_timing.argtypes = [vp, C.POINTER(BsqTiming)]
    L.bsq_multi_result_tuples.argtypes = [vp, C.POINTER(BsqResult), vp, vp, u32, C.POINTER(C.POINTER(BsqTuples))]
    L.bsq_index_bwt_plain.argtypes = [vp, vp]
    L.bsq_index_sa_sampled.argtypes = [vp, vp, u64]
    L.bsq_debug_seed.argtypes = [vp, vp, vp, u64, vp, u32, vp]
    L.bsq_debug_sa_lookup.argtypes = [vp, vp, u64, vp]
    L.bsq_debug_ksw_extend.argtypes = [C.POINTER(BsqOpts), C.c_int, u64, vp, vp, vp, vp, vp, vp, vp, vp]
    L.bsq_debug_ksw_extend_thread.argtypes = [C.POINTER(BsqOpts), C.c_int, u64, vp, vp, vp, vp, vp, vp, vp, vp, C.c_int]
    L.bsq_debug_ksw_global.argtypes = [C.POINTER(BsqOpts), C.c_int, u64, vp, vp, vp, vp, vp, vp, vp, u32, vp]
    L.bsq_bench_gather.argtypes = [vp, u64, C.c_int, C.POINTER(C.c_double)]
    L.bsq_bench_dpx.argtypes = [C.c_int, C.c_int, C.POINTER(C.c_double)]
    L.bsq_set_counters.argtypes = [vp, C.c_int]
    L.bsq_get_counters.argtypes = [vp, vp]
    L.bsq_debug_ctl.argtypes = [vp, vp]
    L.bsq_index_verify.argtypes = [vp, C.c_uint64, C.c_uint64, vp]
    _LIB = L
    return L


ABI_SYMBOLS = [
    "bsq_last_error", "bsq_device_count", "bsq_opts_init", "bsq_index_new", "bsq_index_set_opts", "bsq_index_set_flags", "bsq_index_add_ref", "bsq_index_add_ref_datums", "bsq_index_build",
    "bsq_index_free", "bsq_align_batch", "bsq_align_batch_datums", "bsq_session_lrand48", "bsq_result_free", "bsq_last_timing", "bsq_result_tuples", "bsq_tuples_free", "bsq_nuclseq_from_text_batch", "bsq_nuclseqs_free", "bsq_reads_upload", "bsq_align_resident", "bsq_result_download",
    "bsq_index_get_meta", "bsq_index_device_bytes", "bsq_index_device_ptr", "bsq_index_download", "bsq_index_alloc_replica", "bsq_index_host_state_size", "bsq_index_host_state_get", "bsq_index_replica_finish", "bsq_index_prepare", "bsq_index_save", "bsq_index_load", "bsq_index_last_load", "bsq_multi_new", "bsq_multi_free", "bsq_multi_devices", "bsq_multi_align_batch", "bsq_multi_align_batch_datums", "bsq_multi_last_timing", "bsq_multi_result_tuples", "bsq_index_bwt_plain", "bsq_index_sa_sampled",
    "bsq_debug_seed", "bsq_debug_sa_lookup", "bsq_debug_ksw_extend", "bsq_debug_ksw_extend_thread", "bsq_debug_ksw_global", "bsq_bench_gather", "bsq_bench_dpx", "bsq_set_counters", "bsq_get_counters", "bsq_debug_ctl", "bsq_index_verify",
]


class BsqError(RuntimeError):
    pass


def check(rc):
    if rc != 0:
        raise BsqError(lib().bsq_last_error().decode(errors="replace"))


def ptr(a):
    return a.ctypes.data_as(C.c_void_p)
