"""ctypes binding of libnpore_b200.so (include/npore_b200.h).  No CPU fallback: if the CUDA library is
missing, importing this module's `lib()` raises."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("NPORE_B200_LIB") or os.path.join(HERE, "libnpore_b200.so")   # env override: A/B builds

NPORE_OUT_STANDARDIZE = 1
NPORE_OUT_RLE = 2
NPORE_OUT_NO_EXPANDED = 4
ST_BAD_CIGAR = 16


class Batch(C.Structure):
    _fields_ = [("n_items", C.c_int32),
                ("ref_codes", C.c_void_p), ("ref_start", C.c_void_p), ("ref_len", C.c_void_p), ("ref_total", C.c_int64),
                ("seq_codes", C.c_void_p), ("seq_start", C.c_void_p), ("seq_len", C.c_void_p), ("seq_total", C.c_int64),
                ("cigar_rle", C.c_void_p), ("cigar_off", C.c_void_p),
                ("seq_nib", C.c_void_p), ("seq_nib_start", C.c_void_p), ("seq_nib_bytes", C.c_int64)]


class Result(C.Structure):
    _fields_ = [("ops", C.c_void_p), ("ops_capacity", C.c_int64), ("ops_off", C.c_void_p),
                ("rle", C.c_void_p), ("rle_capacity", C.c_int64), ("rle_off", C.c_void_p),
                ("chunk_scores", C.c_void_p), ("score_capacity", C.c_int64), ("score_off", C.c_void_p),
                ("status", C.c_void_p)]


class Stats(C.Structure):
    _fields_ = [("n_items", C.c_int64), ("n_chunks", C.c_int64), ("n_cu", C.c_int64),
                ("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64), ("tb_bytes", C.c_int64),
                ("ms_plan", C.c_float), ("ms_annotate", C.c_float), ("ms_forward", C.c_float),
                ("ms_traceback", C.c_float), ("ms_finish", C.c_float), ("ms_kernels_total", C.c_float),
                ("ms_h2d", C.c_float), ("ms_d2h", C.c_float),
                ("launches", C.c_int32), ("n_sub_batches", C.c_int32), ("fwd_warps_per_sm", C.c_int32), ("sm_count", C.c_int32)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class BaiLists(C.Structure):
    _fields_ = [("chunks", C.c_void_p), ("n_chunks", C.c_int64), ("refs", C.c_void_p), ("n_refs", C.c_int64),
                ("windows", C.c_void_p), ("n_windows", C.c_int64), ("error_bits", C.c_uint64)]


class PileupBatch(C.Structure):
    _fields_ = [("n_ranges", C.c_int32), ("range_start", C.c_void_p), ("range_end", C.c_void_p),
                ("ref_ascii", C.c_void_p), ("ref_off", C.c_void_p),
                ("n_reads", C.c_int32), ("read_pos", C.c_void_p), ("seq_ascii", C.c_void_p), ("qual", C.c_void_p),
                ("seq_off", C.c_void_p), ("cigar_rle", C.c_void_p), ("cigar_off", C.c_void_p),
                ("range_reads", C.c_void_p), ("range_reads_off", C.c_void_p), ("min_base_q", C.c_int32),
                ("seq_nib", C.c_void_p), ("seq_nib_start", C.c_void_p), ("seq_nib_bytes", C.c_int64), ("has_qual", C.c_void_p)]


EXPORTS = ["npore_ctx_create", "npore_ctx_destroy", "npore_set_stream", "npore_count_chunks", "npore_upload", "npore_run", "npore_download",
           "npore_align_batch", "npore_get_np_info", "npore_get_np_info_batch", "npore_confusion_batch", "npore_last_stats", "npore_strerror", "npore_last_error", "npore_version",
           "npore_bgzf_create", "npore_bgzf_destroy", "npore_bgzf_bound", "npore_bgzf_compress", "npore_bgzf_index"]

IO_EXPORTS = ["npore_io_last_error", "npore_bam_open", "npore_bam_advance", "npore_bam_prefetch", "npore_bam_close", "npore_bam_header_text", "npore_bam_n_refs", "npore_bam_ref",
              "npore_bam_n_records", "npore_bam_columns", "npore_bam_gather", "npore_bam_gather_nib", "npore_sam_bound", "npore_sam_format", "npore_sam_format_fd",
              "npore_bam_bound", "npore_bam_format", "npore_bam_format_offsets",
              "npore_bam_restrict", "npore_bam_voffsets", "npore_bam_bytes_read"]

_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is not built (python -c 'import __graft_entry__ as g; g.build()'); "
                               "npore_b200 has no CPU fallback")
        L = C.CDLL(LIB_PATH)
        L.npore_ctx_create.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                       C.c_float, C.c_float, C.c_int, C.c_int]
        L.npore_ctx_destroy.argtypes = [C.c_void_p]
        L.npore_ctx_destroy.restype = None
        L.npore_set_stream.argtypes = [C.c_void_p, C.c_void_p]
        L.npore_count_chunks.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]
        L.npore_count_chunks.restype = C.c_int64
        L.npore_upload.argtypes = [C.c_void_p, C.POINTER(Batch)]
        L.npore_run.argtypes = [C.c_void_p, C.c_uint32]
        L.npore_download.argtypes = [C.c_void_p, C.POINTER(Result)]
        L.npore_align_batch.argtypes = [C.c_void_p, C.POINTER(Batch), C.c_uint32, C.POINTER(Result)]
        L.npore_get_np_info.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]
        L.npore_get_np_info_batch.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
        L.npore_confusion_batch.argtypes = [C.c_void_p, C.POINTER(PileupBatch), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.npore_last_stats.argtypes = [C.c_void_p, C.POINTER(Stats)]
        L.npore_strerror.argtypes = [C.c_int]
        L.npore_strerror.restype = C.c_char_p
        L.npore_last_error.argtypes = [C.c_void_p]
        L.npore_last_error.restype = C.c_char_p
        L.npore_version.restype = C.c_char_p
        L.npore_bgzf_create.argtypes = [C.POINTER(C.c_void_p), C.c_int]
        L.npore_bgzf_destroy.argtypes = [C.c_void_p]
        L.npore_bgzf_destroy.restype = None
        L.npore_bgzf_bound.argtypes = [C.c_int64]
        L.npore_bgzf_bound.restype = C.c_int64
        L.npore_bgzf_compress.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.POINTER(C.c_int64),
                                          C.POINTER(C.c_float)]
        L.npore_bgzf_index.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_uint64, C.POINTER(BaiLists), C.POINTER(C.c_float)]
        # include/npore_bamio.h
        vp = C.c_void_p
        L.npore_io_last_error.restype = C.c_char_p
        L.npore_bam_open.argtypes = [C.c_char_p, C.c_int, C.POINTER(vp)]
        L.npore_bam_advance.argtypes = [vp, C.c_int64]
        L.npore_bam_advance.restype = C.c_int64
        L.npore_bam_close.argtypes = [vp]
        L.npore_bam_close.restype = None
        L.npore_bam_header_text.argtypes = [vp, C.POINTER(C.c_char_p)]
        L.npore_bam_header_text.restype = C.c_int64
        L.npore_bam_n_refs.argtypes = [vp]
        L.npore_bam_n_refs.restype = C.c_int32
        L.npore_bam_ref.argtypes = [vp, C.c_int32, C.POINTER(C.c_char_p), C.POINTER(C.c_int64)]
        L.npore_bam_n_records.argtypes = [vp]
        L.npore_bam_n_records.restype = C.c_int64
        L.npore_bam_columns.argtypes = [vp] * 11
        L.npore_bam_prefetch.argtypes = [vp, C.c_int64]
        L.npore_bam_restrict.argtypes = [vp, C.c_int64, vp, vp]
        L.npore_bam_voffsets.argtypes = [vp, vp]
        L.npore_bam_bytes_read.argtypes = [vp]
        L.npore_bam_bytes_read.restype = C.c_int64
        L.npore_bam_gather.argtypes = [vp, C.c_int64, vp, C.c_int, vp, vp, vp, vp, vp, vp, vp, vp]
        L.npore_bam_gather_nib.argtypes = [vp, C.c_int64, vp, C.c_int, vp, vp, vp]
        L.npore_sam_bound.argtypes = [C.c_int64, vp, vp, vp, C.c_int64]
        L.npore_sam_bound.restype = C.c_int64
        L.npore_sam_format.argtypes = [C.c_int64, C.c_int] + [vp] * 6 + [C.c_int32] + [vp] * 11 + [C.c_int64]
        L.npore_sam_format.restype = C.c_int64
        L.npore_sam_format_fd.argtypes = [C.c_int64, C.c_int] + [vp] * 6 + [C.c_int32] + [vp] * 11 + [C.c_int64, C.c_int, C.c_int64]
        L.npore_sam_format_fd.restype = C.c_int64
        L.npore_bam_bound.argtypes = [C.c_int64, vp, vp, vp]
        L.npore_bam_bound.restype = C.c_int64
        L.npore_bam_format.argtypes = L.npore_sam_format.argtypes
        L.npore_bam_format.restype = C.c_int64
        L.npore_bam_format_offsets.argtypes = L.npore_sam_format.argtypes + [vp]
        L.npore_bam_format_offsets.restype = C.c_int64
        _lib = L
    return _lib
