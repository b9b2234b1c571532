"""ctypes binding of libckm.so (include/ckm.h).  There is no fallback: if the CUDA library is missing the import
of this module raises, and if no B200 is visible `ckm_init` fails (CKM_ENODEVICE)."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CKM_LIBRARY") or os.path.join(_HERE, "libckm.so")     # CKM_LIBRARY: an experimental build of the same library


class ModelInfo(C.Structure):
    _fields_ = [("name", C.c_char * 128), ("acc", C.c_char * 64), ("desc", C.c_char * 256), ("M", C.c_int32),
                ("has_ga", C.c_int32), ("has_tc", C.c_int32), ("has_nc", C.c_int32),
                ("ga", C.c_float * 2), ("tc", C.c_float * 2), ("nc", C.c_float * 2), ("evparam", C.c_float * 6),
                ("ga_d", C.c_double * 2), ("tc_d", C.c_double * 2), ("nc_d", C.c_double * 2)]


class Hit(C.Structure):
    _fields_ = [("bin", C.c_int32), ("seq", C.c_int32), ("model", C.c_int32), ("tlen", C.c_int32), ("qlen", C.c_int32),
                ("dom", C.c_int32), ("ndom", C.c_int32),
                ("hmm_from", C.c_int32), ("hmm_to", C.c_int32), ("ali_from", C.c_int32), ("ali_to", C.c_int32),
                ("env_from", C.c_int32), ("env_to", C.c_int32),
                ("full_score", C.c_float), ("full_bias", C.c_float), ("dom_score", C.c_float), ("dom_bias", C.c_float),
                ("acc", C.c_float),
                ("full_evalue", C.c_double), ("c_evalue", C.c_double), ("i_evalue", C.c_double),
                ("full_lnP", C.c_double), ("dom_lnP", C.c_double)]


class Stats(C.Structure):
    _fields_ = [("n_pairs", C.c_int64), ("n_cells", C.c_int64), ("n_ssv_cand", C.c_int64), ("n_past_msv", C.c_int64),
                ("n_past_bias", C.c_int64), ("n_past_vit", C.c_int64), ("n_past_fwd", C.c_int64),
                ("n_hits_seq", C.c_int64), ("n_domains", C.c_int64), ("n_reported", C.c_int64),
                ("ms_ssv", C.c_float), ("ms_msv", C.c_float), ("ms_bias", C.c_float), ("ms_vit", C.c_float),
                ("ms_fwd", C.c_float), ("ms_domdef", C.c_float), ("ms_total", C.c_float),
                ("kernel_launches", C.c_int64), ("n_vit_redo", C.c_int64), ("n_msv_exact", C.c_int64),
                ("n_queue_retries", C.c_int64)]


class QaRow(C.Structure):
    _fields_ = [("bin", C.c_int32), ("counts", C.c_int32 * 6), ("n_markers", C.c_int32), ("n_sets", C.c_int32),
                ("unique_hits", C.c_int32), ("multi_hits", C.c_int32),
                ("completeness", C.c_double), ("contamination", C.c_double)]


class MarkerHit(C.Structure):
    _fields_ = [("bin", C.c_int32), ("model", C.c_int32), ("seq_a", C.c_int32), ("seq_b", C.c_int32),
                ("target_length", C.c_int32), ("hmm_from", C.c_int32), ("hmm_to", C.c_int32),
                ("ali_from", C.c_int32), ("ali_to", C.c_int32), ("env_from", C.c_int32), ("env_to", C.c_int32),
                ("order", C.c_int32), ("src_row", C.c_int32), ("dict_key", C.c_int64)]


class ReduceOpts(C.Structure):
    _fields_ = [("ignore_thresholds", C.c_int32), ("skip_pseudogene", C.c_int32), ("skip_adjacent", C.c_int32),
                ("individual_markers", C.c_int32), ("evalue_threshold", C.c_double), ("evalue_exp10", C.c_int32),
                ("pad0", C.c_int32), ("evalue_mant", C.c_double), ("length_threshold", C.c_double),
                ("pseudogene_length", C.c_double)]


class ReduceMeta(C.Structure):
    _fields_ = [("is_pfam", C.c_void_p), ("is_tigr", C.c_void_p), ("clan", C.c_void_p),
                ("nest_off", C.c_void_p), ("nest_idx", C.c_void_p), ("has_cut", C.c_void_p), ("cutoffs", C.c_void_p), ("row_scores", C.c_void_p),
                ("scaffold_id", C.c_void_p), ("orf_num", C.c_void_p), ("name_rank", C.c_void_p),
                ("bin_set_off", C.c_void_p), ("set_marker_off", C.c_void_p), ("set_marker_idx", C.c_void_p)]


# every symbol include/ckm.h declares (tests/test_abi.py checks the .so exports each one)
SYMBOLS = ["ckm_init", "ckm_destroy", "ckm_last_error", "ckm_version", "ckm_device_name",
           "ckm_models_load", "ckm_models_count", "ckm_models_info", "ckm_models_find", "ckm_models_select",
           "ckm_models_write", "ckm_models_free", "ckm_digitize", "ckm_fasta_parse", "ckm_seqdb_create", "ckm_seqdb_free",
           "ckm_search", "ckm_search_per_bin", "ckm_hits_free", "ckm_align", "ckm_last_stats", "ckm_workspace_bytes", "ckm_msv_scores",
           "ckm_filter_scores", "ckm_viterbi_scores", "ckm_write_domtblout", "ckm_reduce", "ckm_genome_check", "ckm_free", "ckm_allgather_qa", "ckm_nccl_unique_id",
           "ckm_nccl_comm_init", "ckm_nccl_comm_destroy", "ckm_fasta_scan_nt", "ckm_scaffold_stats"]

_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError("checkm_b200: %s is missing; run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(there is no CPU fallback)" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp, i32, i64, dbl = C.c_void_p, C.c_int32, C.c_int64, C.c_double
    L.ckm_last_error.restype = C.c_char_p
    L.ckm_version.restype = C.c_char_p
    L.ckm_init.argtypes = [C.c_int, C.POINTER(vp)]
    L.ckm_destroy.argtypes = [vp]
    L.ckm_destroy.restype = None
    L.ckm_device_name.argtypes = [vp, C.c_char_p, C.c_int]
    L.ckm_models_load.argtypes = [vp, C.c_char_p, C.POINTER(vp)]
    L.ckm_models_count.argtypes = [vp]
    L.ckm_models_info.argtypes = [vp, C.c_int, C.POINTER(ModelInfo)]
    L.ckm_models_find.argtypes = [vp, C.c_char_p]
    L.ckm_models_select.argtypes = [vp, C.POINTER(C.c_char_p), C.c_int, vp, C.POINTER(C.c_int)]
    L.ckm_models_write.argtypes = [vp, vp, C.c_int, C.c_char_p]
    L.ckm_models_free.argtypes = [vp]
    L.ckm_models_free.restype = None
    L.ckm_digitize.argtypes = [C.c_char_p, i64, vp]
    L.ckm_fasta_parse.argtypes = [C.c_char_p, i64, vp, vp, i32, vp, i64, C.POINTER(i32), C.POINTER(i64), C.POINTER(i64)]
    L.ckm_fasta_scan_nt.argtypes = [C.c_char_p, i64, vp, i64, vp, vp, i32, vp, i64, C.POINTER(i32), C.POINTER(i64), C.POINTER(i64)]
    L.ckm_scaffold_stats.argtypes = [vp, vp, i64, vp, vp, i32, vp, vp, vp, i64, C.POINTER(i64), C.POINTER(C.c_float)]
    L.ckm_seqdb_create.argtypes = [vp, vp, vp, i32, vp, i32, C.POINTER(vp)]
    L.ckm_seqdb_free.argtypes = [vp]
    L.ckm_seqdb_free.restype = None
    L.ckm_search.argtypes = [vp, vp, vp, i32, vp, dbl, dbl, C.POINTER(C.POINTER(Hit)), C.POINTER(i64)]
    L.ckm_search_per_bin.argtypes = [vp, vp, vp, vp, vp, dbl, dbl, C.POINTER(C.POINTER(Hit)), C.POINTER(i64)]
    L.ckm_align.argtypes = [vp, vp, i32, vp, vp, vp]
    L.ckm_hits_free.argtypes = [C.POINTER(Hit)]
    L.ckm_hits_free.restype = None
    L.ckm_last_stats.argtypes = [vp, C.POINTER(Stats)]
    L.ckm_workspace_bytes.argtypes = [vp, C.POINTER(i64)]
    L.ckm_msv_scores.argtypes = [vp, vp, vp, i32, vp, vp]
    L.ckm_filter_scores.argtypes = [vp, vp, vp, i32, vp, vp, vp, vp, vp]
    L.ckm_viterbi_scores.argtypes = [vp, vp, vp, i32, vp, i32, vp]
    L.ckm_write_domtblout.argtypes = [vp, C.POINTER(Hit), i64, i32, i32, C.POINTER(C.c_char_p), C.POINTER(C.c_char_p),
                                      C.c_char_p]
    L.ckm_reduce.argtypes = [vp, i32, i32, i32, C.POINTER(Hit), i64, C.POINTER(ReduceOpts), C.POINTER(ReduceMeta),
                             C.POINTER(C.POINTER(QaRow)), C.POINTER(i32), C.POINTER(C.POINTER(MarkerHit)),
                             C.POINTER(i64)]
    L.ckm_genome_check.argtypes = [vp, i32, vp, vp, vp, i32, vp]
    L.ckm_free.argtypes = [vp]
    L.ckm_free.restype = None
    L.ckm_allgather_qa.argtypes = [vp, vp, vp, i32, i32, i32, vp, vp]
    L.ckm_nccl_unique_id.argtypes = [vp, i32]
    L.ckm_nccl_comm_init.argtypes = [vp, i32, i32, vp, C.POINTER(vp)]
    L.ckm_nccl_comm_destroy.argtypes = [vp]
    L.ckm_nccl_comm_destroy.restype = None
    _lib = L
    return L


class CkmError(RuntimeError):
    def __init__(self, code, msg):
        RuntimeError.__init__(self, "libckm error %d: %s" % (code, msg))
        self.code = code


def check(rc):
    if rc != 0:
        raise CkmError(rc, lib().ckm_last_error().decode(errors="replace"))
