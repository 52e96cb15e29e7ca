"""ctypes binding of libcobweb_b200.so (include/cobweb_b200.h).

There is no CPU fallback: if the library is missing or CUDA is unavailable, every compute
entry point raises.  Loading the library (symbol checks) works without a GPU.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(HERE, "libcobweb_b200.so")

CW_E_ARG, CW_E_CAPACITY, CW_E_CUDA, CW_E_FANOUT = -1, -2, -3, -4
CW_USE_INFO, CW_USE_KL, CW_ACUITY_CUTOFF, CW_GREEDY = 1, 2, 4, 8
(HDR_ROOT, HDR_N_USED, HDR_FREE_TOP, HDR_POOL_USED, HDR_STATUS, HDR_DONE, HDR_MAX_CHILD, HDR_N_SCORES, _h8, HDR_N_ROWS,
 _h10, HDR_N_LEVELS, _h12) = range(13)
HDR_WORDS = 16
SCRATCH_WORDS = 16384
TILE_N, TILE_K, MAX_K, MAX_D, MAX_CHILDREN = 128, 16, 128, 4096, 2048
IFIT_NODE_SLACK, IFIT_POOL_SLACK = 160, 16384
H_TILE, H_F1, H_F2 = 256, 1, 2
FUSED_MAX_K, FUSED_FB_ROUNDS, SMALL_Q, SID_UNRESOLVED, FUSED_STATS, FUSED_STAGES = 30, 2, 32, -2, 12, 7
PAIR_MAX_M, PAIR_MAX_LEN = 1024, 1024

EXPORTS = ["cw_version", "cw_last_error", "cw_store_init", "cw_store_derive", "cw_ifit", "cw_set_ifit_cluster", "cw_selftest_arith", "cw_categorize_ctas", "cw_categorize",
           "cw_index_build", "cw_xt_floats", "cw_score_ldq", "cw_dense_node_scores", "cw_topk_chunks", "cw_dense_paths_topk",
           "cw_predict_dense_host", "cw_index_rows_build",
           "cw_h_b_bytes", "cw_h_a_bytes", "cw_h_stages", "cw_h_set_build", "cw_h_rows_isotropic", "cw_fused_flag_words", "cw_fused_predict",
           "cw_fused_predict_host", "cw_fused_profile", "cw_small_scratch_words", "cw_small_predict", "cw_small_predict_host",
           "cw_rank_scores_bwd", "cw_pair_scratch_words", "cw_pair_scores", "cw_pair_scores_bwd", "cw_whiten", "cw_ffma_peak", "cw_ffma2_peak",
           "cw_leaf_tags", "cw_dense_paths_topk_tagged", "cw_small_predict_tagged", "cw_fused_predict_tagged"]


class CwStore(C.Structure):
    _fields_ = [("D", C.c_int32), ("cap", C.c_int32), ("pool_cap", C.c_int32), ("flags", C.c_int32),
                ("prior_var", C.c_float), ("reserved", C.c_int32),
                ("mean", C.c_void_p), ("m2", C.c_void_p), ("count", C.c_void_p), ("parent", C.c_void_p),
                ("child_off", C.c_void_p), ("child_cnt", C.c_void_p), ("child_cap", C.c_void_p),
                ("child_pool", C.c_void_p), ("n_sent", C.c_void_p), ("free_list", C.c_void_p), ("hdr", C.c_void_p), ("scratch", C.c_void_p),
                ("var", C.c_void_p), ("tf", C.c_void_p)]


class CwIndex(C.Structure):
    _fields_ = [("D", C.c_int32), ("nn", C.c_int32), ("n_ntiles", C.c_int32), ("n_ktiles", C.c_int32),
                ("R", C.c_void_p), ("MB", C.c_void_p), ("sumlog", C.c_void_p),
                ("n_pos", C.c_int32), ("max_len", C.c_int32),
                ("path_idx", C.c_void_p), ("level_w", C.c_void_p), ("pos_rec", C.c_void_p)]


class CwDenseWork(C.Structure):
    _fields_ = [("Q_dev", C.c_void_p), ("xt_scratch", C.c_void_p), ("node_scores", C.c_void_p), ("ldq", C.c_int64),
                ("out_sid_dev", C.c_void_p), ("out_score_dev", C.c_void_p), ("scratch", C.c_void_p)]


class CwHSet(C.Structure):
    _fields_ = [("n_rows", C.c_int32), ("n_ntiles", C.c_int32), ("n_stages", C.c_int32), ("nprod", C.c_int32),
                ("layout", C.c_int32), ("reserved", C.c_int32), ("B", C.c_void_p), ("rc", C.c_void_p)]


class CwFusedIndex(C.Structure):
    _fields_ = [("ix", CwIndex), ("n_int", C.c_int32), ("n_leaf", C.c_int32), ("n_sample_tiles", C.c_int32),
                ("n_levels", C.c_int32), ("internal", CwHSet), ("leaves", CwHSet),
                ("int_parent", C.c_void_p), ("int_w", C.c_void_p), ("level_off", C.c_void_p), ("leaf_row_b", C.c_void_p),
                ("leaf_pos", C.c_void_p), ("sent_off", C.c_void_p), ("sent_ids", C.c_void_p), ("rows", C.c_void_p),
                ("e1max", C.c_float), ("hmax", C.c_float), ("lmax", C.c_float), ("wfac", C.c_float), ("eps_scale", C.c_float),
                ("prior_var", C.c_float)]


class CwFusedWork(C.Structure):
    _fields_ = [("cap_q", C.c_int64), ("ldq", C.c_int64), ("Q_dev", C.c_void_p), ("A_int", C.c_void_p), ("A_leaf", C.c_void_p),
                ("qv", C.c_void_p), ("S", C.c_void_p), ("slots", C.c_void_p), ("tau", C.c_void_p), ("cap", C.c_int32),
                ("fin_ml", C.c_int32), ("cnt", C.c_void_p), ("cand_val", C.c_void_p), ("cand_row", C.c_void_p),
                ("flag", C.c_void_p), ("out_sid_dev", C.c_void_p), ("out_val_dev", C.c_void_p), ("sm_Q", C.c_void_p),
                ("sm_scores", C.c_void_p), ("sm_scratch", C.c_void_p), ("sm_sid", C.c_void_p), ("sm_val", C.c_void_p),
                ("sm_n", C.c_void_p), ("stats", C.c_void_p), ("audit_every", C.c_int32), ("audit_phase", C.c_int32)]


class CwTagFilter(C.Structure):
    _fields_ = [("query_tags", C.c_void_p), ("pos_tags", C.c_void_p), ("leaf_tags", C.c_void_p), ("sent_tags", C.c_void_p)]


class CobwebB200Error(RuntimeError):
    pass


_lib = None


def load():
    """Load the shared library and declare prototypes.  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO):
        raise CobwebB200Error(
            f"{SO} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  There is no CPU fallback.")
    L = C.CDLL(SO)
    vp, i32, i64 = C.c_void_p, C.c_int, C.c_int64
    L.cw_version.restype = C.c_int
    L.cw_last_error.restype = C.c_char_p
    L.cw_store_init.argtypes = [C.POINTER(CwStore), vp]
    L.cw_store_derive.argtypes = [C.POINTER(CwStore), C.c_int32, vp]
    L.cw_ifit.argtypes = [C.POINTER(CwStore), vp, i64, vp, vp, vp, i64, i32, vp]
    L.cw_set_ifit_cluster.argtypes = [i32]
    L.cw_selftest_arith.argtypes = [i64, i64, C.c_uint32, vp, vp]
    L.cw_categorize_ctas.restype = C.c_int
    L.cw_categorize.argtypes = [C.POINTER(CwStore), vp, i64, i32, i64, i32, i32, i32, vp, i64, vp, vp, vp, vp, vp]
    L.cw_index_build.argtypes = [C.POINTER(CwStore), vp, C.c_int32, C.POINTER(CwIndex), vp]
    L.cw_xt_floats.restype = i64
    L.cw_xt_floats.argtypes = [i64, C.c_int32]
    L.cw_score_ldq.restype = i64
    L.cw_score_ldq.argtypes = [i64]
    L.cw_dense_node_scores.argtypes = [C.POINTER(CwIndex), vp, i64, vp, vp, i64, vp]
    L.cw_topk_chunks.restype = i64
    L.cw_topk_chunks.argtypes = [i64]
    L.cw_dense_paths_topk.argtypes = [C.POINTER(CwIndex), vp, i64, i64, i32, vp, vp, vp, vp, vp]
    L.cw_predict_dense_host.argtypes = [C.POINTER(CwIndex), C.POINTER(CwDenseWork), vp, i64, i32, vp, vp, vp]
    L.cw_index_rows_build.argtypes = [C.POINTER(CwStore), vp, C.c_int32, vp, vp]
    i32c = C.c_int32
    L.cw_h_b_bytes.restype = i64
    L.cw_h_b_bytes.argtypes = [i32c, i32c, i32c, i32c]
    L.cw_h_a_bytes.restype = i64
    L.cw_h_a_bytes.argtypes = [i64, i32c, i32c, i32c]
    L.cw_h_stages.restype = i32c
    L.cw_h_stages.argtypes = [i32c, i32c, i32c]
    L.cw_h_set_build.argtypes = [C.POINTER(CwStore), vp, vp, vp, C.POINTER(CwHSet), vp, vp, vp, vp, vp, vp, vp]
    L.cw_h_rows_isotropic.argtypes = [C.POINTER(CwStore), vp, vp, i32c, vp, vp]
    L.cw_fused_flag_words.restype = i64
    L.cw_fused_flag_words.argtypes = [i64, i32c]
    L.cw_fused_predict.argtypes = [C.POINTER(CwFusedIndex), C.POINTER(CwFusedWork), vp, i64, i32, vp, vp, vp]
    L.cw_fused_predict_host.argtypes = [C.POINTER(CwFusedIndex), C.POINTER(CwFusedWork), vp, i64, i32, vp, vp, vp, vp]
    L.cw_fused_profile.argtypes = [C.POINTER(CwFusedIndex), C.POINTER(CwFusedWork), vp, i64, i32, vp, vp, vp, vp]
    L.cw_small_scratch_words.restype = i64
    L.cw_small_scratch_words.argtypes = [i64, i32]
    L.cw_small_predict.argtypes = [C.POINTER(CwIndex), vp, i64, vp, vp, i32c, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    L.cw_small_predict_host.argtypes = [C.POINTER(CwIndex), vp, i64, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    L.cw_rank_scores_bwd.argtypes = [C.POINTER(CwIndex), vp, i64, vp, vp, i64, vp, vp]
    L.cw_pair_scratch_words.restype = i64
    L.cw_pair_scratch_words.argtypes = [i64, i32c, i32c]
    L.cw_pair_scores.argtypes = [C.POINTER(CwIndex), vp, vp, i32c, vp, i64, vp, i32c, vp, vp, vp]
    L.cw_pair_scores_bwd.argtypes = [C.POINTER(CwIndex), vp, vp, i32c, vp, i64, vp, i32c, vp, vp, vp, vp]
    L.cw_leaf_tags.argtypes = [vp, vp, i32c, vp, vp, vp]
    tfp = C.POINTER(CwTagFilter)
    L.cw_dense_paths_topk_tagged.argtypes = [C.POINTER(CwIndex), tfp, vp, i64, i64, i32, vp, vp, vp, vp]
    L.cw_small_predict_tagged.argtypes = [C.POINTER(CwIndex), tfp, vp, i64, vp, vp, i32c, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp,
                                          vp]
    L.cw_fused_predict_tagged.argtypes = [C.POINTER(CwFusedIndex), C.POINTER(CwFusedWork), tfp, vp, i64, i32, vp, vp, vp]
    L.cw_whiten.argtypes = [vp, i64, C.c_int32, vp, vp, C.c_int32, vp, vp, vp, vp, vp]
    L.cw_ffma_peak.argtypes = [i32, i32, i32, vp, vp]
    L.cw_ffma2_peak.argtypes = [i32, i32, i32, vp, vp]
    for name in EXPORTS:
        getattr(L, name)  # AttributeError here = header and library out of sync
    _lib = L
    return L


def check(rc, what=""):
    if rc == 0:
        return
    msg = load().cw_last_error().decode(errors="replace")
    raise CobwebB200Error(f"{what or 'libcobweb_b200'} failed with code {rc}: {msg}")


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise CobwebB200Error("cobweb-b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    load()


def stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)
