"""ctypes binding of libtfrecomm.so (include/tfrecomm.h).  No torch types cross this boundary: only raw
device pointers (tensor.data_ptr()), sizes and a cudaStream_t handle.

There is NO fallback: if the shared library is missing or a call fails, TfrError is raised.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(HERE, os.environ.get("TFR_SO_NAME", "libtfrecomm.so"))  # TFR_SO_NAME: A/B builds

ABS_ITEM, LOSS_SIGMOID_CE, REG_BIAS, OPT_SGD = 1, 2, 4, 8
README_FLAGS = 0
FORK_FLAGS = ABS_ITEM | LOSS_SIGMOID_CE | REG_BIAS | OPT_SGD
VAR_MU, VAR_UB, VAR_UF, VAR_IB, VAR_IF, VAR_ALL = 1, 2, 4, 8, 16, 31
MAX_PARTIALS = 1024
FM_PRESORTED = 256   # host-side flag of tfr_fm_train_step

vp = C.c_void_p
i64 = C.c_int64
i32 = C.c_int32
f32 = C.c_float


class TfrError(RuntimeError):
    pass


class OptScalars(C.Structure):
    """Mirror of tfr_opt_scalars (device-resident)."""
    _fields_ = [("lr", f32), ("reg", f32), ("beta1", f32), ("beta2", f32), ("eps", f32),
                ("beta1_power", f32), ("beta2_power", f32), ("lr_t", f32),
                ("one_minus_beta1", f32), ("one_minus_beta2", f32),
                ("flags", i32), ("var_mask", i32),
                ("global_step", i64), ("batch_cursor", i64), ("prefetch_cursor", i64), ("se_sum", C.c_double),
                ("g_mu", f32), ("ticket", C.c_uint32), ("se_ring", vp), ("se_ring_len", i64),
                ("chunk_ctr", C.c_uint32 * 4), ("timeline", vp), ("lr_t_prev", f32)]


class SvdTables(C.Structure):
    """Mirror of tfr_svd_tables (host struct of device pointers, passed by pointer)."""
    _fields_ = [("user_num", i32), ("item_num", i32), ("dim", i32), ("feat_stride", i32),
                ("mu", vp), ("user_bias", vp), ("item_bias", vp), ("user_feat", vp), ("item_feat", vp),
                ("m_mu", vp), ("v_mu", vp), ("m_ub", vp), ("v_ub", vp), ("m_ib", vp), ("v_ib", vp),
                ("m_uf", vp), ("v_uf", vp), ("m_if", vp), ("v_if", vp),
                ("user_slot", vp), ("item_slot", vp),
                ("g_user_feat", vp), ("g_item_feat", vp), ("g_user_bias", vp), ("g_item_bias", vp), ("g_stride", i64)]


class StepWs(C.Structure):
    """Mirror of tfr_svd_step_ws."""
    _fields_ = [("err", vp), ("partials", vp), ("se_partials", vp),
                ("su_ids", vp), ("su_pos", vp), ("si_ids", vp), ("si_pos", vp),
                ("gsum_uf", vp), ("gsum_if", vp), ("gsum_ub", vp), ("gsum_ib", vp),
                ("cont_uf", vp), ("cont_if", vp), ("tail_uf", vp), ("tail_if", vp),
                ("cont_ub", vp), ("cont_ib", vp), ("tail_ub", vp), ("tail_ib", vp),
                ("kind_u", vp), ("kind_i", vp), ("fix_list_u", vp), ("fix_list_i", vp), ("fix_count", vp),
                ("sort_ws", vp), ("sort_ws_bytes", i64), ("tile", i32), ("n_tiles", i32)]


class FeedSet(C.Structure):
    """Mirror of tfr_feed_set."""
    _fields_ = [("h_feed", vp), ("d_feed", vp), ("d_out", vp), ("h_out", vp), ("workspace", vp), ("workspace_bytes", i64),
                ("ev_h2d", vp), ("ev_sorted", vp), ("ev_pred", vp), ("ev_d2h", vp), ("ev_done", vp),
                ("used", i32), ("copied", i32), ("sorted", i32), ("staged", i32),
                ("d_sync", vp), ("h_flag", vp), ("deliver_seq", C.c_uint32), ("reserved", C.c_uint32)]


class FmTables(C.Structure):
    """Mirror of tfr_fm_tables."""
    _fields_ = [("n_feat", i32), ("dim", i32), ("w0", vp), ("W", vp), ("V", vp), ("m_w0", vp), ("v_w0", vp),
                ("m_W", vp), ("v_W", vp), ("m_V", vp), ("v_V", vp), ("slot", vp)]


class AdamTable(C.Structure):
    """Mirror of tfr_adam_table."""
    _fields_ = [("var", vp), ("m", vp), ("v", vp), ("rows", i64), ("width", i32), ("slot", vp), ("gsum", vp),
                ("stride", i64)]


class SliceUpdate(C.Structure):
    """Mirror of tfr_slice_update."""
    _fields_ = [("var", vp), ("m", vp), ("v", vp), ("bvar", vp), ("bm", vp), ("bv", vp), ("sorted_ids", vp),
                ("gsum", vp), ("bgsum", vp), ("stride", i64)]


# name -> (restype, argtypes).  Every symbol include/tfrecomm.h declares is listed here; the CPU test
# suite checks that the library exports all of them.
_PROTOS = {
    "tfr_last_error": (C.c_char_p, []),
    "tfr_abi_version": (C.c_int, []),
    "tfr_device_sm_count": (C.c_int, []),
    "tfr_tune_set": (C.c_int, [C.c_char_p, i32]),
    "tfr_tune_get": (C.c_int, [C.c_char_p, C.POINTER(i32)]),
    "tfr_opt_init": (C.c_int, [vp, f32, f32, f32, f32, f32, i32, i32, vp]),
    "tfr_opt_set_se_ring": (C.c_int, [vp, vp, i64, vp]),
    "tfr_opt_set_timeline": (C.c_int, [vp, vp, vp]),
    "tfr_svd_forward": (C.c_int, [C.POINTER(SvdTables), vp, vp, i64, i32, vp, vp, vp]),
    "tfr_svd_batch_assemble": (C.c_int, [C.POINTER(SvdTables), vp, vp, vp, vp, vp, i64, i64, vp, vp, vp, vp]),
    "tfr_dedup_workspace_bytes": (i64, [i64]),
    "tfr_dedup_sort_pairs": (C.c_int, [vp, i64, vp, vp, vp, i64, vp, vp, i64, vp, i64, vp]),
    "tfr_dedup_sort_pairs_tl": (C.c_int, [vp, i64, vp, vp, vp, i64, vp, vp, i64, vp, i64, vp, vp]),
    "tfr_unique_first_occurrence": (C.c_int, [vp, vp, i64, vp, vp, vp, vp, vp]),
    "tfr_svd_step_workspace_bytes": (i64, [i64, i32]),
    "tfr_svd_train_step": (C.c_int, [C.POINTER(SvdTables), vp, vp, vp, vp, i64, vp, vp, i32, i32, vp, i64, vp,
                                     C.POINTER(vp), i32, C.POINTER(vp)]),
    "tfr_svd_feed_prefetch": (C.c_int, [C.POINTER(SvdTables), vp, C.POINTER(FeedSet), vp, i32, i64, vp, i32, i64, vp, i32, i64,
                                        i64, vp]),
    "tfr_svd_feed_stage": (C.c_int, [C.POINTER(SvdTables), C.POINTER(FeedSet), vp, i32, i64, vp, i32, i64, vp, i32, i64, i64]),
    "tfr_svd_feed_graph_create": (C.c_int, [C.POINTER(SvdTables), vp, C.POINTER(FeedSet), C.POINTER(FeedSet), i64, i32, i32, i32,
                                            i32, vp, vp, C.POINTER(vp)]),
    "tfr_svd_feed_graph_launch": (C.c_int, [vp, C.POINTER(FeedSet), C.POINTER(FeedSet), i32, vp]),
    "tfr_svd_feed_sort": (C.c_int, [C.POINTER(SvdTables), vp, C.POINTER(FeedSet), i64, vp, vp]),
    "tfr_svd_feed_step": (C.c_int, [C.POINTER(SvdTables), vp, C.POINTER(FeedSet), i64, i32, i32, i32, vp, vp,
                                    C.POINTER(FeedSet), vp]),
    "tfr_event_synchronize": (C.c_int, [vp]),
    "tfr_host_wait_flag": (C.c_int, [vp, C.c_uint32, i64]),
    "tfr_binary_metrics_workspace_bytes": (i64, [i64]),
    "tfr_binary_metrics": (C.c_int, [vp, vp, i64, vp, i64, vp, vp]),
    "tfr_ktm_workspace_bytes": (i64, [i64]),
    "tfr_ktm_csr_indptr": (C.c_int, [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i64, C.POINTER(i32), C.POINTER(i32), i32,
                                     vp, vp, i64, vp]),
    "tfr_ktm_csr_fill": (C.c_int, [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i64, C.POINTER(i32), C.POINTER(i32), i32,
                                   vp, vp, vp, vp]),
    "tfr_event_create": (C.c_int, [C.POINTER(vp)]),
    "tfr_event_destroy": (C.c_int, [vp]),
    "tfr_svd_prefetch_batch": (C.c_int, [C.POINTER(SvdTables), vp, vp, vp, vp, vp, i64, i64, vp, vp, vp, vp, i64, vp]),
    "tfr_svd_train_step_presorted": (C.c_int, [C.POINTER(SvdTables), vp, vp, vp, vp, i64, vp, vp, i32, i32, i32, vp, i64,
                                               vp]),
    "tfr_svd_pair_bring": (C.c_int, [C.POINTER(SvdTables), vp, i64, i32, i32, vp, i64, vp, i64, vp]),
    "tfr_svd_pair_pass": (C.c_int, [C.POINTER(SvdTables), vp, i64, i32, i32, vp, i64, vp, i64, vp]),
    "tfr_svd_step_carve": (C.c_int, [vp, i64, i64, i32, C.POINTER(StepWs)]),
    "tfr_svd_fwd_err": (C.c_int, [C.POINTER(SvdTables), vp, vp, vp, vp, i64, vp, vp, C.POINTER(StepWs), vp]),
    "tfr_svd_fwd_segment_grads": (C.c_int, [C.POINTER(SvdTables), vp, vp, vp, vp, i64, vp, vp, i32, C.POINTER(StepWs), vp]),
    "tfr_svd_fused_n_partials": (C.c_int, [i32, i64]),
    "tfr_svd_begin_step": (C.c_int, [vp, vp]),
    "tfr_svd_segment_grads": (C.c_int, [C.POINTER(SvdTables), vp, vp, vp, i64, C.POINTER(StepWs), vp]),
    "tfr_adam_stream_multi": (C.c_int, [C.POINTER(AdamTable), i32, vp, i32, vp]),
    "tfr_adam_touched": (C.c_int, [vp, vp, vp, i32, vp, i64, vp, vp, vp]),
    "tfr_adam_slice_multi": (C.c_int, [C.POINTER(SliceUpdate), i32, i32, i64, vp, i32, i32, vp]),
    "tfr_sgd_apply": (C.c_int, [vp, i32, vp, i64, vp, vp]),
    "tfr_svd_finish_step": (C.c_int, [C.POINTER(SvdTables), vp, vp, vp, i64, C.POINTER(StepWs), i32, vp]),
    "tfr_shard_gather_rows": (C.c_int, [vp, vp, i64, i32, i64, vp, i64, i32, i32, vp, vp, vp, vp]),
    "tfr_shard_bucket_workspace_bytes": (i64, [i64]),
    "tfr_shard_bucket": (C.c_int, [vp, vp, i64, i32, vp, vp, vp, vp, vp, i64, vp]),
    "tfr_shard_gather_records": (C.c_int, [C.POINTER(SvdTables), vp, C.POINTER(i32), C.POINTER(i32), i32, vp, vp]),
    "tfr_shard_fwd_records": (C.c_int, [C.POINTER(SvdTables), vp, vp, vp, vp, vp, i64, vp, vp, vp, vp, vp, vp, vp]),
    "tfr_shard_owner_prepare": (C.c_int, [vp, vp, C.POINTER(i32), C.POINTER(i32), i32, i32, i64, i64, vp, vp, vp, vp, vp, vp, vp]),
    "tfr_shard_excl_workspace_bytes": (i64, [i64]),
    "tfr_shard_excl_indptr": (C.c_int, [vp, vp, i64, vp, i64, i32, i32, vp, vp, i64, vp]),
    "tfr_shard_excl_fill": (C.c_int, [vp, vp, i64, vp, i64, i32, i32, vp, vp, vp]),
    "tfr_shard_topk_merge": (C.c_int, [vp, vp, i32, i64, i32, vp, vp, vp]),
    "tfr_svd_train_step_gathered": (C.c_int, [C.POINTER(SvdTables), vp, vp, vp, i64, i32, i32, vp, vp, vp, i64, vp]),
    "tfr_fm_forward": (C.c_int, [i64, vp, vp, vp, vp, vp, vp, i32, vp, vp, vp]),
    "tfr_fm_segment_grads": (C.c_int, [vp, vp, vp, i32, i32, vp, vp, vp, vp, vp, i64, C.POINTER(StepWs), vp]),
    "tfr_fm_train_step": (C.c_int, [C.POINTER(FmTables), vp, i64, vp, vp, vp, vp, i64, vp, vp, vp, vp, i32, vp, i64, vp]),
    "tfr_allpairs_workspace_bytes": (i64, [i64, i64, i32, i32]),
    "tfr_allpairs": (C.c_int, [vp, vp, vp, vp, vp, i64, i64, i32, i64, i64, i32, vp, vp, vp, vp, i64, vp]),
    "tfr_allpairs_topk_workspace_bytes": (i64, [i64, i64, i32, i32]),
    "tfr_allpairs_consume": (C.c_int, [vp, vp, vp, vp, vp, i64, i64, i32, i64, i64, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp,
                                       i64, vp]),
    "tfr_allpairs_rank_excluding": (C.c_int, [vp, vp, vp, vp, vp, i64, i64, i32, i64, i64, i32, i32, vp, vp, vp, vp, vp, vp,
                                              i64, vp]),
    "tfr_rank_users_workspace_bytes": (i64, [i64, i64, i32]),
    "tfr_rank_users": (C.c_int, [vp, vp, vp, vp, vp, i64, i64, i32, i64, i64, i32, vp, i64, i32, vp, vp, vp, vp, vp, i64, vp]),
    "tfr_similar_rows_workspace_bytes": (i64, [i64, i64, i32]),
    "tfr_similar_rows": (C.c_int, [vp, i64, i64, vp, vp, i64, vp, i64, i64, i32, i32, i32, vp, vp, vp, i64, vp]),
    "tfr_fold_in_users": (C.c_int, [vp, vp, vp, i64, i32, i64, i32, f32, vp, vp, vp, i64, vp, vp, vp, vp]),
    "tfr_als_chunk": (i32, []),
    "tfr_als_workspace_bytes": (i64, [i64, i32]),
    "tfr_als_half_sweep": (C.c_int, [vp, vp, vp, i64, i32, i64, i32, i32, f32, vp, vp, vp, vp, i64, vp, vp, i64, vp, i64, i32,
                                     vp, i64, vp, vp, vp, i64, vp]),
    "tfr_svd_objective_workspace_bytes": (i64, [i64, i64]),
    "tfr_svd_objective": (C.c_int, [vp, vp, vp, vp, vp, i64, i64, i32, i64, i64, i32, f32, vp, vp, vp, vp, vp, vp, vp, i64,
                                    vp]),
    "tfr_gram_workspace_bytes": (i64, [i64, i32]),
    "tfr_gram_rows": (C.c_int, [vp, i64, i32, i64, vp, vp, i64, vp]),
    "tfr_ials_workspace_bytes": (i64, [i64, i32]),
    "tfr_ials_half_sweep": (C.c_int, [vp, i64, i32, i64, vp, f32, f32, vp, vp, vp, vp, i64, vp, vp, i64, vp, i64, i32, vp, i64,
                                      vp, vp, vp, i64, vp]),
    "tfr_ials_objective_workspace_bytes": (i64, [i64]),
    "tfr_ials_objective": (C.c_int, [vp, vp, i64, i64, i32, i64, i64, vp, vp, f32, f32, vp, vp, vp, vp, vp, i64, vp]),
    "tfr_ranking_metrics_workspace_bytes": (i64, [i64, i32]),
    "tfr_ranking_metrics": (C.c_int, [vp, i64, i32, vp, vp, vp, vp, vp, i64, vp]),
    "tfr_host_pack_feed": (C.c_int, [vp, i32, i64, vp, i32, i64, vp, i32, i64, i64, vp]),
    "tfr_host_pack_feed_checked": (C.c_int, [vp, i32, i64, vp, i32, i64, vp, i32, i64, i64, vp, i64, i64]),
    "tfr_opt_set_cursor": (C.c_int, [vp, i64, vp]),
    "tfr_topk_rows": (C.c_int, [vp, i64, i64, i64, i32, vp, vp, vp]),
    "tfr_graph_begin_capture": (C.c_int, [vp]),
    "tfr_graph_end_capture": (C.c_int, [vp, C.POINTER(vp)]),
    "tfr_graph_launch": (C.c_int, [vp, vp]),
    "tfr_graph_destroy": (C.c_int, [vp]),
}

_lib = None


def load():
    """dlopen the in-tree library; raise loudly if it has not been built (no CPU fallback exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise TfrError(
            "libtfrecomm.so is not built (%s). Run `python __graft_entry__.py build` (nvcc, sm_100a). "
            "There is no CPU fallback for this path." % SO_PATH)
    L = C.CDLL(SO_PATH)
    for name, (res, args) in _PROTOS.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    if L.tfr_abi_version() != 1:
        raise TfrError("libtfrecomm.so ABI version mismatch")
    _lib = L
    return L


def check(rc):
    if rc < 0:
        raise TfrError("libtfrecomm: %s (status %d)" % (load().tfr_last_error().decode(), rc))
    return rc


def tune_set(name, value):
    """Process-wide tuning knob (tfr_tune_set).  Most knobs change launch geometry only and keep results bit for bit;
    SEG_TILE and SEG_MAX_UNITS change the fp32 rounding of the training step (within the oracle's 1e-5 bar); ALS_CHUNK
    changes the float64 summation order of the ALS half-sweep's heavy rows (parity with the exact solution, not bits);
    STREAM_COPY_ONLY, RING_SLOT_MODE=3, AP_STAGES and RANK_STAGES are debug knobs that change results on purpose
    (include/tfrecomm.h lists them all)."""
    check(load().tfr_tune_set(name.encode(), int(value)))


def tune_get(name):
    v = i32()
    check(load().tfr_tune_get(name.encode(), C.byref(v)))
    return v.value


def exported_symbols():
    return sorted(_PROTOS)
