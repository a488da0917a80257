"""ctypes binding of libmovierec_b200.so (C ABI: include/movierec_b200.h).

The library is built in-tree by `make -C movierecommender-tf-trt_b200/csrc` (or
`__graft_entry__.build()`).  There is no fallback: if the shared object is missing the import of
this module raises, and every call that returns a non-zero status raises `MovierecNativeError`
with the library's message.
"""

import ctypes as C
import os

MR_MAX_LAYERS = 8
MR_MAX_WIDTH = 1024
MR_MAX_NEGS = 1023
MR_MAX_TOPK = 256
MR_MAX_CUTOFFS = 8
# sums of mr_targets_scores / mr_catalogue_targets: [users, mrr] then TGT_PER_CUTOFF metrics per cutoff
TGT_USERS, TGT_MRR, TGT_CUTOFF0, TGT_PER_CUTOFF = 0, 1, 2, 5
TGT_METRICS = ("hr", "precision", "recall", "ndcg", "map")  # MR_TGT_HIT .. MR_TGT_MAP
MR_STEP_OUT_FLOATS = 8
OUT_LOSS_SUM, OUT_HIT_SUM, OUT_DCG_SUM, OUT_L2_PENALTY, OUT_BAD_IDS = 0, 1, 2, 3, 4
TRAIN_USERS_GROUPED = 1  # MR_TRAIN_USERS_GROUPED
TRAIN_NO_DENSE_L2 = 2    # MR_TRAIN_NO_DENSE_L2
OPT_ADAM, OPT_SGD = 0, 1
TABLES_DENSE, TABLES_SPARSE = 0, 1

LIB_NAME = "libmovierec_b200.so"
# MR_LIB_PATH points at another build of the same library (A/B runs of kernel variants); the default is the
# in-tree build next to this file.
LIB_PATH = os.environ.get("MR_LIB_PATH") or os.path.join(os.path.dirname(os.path.abspath(__file__)), LIB_NAME)


class MovierecNativeError(RuntimeError):
    pass


_fp = C.POINTER(C.c_float)


class MrModel(C.Structure):
    _fields_ = [
        ("user_mlp", C.c_void_p), ("item_mlp", C.c_void_p), ("user_gmf", C.c_void_p), ("item_gmf", C.c_void_p),
        ("dense", C.c_void_p),
        ("W", C.c_void_p * MR_MAX_LAYERS), ("b", C.c_void_p * MR_MAX_LAYERS),
        ("w_out", C.c_void_p), ("b_out", C.c_void_p),
        ("dense_count", C.c_int64),
        ("num_users", C.c_int32), ("num_items", C.c_int32),
        ("n_layers", C.c_int32),
        ("L", C.c_int32 * MR_MAX_LAYERS),
        ("mf_dim", C.c_int32),
        ("l2", C.c_float * MR_MAX_LAYERS),
        ("compute_path", C.c_int32), ("item_projection", C.c_int32), ("fused_train", C.c_int32),
    ]


class MrOptState(C.Structure):
    _fields_ = [
        ("optimizer", C.c_int32), ("table_mode", C.c_int32),
        ("lr", C.c_float), ("beta_1", C.c_float), ("beta_2", C.c_float), ("epsilon", C.c_float),
        ("iterations", C.c_int64),
        ("m_user_mlp", C.c_void_p), ("m_item_mlp", C.c_void_p), ("m_user_gmf", C.c_void_p),
        ("m_item_gmf", C.c_void_p), ("m_dense", C.c_void_p),
        ("v_user_mlp", C.c_void_p), ("v_item_mlp", C.c_void_p), ("v_user_gmf", C.c_void_p),
        ("v_item_gmf", C.c_void_p), ("v_dense", C.c_void_p),
    ]


class MrGrads(C.Structure):
    _fields_ = [("dense", C.c_void_p), ("user_mlp", C.c_void_p), ("item_mlp", C.c_void_p),
                ("user_gmf", C.c_void_p), ("item_gmf", C.c_void_p), ("user_tables_ready", C.c_void_p),
                ("user_gmf_ready", C.c_void_p)]


class MrFoldIn(C.Structure):
    _fields_ = [("steps", C.c_int32), ("negs", C.c_int32), ("optimizer", C.c_int32),
                ("lr", C.c_float), ("beta_1", C.c_float), ("beta_2", C.c_float), ("epsilon", C.c_float),
                ("seed", C.c_uint64)]


# name -> (restype, argtypes); every symbol declared in include/movierec_b200.h
_vp, _i32, _i64, _u64, _f, _sz = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64, C.c_float, C.c_size_t
_PM, _PO, _PG = C.POINTER(MrModel), C.POINTER(MrOptState), C.POINTER(MrGrads)
_PF = C.POINTER(MrFoldIn)
SIGNATURES = {
    "mr_version": (C.c_int, []),
    "mr_last_error": (C.c_char_p, []),
    "mr_device_sm_count": (C.c_int, []),
    "mr_gather_rows": (C.c_int, [_vp, _i64, _i32, _vp, _i64, _vp, _vp]),
    "mr_forward_workspace_bytes": (_sz, [_PM, _i64]),
    "mr_neumf_forward": (C.c_int, [_PM, _vp, _vp, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "mr_train_workspace_bytes": (_sz, [_PM, _i64]),
    "mr_neumf_train_step": (C.c_int, [_PM, _PO, _PG, _vp, _vp, _vp, _i64, _i32, _i32, _i32, _f, _vp, _vp, _sz, _vp]),
    "mr_neumf_train_grads": (C.c_int, [_PM, _PO, _PG, _vp, _vp, _vp, _i64, _i32, _i32, _i32, _f, _vp, _vp, _sz, _vp]),
    "mr_users_grouped": (C.c_int, [_vp, _i64, _i32, _vp, _vp]),
    "mr_neumf_apply": (C.c_int, [_PM, _PO, _PG, _vp]),
    "mr_rank_eval_workspace_bytes": (_sz, [_PM, _i64, _i32]),
    "mr_rank_eval": (C.c_int, [_PM, _vp, _vp, _i64, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "mr_rank_scores_workspace_bytes": (_sz, [_i64]),
    "mr_rank_scores": (C.c_int, [_vp, _i64, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "mr_topk_scores_workspace_bytes": (_sz, [_i64, _i32, _i32]),
    "mr_topk_scores": (C.c_int, [_vp, _i64, _i32, _i32, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "mr_catalogue_topk_workspace_bytes": (_sz, [_PM, _i64, _i32]),
    "mr_catalogue_topk": (C.c_int, [_PM, _vp, _i64, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "mr_targets_scores_workspace_bytes": (_sz, [_i64, _i32, _i64]),
    "mr_targets_scores": (C.c_int, [_vp, _i64, _i32, _vp, _i32, _vp, _vp, _vp, _vp, _i64, _vp, _i32, _vp, _vp, _vp, _sz,
                                    _vp]),
    "mr_catalogue_targets_workspace_bytes": (_sz, [_PM, _i64, _i64]),
    "mr_catalogue_targets": (C.c_int, [_PM, _vp, _i64, _i32, _vp, _vp, _vp, _vp, _i64, _vp, _i32, _vp, _vp, _vp, _sz,
                                       _vp]),
    "mr_topk_lists_workspace_bytes": (_sz, [_i64, _i64, _i32]),
    "mr_topk_lists": (C.c_int, [_vp, _i64, _vp, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "mr_rank_lists_workspace_bytes": (_sz, [_PM, _i64, _i64, _i32]),
    "mr_rank_lists": (C.c_int, [_PM, _vp, _i64, _vp, _vp, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz,
                                _vp]),
    "mr_fold_in_workspace_bytes": (_sz, [_PM, _i64, _i64]),
    "mr_fold_in_users": (C.c_int, [_PM, _vp, _vp, _i64, _i64, _vp, _PF, _vp, _vp, _vp, _vp, _sz, _vp]),
    "mr_fold_in_items_workspace_bytes": (_sz, [_PM, _i64, _i64]),
    "mr_fold_in_items": (C.c_int, [_PM, _vp, _vp, _i64, _i64, _vp, _PF, _vp, _vp, _vp, _vp, _sz, _vp]),
    "mr_sample_negatives": (C.c_int, [_vp, _vp, _i32, _vp, _vp, _i64, _i64, _i32, _u64, _u64, _vp, _vp, _vp, _vp]),
    "mr_sort_workspace_bytes": (_sz, [_i64]),
    "mr_sort_pairs": (C.c_int, [_vp, _i64, _i32, _vp, _vp, _vp, _sz, _vp]),
    "mr_gather_rows_sharded": (C.c_int, [_vp, _i32, _i64, _i32, _vp, _i64, _vp, _vp]),
    "mr_sparse_rows_workspace_bytes": (_sz, [_i64, _i32, _i32]),
    "mr_sparse_rows_update": (C.c_int, [_vp, _vp, _vp, _i32, _vp, _vp, _vp, _i32, _i32, _vp, _vp, _i64, _i32, _f, _f, _f, _f,
                                        _f, _vp, _sz, _vp]),
    "mr_remap_workspace_bytes": (C.c_size_t, [_i64]),
    "mr_remap_ids": (C.c_int, [_vp, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "mr_split_workspace_bytes": (C.c_size_t, [_i64]),
    "mr_split_last_two": (C.c_int, [_vp, _i64, _i32, _vp, _vp, _vp, _vp, _sz, _vp]),
    "mr_user_csr_workspace_bytes": (C.c_size_t, [_i64]),
    "mr_build_user_csr": (C.c_int, [_vp, _vp, _i64, _i32, _i32, _vp, _vp, _vp, _vp, _sz, _vp]),
    "mr_uses_tensor_cores": (C.c_int, [_PM]),
    "mr_uses_item_projection": (C.c_int, [_PM, _i64]),
    "mr_uses_user_projection": (C.c_int, [_PM, _i64, _i32]),
    "mr_uses_small_tower": (C.c_int, [_PM, _i64, _i32]),
    "mr_profile_begin": (C.c_int, []),
    "mr_profile_end": (C.c_int, [C.POINTER(C.c_float), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "mr_optimizer_flat": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _i32, _f, _f, _f, _f, _f, _vp]),
    "mr_dp_reduce_apply": (C.c_int, [_vp, _vp, _i32, _i32, _vp, _vp, _i64, _i64, _i32, _f, _f, _f, _f, _f, _vp, _vp, _vp]),
}


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "{} not found at {}: build it with `make -C movierecommender-tf-trt_b200/csrc` or "
            "`python -c 'import __graft_entry__ as g; g.build()'` (there is no CPU fallback)".format(LIB_NAME, LIB_PATH))
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here = header and library disagree
        fn.restype = res
        fn.argtypes = args
    return lib


lib = _load()


def last_error():
    msg = lib.mr_last_error()
    return msg.decode("utf-8", "replace") if msg else ""


def check(rc, what):
    if rc != 0:
        raise MovierecNativeError("{} failed (status {}): {}".format(what, rc, last_error()))


NUM_PHASES = 14
PHASE_NAMES = ["tile_train", "misc", "sort", "segreduce", "optimizer", "tile_forward", "rank", "sampler",
               "tc_dense_fwd", "tc_dense_bwd", "tc_wgrad", "head", "h1_gather", "fused_tile"]


def profile_begin():
    check(lib.mr_profile_begin(), "mr_profile_begin")


def profile_end():
    """-> ({phase: (ms, intervals)}, kernel launches since profile_begin)."""
    ms = (C.c_float * NUM_PHASES)()
    cnt = (C.c_int64 * NUM_PHASES)()
    launches = C.c_int64(0)
    check(lib.mr_profile_end(ms, cnt, C.byref(launches)), "mr_profile_end")
    return {PHASE_NAMES[i]: (float(ms[i]), int(cnt[i])) for i in range(NUM_PHASES)}, int(launches.value)


def version():
    return lib.mr_version()
