"""ctypes binding of librecad_b200.so (the C ABI declared in include/recad_b200.h).

There is NO fallback: if the shared library is missing or a call fails, a
RuntimeError is raised.  Nothing in this package imports ``oracle``.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "librecad_b200.so")

i32, i64, f32, vp = C.c_int32, C.c_int64, C.c_float, C.c_void_p


class RecadError(RuntimeError):
    pass


class CSR(C.Structure):
    """struct recad_csr"""
    _fields_ = [
        ("n_rows", i64), ("n_cols", i64), ("nnz", i64), ("rowptr", vp), ("colidx", vp), ("vals", vp), ("cv", vp),
        ("n_seg", i64), ("seg_meta", vp), ("n_mrow", i64), ("row_mseg", vp), ("row_cnt", vp), ("partials", vp),
    ]


class LightGCN(C.Structure):
    """struct recad_lightgcn"""
    _fields_ = [
        ("graph", C.POINTER(CSR)), ("n_users", i64), ("n_items", i64), ("D", i32), ("n_layers", i32),
        ("lam", f32), ("lr", f32), ("beta1", f32), ("beta2", f32), ("eps", f32), ("_pad", i32),
        ("E", vp), ("m", vp), ("v", vp), ("O", vp), ("X0", vp), ("X1", vp), ("g", vp), ("cnt", vp), ("loss_acc", vp),
        ("graph_t", C.POINTER(CSR)),
    ]


class EpochSamples(C.Structure):
    """struct recad_epoch_samples"""
    _fields_ = [("n_samples", i64), ("rows", vp), ("perm64", vp), ("users", vp), ("rel", vp), ("negs", vp), ("perm32", vp)]


class LightGCNShard(C.Structure):
    """struct recad_lightgcn_shard"""
    _fields_ = [
        ("rank", i32), ("world", i32), ("D", i32), ("n_layers", i32),
        ("n_users_local", i64), ("n_items", i64), ("user_lo", i64), ("slice", i64),
        ("lam", f32), ("lr", f32), ("beta1", f32), ("beta2", f32), ("eps", f32), ("_pad", i32),
        ("g_user", C.POINTER(CSR)), ("g_item", C.POINTER(CSR)),
        ("pos_rowptr", vp), ("pos_col", vp), ("pos_col_offset", i64),
        ("E", vp), ("m", vp), ("v", vp), ("loss_acc", vp),
        ("peer_base", C.POINTER(vp)), ("mc_base", vp), ("peer_users", C.POINTER(i64)),
        ("off_X0", i64), ("off_X1", i64), ("off_O", i64), ("off_g", i64), ("off_cnt", i64), ("off_stage", i64), ("off_signal", i64),
    ]


class WMF(C.Structure):
    """struct recad_wmf"""
    _fields_ = [("n_rows", i64), ("n_items", i64), ("dim", i32), ("batch", i32), ("lr", f32), ("beta1", f32), ("beta2", f32),
                ("eps", f32), ("weight_decay", f32), ("weight_pos", f32), ("weight_neg", f32), ("_pad", i32),
                ("P", vp), ("Q", vp), ("mP", vp), ("vP", vp), ("mQ", vp), ("vQ", vp)]


class Aush(C.Structure):
    """struct recad_aush"""
    _fields_ = [("n_items", i64), ("n_sel", i32), ("filler_num", i32), ("lr", f32), ("beta1", f32), ("beta2", f32), ("eps", f32),
                ("G_W1t", vp), ("G_b1", vp), ("G_W2", vp), ("G_b2", vp), ("D", vp), ("Dm", vp), ("Dv", vp), ("selected", vp), ("work", vp)]


class AushEpoch(C.Structure):
    """struct recad_aush_epoch"""
    _fields_ = [("n_rows", i64), ("batch", i32), ("_pad", i32), ("cols", vp), ("tval", vp), ("dval", vp), ("rsel", vp), ("tsel", vp),
                ("msel", vp), ("zr", vp), ("colptr", vp), ("ent", vp)]


class MF(C.Structure):
    """struct recad_mf"""
    _fields_ = [
        ("n_users", i64), ("n_items", i64), ("D", i32), ("mean", f32), ("lr", f32), ("beta1", f32), ("beta2", f32),
        ("eps", f32),
        ("Ue", vp), ("Ub", vp), ("Ie", vp), ("Ib", vp),
        ("mUe", vp), ("mUb", vp), ("mIe", vp), ("mIb", vp),
        ("vUe", vp), ("vUb", vp), ("vIe", vp), ("vIb", vp),
        ("gUe", vp), ("gUb", vp), ("gIe", vp), ("gIb", vp),
        ("loss_acc", vp),
    ]


class NCF(C.Structure):
    """struct recad_ncf"""
    _fields_ = [
        ("n_users", i64), ("n_items", i64), ("factor", i32), ("n_layers", i32),
        ("lr", f32), ("beta1", f32), ("beta2", f32), ("eps", f32), ("tower_fp32", i32), ("variant", i32),
        ("params", vp), ("m", vp), ("v", vp), ("grads", vp), ("n_params", i64),
        ("work", vp), ("work_floats", i64), ("max_batch", i64), ("loss_acc", vp),
    ]


# name -> (restype, argtypes); every symbol of include/recad_b200.h
SIGNATURES = {
    "recad_abi_version": (C.c_int, []),
    "recad_last_error": (C.c_char_p, []),
    "recad_device_info": (C.c_int, [C.POINTER(C.c_int)] * 3),
    "recad_csr_build_scratch_bytes": (i64, [i64, i64, i64]),
    "recad_csr_build_structure": (C.c_int, [vp, vp, i64, i64, i64, vp, vp, vp, vp, C.POINTER(i64), vp, i64, vp]),
    "recad_csr_normalize": (C.c_int, [vp, vp, vp, vp, i64, vp, vp]),
    "recad_csr_append_users": (C.c_int, [vp, vp, vp, i64, i64, i64, vp, vp, i64, vp, vp, vp, vp, vp, i64, vp]),
    "recad_csr_append_scratch_bytes": (i64, [i64, i64, i64, i64]),
    "recad_spmm": (C.c_int, [C.POINTER(CSR), vp, vp, vp, vp, f32, i32, vp]),
    "recad_spmm_pack_cv": (C.c_int, [vp, vp, i64, vp, vp]),
    "recad_spmm_scatter": (C.c_int, [C.POINTER(CSR), vp, C.POINTER(vp), i32, i64, i32, vp]),
    "recad_peer_reduce_bcast": (C.c_int, [vp, i32, i64, i64, C.POINTER(vp), i32, i32, vp]),
    "recad_bpr_fwd_bwd": (C.c_int, [vp, vp, i64, i64, vp, vp, i64, i64, f32, vp, vp, vp, i32, vp]),
    "recad_axpby": (C.c_int, [vp, f32, vp, f32, vp, i64, vp]),
    "recad_adam": (C.c_int, [vp, vp, vp, f32, vp, vp, i64, i32, f32, f32, f32, f32, i64, vp]),
    "recad_lightgcn_propagate": (C.c_int, [C.POINTER(LightGCN), vp]),
    "recad_lightgcn_train_epoch": (C.c_int, [C.POINTER(LightGCN), vp, vp, i64, i64, i64, vp]),
    "recad_bpr_fwd_bwd_i32": (C.c_int, [vp, vp, i64, i64, vp, vp, i64, i64, f32, vp, vp, vp, i32, vp]),
    "recad_lightgcn_train_epoch_i32": (C.c_int, [C.POINTER(LightGCN), vp, vp, i64, i64, i64, vp]),
    "recad_lightgcn_shard_propagate": (C.c_int, [C.POINTER(LightGCNShard), vp]),
    "recad_lightgcn_shard_train_epoch": (C.c_int, [C.POINTER(LightGCNShard), C.POINTER(EpochSamples), i64, i64, C.POINTER(C.c_double), vp]),
    "recad_lightgcn_shard_barrier_state": (C.c_int, [C.POINTER(LightGCNShard), C.POINTER(C.c_uint32), vp]),
    "recad_wmf_snapshot_floats": (i64, [C.POINTER(WMF), i32]),
    "recad_wmf_fit": (C.c_int, [C.POINTER(WMF), vp, vp, i32, i64, i32, vp, vp]),
    "recad_wmf_backward": (C.c_int, [C.POINTER(WMF), vp, vp, i32, i64, vp, vp, vp, vp, vp, vp]),
    "recad_aush_d_layout": (C.c_int, [i64, C.POINTER(i64)]),
    "recad_aush_work_floats": (i64, [i64, i64, i32, i32]),
    "recad_aush_plan_columns": (C.c_int, [vp, i64, i32, i32, i64, vp, vp]),
    "recad_aush_train_epoch": (C.c_int, [C.POINTER(Aush), C.POINTER(AushEpoch), i64, vp, vp]),
    "recad_aush_generate": (C.c_int, [C.POINTER(Aush), vp, vp, i64, vp, vp]),
    "recad_mt19937_aush_batch": (C.c_int, [vp, C.POINTER(i32), i64, vp, vp, vp, vp, i32, i32, vp, C.c_double, vp, vp, vp]),
    "recad_dot_scores": (C.c_int, [vp, i64, vp, vp, i64, i32, vp, vp]),
    "recad_pair_scores_backward_scratch_bytes": (i64, [i64]),
    "recad_pair_scores_backward": (C.c_int, [vp, i64, vp, i64, i32, vp, vp, i64, vp, vp, vp, vp, vp, vp, i64, vp]),
    "recad_lightgcn_backward": (C.c_int, [C.POINTER(LightGCN), vp, vp, vp]),
    "recad_lightgcn_backward_values": (C.c_int, [C.POINTER(LightGCN), vp, C.POINTER(vp), vp, vp, vp]),
    "recad_pair_scores_hvp": (C.c_int, [vp, vp, i64, vp, vp, i64, i32, vp, vp, i64, vp, vp, vp, vp, vp, vp, vp, i64, vp]),
    "recad_bpr_hvp_seeds": (C.c_int, [vp, vp, i64, i64, vp, i64, i64, i32, vp, vp, f32, vp, vp, vp, vp, vp]),
    "recad_lightgcn_loss_mixed_values_work_bytes": (i64, [i64, i32, i32, i64]),
    "recad_lightgcn_loss_mixed_values": (C.c_int, [C.POINTER(LightGCN), C.POINTER(CSR), vp, vp, i64, vp, vp, i64, vp]),
    "recad_index_sums": (C.c_int, [vp, vp, i64, i64, vp, vp, i64, vp]),
    "recad_lightgcn_candidate_weight_grads_work_bytes": (i64, [i64, i64, i32, i32, i64, i64, i64]),
    "recad_lightgcn_candidate_weight_grads": (C.c_int, [C.POINTER(LightGCN), C.POINTER(CSR), vp, vp, vp, vp, vp, vp, i64, f32,
                                                        vp, i64, vp, vp, i64, vp]),
    "recad_csr_sddmm": (C.c_int, [C.POINTER(CSR), vp, vp, i32, f32, i32, vp, vp]),
    "recad_csr_row_sums": (C.c_int, [vp, vp, i64, i64, vp, vp]),
    "recad_csr_normalize_backward": (C.c_int, [vp, vp, vp, vp, vp, vp, i64, i64, vp, vp, vp]),
    "recad_mf_forward": (C.c_int, [C.POINTER(MF), vp, vp, i64, vp, vp]),
    "recad_mf_train_epoch": (C.c_int, [C.POINTER(MF), vp, vp, i64, i64, i64, vp]),
    "recad_mf_grad": (C.c_int, [C.POINTER(MF), vp, vp, i64, i64, vp]),
    "recad_mf_hvp_seeds": (C.c_int, [C.POINTER(MF), vp, vp, vp, vp, vp, i64, i64, vp, vp, vp, vp, vp]),
    "recad_ncf_layout": (C.c_int, [i32, i32, i64, i64, C.POINTER(i64)]),
    "recad_ncf_work_floats": (i64, [i32, i32, i64]),
    "recad_ncf_forward": (C.c_int, [C.POINTER(NCF), vp, vp, i64, vp, vp]),
    "recad_ncf_rank_work_floats": (i64, [i32, i32, i64]),
    "recad_ncf_rank_floats": (i64, [C.POINTER(NCF), i64]),
    "recad_ncf_rank_prepare": (C.c_int, [C.POINTER(NCF), vp, i64, vp, vp, i64, i64, vp]),
    "recad_ncf_rank_block": (C.c_int, [C.POINTER(NCF), vp, vp, i64, i64, i64, vp, vp, i64, i64, vp]),
    "recad_ncf_train_epoch": (C.c_int, [C.POINTER(NCF), vp, vp, i64, i64, i64, vp]),
    "recad_ncf_graph_launches": (i64, []),
    "recad_ncf_grad": (C.c_int, [C.POINTER(NCF), vp, vp, i64, i64, vp]),
    "recad_ncf_backward": (C.c_int, [C.POINTER(NCF), vp, vp, i64, vp, vp, vp]),
    "recad_ncf_hvp_work_floats": (i64, [i32, i32, i64]),
    "recad_ncf_hvp": (C.c_int, [C.POINTER(NCF), vp, i64, vp, vp, vp, vp, i64, vp]),
    "recad_gemm_tn_tf32x3": (C.c_int, [vp, vp, i32, i32, i32, vp, i32, vp, vp, vp]),
    "recad_transpose_items": (C.c_int, [vp, i64, i32, vp, i64, vp]),
    "recad_fullrank_eval": (C.c_int, [vp, vp, i64, i64, i32, vp, i64, vp, vp, vp, i32, i32, vp, vp, vp, vp, vp]),
    "recad_fullrank_tc_scratch_floats": (i64, [i64, i64]),
    "recad_fullrank_eval_tc": (C.c_int, [vp, vp, i64, i32, vp, i64, vp, vp, vp, i32, i32, vp, vp, vp, vp, vp, vp, i64, vp]),
    "recad_eligible_users_scratch_bytes": (i64, [i64]),
    "recad_eligible_users": (C.c_int, [vp, vp, i64, i64, vp, i32, vp, vp, C.POINTER(i64), vp, i64, vp]),
    "recad_recall_ndcg": (C.c_int, [vp, i64, i32, vp, vp, vp, vp, vp]),
    "recad_rank_from_scores": (C.c_int, [vp, i64, i64, vp, vp, vp, vp, i32, i32, vp, vp, vp, vp, vp]),
    "recad_mt19937_pairwise": (C.c_int, [vp, C.POINTER(i32), i64, i64, i64, vp, vp, vp, C.POINTER(i64)]),
    "recad_host_advise_huge": (C.c_int, [vp, i64]),
    "recad_pairwise_filter_build_range": (C.c_int, [vp, vp, i64, i64, vp, vp, i32]),
    "recad_mt19937_pointwise": (C.c_int, [vp, C.POINTER(i32), i64, vp, vp, vp, vp, i64, i32, vp]),
    "recad_mt19937_permutation": (C.c_int, [vp, C.POINTER(i32), i64, vp]),
    "recad_mt19937_permutation_draw": (C.c_int, [vp, C.POINTER(i32), i64, vp]),
    "recad_permutation_apply": (C.c_int, [i64, vp, vp]),
    "recad_mt19937_pairwise_soa": (C.c_int, [vp, C.POINTER(i32), i64, i64, i64, vp, vp, vp, vp, i32, vp, vp, vp, C.POINTER(i64), vp]),
    "recad_permutation_apply32": (C.c_int, [i64, vp, vp]),
    "recad_samples_expand": (C.c_int, [vp, vp, vp, vp, vp, i64, vp, vp]),
}

_lib = None


def lib():
    """Load (once) and return the shared library; raise loudly if it is absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RecadError(
                f"{LIB_PATH} not found: build it with `python -m recad_b200.csrc.build` "
                "(recad_b200 has no CPU or PyTorch fallback)")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)   # AttributeError if the library lacks a declared symbol
            fn.restype, fn.argtypes = res, args
        if handle.recad_abi_version() != 2:
            raise RecadError("librecad_b200.so ABI version mismatch; rebuild")
        _lib = handle
    return _lib


def check(rc, what=""):
    if rc != 0:
        msg = lib().recad_last_error()
        raise RecadError(f"{what} failed (code {rc}): {msg.decode() if msg else ''}")
