"""ctypes binding of csrc/libcbrs_b200.so (the C ABI declared in include/cbrs_b200.h).

There is no fallback: if the library is missing or a call fails, a RuntimeError
is raised.  PyTorch is used by the callers for device memory and streams only.
"""
import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_size_t, c_uint64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libcbrs_b200.so")


class CbrsError(RuntimeError):
    pass


class CsrDesc(Structure):
    """Mirror of cbrs_csr_t."""
    _fields_ = [
        ("n_rows", c_int64), ("nnz", c_int64),
        ("rowptr", c_void_p), ("colidx", c_void_p), ("vals", c_void_p),
        ("chunk_edges", c_int32), ("n_chunks", c_int64),
        ("chunk_row", c_void_p), ("chunk_begin", c_void_p), ("chunk_slot", c_void_p),
        ("n_heavy", c_int64), ("heavy_row", c_void_p), ("heavy_slot_ptr", c_void_p),
        ("n_slots", c_int64), ("chunk_len", c_void_p),
    ]


P = c_void_p
_SIGS = {
    "cbrs_version": (c_int, []),
    "cbrs_last_error": (c_char_p, []),
    "cbrs_check_device": (c_int, []),
    "cbrs_graph_build_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int]),
    "cbrs_graph_build_csr": (c_int, [P, P, P, c_int64, c_int64, c_int, P, P, P, P, P, c_size_t, P]),
    "cbrs_graph_build_csr_rel": (c_int, [P, P, P, P, c_int64, c_int64, c_int32, c_int32, c_int, P, P, P, P, P, c_size_t, P]),
    "cbrs_chunks_workspace_bytes": (c_size_t, [c_int64]),
    "cbrs_chunks_count": (c_int, [P, c_int64, c_int32, P, P, c_size_t, P]),
    "cbrs_chunks_fill": (c_int, [P, c_int64, c_int32, P, P, P, P, P, P, c_size_t, P]),
    "cbrs_chunks_blocked_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64, c_int32, c_int64]),
    "cbrs_chunks_blocked_count": (c_int, [P, P, c_int64, c_int64, c_int64, c_int32, c_int32, c_int64, P, P, c_size_t, P]),
    "cbrs_chunks_blocked_fill": (c_int, [P, P, c_int64, c_int64, c_int64, c_int32, c_int32, c_int64, P, P, P, P, P, P, P,
                                         c_size_t, P]),
    "cbrs_spmm_workspace_bytes": (c_size_t, [POINTER(CsrDesc), c_int32]),
    "cbrs_spmm_csr": (c_int, [POINTER(CsrDesc), P, c_int64, P, c_int64, c_int32, c_int, P, c_int, c_int, P, c_size_t, P]),
    "cbrs_gat_workspace_bytes": (c_size_t, [POINTER(CsrDesc), c_int32]),
    "cbrs_gat_csr": (c_int, [POINTER(CsrDesc), c_int64, P, c_int64, P, P, P, c_int64, c_int32, P, c_int, P, c_size_t, P]),
    "cbrs_dense": (c_int, [P, c_int64, P, c_int32, P, c_int64, P, c_int32, P, P, c_int64, c_int32, c_int, c_int,
                           P, P, P, P, P, c_int64, P]),
    "cbrs_dense_ex": (c_int, [P, c_int64, P, c_int32, P, c_int64, P, c_int32, P, P, c_int64, c_int32, c_int, c_int,
                              P, P, P, P, P, c_int64, c_int, POINTER(c_void_p), POINTER(c_void_p), c_int, P]),
    "cbrs_dense_tc_image_bytes": (c_size_t, [c_int32, c_int32]),
    "cbrs_dense_tc_prepare": (c_int, [P, c_int32, c_int32, P, P]),
    "cbrs_dense_tc": (c_int, [P, c_int64, P, c_int32, P, c_int64, P, c_int32, P, P, c_int64, c_int32, c_int, P, c_int64, P]),
    "cbrs_convert_f32_bf16": (c_int, [P, c_int64, c_int64, c_int32, P, c_int64, P]),
    "cbrs_dense_tc_bf16_eligible": (c_int, [c_int32, c_int32, c_int32]),
    "cbrs_dense_tc_bf16": (c_int, [P, c_int64, c_int64, P, c_int32, P, c_int64, c_int64, P, c_int32, P, P, c_int64, c_int32, c_int,
                                   P, c_int64, c_int, P]),
    "cbrs_score_hybrid_topk_bf16_workspace_bytes": (c_size_t, []),
    "cbrs_score_hybrid_topk_bf16": (c_int, [P, P, P, P, c_int64, c_int32, c_int32, P, P, P, P, P, P, P, P, P, P, c_int32, P, P, P,
                                            c_size_t, P]),
    "cbrs_score_hybrid_topk_bf16_ex": (c_int, [P, P, P, P, c_int64, c_int32, c_int32, P, P, P, P, P, P, P, P, P, P, c_int32, P, P,
                                               P, P, P, c_size_t, P]),
    "cbrs_score_hybrid_topk_tf32x3_workspace_bytes": (c_size_t, []),
    "cbrs_score_hybrid_topk_tf32x3": (c_int, [P, P, P, P, c_int64, c_int32, c_int32, P, P, P, P, P, P, P, P, P, P, c_int32, P, P,
                                              P, P, P, c_size_t, P]),
    "cbrs_dense_grouped": (c_int, [P, c_int64, P, c_int64, c_int32, c_int32, c_int32, P, c_int64, c_int64, c_int,
                                   POINTER(c_void_p), c_int, P]),
    "cbrs_dense_tf32x3_eligible": (c_int, [c_int32, c_int32]),
    "cbrs_dense_tf32x3_image_bytes": (c_size_t, [c_int32, c_int32]),
    "cbrs_dense_tf32x3_prepare": (c_int, [P, c_int32, c_int32, P, P]),
    "cbrs_dense_tf32x3": (c_int, [P, c_int64, P, P, c_int64, c_int32, c_int32, c_int, P, c_int64, c_int, POINTER(c_void_p), c_int, P]),
    "cbrs_dense_tf32x3_ex": (c_int, [P, c_int64, P, P, P, c_int64, c_int, c_int64, c_int32, c_int32, c_int, P, c_int64, c_int,
                                     POINTER(c_void_p), c_int, P]),
    "cbrs_dense_tf32x3_attn": (c_int, [P, c_int64, P, c_int64, c_int32, c_int32, P, P, P, P, P, c_int64, POINTER(c_void_p),
                                       POINTER(c_void_p), c_int, P]),
    "cbrs_reduce_layers": (c_int, [POINTER(c_void_p), POINTER(c_int64), c_int32, POINTER(c_float), c_float,
                                   c_int64, c_int32, P, c_int64, P]),
    "cbrs_gather_rows": (c_int, [P, c_int64, P, c_int64, c_int32, P, c_int64, P]),
    "cbrs_topk_rows": (c_int, [P, c_int64, c_int64, c_int32, c_int32, P, P, P]),
    "cbrs_exclude_cols": (c_int, [P, c_int64, c_int64, c_int32, c_int32, P, P, P]),
    "cbrs_rank_metrics_workspace_bytes": (c_size_t, [c_int64, c_int32]),
    "cbrs_rank_metrics": (c_int, [P, c_int64, c_int64, c_int32, c_int32, P, c_int64, P, P, POINTER(c_int32), c_int32, P, P,
                                  P, c_size_t, P]),
    "cbrs_topk_pairs_workspace_bytes": (c_size_t, [c_int64]),
    "cbrs_topk_pairs": (c_int, [P, P, c_int64, c_int64, P, P, P, c_size_t, P]),
    "cbrs_score_catalog_topk": (c_int, [P, c_int64, P, c_int64, c_int64, c_int32, c_int32, P, P, c_int32, P, P, c_int32,
                                        P, P, P]),
    "cbrs_score_catalog_topk_ex": (c_int, [P, c_int64, P, c_int64, c_int64, c_int32, c_int32, P, P, c_int32, P, P, c_int32,
                                           P, P, P, P, P]),
    "cbrs_score_catalog_topk_tf32x3_eligible": (c_int, [c_int32, c_int32]),
    "cbrs_score_catalog_topk_tf32x3_workspace_bytes": (c_size_t, [c_int32, c_int32]),
    "cbrs_score_catalog_topk_tf32x3": (c_int, [P, c_int64, P, c_int64, c_int64, c_int32, c_int32, P, P, c_int32, P, P, c_int32,
                                               P, P, P, c_size_t, P]),
    "cbrs_score_catalog_topk_tf32x3_ex": (c_int, [P, c_int64, P, c_int64, c_int64, c_int32, c_int32, P, P, c_int32, P, P,
                                                  c_int32, P, P, P, P, P, c_size_t, P]),
    "cbrs_score_catalog_topk_bf16_workspace_bytes": (c_size_t, [c_int32, c_int32, c_int32]),
    "cbrs_score_catalog_topk_bf16": (c_int, [P, c_int64, P, c_int64, c_int64, c_int32, c_int32, P, P, c_int32, P, P,
                                             c_int32, P, P, P, c_size_t, P]),
    "cbrs_score_catalog_topk_bf16_ex": (c_int, [P, c_int64, P, c_int64, c_int64, c_int32, c_int32, P, P, c_int32, P, P,
                                                c_int32, P, P, P, P, P, c_size_t, P]),
    "cbrs_peer_alloc": (c_int, [c_size_t, POINTER(c_void_p)]),
    "cbrs_peer_free": (c_int, [P]),
    "cbrs_peer_export": (c_int, [P, P]),
    "cbrs_peer_open": (c_int, [P, POINTER(c_void_p)]),
    "cbrs_peer_close": (c_int, [P]),
    "cbrs_push_rows": (c_int, [P, c_int64, P, c_int64, c_int64, c_int32, P]),
    "cbrs_peer_copy": (c_int, [P, P, c_size_t, P]),
    "cbrs_peer_barrier": (c_int, [POINTER(c_void_p), c_int, c_int, c_uint64, P, c_double, P]),
    "cbrs_spmm_csr_bcast": (c_int, [POINTER(CsrDesc), P, c_int64, P, c_int64, c_int32, c_int, P, c_int, c_int,
                                    POINTER(c_void_p), c_int, P, c_size_t, P]),
    "cbrs_spmm_gcn_fused": (c_int, [POINTER(CsrDesc), P, c_int64, P, c_int64, P, c_int, P, P, c_int64, POINTER(c_void_p), c_int,
                                    POINTER(c_void_p), c_int, P, c_size_t, P]),
    "cbrs_gat_csr_bcast": (c_int, [POINTER(CsrDesc), c_int64, P, c_int64, P, P, P, c_int64, c_int32, P, c_int,
                                   POINTER(c_void_p), c_int, P, c_size_t, P]),
    "cbrs_dense_bcast": (c_int, [P, c_int64, P, c_int32, P, c_int64, P, c_int32, P, P, c_int64, c_int32, c_int, c_int,
                                 P, P, P, P, P, c_int64, POINTER(c_void_p), POINTER(c_void_p), c_int, P]),
    "cbrs_compact_ids_workspace_bytes": (c_size_t, [c_int64]),
    "cbrs_compact_ids": (c_int, [P, c_int64, P, P, P, P, c_size_t, P]),
    "cbrs_lookup_ids": (c_int, [P, c_int64, P, c_int64, P, P]),
    "cbrs_spgemm_workspace_bytes": (c_size_t, [c_int64]),
    "cbrs_spgemm_count": (c_int, [POINTER(CsrDesc), POINTER(CsrDesc), P, P, P, c_size_t, P]),
    "cbrs_spgemm_expand": (c_int, [POINTER(CsrDesc), POINTER(CsrDesc), P, P, P, P, P]),
    "cbrs_count_above": (c_int, [P, c_int64, POINTER(c_float), c_int32, P, P]),
    "cbrs_csr_filter_above_workspace_bytes": (c_size_t, [c_int64]),
    "cbrs_csr_filter_above": (c_int, [POINTER(CsrDesc), c_float, P, P, P, P, c_size_t, P]),
    "cbrs_row_gate": (c_int, [P, c_int64, P, c_int64, c_int32, P, c_int64, P]),
    "cbrs_row_gate_grad": (c_int, [P, c_int64, P, c_int64, P, c_int64, c_int32, P, c_int64, P, P]),
    "cbrs_act_grad": (c_int, [P, c_int64, P, c_int64, c_int64, c_int32, c_int, P, c_int64, P]),
    "cbrs_dense_grad_w_workspace_bytes": (c_size_t, [c_int64, c_int32, c_int32]),
    "cbrs_dense_grad_w": (c_int, [P, c_int64, P, c_int32, P, c_int64, P, c_int32, P, c_int64, c_int64, c_int32, P, P,
                                  P, c_size_t, P]),
    "cbrs_transpose_f32": (c_int, [P, c_int32, c_int32, P, P]),
    "cbrs_scatter_add_rows_workspace_bytes": (c_size_t, [c_int64]),
    "cbrs_scatter_add_rows": (c_int, [P, c_int64, P, c_int64, c_int32, c_int64, P, c_int64, P, c_size_t, P]),
    "cbrs_l2norm_act": (c_int, [P, c_int64, c_int64, c_int32, c_int, P, c_int64, P]),
    "cbrs_l2norm_relu_grad": (c_int, [P, c_int64, P, c_int64, c_int64, c_int32, c_int, P, c_int64, P]),
    "cbrs_scale_rows_inv_degree": (c_int, [P, c_int64, P, c_int64, c_int32, P, c_int64, P]),
    "cbrs_axpby2d": (c_int, [P, c_int64, c_float, P, c_int64, c_float, c_int64, c_int32, P, c_int64, P]),
    "cbrs_bce": (c_int, [P, P, c_int64, P, P, P, P]),
    "cbrs_sum_squares_workspace_bytes": (c_size_t, []),
    "cbrs_sum_squares": (c_int, [P, c_int64, c_float, P, c_int, P, c_size_t, P]),
    "cbrs_adam_step": (c_int, [P, P, P, P, c_int64, c_float, P, c_float, c_float, c_float, c_float, P]),
    "cbrs_attn_fuse": (c_int, [P, c_int64, P, c_int64, P, P, c_int64, c_int32, P, c_int64, P]),
    "cbrs_attn_fuse_grad": (c_int, [P, c_int64, P, c_int64, P, c_int64, P, P, c_int64, c_int32, P, P, P, P, P]),
    "cbrs_add3_act": (c_int, [P, c_int64, P, c_int64, P, c_int64, c_int64, c_int32, c_int, P, c_int64, P]),
    "cbrs_gat_backward_workspace_bytes": (c_size_t, [c_int64]),
    "cbrs_gat_backward": (c_int, [POINTER(CsrDesc), P, c_int64, P, P, P, c_int64, P, P, c_int64, c_int32, P, P, P, c_int64,
                                  P, P, P, c_size_t, P]),
    "cbrs_adam_step_multi": (c_int, [c_int32, POINTER(c_void_p), POINTER(c_void_p), POINTER(c_void_p), POINTER(c_void_p),
                                     POINTER(c_int64), POINTER(c_float), c_float, P, c_float, c_float, c_float, P]),
    "cbrs_synth_bipartite": (c_int, [c_int64, c_int64, c_int64, c_uint64, P, P, P]),
    "cbrs_synth_bipartite_ex": (c_int, [c_int64, c_int64, c_int64, c_uint64, c_int, P, P, P]),
    "cbrs_sort_workspace_bytes": (c_size_t, [c_int64]),
    "cbrs_sort_pairs_u64": (c_int, [P, P, c_int64, c_int, P, c_size_t, P]),
}

# constants of include/cbrs_b200.h
GRAPH_DEDUP_SUM, GRAPH_ADD_SELF_LOOPS, GRAPH_SYM_NORM, GRAPH_DROP_DIAG = 1, 2, 4, 8
AGG_WEIGHTED, AGG_SUM, AGG_MEAN = 0, 1, 2
DTYPE_F32, DTYPE_BF16 = 0, 1
ACT_NONE, ACT_RELU, ACT_SIGMOID, ACT_TANH = 0, 1, 2, 3
ROWOP_NONE, ROWOP_L2NORM, ROWOP_ATTN = 0, 1, 2
MAX_PEERS, IPC_HANDLE_BYTES = 8, 64
ACTS = {None: ACT_NONE, "linear": ACT_NONE, "relu": ACT_RELU, "sigmoid": ACT_SIGMOID, "tanh": ACT_TANH}

_lib = None


def exported_symbols():
    return sorted(_SIGS)


def load():
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise CbrsError(
            "CUDA library not built: {} is missing. Run `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C deep_cbrs_amar_renaissance_b200/csrc`). There is no CPU fallback.".format(LIB_PATH))
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in _SIGS.items():
        fn = getattr(lib, name)  # AttributeError here == header / library drift
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().cbrs_last_error()
        raise CbrsError("{} failed (code {}): {}".format(what, rc, msg.decode() if msg else "?"))
