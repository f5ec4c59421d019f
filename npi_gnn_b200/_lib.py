"""ctypes binding of libnpi.so (the C ABI declared in include/npi.h).

The library is built in-tree by ``npi_gnn_b200.build`` / ``__graft_entry__.build()``.  There is
NO fallback: if the shared object is missing or a call fails, an exception is raised.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("NPI_LIB") or os.path.join(_HERE, "libnpi.so")     # NPI_LIB: a tuning variant (build.py --variant)


class NPIError(RuntimeError):
    pass


class Features(C.Structure):
    """npi_features_t"""
    _fields_ = [("x", C.c_void_p), ("ldx", C.c_int32), ("table", C.c_void_p), ("ld", C.c_int32),
                ("gid", C.c_void_p), ("dist", C.c_void_p), ("F", C.c_int32)]


class TinyArgs(C.Structure):
    """npi_tiny_args_t (include/npi.h): the buffers of the small-subgraph path, filled once per engine slot"""
    _fields_ = [("B", C.c_int32), ("max_graph_nodes", C.c_int32), ("graph_ptr", C.c_void_p * 4),
                ("T", C.c_void_p), ("w_label", C.c_void_p), ("gid", C.c_void_p), ("dist", C.c_void_p),
                ("rowptr0", C.c_void_p), ("col0", C.c_void_p),
                ("weight", C.c_void_p * 3), ("bias", C.c_void_p * 3), ("pool_w", C.c_void_p * 3), ("weight_t", C.c_void_p * 3),
                ("h", C.c_void_p * 3), ("z", C.c_void_p * 3), ("s", C.c_void_p * 3),
                ("perm", C.c_void_p * 3), ("new_id", C.c_void_p * 3), ("batch", C.c_void_p * 3),
                ("xp", C.c_void_p * 3), ("argmax", C.c_void_p * 3),
                ("rowptr_f", C.c_void_p * 2), ("col_f", C.c_void_p * 2),
                ("y", C.c_void_p * 3), ("readout", C.c_void_p), ("d_readout", C.c_void_p),
                ("dpre", C.c_void_p * 3), ("dxa", C.c_void_p * 3), ("dxp", C.c_void_p * 2),
                ("partials", C.c_void_p), ("d_pool_w", C.c_void_p * 3), ("d_bias", C.c_void_p * 3)]


_vp, _i32, _i64, _f32, _u64 = C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_uint64
_f64, _u32 = C.c_double, C.c_uint32
_FP = C.POINTER(Features)
_TP = C.POINTER(TinyArgs)

# name -> (restype, argtypes); mirrors include/npi.h one to one
SIGNATURES = {
    "npi_last_error": (C.c_char_p, []),
    "npi_version": (C.c_int, []),
    "npi_sm_count": (C.c_int, [C.POINTER(_i32)]),
    "npi_csr_build_host": (C.c_int, [_vp, _i64, _i32, _vp, _vp, _vp, _vp, C.POINTER(_i64)]),
    "npi_khop_workspace_bytes": (_i64, [_i32, _i32]),
    "npi_csr_fold_mask": (C.c_int, [_vp, _vp, _vp, _i64, _vp, _vp]),
    "npi_khop_count": (C.c_int, [_vp, _vp, _i32, _vp, _i32, _i32, _vp, _vp, _vp, _i64, _i32, _vp]),
    "npi_khop_fill": (C.c_int, [_vp, _vp, _i32, _vp, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _vp, _vp, _i64, _i32, _vp]),
    "npi_batch_prepare": (C.c_int, [_vp, _i32, _i32, _vp, _vp, _vp, _vp, _f32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "npi_subgraph_coo": (C.c_int, [_vp, _vp, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i32, _vp]),
    "npi_gather_features": (C.c_int, [_FP, _vp, _i32, _vp, _vp]),
    "npi_coo_to_csr_workspace_bytes": (_i64, [_i32, _i64]),
    "npi_edge_symmetry_sums": (C.c_int, [_vp, _i64, _vp, _vp]),
    "npi_coo_to_csr": (C.c_int, [_vp, _i64, _i32, _vp, _vp, _vp, _i64, _vp]),
    "npi_sage_fwd": (C.c_int, [_FP, _vp, _vp, _vp, _i32, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp]),
    "npi_sage_bwd_weight_workspace_bytes": (_i64, [_i32]),
    "npi_sage_bwd_weight": (C.c_int, [_FP, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _i64, _vp]),
    "npi_sage_bwd_input": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp]),
    "npi_topk_score": (C.c_int, [_vp, _vp, _i32, _vp, _vp, _vp, _vp]),
    "npi_topk_select_workspace_bytes": (_i64, [_i32, _i32]),
    "npi_topk_select": (C.c_int, [_vp, _vp, _vp, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp]),
    "npi_pool_gate_readout_workspace_bytes": (_i64, [_i32]),
    "npi_pool_gate_readout": (C.c_int, [_vp, _vp, _vp, _vp, _i32, _vp, _vp, _i32, _vp, _vp, _i64, _i32, _vp]),
    "npi_filter_adj_workspace_bytes": (_i64, [_i32]),
    "npi_filter_adj": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _i64, _vp, _vp, _i64, _vp]),
    "npi_hub_rows_reset": (C.c_int, [_vp, _vp]),
    "npi_pool_bwd_workspace_bytes": (_i64, []),
    "npi_pool_bwd": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _vp, _i32, _vp, _vp, _vp, _vp, _i64, _i32, _vp]),
    "npi_filter_edges_coo_workspace_bytes": (_i64, [_i64]),
    "npi_filter_edges_coo": (C.c_int, [_vp, _i64, _vp, _vp, _vp, _vp, _i64, _vp]),
    "npi_readout_bwd": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _i32, _i32, _vp, _vp]),
    "npi_gemm_nn": (C.c_int, [_vp, _i32, _vp, _i32, _i32, _vp, _i32, _vp, _vp]),
    "npi_gemm_nn_tc": (C.c_int, [_vp, _i32, _vp, _i32, _i32, _vp, _i32, _vp, _i32, _vp]),
    "npi_gemm_tn_tc_workspace_bytes": (_i64, []),
    "npi_gemm_tn_tc": (C.c_int, [_vp, _i32, _i32, _vp, _vp, _i32, _vp, _i32, _vp, _i32, _vp, _i64, _vp]),
    "npi_gemm_tn_workspace_bytes": (_i64, [_i32]),
    "npi_gemm_tn": (C.c_int, [_vp, _i32, _vp, _vp, _i32, _i32, _vp, _i32, _vp, _vp, _i64, _vp]),
    "npi_hub_rows_bytes": (_i64, [_i64]),
    "npi_hub_rows_build": (C.c_int, [_vp, _vp, _i32, _i64, _vp, _i64, _vp, _vp, _vp, _vp, _vp]),
    "npi_debug_stamp": (C.c_int, [_vp, _i32, _vp]),
    "npi_table_grad_workspace_bytes": (_i64, [_i32]),
    "npi_table_grad": (C.c_int, [_vp, _i32, _i32, _vp, _i32, _vp, _i32, _vp, _vp, _i64, _vp]),
    "npi_ctx_workspace_bytes": (_i64, [_i32]),
    "npi_ctx_build": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _i64, _vp]),
    "npi_sort_workspace_bytes": (_i64, [_i64]),
    "npi_sort_passes": (_i32, [_i32]),
    "npi_sort_pairs_u32": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _i32, _vp, _i64, _vp]),
    "npi_ctx_index_workspace_bytes": (_i64, [_i32, _i64]),
    "npi_ctx_class_result_in_b": (_i32, [_i32]),
    "npi_ctx_index_build": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i32, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp]),
    "npi_ctx_class_pack": (C.c_int, [_vp, _vp, _i32, _vp, _vp, _vp, _i32, _vp, _vp]),
    "npi_ctx_scatter_max": (C.c_int, [_vp, _vp, _i32, _vp, _vp]),
    "npi_ctx_finish_partials": (_i32, []),
    "npi_ctx_finish": (C.c_int, [_vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _i64, _vp]),
    "npi_csr_gather_sum": (C.c_int, [_vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp]),
    "npi_entry_pack_virt": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i32, _i32, _i64, _vp, _vp]),
    "npi_entry_pack_sel": (C.c_int, [_vp, _vp, _vp, _vp, _i32, _i64, _vp, _vp]),
    "npi_sage_aggregate_fwd": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _vp]),
    "npi_sage_aggregate_bwd": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp]),
    "npi_gid_index_workspace_bytes": (_i64, [_i32, _i32]),
    "npi_gid_index_build": (C.c_int, [_vp, _vp, _i32, _i32, _vp, _vp, _vp, _i64, _vp]),
    "npi_gid_reduce_partials": (_i32, []),
    "npi_gid_reduce": (C.c_int, [_vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp]),
    "npi_head_fwd": (C.c_int, [_vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _vp, _u64, _vp, _vp, _i32, _vp, _f32,
                               _vp, _vp, _vp, _vp, _vp, _i32, _vp]),
    "npi_head_bwd_workspace_bytes": (_i64, [_i32]),
    "npi_head_fwd_delta": (C.c_int, [_vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _vp, _u64, _vp, _vp, _i32, _vp, _f32,
                                     _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp]),
    "npi_head_bwd": (C.c_int, [_vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _f32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                               _vp, _i64, _i32, _vp]),
    "npi_adam_l2_step": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _vp, _vp, _f32, _f32, _f32, _f32, _f32, _vp]),
    "npi_confusion_counts": (C.c_int, [_vp, _vp, _i32, _f32, _vp, _vp]),
    "npi_rank_workspace_bytes": (_i64, [_i64]),
    "npi_rank_curve": (C.c_int, [_vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp]),
    "npi_group_topk_workspace_bytes": (_i64, [_i64, _i32]),
    "npi_group_topk": (C.c_int, [_vp, _vp, _i64, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _i64, _vp]),
    "npi_group_rank_workspace_bytes": (_i64, [_i64, _i32]),
    "npi_group_rank": (C.c_int, [_vp, _vp, _vp, _i64, _i32, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp]),
    "npi_input_attribution_workspace_bytes": (_i64, [_i32, _i32, _i32]),
    "npi_input_attribution": (C.c_int, [_vp, _vp, _vp, _vp, _i32, _i32, _vp, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _i64, _vp]),
    "npi_scalar_axpy": (C.c_int, [_vp, _vp, _f32, _vp]),
    "npi_peer_header_bytes": (_i64, []),
    "npi_peer_alloc": (C.c_int, [_i64, C.POINTER(_vp), C.c_char_p]),
    "npi_peer_open": (C.c_int, [C.c_char_p, C.POINTER(_vp)]),
    "npi_peer_close": (C.c_int, [_vp]),
    "npi_peer_free": (C.c_int, [_vp]),
    "npi_allreduce_adam_fused": (C.c_int, [C.POINTER(_vp), _i32, _i32, _vp, _vp, _vp, _i64, _vp, _vp, _vp, _f32, _f32, _f32, _f32,
                                           _f32, _i32, _i64, _i32, _vp]),
    "npi_peer_barrier": (C.c_int, [C.POINTER(_vp), _i32, _i32, _vp, _i32, _vp]),
    "npi_tiny_max_nodes": (_i32, []),
    "npi_tiny_partials_bytes": (_i64, [_i32]),
    "npi_tiny_transpose": (C.c_int, [_vp, _vp, _vp, _vp, _vp]),
    "npi_tiny_fwd": (C.c_int, [_TP, _vp]),
    "npi_tiny_bwd": (C.c_int, [_TP, _i32, _vp]),
    "npi_tiny_weight_grads_workspace_bytes": (_i64, [_i32]),
    "npi_tiny_weight_grads": (C.c_int, [_vp, _i32, _i32, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _i32, _vp,
                                        _vp, _vp, _vp, _i32, _vp, _vp, _i64, _vp]),
    "npi_n2v_etab_scan": (C.c_int, [_vp, _vp, _i32, _i64, _vp, _vp]),
    "npi_n2v_alias_tables": (C.c_int, [_vp, _vp, _vp, _i32, _i64, _f64, _f64, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _vp]),
    "npi_n2v_alias_from_probs": (C.c_int, [_vp, _i32, _vp, _vp, _vp, _vp]),
    "npi_n2v_walks": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i64, _i32, _u64, _u32, _vp, _vp, _vp]),
    "npi_n2v_vocab_count": (C.c_int, [_vp, _vp, _i64, _i32, _i32, _vp, _vp]),
    "npi_n2v_init_vectors": (C.c_int, [_vp, _i64, _i32, _u64, _vp]),
    "npi_n2v_skipgram": (C.c_int, [_vp, _vp, _vp, _i64, _i32, _i64, _vp, _vp, _i32, _i32, _vp, _vp, _vp, _i32, _i32,
                                   _f64, _f64, _u64, _u32, _i32, _i32, _vp]),
}

_lib = None


def load():
    """Load libnpi.so (raises if it has not been built)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NPIError("libnpi.so is missing at %s -- build it with `python -m npi_gnn_b200.build` "
                           "(or __graft_entry__.build()); there is no CPU/PyTorch fallback" % LIB_PATH)
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)          # AttributeError if a declared symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def last_error():
    return load().npi_last_error().decode("utf-8", "replace")


# kernels launched by one call of each entry point (for the bench's gpu_launches claim)
KERNELS_PER_CALL = {
    "npi_csr_fold_mask": 1, "npi_khop_count": 1, "npi_khop_fill": 1, "npi_batch_prepare": 1, "npi_subgraph_coo": 1,
    "npi_gather_features": 1, "npi_coo_to_csr": 6, "npi_edge_symmetry_sums": 1, "npi_sage_fwd": 1, "npi_sage_bwd_weight": 2,
    "npi_sage_bwd_input": 1, "npi_topk_score": 1, "npi_topk_select": 1, "npi_pool_gate_readout": 2,
    "npi_filter_adj": 3, "npi_pool_bwd": 2, "npi_gemm_nn": 1, "npi_gemm_nn_tc": 1, "npi_gemm_tn": 2, "npi_gemm_tn_tc": 2, "npi_gemm_tn_tc/wide": 4, "npi_sage_aggregate_fwd": 1,
    "npi_sage_aggregate_bwd": 1, "npi_entry_pack_virt": 1, "npi_entry_pack_sel": 1, "npi_hub_rows_build": 1, "npi_hub_rows_build/order": 2, "npi_gid_index_build": 4, "npi_gid_reduce": 1,
    "npi_filter_edges_coo": 3, "npi_readout_bwd": 1, "npi_head_fwd": 2, "npi_head_bwd": 2, "npi_head_bwd/phase": 1, "npi_pool_bwd/phase": 1, "npi_head_fwd/phase": 1, "npi_pool_gate_readout/phase": 1, "npi_adam_l2_step": 1,
    "npi_confusion_counts": 1, "npi_rank_curve": 17, "npi_group_topk": 9, "npi_group_topk/1pass": 6, "npi_group_topk/3pass": 12,
    "npi_group_rank": 27, "npi_group_rank/1pass": 24, "npi_group_rank/3pass": 30,
    "npi_input_attribution": 3, "npi_input_attribution/no_rows": 2,
    "npi_debug_stamp": 1, "npi_hub_rows_reset": 0, "npi_table_grad": 2, "npi_ctx_build": 2, "npi_sort_pairs_u32": 6, "npi_ctx_index_build": 22, "npi_ctx_class_pack": 1,
    "npi_ctx_scatter_max": 1, "npi_ctx_finish": 1, "npi_csr_gather_sum": 1, "npi_allreduce_adam_fused": 1, "npi_scalar_axpy": 1, "npi_peer_barrier": 1,
    "npi_head_fwd_delta": 1, "npi_tiny_transpose": 1, "npi_tiny_fwd": 1, "npi_tiny_bwd": 2, "npi_tiny_bwd/phase": 1, "npi_tiny_weight_grads": 1,
    "npi_n2v_etab_scan": 1, "npi_n2v_alias_tables": 1, "npi_n2v_alias_from_probs": 1, "npi_n2v_walks": 1,
    "npi_n2v_vocab_count": 1, "npi_n2v_init_vectors": 1, "npi_n2v_skipgram": 1,
}
CALL_COUNTS = {}
TIMER = None        # optional: object with .begin(name) / .end(name) bracketing every call (bench.py)


def launches_since(snapshot=None):
    """Kernel launches issued through the C ABI (optionally since a snapshot of CALL_COUNTS)."""
    tot = 0
    for k, v in CALL_COUNTS.items():
        d = v - (snapshot.get(k, 0) if snapshot else 0)
        tot += d * KERNELS_PER_CALL.get(k, 0)
    return tot


def call(name, *args, count_as=None):
    """Call an int-returning entry point and raise NPIError on a non-zero status.  ``count_as``:
    key of KERNELS_PER_CALL to book the launches under (calls that run one phase of an entry point)."""
    fn = getattr(load(), name)
    t = TIMER
    if t is not None:
        t.begin(name)
    rc = fn(*args)
    if t is not None:
        t.end(name)
    ck = count_as or name
    CALL_COUNTS[ck] = CALL_COUNTS.get(ck, 0) + 1
    if rc != 0:
        raise NPIError("%s failed (rc=%d): %s" % (name, rc, last_error()))


def query(name, *args):
    return getattr(load(), name)(*args)


def ptr(t):
    """Device (or host) pointer of a tensor / None."""
    if t is None:
        return None
    return C.c_void_p(t.data_ptr())


def stream_ptr(device=None):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise NPIError("npi_gnn_b200 kernels need CUDA tensors; got a %s tensor (there is no CPU fallback)" % t.device)


def features_dense(x):
    f = Features()
    f.x = x.data_ptr(); f.ldx = x.stride(0); f.table = None; f.ld = 0; f.gid = None; f.dist = None
    f.F = x.shape[1]
    return f


def features_virtual(table, gid, dist, F):
    f = Features()
    f.x = None; f.ldx = 0; f.table = table.data_ptr(); f.ld = table.stride(0)
    f.gid = gid.data_ptr(); f.dist = dist.data_ptr(); f.F = F
    return f
