"""Tensor-level wrappers over the libnpi C ABI (no autograd, no allocation policy).

Every function takes CUDA tensors, enqueues kernels on the current stream and returns
immediately.  Sizes that depend on data are passed as ``(n_dev, n_host)``: a 1-element int32
CUDA tensor (or None) plus a host upper bound.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib as L

H = 128
_i32, _i64, _f32, _u64 = C.c_int32, C.c_int64, C.c_float, C.c_uint64


def _s():
    return L.stream_ptr()


def sm_count():
    out = _i32(0)
    L.call("npi_sm_count", C.byref(out))
    return out.value


# ----------------------------------------------------------------------------- graph prep (host)
def csr_build_host(edges, num_nodes):
    """edges: int32 numpy [E,2] (rna, protein) in interaction_list order.  Returns numpy
    rowptr[V+1], col[2E'], eid[2E'], edge_id[E] (-1 = duplicate), E'."""
    edges = np.ascontiguousarray(edges, dtype=np.int32)
    E = edges.shape[0]
    rowptr = np.zeros(num_nodes + 1, dtype=np.int32)
    col = np.zeros(2 * E, dtype=np.int32)
    eid = np.zeros(2 * E, dtype=np.int32)
    edge_id = np.zeros(E, dtype=np.int32)
    nu = _i64(0)
    L.call("npi_csr_build_host", edges.ctypes.data_as(C.c_void_p), _i64(E), _i32(num_nodes),
           rowptr.ctypes.data_as(C.c_void_p), col.ctypes.data_as(C.c_void_p), eid.ctypes.data_as(C.c_void_p),
           edge_id.ctypes.data_as(C.c_void_p), C.byref(nu))
    nu = nu.value
    return rowptr, col[:2 * nu].copy(), eid[:2 * nu].copy(), edge_id, nu


# ----------------------------------------------------------------------------- extraction
def khop_workspace_bytes(V, num_ctas):
    return L.query("npi_khop_workspace_bytes", _i32(V), _i32(num_ctas))


def csr_fold_mask(col, eid, mask, colm):
    L.call("npi_csr_fold_mask", L.ptr(col), L.ptr(eid), L.ptr(mask), _i64(col.numel()), L.ptr(colm), _s())


def khop_count(g, pairs, h, n_out, e_out, ws, num_ctas):
    L.call("npi_khop_count", L.ptr(g.rowptr), L.ptr(g.colm), _i32(g.num_nodes),
           L.ptr(pairs), _i32(pairs.shape[0]), _i32(h), L.ptr(n_out), L.ptr(e_out),
           L.ptr(ws), _i64(ws.numel() * ws.element_size()), _i32(num_ctas), _s())


def khop_fill(g, pairs, num_pairs, h, max_graph_nodes, graph_ptr, edge_ptr, gid, dist, sub_rowptr, sub_col, ws, num_ctas,
              overflow=None):
    L.call("npi_khop_fill", L.ptr(g.rowptr), L.ptr(g.colm), _i32(g.num_nodes),
           L.ptr(pairs), _i32(num_pairs), _i32(h), _i32(max_graph_nodes), L.ptr(graph_ptr), L.ptr(edge_ptr),
           L.ptr(gid), L.ptr(dist), L.ptr(sub_rowptr), L.ptr(sub_col),
           _i32(min(gid.numel(), dist.numel(), sub_rowptr.numel() - 1)), _i32(sub_col.numel()), L.ptr(overflow),
           L.ptr(ws), _i64(ws.numel() * ws.element_size()), _i32(num_ctas), _s())


def batch_prepare(pair_index, first, B, pairs_all, y_all, n_all, e_all, ratio, pairs_b, y_b, graph_ptrs, edge_ptr, sizes):
    L.call("npi_batch_prepare", L.ptr(pair_index), _i32(first), _i32(B), L.ptr(pairs_all), L.ptr(y_all),
           L.ptr(n_all), L.ptr(e_all), _f32(ratio), L.ptr(pairs_b), L.ptr(y_b), L.ptr(graph_ptrs), L.ptr(edge_ptr),
           L.ptr(sizes), _s())


def subgraph_coo(graph_ptr, edge_ptr, B, h, gid, dist, is_rna, sub_rowptr, sub_col, edge_index, local_ids):
    L.call("npi_subgraph_coo", L.ptr(graph_ptr), L.ptr(edge_ptr), _i32(B), _i32(h), L.ptr(gid), L.ptr(dist),
           L.ptr(is_rna), L.ptr(sub_rowptr), L.ptr(sub_col), L.ptr(edge_index), _i64(edge_index.shape[1]),
           _i32(1 if local_ids else 0), _s())


def gather_features(feat, n_dev, n_host, x_out):
    L.call("npi_gather_features", C.byref(feat), L.ptr(n_dev), _i32(n_host), L.ptr(x_out), _s())


def coo_to_csr(edge_index, N, rowptr_out, col_out):
    E = edge_index.shape[1]
    nbytes = L.query("npi_coo_to_csr_workspace_bytes", _i32(N), _i64(E))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=edge_index.device)
    ei = edge_index.contiguous()
    L.call("npi_coo_to_csr", L.ptr(ei), _i64(E), _i32(N), L.ptr(rowptr_out), L.ptr(col_out), L.ptr(ws), _i64(nbytes), _s())


def edge_symmetry_sums(edge_index):
    """uint64[2] fingerprints of the edge multiset and of its transpose (equal <=> symmetric)."""
    ei = edge_index.contiguous()
    out = torch.empty(2, dtype=torch.int64, device=edge_index.device)
    L.call("npi_edge_symmetry_sums", L.ptr(ei), _i64(ei.shape[1]), L.ptr(out), _s())
    return out


# ----------------------------------------------------------------------------- SAGEConv
def sage_fwd(feat, rowptr, col, n_dev, n_host, W, b, relu, pool_w, h_out, z_out, s_out):
    L.call("npi_sage_fwd", C.byref(feat), L.ptr(rowptr), L.ptr(col), L.ptr(n_dev), _i32(n_host), L.ptr(W), L.ptr(b),
           _i32(1 if relu else 0), L.ptr(pool_w), L.ptr(h_out), L.ptr(z_out), L.ptr(s_out), _s())


def sage_bwd_weight_workspace_bytes(F):
    return L.query("npi_sage_bwd_weight_workspace_bytes", _i32(F))


def sage_bwd_weight(feat, rowptr, col, sel, nsel_dev, nsel_host, dpre, dW, db, ws):
    L.call("npi_sage_bwd_weight", C.byref(feat), L.ptr(rowptr), L.ptr(col), L.ptr(sel), L.ptr(nsel_dev), _i32(nsel_host),
           L.ptr(dpre), L.ptr(dW), L.ptr(db), L.ptr(ws), _i64(ws.numel() * ws.element_size()), _s())


def sage_bwd_input(dpre, new_id, rowptr, col, n_dev, n_host, W, dx):
    L.call("npi_sage_bwd_input", L.ptr(dpre), L.ptr(new_id), L.ptr(rowptr), L.ptr(col), L.ptr(n_dev), _i32(n_host),
           L.ptr(W), L.ptr(dx), _s())


# ----------------------------------------------------------------------------- TopKPooling / readout
def topk_score(h, n_dev, n_host, pool_w, z_out, s_out):
    L.call("npi_topk_score", L.ptr(h), L.ptr(n_dev), _i32(n_host), L.ptr(pool_w), L.ptr(z_out), L.ptr(s_out), _s())


def topk_select_workspace_bytes(B, max_graph_nodes):
    return L.query("npi_topk_select_workspace_bytes", _i32(B), _i32(max_graph_nodes))


def topk_select(s, gptr_in, gptr_out, B, max_graph_nodes, perm, new_id, batch_out, ws, row_map=None, perm_src=None):
    """row_map/perm_src: scores are read through row_map (rows sharing a layer-1 context, ctx_build) and
    perm_src[r] = row_map[perm[r]] is emitted next to perm."""
    L.call("npi_topk_select", L.ptr(s), L.ptr(gptr_in), L.ptr(gptr_out), _i32(B), _i32(max_graph_nodes), L.ptr(perm),
           L.ptr(new_id), L.ptr(batch_out), L.ptr(row_map), L.ptr(perm_src), L.ptr(ws), _i64(ws.numel() * ws.element_size()), _s())


def pool_gate_readout_workspace_bytes(B):
    return L.query("npi_pool_gate_readout_workspace_bytes", _i32(B))


def pool_gate_readout(h, s, perm, gptr_out, B, xp, readout, accumulate, argmax, ws=None, phases=0):
    """phases 0: everything; 1: gating + per-range partials (in ws); 2: readout / argmax from those partials."""
    if ws is None:
        if phases:
            raise L.NPIError("pool_gate_readout: the two phases share a workspace, pass ws")
        ws = torch.empty(pool_gate_readout_workspace_bytes(B), dtype=torch.uint8, device=h.device)
    L.call("npi_pool_gate_readout", L.ptr(h), L.ptr(s), L.ptr(perm), L.ptr(gptr_out), _i32(B), L.ptr(xp), L.ptr(readout),
           _i32(1 if accumulate else 0), L.ptr(argmax), L.ptr(ws), _i64(ws.numel() * ws.element_size()), _i32(phases), _s(),
           count_as=None if phases == 0 else "npi_pool_gate_readout/phase")


def filter_adj_workspace_bytes(n_new_max):
    return L.query("npi_filter_adj_workspace_bytes", _i32(n_new_max))


def filter_adj(rowptr, col, perm, new_id, nnew_dev, nnew_host, rowptr_out, col_out, ws, hubq=None, hub_e_max=0, row_order=None):
    """hubq / row_order: hub queue and binned row order of the NEW CSR built on the way (header zeroed by hub_rows_reset)."""
    L.call("npi_filter_adj", L.ptr(rowptr), L.ptr(col), L.ptr(perm), L.ptr(new_id), L.ptr(nnew_dev), _i32(nnew_host),
           L.ptr(rowptr_out), L.ptr(col_out), L.ptr(hubq), _i64(hub_e_max), L.ptr(row_order),
           L.ptr(ws), _i64(ws.numel() * ws.element_size()), _s())


def hub_rows_reset(hubq):
    L.call("npi_hub_rows_reset", L.ptr(hubq), _s())


def pool_bwd_workspace_bytes():
    return L.query("npi_pool_bwd_workspace_bytes")


def pool_bwd(d_xp, d_readout, h, z, s, perm, batch_out, argmax, gptr_out, nnew_dev, nnew_host, B, pool_w, relu,
             dpre, d_pool_w, ws, d_bias=None, phases=0):
    """phases 0: everything; 1: dpre + per-CTA partials (in ws); 2: d_pool_w / d_bias from those partials."""
    L.call("npi_pool_bwd", L.ptr(d_xp), L.ptr(d_readout), L.ptr(h), L.ptr(z), L.ptr(s), L.ptr(perm), L.ptr(batch_out),
           L.ptr(argmax), L.ptr(gptr_out), L.ptr(nnew_dev), _i32(nnew_host), _i32(B), L.ptr(pool_w),
           _i32(1 if relu else 0), L.ptr(dpre), L.ptr(d_pool_w), L.ptr(d_bias), L.ptr(ws),
           _i64(ws.numel() * ws.element_size()), _i32(phases), _s(),
           count_as=None if phases == 0 else "npi_pool_bwd/phase")


# ----------------------------------------------------------------------------- decomposed SAGEConv
def gemm_nn(A, m_dev, m_host, K, B, transB, C):
    L.call("npi_gemm_nn", L.ptr(A), _i32(A.stride(0)), L.ptr(m_dev), _i32(m_host), _i32(K), L.ptr(B),
           _i32(1 if transB else 0), L.ptr(C), _s())


def gemm_nn_tc(A, m_dev, m_host, K, B, transB, C, single_pass=False):
    L.call("npi_gemm_nn_tc", L.ptr(A), _i32(A.stride(0)), L.ptr(m_dev), _i32(m_host), _i32(K), L.ptr(B),
           _i32(1 if transB else 0), L.ptr(C), _i32(int(single_pass)), _s())


def gemm_tn_workspace_bytes(K):
    return L.query("npi_gemm_tn_workspace_bytes", _i32(K))


def gemm_tn(A, D, m_dev, m_host, K, row0_partials, out, ws):
    R = 0 if row0_partials is None else row0_partials.shape[0]
    L.call("npi_gemm_tn", L.ptr(A), _i32(A.stride(0)), L.ptr(D), L.ptr(m_dev), _i32(m_host), _i32(K),
           L.ptr(row0_partials), _i32(R), L.ptr(out), L.ptr(ws), _i64(ws.numel() * ws.element_size()), _s())


def gemm_tn_tc_workspace_bytes():
    return L.query("npi_gemm_tn_tc_workspace_bytes")


def gemm_tn_tc(A, D, m_dev, m_host, row0_partials, out, ws, single_pass=0, K=128):
    """out[K,128] = A[:, :K]^T . D; K > 128 runs one pass per 128 columns (columns K..ld-1 of A must be zero)."""
    R = 0 if row0_partials is None else row0_partials.shape[0]
    L.call("npi_gemm_tn_tc", L.ptr(A), _i32(A.stride(0)), _i32(K), L.ptr(D), L.ptr(m_dev), _i32(m_host),
           L.ptr(row0_partials), _i32(R), L.ptr(out), _i32(int(single_pass)), L.ptr(ws),
           _i64(ws.numel() * ws.element_size()), _s(), count_as="npi_gemm_tn_tc/wide" if K > 128 else None)


def table_grad_workspace_bytes(K):
    return L.query("npi_table_grad_workspace_bytes", _i32(K))


def table_grad(table, G, V, row0_partials, out, ws, K):
    """out[K,128] = table[:V, :K]^T . G[:V] (+ row0 partials on row 0): small-table layer-1 weight gradient, two launches."""
    R = 0 if row0_partials is None else row0_partials.shape[0]
    L.call("npi_table_grad", L.ptr(table), _i32(table.stride(0)), _i32(K), L.ptr(G), _i32(V), L.ptr(row0_partials), _i32(R),
           L.ptr(out), L.ptr(ws), _i64(ws.numel() * ws.element_size()), _s())


def hub_rows_bytes(e_max):
    return L.query("npi_hub_rows_bytes", _i64(e_max))


def ctx_workspace_bytes(n_max):
    return L.query("npi_ctx_workspace_bytes", _i32(n_max))


def ctx_build(rowptr, packed, gid, dist, n_dev, n_host, rep_of, stats, ws, label_sum=None):
    """rep_of[i] = first row of the batch with row i's layer-1 context (csrc/ctx.cu); packed = entry_pack_virt."""
    L.call("npi_ctx_build", L.ptr(rowptr), L.ptr(packed), L.ptr(gid), L.ptr(dist), L.ptr(n_dev), _i32(n_host), L.ptr(rep_of),
           L.ptr(stats), L.ptr(label_sum), L.ptr(ws), _i64(ws.numel() * ws.element_size()), _s())


def sort_workspace_bytes(n_max):
    return L.query("npi_sort_workspace_bytes", _i64(n_max))


def sort_pairs_u32(keys_a, vals_a, keys_b, vals_b, n, key_bits, ws):
    """Stable LSD radix sort of (uint32-as-int32 key, int32 value) pairs; returns the (keys, vals) pair holding the result."""
    L.call("npi_sort_pairs_u32", L.ptr(keys_a), L.ptr(vals_a), L.ptr(keys_b), L.ptr(vals_b), _i64(n), _i32(key_bits),
           L.ptr(ws), _i64(ws.numel() * ws.element_size()), _s())
    return (keys_b, vals_b) if L.query("npi_sort_passes", _i32(key_bits)) & 1 else (keys_a, vals_a)


def ctx_index_workspace_bytes(n_max, e_max):
    return L.query("npi_ctx_index_workspace_bytes", _i32(n_max), _i64(e_max))


def ctx_class_result_in_b(n_max):
    return bool(L.query("npi_ctx_class_result_in_b", _i32(n_max)))


def ctx_index_build(rowptr, packed, gid, rep_of, n_dev, n_host, e_max, V, ck_a, cr_a, ck_b, cr_b, class_ptr2, class_rep, n_ctx,
                    inv_ptr, inv_sel, ws):
    L.call("npi_ctx_index_build", L.ptr(rowptr), L.ptr(packed), L.ptr(gid), L.ptr(rep_of), L.ptr(n_dev), _i32(n_host), _i64(e_max),
           _i32(V), L.ptr(ck_a), L.ptr(cr_a), L.ptr(ck_b), L.ptr(cr_b), L.ptr(class_ptr2), L.ptr(class_rep), L.ptr(n_ctx),
           L.ptr(inv_ptr), L.ptr(inv_sel), L.ptr(ws), _i64(ws.numel() * ws.element_size()), _s())


def ctx_class_pack(class_rows, n_dev, n_host, new_id, batch_out, gptr_out, readout_row0, class_sel):
    L.call("npi_ctx_class_pack", L.ptr(class_rows), L.ptr(n_dev), _i32(n_host), L.ptr(new_id), L.ptr(batch_out), L.ptr(gptr_out),
           _i32(readout_row0), L.ptr(class_sel), _s())


def ctx_scatter_max(d_readout, argmax, B, d_xp):
    L.call("npi_ctx_scatter_max", L.ptr(d_readout), L.ptr(argmax), _i32(B), L.ptr(d_xp), _s())


def ctx_finish_partials():
    return L.query("npi_ctx_finish_partials")


def ctx_finish(XU, class_rep, n_ctx_dev, n_ctx_host, h, z, s, pool_w, relu, rowptr, label_sum, label_partials, ws):
    L.call("npi_ctx_finish", L.ptr(XU), L.ptr(class_rep), L.ptr(n_ctx_dev), _i32(n_ctx_host), L.ptr(h), L.ptr(z), L.ptr(s),
           L.ptr(pool_w), _i32(1 if relu else 0), L.ptr(rowptr), L.ptr(label_sum), L.ptr(label_partials), L.ptr(ws),
           _i64(ws.numel() * ws.element_size()), _s())


def csr_gather_sum(src, rowptr, packed, n_rows, out, hubq, row_order):
    """out[r] = sum over the packed entries {row, weight} of CSR row r of src[row] * weight (no self term)."""
    L.call("npi_csr_gather_sum", L.ptr(src), L.ptr(rowptr), L.ptr(packed), _i32(n_rows), L.ptr(out), L.ptr(hubq), L.ptr(row_order), _s())


def hub_rows_build(rowptr, n_dev, n_host, e_max, hubq, gid=None, dist=None, row_order=None, keep=None):
    """List the hub-row segments of a CSR of at most e_max entries into ``hubq`` (uint8 buffer of
    hub_rows_bytes(e_max), any contents: the header and the counters of every listed segment are
    written here); with ``row_order`` (int32 [>= n_host, 4], 16-byte aligned) also the rows of at most
    16 entries binned by length class (what the pipelined aggregation kernels walk).  Hub rows have
    more than 16 entries and are cut into segments of 32."""
    L.call("npi_hub_rows_build", L.ptr(rowptr), L.ptr(n_dev), _i32(n_host), _i64(e_max), L.ptr(hubq),
           _i64(hubq.numel() * hubq.element_size()), L.ptr(gid), L.ptr(dist), L.ptr(row_order), L.ptr(keep), _s(),
           count_as=None if row_order is None else "npi_hub_rows_build/order")
    return hubq


def _hub_queue(hubq, rowptr, col, n_dev, n_host):
    """The queue the caller built when it produced the CSR, or a temporary one built here."""
    if hubq is None:
        e_max = col.numel()
        hubq = hub_rows_build(rowptr, n_dev, n_host, e_max,
                              torch.empty(hub_rows_bytes(e_max), dtype=torch.uint8, device=rowptr.device))
    return hubq


def entry_pack_virt(rowptr, col, gid, dist, n_dev, n_host, V, packed):
    """packed[k] = gid[col[k]] | dist[col[k]] << 29 for every entry of the CSR (int32 [>= E])."""
    L.call("npi_entry_pack_virt", L.ptr(rowptr), L.ptr(col), L.ptr(gid), L.ptr(dist), L.ptr(n_dev), _i32(n_host), _i32(V),
           _i64(packed.numel()), L.ptr(packed), _s())
    return packed


def entry_pack_sel(rowptr, col, new_id, n_dev, n_host, packed):
    """packed[k] = (new_id[col[k]], bits of 1/(deg_col+1) or 0) for every entry of the CSR (int32 [>= E, 2])."""
    L.call("npi_entry_pack_sel", L.ptr(rowptr), L.ptr(col), L.ptr(new_id), L.ptr(n_dev), _i32(n_host),
           _i64(packed.numel() // 2), L.ptr(packed), _s())
    return packed


def sage_aggregate_fwd(Y, gid, dist, w0, rowptr, col, n_dev, n_host, bias, relu, pool_w, h, z, s, hubq=None, packed=None,
                       row_order=None, pipelined=False):
    """``pipelined``: rows in the length-class order ``row_order`` (hub_rows_build of this CSR), software
    pipelined; on the virtual input layer it also needs ``packed`` (entry_pack_virt of this CSR)."""
    hubq = _hub_queue(hubq, rowptr, col, n_dev, n_host)
    if pipelined and (row_order is None or (gid is not None and packed is None)):
        raise L.NPIError("sage_aggregate_fwd: the pipelined kernel needs row_order (ops.hub_rows_build) and, on the "
                         "virtual layer, packed entries (ops.entry_pack_virt)")
    L.call("npi_sage_aggregate_fwd", L.ptr(Y), L.ptr(gid), L.ptr(dist), L.ptr(w0), L.ptr(rowptr), L.ptr(col),
           L.ptr(n_dev), _i32(n_host), L.ptr(bias), _i32(1 if relu else 0), L.ptr(pool_w), L.ptr(h), L.ptr(z), L.ptr(s),
           L.ptr(hubq), L.ptr(packed), L.ptr(row_order), _i32(1 if pipelined else 0), _s())


def sage_aggregate_bwd(dpre, new_id, rowptr, col, n_dev, n_host, dxa, hubq=None, packed=None, row_order=None):
    """``packed`` (entry_pack_sel of this CSR and new_id) + ``row_order`` select the pipelined kernel."""
    hubq = _hub_queue(hubq, rowptr, col, n_dev, n_host)
    if packed is not None and row_order is None:
        raise L.NPIError("sage_aggregate_bwd: the pipelined kernel needs row_order (ops.hub_rows_build)")
    L.call("npi_sage_aggregate_bwd", L.ptr(dpre), L.ptr(new_id), L.ptr(rowptr), L.ptr(col), L.ptr(n_dev), _i32(n_host),
           L.ptr(dxa), L.ptr(hubq), L.ptr(packed), L.ptr(row_order), _s())


def gid_index_workspace_bytes(V, n_max):
    return L.query("npi_gid_index_workspace_bytes", _i32(V), _i32(n_max))


def gid_index_build(gid, n_dev, n_host, V, occ_ptr, occ_node, ws):
    L.call("npi_gid_index_build", L.ptr(gid), L.ptr(n_dev), _i32(n_host), _i32(V), L.ptr(occ_ptr), L.ptr(occ_node),
           L.ptr(ws), _i64(ws.numel() * ws.element_size()), _s())


def gid_reduce_partials():
    return L.query("npi_gid_reduce_partials")


def gid_reduce(dxa, dist, occ_ptr, occ_node, V, G, label_partials):
    L.call("npi_gid_reduce", L.ptr(dxa), L.ptr(dist), L.ptr(occ_ptr), L.ptr(occ_node), _i32(V), L.ptr(G),
           L.ptr(label_partials), _s())


# ----------------------------------------------------------------------------- small-subgraph path (csrc/tiny.cu)
def tiny_max_nodes():
    return L.query("npi_tiny_max_nodes")


def tiny_partials_bytes(B):
    return L.query("npi_tiny_partials_bytes", _i32(B))


def tiny_transpose(w2, w3, w2_t, w3_t):
    L.call("npi_tiny_transpose", L.ptr(w2), L.ptr(w3), L.ptr(w2_t), L.ptr(w3_t), _s())


def tiny_args(**kw):
    """npi_tiny_args_t from keyword arguments: scalars, tensors, or lists of tensors for the per-layer arrays."""
    a = L.TinyArgs()
    for name, val in kw.items():
        if isinstance(val, (list, tuple)):
            arr = getattr(a, name)
            if len(val) != len(arr):
                raise L.NPIError("tiny_args: %s takes %d entries" % (name, len(arr)))
            for i, t in enumerate(val):
                L.require_cuda(t)
                arr[i] = None if t is None else t.data_ptr()
        elif isinstance(val, int):
            setattr(a, name, val)
        else:
            L.require_cuda(val)
            setattr(a, name, None if val is None else val.data_ptr())
    return a


def tiny_weight_grads_workspace(F, device):
    """Zeroed workspace of tiny_weight_grads (its ticket counters must start at zero; every call leaves them zero)."""
    return torch.zeros(L.query("npi_tiny_weight_grads_workspace_bytes", _i32(F)), dtype=torch.uint8, device=device)


def tiny_weight_grads(table, F, gid, dist, dxa1, n0_dev, n0_host, d_w1, ws, x1=None, dxa2=None, n1_dev=None, n1_host=0, d_w2=None,
                      x2=None, dxa3=None, n2_dev=None, n2_host=0, d_w3=None):
    """d conv1.weight = sum_j [dist_j | table[gid_j][1:F]]^T . dxa1_j over the batch rows and (optionally) the dense
    d conv2.weight = x1^T . dxa2, d conv3.weight = x2^T . dxa3 -- one launch."""
    for t in (x1, x2):
        if t is not None and (t.stride(0) != 128 or t.stride(1) != 1):
            raise L.NPIError("tiny_weight_grads: x1 / x2 must be contiguous [n,128]")
    L.call("npi_tiny_weight_grads", L.ptr(table), _i32(table.stride(0)), _i32(F), L.ptr(gid), L.ptr(dist), L.ptr(dxa1),
           L.ptr(n0_dev), _i32(n0_host), L.ptr(d_w1),
           L.ptr(x1), L.ptr(dxa2), L.ptr(n1_dev), _i32(n1_host), L.ptr(d_w2),
           L.ptr(x2), L.ptr(dxa3), L.ptr(n2_dev), _i32(n2_host), L.ptr(d_w3),
           L.ptr(ws), _i64(ws.numel() * ws.element_size()), _s())


def tiny_fwd(args):
    L.call("npi_tiny_fwd", C.byref(args), _s())


def tiny_bwd(args, phases=0):
    """phases 0: everything; 1: the per-subgraph backward kernel; 2: d_pool_w / d_bias from its partials."""
    L.call("npi_tiny_bwd", C.byref(args), _i32(phases), _s(), count_as=None if phases == 0 else "npi_tiny_bwd/phase")


# ----------------------------------------------------------------------------- head / loss / optimizer
def head_fwd(readout, B, w1, b1, w2, b2, w3, b3, training, drop_mask_in, seed, step_dev, sample_ids, sample_id_base,
             y, loss_scale, a1, drop_mask_out, a2, logp, loss_out, phases=0):
    """phases 0: everything; 1: the MLP; 2: the scalar loss from logp."""
    with_loss = y is not None and loss_out is not None
    L.call("npi_head_fwd", L.ptr(readout), _i32(B), L.ptr(w1), L.ptr(b1), L.ptr(w2), L.ptr(b2), L.ptr(w3), L.ptr(b3),
           _i32(1 if training else 0), L.ptr(drop_mask_in), _u64(seed), L.ptr(step_dev), L.ptr(sample_ids),
           _i32(sample_id_base), L.ptr(y), _f32(loss_scale), L.ptr(a1), L.ptr(drop_mask_out), L.ptr(a2), L.ptr(logp),
           L.ptr(loss_out), _i32(phases), _s(),
           count_as="npi_head_fwd/phase" if (phases or not with_loss) else None)


def head_fwd_delta(readout, B, w1, b1, w2, b2, w3, b3, training, drop_mask_in, seed, step_dev, sample_ids, sample_id_base,
                   y, loss_scale, a1, drop_mask_out, a2, logp, d_readout, ws):
    """head_fwd(phases=1) + head_bwd(phases=1) of the mean-NLL loss in one launch (training step)."""
    L.call("npi_head_fwd_delta", L.ptr(readout), _i32(B), L.ptr(w1), L.ptr(b1), L.ptr(w2), L.ptr(b2), L.ptr(w3), L.ptr(b3),
           _i32(1 if training else 0), L.ptr(drop_mask_in), _u64(seed), L.ptr(step_dev), L.ptr(sample_ids),
           _i32(sample_id_base), L.ptr(y), _f32(loss_scale), L.ptr(a1), L.ptr(drop_mask_out), L.ptr(a2), L.ptr(logp),
           L.ptr(d_readout), L.ptr(ws), _i64(ws.numel() * ws.element_size()), _s())


def head_bwd_workspace_bytes(B):
    return L.query("npi_head_bwd_workspace_bytes", _i32(B))


def head_bwd(readout, B, w1, w2, w3, a1, drop_mask, a2, logp, y, loss_scale, d_logp, dw1, db1, dw2, db2, dw3, db3,
             d_readout, ws, phases=0):
    """phases 0: everything; 1: per-sample deltas + d_readout; 2: the weight gradients from those deltas."""
    L.call("npi_head_bwd", L.ptr(readout), _i32(B), L.ptr(w1), L.ptr(w2), L.ptr(w3), L.ptr(a1), L.ptr(drop_mask), L.ptr(a2),
           L.ptr(logp), L.ptr(y), _f32(loss_scale), L.ptr(d_logp), L.ptr(dw1), L.ptr(db1), L.ptr(dw2), L.ptr(db2),
           L.ptr(dw3), L.ptr(db3), L.ptr(d_readout), L.ptr(ws), _i64(ws.numel() * ws.element_size()), _i32(phases), _s(),
           count_as=None if phases == 0 else "npi_head_bwd/phase")


def adam_l2_step(params, grads, m, v, lr_dev, step_dev, beta1, beta2, eps, weight_decay, grad_scale):
    L.call("npi_adam_l2_step", L.ptr(params), L.ptr(grads), L.ptr(m), L.ptr(v), _i64(params.numel()), L.ptr(lr_dev),
           L.ptr(step_dev), _f32(beta1), _f32(beta2), _f32(eps), _f32(weight_decay), _f32(grad_scale), _s())


def confusion_counts(logp, y, B, threshold, counts):
    L.call("npi_confusion_counts", L.ptr(logp), L.ptr(y), _i32(B), _f32(threshold), L.ptr(counts), _s())


def rank_workspace_bytes(n_max):
    return L.query("npi_rank_workspace_bytes", _i64(n_max))


def rank_curve(scores, labels, summary, areas, status, ws, thresholds=None, tps=None, fps=None):
    """ROC / PR curve and areas of float32 ``scores`` against int32 ``labels`` (include/npi.h npi_rank_curve):
    summary int64[4] = {n_pos, n_neg, n_thresholds, twice_u}, areas float64[2] = {AP, trapezoidal PR AUC},
    status int32[1]; the optional curve arrays take n entries each."""
    n = scores.numel()
    if labels.numel() != n or scores.dtype != torch.float32 or labels.dtype != torch.int32 \
            or not (scores.is_contiguous() and labels.is_contiguous()):
        raise L.NPIError("rank_curve: contiguous float32 scores and int32 labels of equal length expected")
    L.call("npi_rank_curve", L.ptr(scores), L.ptr(labels), _i64(n), L.ptr(summary), L.ptr(areas), L.ptr(thresholds),
           L.ptr(tps), L.ptr(fps), L.ptr(status), L.ptr(ws), _i64(ws.numel() * ws.element_size()), _s())


def _group_sort_count_as(entry, num_groups):
    """Launch-count key of npi_group_topk / npi_group_rank: their launches grow with the passes of the sort by group id
    (ceil(log2 num_groups) key bits); None for the two-pass default."""
    passes = L.query("npi_sort_passes", _i32(max(1, (int(num_groups) - 1).bit_length())))
    return None if passes == 2 else "%s/%dpass" % (entry, passes)


def group_topk_workspace_bytes(n_max, num_groups):
    return L.query("npi_group_topk_workspace_bytes", _i64(n_max), _i32(num_groups))


def group_topk(scores, group, num_groups, k, out_pos, out_score, out_count, status, ws):
    """Top-``k`` items of every group of float32 ``scores`` / int32 ``group`` ids, by descending score with ties by
    ascending position (include/npi.h npi_group_topk): out_pos int32 / out_score float32 [num_groups, k] (-1 / NaN past
    the group's count), out_count int32[num_groups], status int32[1] (bit 0 NaN score, bit 1 group id out of range)."""
    n = scores.numel()
    if group.numel() != n or scores.dtype != torch.float32 or group.dtype != torch.int32 \
            or not (scores.is_contiguous() and group.is_contiguous()):
        raise L.NPIError("group_topk: contiguous float32 scores and int32 group ids of equal length expected")
    if out_pos.numel() < num_groups * k or out_score.numel() < num_groups * k or out_count.numel() < num_groups:
        raise L.NPIError("group_topk: outputs hold fewer than num_groups x k entries")
    L.call("npi_group_topk", L.ptr(scores), L.ptr(group), _i64(n), _i32(num_groups), _i32(k), L.ptr(out_pos),
           L.ptr(out_score), L.ptr(out_count), L.ptr(status), L.ptr(ws), _i64(ws.numel() * ws.element_size()), _s(),
           count_as=_group_sort_count_as("npi_group_topk", num_groups))


def group_rank_workspace_bytes(n_max, num_groups):
    return L.query("npi_group_rank_workspace_bytes", _i64(n_max), _i32(num_groups))


def group_rank(scores, labels, group, num_groups, hits_k, n_pos, n_neg, twice_u, summary, sum_rr, status, ws, above=None, tied=None):
    """Filtered rank of every query (label 1) among the competitors (label 0) of its group (include/npi.h npi_group_rank):
    float32 ``scores``, int32 ``labels`` / ``group`` ids; ``hits_k`` a host sequence of 1..8 cut-offs K.  Outputs: n_pos /
    n_neg int32 and twice_u int64 [num_groups]; summary int64[3 + len(hits_k)] = {n_queries, n_unranked, n_groups_scored,
    hits...}; sum_rr float64[1]; status int32[1] (bit 0 NaN score, bit 1 label not 0/1, bit 2 group id out of range);
    optional above / tied int32[n] in input order (-1 for competitors)."""
    n = scores.numel()
    if labels.numel() != n or group.numel() != n or scores.dtype != torch.float32 or labels.dtype != torch.int32 \
            or group.dtype != torch.int32 or not (scores.is_contiguous() and labels.is_contiguous() and group.is_contiguous()):
        raise L.NPIError("group_rank: contiguous float32 scores, int32 labels and int32 group ids of equal length expected")
    G, nh = int(num_groups), len(hits_k)
    outs = ((n_pos, torch.int32, G), (n_neg, torch.int32, G), (twice_u, torch.int64, G), (summary, torch.int64, 3 + nh),
            (sum_rr, torch.float64, 1), (status, torch.int32, 1), (above, torch.int32, n), (tied, torch.int32, n))
    for t, dt, size in outs:
        if t is not None and (t.dtype != dt or not t.is_contiguous() or t.numel() < size):
            raise L.NPIError("group_rank: outputs of the wrong dtype or holding too few entries (num_groups = %d, n = %d, %d hits)"
                             % (G, n, nh))
    ks = (_i32 * max(nh, 1))(*[int(k) for k in hits_k])
    L.call("npi_group_rank", L.ptr(scores), L.ptr(labels), L.ptr(group), _i64(n), _i32(G), ks, _i32(nh), L.ptr(n_pos),
           L.ptr(n_neg), L.ptr(twice_u), L.ptr(summary), L.ptr(sum_rr), L.ptr(above), L.ptr(tied), L.ptr(status), L.ptr(ws),
           _i64(ws.numel() * ws.element_size()), _s(), count_as=_group_sort_count_as("npi_group_rank", G))


def input_attribution_workspace_bytes(n_rows, B, F):
    return L.query("npi_input_attribution_workspace_bytes", _i32(n_rows), _i32(B), _i32(F))


def input_attribution(dxa, gid, dist, graph_ptr, B, n_rows, table, F, w1, node_attr, feature_attr, ws, grad_x=None):
    """Gradient x input of every pair's target over the layer-1 input rows of its subgraph (include/npi.h
    npi_input_attribution): dxa float32 [>= n_rows, 128], gid int32 / dist uint8 [>= n_rows], graph_ptr int32 [>= B + 1],
    table float32 [V, ld] (row stride ld >= F, unit column stride), w1 float32 [F, 128].  Outputs: node_attr float32
    [>= n_rows], feature_attr float32 [B, F] and optional grad_x float32 [n_rows, F], all contiguous."""
    B, n_rows, F = int(B), int(n_rows), int(F)
    f32 = torch.float32
    ok = (dxa.dtype == f32 and dxa.dim() == 2 and dxa.shape[1] == H and dxa.is_contiguous() and dxa.shape[0] >= n_rows
          and gid.dtype == torch.int32 and gid.is_contiguous() and gid.numel() >= n_rows
          and dist.dtype == torch.uint8 and dist.is_contiguous() and dist.numel() >= n_rows
          and graph_ptr.dtype == torch.int32 and graph_ptr.is_contiguous() and graph_ptr.numel() >= B + 1
          and table.dtype == f32 and table.dim() == 2 and table.stride(1) == 1 and table.stride(0) >= F
          and w1.dtype == f32 and w1.is_contiguous() and tuple(w1.shape) == (F, H)
          and node_attr.dtype == f32 and node_attr.is_contiguous() and node_attr.numel() >= n_rows
          and feature_attr.dtype == f32 and feature_attr.is_contiguous() and feature_attr.numel() >= B * F
          and (grad_x is None or (grad_x.dtype == f32 and grad_x.is_contiguous() and grad_x.numel() >= n_rows * F)))
    if not ok:
        raise L.NPIError("input_attribution: expected contiguous float32 dxa [>= %d, 128], int32 gid, uint8 dist, int32 graph_ptr "
                         "[>= %d], a float32 table of row stride >= F, w1 [%d, 128] and float32 outputs node_attr [>= %d], "
                         "feature_attr [%d, %d] (and grad_x [%d, %d])" % (n_rows, B + 1, F, n_rows, B, F, n_rows, F))
    L.call("npi_input_attribution", L.ptr(dxa), L.ptr(gid), L.ptr(dist), L.ptr(graph_ptr), _i32(B), _i32(n_rows), L.ptr(table),
           _i32(table.stride(0)), _i32(F), L.ptr(w1), L.ptr(node_attr), L.ptr(feature_attr), L.ptr(grad_x), L.ptr(ws),
           _i64(ws.numel() * ws.element_size()), _s(), count_as=None if n_rows > 0 else "npi_input_attribution/no_rows")


# ----------------------------------------------------------------------------- operator-API helpers
def filter_edges_coo(edge_index, new_id, out, count_dev):
    E = edge_index.shape[1]
    nbytes = L.query("npi_filter_edges_coo_workspace_bytes", _i64(E))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=edge_index.device)
    L.call("npi_filter_edges_coo", L.ptr(edge_index), _i64(E), L.ptr(new_id), L.ptr(out), L.ptr(count_dev), L.ptr(ws),
           _i64(nbytes), _s())


def readout_bwd(d_readout, argmax, graph_ptr, batch, n, use_max, use_mean, dx):
    L.call("npi_readout_bwd", L.ptr(d_readout), L.ptr(argmax), L.ptr(graph_ptr), L.ptr(batch), _i64(n),
           _i32(1 if use_max else 0), _i32(1 if use_mean else 0), L.ptr(dx), _s())


def scalar_axpy(acc, x, a):
    """acc[0] += a * x[0] (device scalars)."""
    L.call("npi_scalar_axpy", L.ptr(acc), L.ptr(x), _f32(a), _s())
