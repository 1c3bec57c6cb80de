"""Thin tensor -> pointer wrappers over the C ABI (include/cbrs_b200.h).

Every function takes CUDA torch tensors, launches on torch's current stream and
returns torch tensors.  No CPU path exists: a non-CUDA tensor raises.
"""
import ctypes

import torch

from . import _lib as L


# bench instrumentation: kernel launches issued through this module, and (when PROFILE_ON) CUDA
# events on the launching stream around each propagation call
LAUNCHES = 0
PROFILE_ON = False
PROFILE = []


def _count(n):
    global LAUNCHES
    LAUNCHES += n


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t, dtype=None):
    if t is None:
        return None
    if not t.is_cuda:
        raise L.CbrsError("expected a CUDA tensor (there is no CPU path)")
    if dtype is not None and t.dtype != dtype:
        raise L.CbrsError("expected dtype {}, got {}".format(dtype, t.dtype))
    return ctypes.c_void_p(t.data_ptr())


def _rowmajor(t, dtypes=(torch.float32,)):
    """(tensor, leading dimension in elements) of a 2-D view whose rows are contiguous."""
    if t.dim() != 2 or t.dtype not in dtypes or (t.shape[1] > 1 and t.stride(1) != 1):
        raise L.CbrsError("expected a 2-D {} tensor with unit column stride".format("/".join(str(d) for d in dtypes)))
    return t, (t.stride(0) if t.shape[0] > 1 else max(t.stride(0), t.shape[1]))


def _ws(nbytes, device):
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)


def check_device():
    L.check(L.load().cbrs_check_device(), "cbrs_check_device")


# ------------------------------------------------------------------ graph build
def graph_build_csr(row, col, val, n_nodes, flags, rel=None, n_rel=1, self_rel=0):
    """COO (int32 row/col [, float32 val] [, int32 rel]) -> (rowptr int64, colidx int32, vals float32)."""
    lib = L.load()
    dev = row.device
    nnz = row.numel()
    cap = nnz + (n_nodes if flags & L.GRAPH_ADD_SELF_LOOPS else 0)
    rowptr = torch.empty(n_nodes + 1, dtype=torch.int64, device=dev)
    colidx = torch.empty(max(cap, 1), dtype=torch.int32, device=dev)
    vals = torch.empty(max(cap, 1), dtype=torch.float32, device=dev)
    ws_bytes = lib.cbrs_graph_build_workspace_bytes(nnz, n_nodes, flags)
    ws = _ws(ws_bytes, dev)
    if rel is None and n_rel == 1:
        rc = lib.cbrs_graph_build_csr(_ptr(row, torch.int32), _ptr(col, torch.int32), _ptr(val, torch.float32), nnz,
                                      n_nodes, flags, _ptr(rowptr), _ptr(colidx), _ptr(vals), None, _ptr(ws),
                                      ws.numel(), _stream())
    else:
        rc = lib.cbrs_graph_build_csr_rel(_ptr(row, torch.int32), _ptr(col, torch.int32), _ptr(rel, torch.int32),
                                          _ptr(val, torch.float32), nnz, n_nodes, n_rel, self_rel, flags,
                                          _ptr(rowptr), _ptr(colidx), _ptr(vals), None, _ptr(ws), ws.numel(),
                                          _stream())
    L.check(rc, "cbrs_graph_build_csr")
    n_out = int(rowptr[-1].item())
    return rowptr, colidx[:n_out], vals[:n_out]


# ------------------------------------------------------------------ partitioned build (rows of one block only)
def coo_row_histogram(row, n_rows, counts=None):
    """counts[r] += number of entries of row r (int64 [n_rows], created zeroed when None); rows outside are ignored."""
    lib = L.load()
    if counts is None:
        counts = torch.zeros(n_rows, dtype=torch.int64, device=row.device)
    L.check(lib.cbrs_coo_row_histogram(_ptr(row, torch.int32), row.numel(), n_rows, _ptr(counts, torch.int64), _stream()),
            "cbrs_coo_row_histogram")
    return counts


def coo_select_rows(row, col, val, row_lo, row_hi, out_row, out_col, out_val, cursor, rebase=False):
    """Appends the entries of rows [row_lo, row_hi), in input order, to out_* at the device int64 `cursor`, which
    advances by their number (cbrs_coo_select_rows).  Nothing is written past the outputs' length."""
    lib = L.load()
    n = row.numel()
    if n == 0:
        return cursor
    ws = _ws(lib.cbrs_coo_select_rows_workspace_bytes(n), row.device)
    L.check(lib.cbrs_coo_select_rows(_ptr(row, torch.int32), _ptr(col, torch.int32), _ptr(val, torch.float32), n,
                                     int(row_lo), int(row_hi), 1 if rebase else 0, _ptr(out_row, torch.int32),
                                     _ptr(out_col, torch.int32), _ptr(out_val, torch.float32), _ptr(cursor, torch.int64),
                                     out_row.numel(), _ptr(ws), ws.numel(), _stream()), "cbrs_coo_select_rows")
    return cursor


def graph_build_block(row, col, val, row_lo, row_hi, n_nodes, flags):
    """Phase 1 of a row block's build (cbrs_graph_build_block): COO entries of rows [row_lo, row_hi) (global ids) ->
    (rowptr int64, colidx int32, vals float32, dinv float32 [row_hi - row_lo] or None).  With GRAPH_SYM_NORM the
    values are left unscaled and dinv holds the block's degrees; graph_block_scale finishes them."""
    lib = L.load()
    dev = row.device
    nnz, n_rows = row.numel(), int(row_hi) - int(row_lo)
    cap = nnz + (n_rows if flags & L.GRAPH_ADD_SELF_LOOPS else 0)
    rowptr = torch.empty(n_rows + 1, dtype=torch.int64, device=dev)
    colidx = torch.empty(max(cap, 1), dtype=torch.int32, device=dev)
    vals = torch.empty(max(cap, 1), dtype=torch.float32, device=dev)
    dinv = torch.empty(n_rows, dtype=torch.float32, device=dev) if flags & L.GRAPH_SYM_NORM else None
    ws = _ws(lib.cbrs_graph_build_block_workspace_bytes(nnz, n_rows, flags), dev)
    L.check(lib.cbrs_graph_build_block(_ptr(row, torch.int32), _ptr(col, torch.int32), _ptr(val, torch.float32), nnz,
                                       int(row_lo), int(row_hi), int(n_nodes), flags, _ptr(rowptr), _ptr(colidx),
                                       _ptr(vals), _ptr(dinv), None, _ptr(ws), ws.numel(), _stream()),
            "cbrs_graph_build_block")
    del ws
    n_out = int(rowptr[-1].item())
    return rowptr, colidx[:n_out], vals[:n_out], dinv


def graph_block_scale(rowptr, colidx, vals, row_lo, n_nodes, dinv):
    """Phase 2: vals = fl32(fl32(d_i * m_ij) * d_j) in place, d = every node's degree (float32 [n_nodes])."""
    lib = L.load()
    if dinv.numel() != n_nodes:
        raise L.CbrsError("graph_block_scale: {} degrees for {} nodes".format(dinv.numel(), n_nodes))
    L.check(lib.cbrs_graph_block_scale(_ptr(rowptr, torch.int64), _ptr(colidx, torch.int32), _ptr(vals, torch.float32),
                                       rowptr.numel() - 1, int(row_lo), int(n_nodes), _ptr(dinv, torch.float32),
                                       _stream()), "cbrs_graph_block_scale")
    return vals


def build_chunks(rowptr, chunk_edges, colidx=None, n_cols=0, block_cols=0, block_min_len=0):
    """Chunk decomposition of a CSR row-pointer (see cbrs_csr_t).  With block_cols > 0 rows of at least
    block_min_len edges are cut at column-block borders and scheduled by (column block, row)
    (cbrs_chunks_blocked_*): the gather then works on an L2-resident window of the operand table."""
    lib = L.load()
    dev = rowptr.device
    n_rows = rowptr.numel() - 1
    blocked = block_cols > 0 and colidx is not None and n_rows > 0
    counts = torch.zeros(3, dtype=torch.int64, device=dev)
    if blocked:
        nnz = colidx.numel()
        geo = (n_rows, nnz, int(n_cols), int(chunk_edges), int(block_min_len), int(block_cols))
        ws = _ws(lib.cbrs_chunks_blocked_workspace_bytes(n_rows, nnz, int(n_cols), int(block_min_len), int(block_cols)), dev)
        L.check(lib.cbrs_chunks_blocked_count(_ptr(rowptr, torch.int64), _ptr(colidx, torch.int32), *geo, _ptr(counts),
                                              _ptr(ws), ws.numel(), _stream()), "cbrs_chunks_blocked_count")
    else:
        ws = _ws(lib.cbrs_chunks_workspace_bytes(n_rows), dev)
        L.check(lib.cbrs_chunks_count(_ptr(rowptr, torch.int64), n_rows, chunk_edges, _ptr(counts), _ptr(ws), ws.numel(),
                                      _stream()), "cbrs_chunks_count")
    n_chunks, n_heavy, n_slots = (int(v) for v in counts.tolist())
    chunk_row = torch.empty(max(n_chunks, 1), dtype=torch.int32, device=dev)
    chunk_begin = torch.empty(max(n_chunks, 1), dtype=torch.int64, device=dev)
    chunk_slot = torch.empty(max(n_chunks, 1), dtype=torch.int32, device=dev)
    heavy_row = torch.empty(max(n_heavy, 1), dtype=torch.int32, device=dev)
    heavy_slot_ptr = torch.zeros(n_heavy + 1, dtype=torch.int64, device=dev)
    chunk_len = None
    if blocked:
        chunk_len = torch.empty(max(n_chunks, 1), dtype=torch.int32, device=dev)
        L.check(lib.cbrs_chunks_blocked_fill(_ptr(rowptr), _ptr(colidx), *geo, _ptr(chunk_row), _ptr(chunk_begin),
                                             _ptr(chunk_len), _ptr(chunk_slot), _ptr(heavy_row), _ptr(heavy_slot_ptr),
                                             _ptr(ws), ws.numel(), _stream()), "cbrs_chunks_blocked_fill")
        chunk_len = chunk_len[:n_chunks]
    else:
        L.check(lib.cbrs_chunks_fill(_ptr(rowptr), n_rows, chunk_edges, _ptr(chunk_row), _ptr(chunk_begin),
                                     _ptr(chunk_slot), _ptr(heavy_row), _ptr(heavy_slot_ptr), _ptr(ws), ws.numel(),
                                     _stream()), "cbrs_chunks_fill")
    return dict(n_chunks=n_chunks, n_heavy=n_heavy, n_slots=n_slots, chunk_row=chunk_row[:n_chunks],
                chunk_begin=chunk_begin[:n_chunks], chunk_slot=chunk_slot[:n_chunks], heavy_row=heavy_row[:n_heavy],
                heavy_slot_ptr=heavy_slot_ptr, chunk_len=chunk_len)


def csr_subset(csr, ids):
    """Chunk decomposition of the rows `ids` (int64, any order, duplicates allowed, out-of-range ids ignored) of a
    graph.CsrSlice, as build_chunks returns it plus rows / edges (the distinct needed rows and their edge count).
    One device-to-host copy of the counts (cbrs_csr_subset_*)."""
    lib = L.load()
    dev = csr.rowptr.device
    desc = ctypes.byref(csr.desc)
    ws = _ws(lib.cbrs_csr_subset_workspace_bytes(desc), dev)
    counts = torch.empty(5, dtype=torch.int64, device=dev)
    L.check(lib.cbrs_csr_subset_count(desc, _ptr(ids, torch.int64), ids.numel(), _ptr(counts), _ptr(ws), ws.numel(),
                                      _stream()), "cbrs_csr_subset_count")
    n_chunks, n_heavy, n_slots, rows, edges = (int(v) for v in counts.tolist())
    chunk_row = torch.empty(max(n_chunks, 1), dtype=torch.int32, device=dev)
    chunk_begin = torch.empty(max(n_chunks, 1), dtype=torch.int64, device=dev)
    chunk_slot = torch.empty(max(n_chunks, 1), dtype=torch.int32, device=dev)
    chunk_len = torch.empty(max(n_chunks, 1), dtype=torch.int32, device=dev) if csr.desc.chunk_len else None
    heavy_row = torch.empty(max(n_heavy, 1), dtype=torch.int32, device=dev)
    heavy_slot_ptr = torch.zeros(n_heavy + 1, dtype=torch.int64, device=dev)
    L.check(lib.cbrs_csr_subset_fill(desc, _ptr(chunk_row), _ptr(chunk_begin), _ptr(chunk_len), _ptr(chunk_slot),
                                     _ptr(heavy_row), _ptr(heavy_slot_ptr), _ptr(ws), ws.numel(), _stream()),
            "cbrs_csr_subset_fill")
    return dict(n_chunks=n_chunks, n_heavy=n_heavy, n_slots=n_slots, chunk_row=chunk_row[:n_chunks],
                chunk_begin=chunk_begin[:n_chunks], chunk_slot=chunk_slot[:n_chunks], heavy_row=heavy_row[:n_heavy],
                heavy_slot_ptr=heavy_slot_ptr, chunk_len=chunk_len[:n_chunks] if chunk_len is not None else None,
                rows=rows, edges=edges)


# ------------------------------------------------------------------ propagation
def _ptr_array(addresses):
    """host array of device addresses for the *_bcast entry points"""
    return (ctypes.c_void_p * max(len(addresses), 1))(*addresses)


def spmm(csr, x, out, agg=L.AGG_WEIGHTED, bias=None, relu=False, workspace=None, peers=None, mc=None):
    """out[:, :] = epilogue(A @ x) for the rows held by `csr` (a graph.CsrSlice).
    peers: device addresses of the same `out` view in the other ranks' symmetric buffers; every
    finished row is stored there too (cbrs_spmm_csr_bcast).
    mc: address of the same `out` view in the NVSwitch MULTICAST mapping of the symmetric buffer: the kernel then
    stores every finished row ONCE, to that address, and the switch delivers it to all ranks' copies (this rank's
    included) - one store per row instead of 1 + n_peers (multimem.st is a plain store on a multicast address)."""
    lib = L.load()
    x, ldx = _rowmajor(x, (torch.float32, torch.bfloat16))
    xdt = L.DTYPE_BF16 if x.dtype == torch.bfloat16 else L.DTYPE_F32
    out, ldy = _rowmajor(out)
    d = x.shape[1]
    if out.shape[1] != d or out.shape[0] != csr.n_rows:
        raise L.CbrsError("spmm: output shape {} does not match [{}, {}]".format(tuple(out.shape), csr.n_rows, d))
    need = lib.cbrs_spmm_workspace_bytes(ctypes.byref(csr.desc), d)
    ws = workspace if workspace is not None and workspace.numel() >= need else _ws(need, x.device)
    if PROFILE_ON:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    if mc:
        L.check(lib.cbrs_spmm_csr(ctypes.byref(csr.desc), _ptr(x), ldx, ctypes.c_void_p(int(mc)), ldy, d, agg,
                                  _ptr(bias, torch.float32), 1 if relu else 0, xdt, _ptr(ws), ws.numel(),
                                  _stream()), "cbrs_spmm_csr")
    elif peers:
        L.check(lib.cbrs_spmm_csr_bcast(ctypes.byref(csr.desc), _ptr(x), ldx, _ptr(out), ldy, d, agg,
                                        _ptr(bias, torch.float32), 1 if relu else 0, xdt, _ptr_array(peers),
                                        len(peers), _ptr(ws), ws.numel(), _stream()), "cbrs_spmm_csr_bcast")
    else:
        L.check(lib.cbrs_spmm_csr(ctypes.byref(csr.desc), _ptr(x), ldx, _ptr(out), ldy, d, agg,
                                  _ptr(bias, torch.float32), 1 if relu else 0, xdt, _ptr(ws), ws.numel(),
                                  _stream()), "cbrs_spmm_csr")
    if PROFILE_ON:
        e1.record()
        # algorithmic bytes of this launch (SURVEY 8d): nnz*(4 col + 4 val + d*4 row) + rows*(d*4 out + 8 rowptr)
        # (a graph.CsrSubset counts the rows and edges it computes)
        xb = x.element_size()
        rows = getattr(csr, "n_needed", csr.n_rows)
        PROFILE.append(("spmm", e0, e1, {"nnz": csr.nnz, "rows": rows, "d": d,
                                         "bytes": csr.nnz * (8 + xb * d) + rows * (4 * d + 8)}))
    _count(1 + (1 if csr.chunks["n_heavy"] else 0))
    return out


def gat(csr, z, p, q, out, bias=None, relu=True, row_offset=0, workspace=None, peers=None, mc=None):
    """mc: as for spmm, the multicast address of `out` (the kernel only stores to its output)"""
    lib = L.load()
    z, ldz = _rowmajor(z)
    out, ldy = _rowmajor(out)
    h = z.shape[1]
    need = lib.cbrs_gat_workspace_bytes(ctypes.byref(csr.desc), h)
    ws = workspace if workspace is not None and workspace.numel() >= need else _ws(need, z.device)
    if mc:
        L.check(lib.cbrs_gat_csr(ctypes.byref(csr.desc), row_offset, _ptr(z), ldz, _ptr(p, torch.float32),
                                 _ptr(q, torch.float32), ctypes.c_void_p(int(mc)), ldy, h, _ptr(bias, torch.float32),
                                 1 if relu else 0, _ptr(ws), ws.numel(), _stream()), "cbrs_gat_csr")
    elif peers:
        L.check(lib.cbrs_gat_csr_bcast(ctypes.byref(csr.desc), row_offset, _ptr(z), ldz, _ptr(p, torch.float32),
                                       _ptr(q, torch.float32), _ptr(out), ldy, h, _ptr(bias, torch.float32),
                                       1 if relu else 0, _ptr_array(peers), len(peers), _ptr(ws), ws.numel(),
                                       _stream()), "cbrs_gat_csr_bcast")
    else:
        L.check(lib.cbrs_gat_csr(ctypes.byref(csr.desc), row_offset, _ptr(z), ldz, _ptr(p, torch.float32),
                                 _ptr(q, torch.float32), _ptr(out), ldy, h, _ptr(bias, torch.float32),
                                 1 if relu else 0, _ptr(ws), ws.numel(), _stream()), "cbrs_gat_csr")
    _count(1 + (1 if csr.chunks["n_heavy"] else 0))
    return out


def dense(x1, w, b=None, act=None, x2=None, idx1=None, idx2=None, rowop=L.ROWOP_NONE, a_self=None, a_neigh=None,
          out=None, m=None, peers=None, q_out=None, q_peers=None, out_dtype=None):
    """act(rowop([x1[idx1] || x2[idx2]] @ w + b)); returns out (and (p, q) for the attention row-op).
    peers / q_peers: device addresses of the same `out` (and q) views in the other ranks' symmetric
    buffers; finished rows are stored there too (cbrs_dense_bcast)."""
    lib = L.load()
    x1, ld1 = _rowmajor(x1)
    f1 = x1.shape[1]
    f2 = 0
    ld2 = 0
    if x2 is not None:
        x2, ld2 = _rowmajor(x2)
        f2 = x2.shape[1]
    if m is None:
        m = idx1.numel() if idx1 is not None else x1.shape[0]
    if w.dim() != 2 or w.shape[0] != f1 + f2 or not w.is_contiguous():
        raise L.CbrsError("dense: kernel must be contiguous [{}, n], got {}".format(f1 + f2, tuple(w.shape)))
    n = w.shape[1]
    if out is None:
        out = torch.empty(m, n, dtype=out_dtype or torch.float32, device=x1.device)
    out, ldo = _rowmajor(out, (torch.float32, torch.bfloat16))
    p_out = None
    if rowop != L.ROWOP_ATTN:
        q_out = None
    if rowop == L.ROWOP_ATTN:
        p_out = torch.empty(m, dtype=torch.float32, device=x1.device)
        if q_out is None:
            q_out = torch.empty(m, dtype=torch.float32, device=x1.device)
    code = act if isinstance(act, int) else L.ACTS[act]
    if PROFILE_ON:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    if out.dtype == torch.bfloat16:
        L.check(lib.cbrs_dense_ex(_ptr(x1), ld1, _ptr(idx1, torch.int64), f1, _ptr(x2), ld2, _ptr(idx2, torch.int64), f2,
                                  _ptr(w, torch.float32), _ptr(b, torch.float32), m, n, code, rowop,
                                  _ptr(a_self, torch.float32), _ptr(a_neigh, torch.float32), _ptr(p_out), _ptr(q_out),
                                  _ptr(out), ldo, L.DTYPE_BF16, _ptr_array(peers) if peers else None,
                                  _ptr_array(q_peers) if q_peers else None, len(peers) if peers else 0, _stream()),
                "cbrs_dense_ex")
    elif peers:
        L.check(lib.cbrs_dense_bcast(_ptr(x1), ld1, _ptr(idx1, torch.int64), f1, _ptr(x2), ld2,
                                     _ptr(idx2, torch.int64), f2, _ptr(w, torch.float32), _ptr(b, torch.float32), m, n,
                                     code, rowop, _ptr(a_self, torch.float32), _ptr(a_neigh, torch.float32),
                                     _ptr(p_out), _ptr(q_out), _ptr(out), ldo, _ptr_array(peers),
                                     _ptr_array(q_peers) if q_peers else None, len(peers), _stream()),
                "cbrs_dense_bcast")
    else:
        L.check(lib.cbrs_dense(_ptr(x1), ld1, _ptr(idx1, torch.int64), f1, _ptr(x2), ld2, _ptr(idx2, torch.int64), f2,
                               _ptr(w, torch.float32), _ptr(b, torch.float32), m, n, code, rowop,
                               _ptr(a_self, torch.float32), _ptr(a_neigh, torch.float32), _ptr(p_out), _ptr(q_out),
                               _ptr(out), ldo, _stream()), "cbrs_dense")
    _count(2 if (rowop == L.ROWOP_L2NORM and n > 128) else 1)
    if PROFILE_ON:
        e1.record()
        PROFILE.append(("dense", e0, e1, m * n))
    if rowop == L.ROWOP_ATTN:
        return out, p_out, q_out
    return out


# ---- the GCN transform Z = X W: fp32 FFMA kernel or the fp32-accurate tensor-core kernel (3xTF32) ----------------
# "auto": tensor cores from TF32X3_MIN_ROWS graph nodes up (below that the layer is launch-latency bound and the FFMA
# kernel keeps the round-1 bits of every MovieLens-sized parity case).  The choice is made on the GLOBAL node count, so
# all ranks of a row partition and the single-GPU run take the same kernel.  Setting GCN_TRANSFORM to "ffma" or "tf32x3"
# forces one.
GCN_TRANSFORM = "auto"
TF32X3_MIN_ROWS = 1 << 16


def tf32x3_chosen(rows_total, k, n, x=None, out=None):
    if GCN_TRANSFORM == "ffma" or (GCN_TRANSFORM == "auto" and rows_total < TF32X3_MIN_ROWS):
        return False
    if not L.load().cbrs_dense_tf32x3_eligible(int(k), int(n)):
        return False
    if x is not None and (x.dtype != torch.float32 or x.stride(1) != 1 or x.stride(0) % 4 or x.data_ptr() % 16):
        return False
    if out is not None:
        if out.dtype == torch.bfloat16:
            if out.stride(1) != 1 or out.stride(0) % 16 or out.data_ptr() % 32:
                return False
        elif out.dtype != torch.float32 or out.stride(1) != 1 or out.stride(0) % 4 or out.data_ptr() % 16:
            return False
    return True


def dense_tf32x3(x, w, b=None, act=None, out=None, peers=None, out_dtype=None):
    """act(x @ w + b) with the product as three TF32 tcgen05 MMAs (fp32-accurate, cbrs_dense_tf32x3); the result can be
    stored rounded to bf16 (out_dtype=torch.bfloat16 / a bf16 `out`), as cbrs_dense_ex does for the FFMA kernel."""
    lib = L.load()
    x, ldx = _rowmajor(x)
    m, k = x.shape
    if w.dim() != 2 or w.shape[0] != k or not w.is_contiguous():
        raise L.CbrsError("dense_tf32x3: kernel must be contiguous [{}, n], got {}".format(k, tuple(w.shape)))
    n = w.shape[1]
    if out is None:
        out = torch.empty(m, n, dtype=out_dtype or torch.float32, device=x.device)
    out, ldo = _rowmajor(out, (torch.float32, torch.bfloat16))
    image = torch.empty(lib.cbrs_dense_tf32x3_image_bytes(k, n), dtype=torch.uint8, device=x.device)
    if PROFILE_ON:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    L.check(lib.cbrs_dense_tf32x3_prepare(_ptr(w, torch.float32), k, n, _ptr(image), _stream()), "cbrs_dense_tf32x3_prepare")
    code = act if isinstance(act, int) else L.ACTS[act]
    L.check(lib.cbrs_dense_tf32x3(_ptr(x), ldx, _ptr(image), _ptr(b, torch.float32), m, k, n, code, _ptr(out), ldo,
                                  L.DTYPE_BF16 if out.dtype == torch.bfloat16 else L.DTYPE_F32,
                                  _ptr_array(peers) if peers else None, len(peers) if peers else 0, _stream()),
            "cbrs_dense_tf32x3")
    _count(2)
    if PROFILE_ON:
        e1.record()
        PROFILE.append(("dense", e0, e1, m * n))
    return out


def sage_dense(x_self, agg, kernel, bias, act, rows_total, out=None, peers=None):
    """GraphSageConv's dense part act(l2_normalize([x_self || agg] @ kernel + bias)) (spektral GraphSageConv.call).
    From TF32X3_MIN_ROWS graph nodes up (the same GLOBAL rule as the GCN transform, so every rank of a row partition and
    the single-GPU run take the same kernel) it runs on the tensor cores at fp32 accuracy as two products - the operand
    images of a 2f-deep kernel do not fit shared memory at once: t = x_self @ kernel[:f], then
    act(l2norm(agg @ kernel[f:] + t + bias)) with the normalisation in the second product's epilogue
    (cbrs_dense_tf32x3_ex); below that, and for shapes the kernel does not take, the FFMA kernel (cbrs_dense)."""
    f, n = x_self.shape[1], kernel.shape[1]
    if not (agg.shape[1] == f and tf32x3_chosen(rows_total, f, n, x_self, out) and tf32x3_chosen(rows_total, f, n, agg)
            and (out is None or out.dtype == torch.float32)):
        return dense(x_self, kernel, bias, act, x2=agg, rowop=L.ROWOP_L2NORM, out=out, peers=peers)
    lib = L.load()
    x_self, ld1 = _rowmajor(x_self)
    agg, ld2 = _rowmajor(agg)
    m = x_self.shape[0]
    if out is None:
        out = torch.empty(m, n, dtype=torch.float32, device=x_self.device)
    out, ldo = _rowmajor(out)
    t = torch.empty(m, n, dtype=torch.float32, device=x_self.device)
    nbytes = lib.cbrs_dense_tf32x3_image_bytes(f, n)
    images = torch.empty(2 * nbytes, dtype=torch.uint8, device=x_self.device)
    top, bot = images[:nbytes], images[nbytes:]
    if PROFILE_ON:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    L.check(lib.cbrs_dense_tf32x3_prepare(_ptr(kernel[:f], torch.float32), f, n, _ptr(top), _stream()), "cbrs_dense_tf32x3_prepare")
    L.check(lib.cbrs_dense_tf32x3_prepare(_ptr(kernel[f:], torch.float32), f, n, _ptr(bot), _stream()), "cbrs_dense_tf32x3_prepare")
    L.check(lib.cbrs_dense_tf32x3(_ptr(x_self), ld1, _ptr(top), None, m, f, n, L.ACT_NONE, _ptr(t), n, L.DTYPE_F32, None, 0,
                                  _stream()), "cbrs_dense_tf32x3")
    code = act if isinstance(act, int) else L.ACTS[act]
    L.check(lib.cbrs_dense_tf32x3_ex(_ptr(agg), ld2, _ptr(bot), _ptr(bias, torch.float32), _ptr(t), n, L.ROWOP_L2NORM, m, f, n,
                                     code, _ptr(out), ldo, L.DTYPE_F32, _ptr_array(peers) if peers else None,
                                     len(peers) if peers else 0, _stream()), "cbrs_dense_tf32x3_ex")
    _count(4)
    if PROFILE_ON:
        e1.record()
        PROFILE.append(("dense", e0, e1, m * n))
    return out


def gat_transform(x, w, a_self, a_neigh, rows_total, out=None, q_out=None, peers=None, q_peers=None):
    """(z, p, q) = (x @ w, z . a_self, z . a_neigh) for a GAT layer: the tensor-core kernel with the attention row-op from
    TF32X3_MIN_ROWS graph nodes up (cbrs_dense_tf32x3_attn), else cbrs_dense with CBRS_ROWOP_ATTN."""
    k, n = x.shape[1], w.shape[1]
    if not tf32x3_chosen(rows_total, k, n, x, out):
        return dense(x, w, rowop=L.ROWOP_ATTN, a_self=a_self, a_neigh=a_neigh, out=out, q_out=q_out, peers=peers, q_peers=q_peers)
    lib = L.load()
    x, ldx = _rowmajor(x)
    m = x.shape[0]
    if out is None:
        out = torch.empty(m, n, dtype=torch.float32, device=x.device)
    out, ldo = _rowmajor(out)
    p_out = torch.empty(m, dtype=torch.float32, device=x.device)
    if q_out is None:
        q_out = torch.empty(m, dtype=torch.float32, device=x.device)
    image = torch.empty(lib.cbrs_dense_tf32x3_image_bytes(k, n), dtype=torch.uint8, device=x.device)
    if PROFILE_ON:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    L.check(lib.cbrs_dense_tf32x3_prepare(_ptr(w.contiguous(), torch.float32), k, n, _ptr(image), _stream()), "cbrs_dense_tf32x3_prepare")
    L.check(lib.cbrs_dense_tf32x3_attn(_ptr(x), ldx, _ptr(image), m, k, n, _ptr(a_self, torch.float32), _ptr(a_neigh, torch.float32),
                                       _ptr(p_out), _ptr(q_out), _ptr(out), ldo, _ptr_array(peers) if peers else None,
                                       _ptr_array(q_peers) if q_peers else None, len(peers) if peers else 0, _stream()),
            "cbrs_dense_tf32x3_attn")
    _count(2)
    if PROFILE_ON:
        e1.record()
        PROFILE.append(("dense", e0, e1, m * n))
    return out, p_out, q_out


def gcn_transform(x, w, rows_total, out=None, out_dtype=None, peers=None):
    """Z = x @ w for a GCN layer; rows_total = node count of the whole graph (decides the kernel, see above)."""
    if out is None and out_dtype is not None:
        out = torch.empty(x.shape[0], w.shape[1], dtype=out_dtype, device=x.device)
    if tf32x3_chosen(rows_total, x.shape[1], w.shape[1], x, out):
        return dense_tf32x3(x, w, out=out, peers=peers)
    return dense(x, w, out=out, out_dtype=out_dtype, peers=peers)


def dense_grouped(x, kernels, out, group_rows, peers=None):
    """Relational transform in one launch: out[r * group_rows + m, :] = x[m] @ kernels[r] for every relation r
    (cbrs_dense_grouped).  `out` is the stacked operand [R * group_rows, h] (or a row-offset view of it)."""
    lib = L.load()
    x, ldx = _rowmajor(x)
    m, f = x.shape
    h = kernels[0].shape[1]
    w_cat = kernels[0].contiguous() if len(kernels) == 1 else torch.cat(list(kernels), dim=1).contiguous()
    out, ldo = _rowmajor(out, (torch.float32, torch.bfloat16))
    if out.shape[1] != h or out.shape[0] < (len(kernels) - 1) * group_rows + m:
        raise L.CbrsError("dense_grouped: stacked output {} too small for {} x [{}, {}] at stride {}".format(
            tuple(out.shape), len(kernels), m, h, group_rows))
    if PROFILE_ON:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    L.check(lib.cbrs_dense_grouped(_ptr(x), ldx, _ptr(w_cat, torch.float32), m, f, h, len(kernels), _ptr(out), ldo,
                                   int(group_rows), L.DTYPE_BF16 if out.dtype == torch.bfloat16 else L.DTYPE_F32,
                                   _ptr_array(peers) if peers else None, len(peers) if peers else 0, _stream()),
            "cbrs_dense_grouped")
    _count(1)
    if PROFILE_ON:
        e1.record()
        PROFILE.append(("dense", e0, e1, m * h * len(kernels)))
    return out


def dense_tc_eligible(f1, f2, n):
    """shapes cbrs_dense_tc takes: source widths multiples of 8, at most 256 outputs"""
    return f1 > 0 and f1 % 8 == 0 and f2 % 8 == 0 and 0 < n <= 256


def dense_tc(x1, w, b=None, act=None, x2=None, idx1=None, idx2=None, out=None, image=None):
    """cbrs_dense on the tensor cores: act(bf16([x1[idx1] || x2[idx2]]) @ bf16(w) + b), fp32 accumulate and output.
    `image` = a previously prepared operand image of w (dense_tc_image); built here (one small kernel) when absent."""
    lib = L.load()
    x1, ld1 = _rowmajor(x1)
    f1, f2, ld2 = x1.shape[1], 0, 0
    if x2 is not None:
        x2, ld2 = _rowmajor(x2)
        f2 = x2.shape[1]
    m = idx1.numel() if idx1 is not None else x1.shape[0]
    if w.dim() != 2 or w.shape[0] != f1 + f2 or not w.is_contiguous():
        raise L.CbrsError("dense_tc: kernel must be contiguous [{}, n], got {}".format(f1 + f2, tuple(w.shape)))
    n = w.shape[1]
    if image is None:
        image = dense_tc_image(w)
    if out is None:
        out = torch.empty(m, n, dtype=torch.float32, device=x1.device)
    out, ldo = _rowmajor(out)
    code = act if isinstance(act, int) else L.ACTS[act]
    L.check(lib.cbrs_dense_tc(_ptr(x1), ld1, _ptr(idx1, torch.int64), f1, _ptr(x2), ld2, _ptr(idx2, torch.int64), f2,
                              _ptr(image), _ptr(b, torch.float32), m, n, code, _ptr(out), ldo, _stream()), "cbrs_dense_tc")
    _count(1)
    return out


def to_bf16(x, out=None):
    """row-major fp32 matrix -> bf16 copy, round to nearest even (cbrs_convert_f32_bf16): how a static table (the
    content embeddings) is stored once for cbrs_dense_tc_bf16"""
    lib = L.load()
    x, ldx = _rowmajor(x)
    m, k = x.shape
    if k % 8 != 0:
        raise L.CbrsError("to_bf16: width must be a multiple of 8 (16-byte bf16 rows), got {}".format(k))
    if out is None:
        out = torch.empty(m, k, dtype=torch.bfloat16, device=x.device)
    if out.dtype != torch.bfloat16 or out.stride(1) != 1 or tuple(out.shape) != (m, k):
        raise L.CbrsError("to_bf16: out must be a row-major bf16 [{}, {}]".format(m, k))
    L.check(lib.cbrs_convert_f32_bf16(_ptr(x), ldx, m, k, _ptr(out, torch.bfloat16), out.stride(0) if m > 1 else k, _stream()),
            "cbrs_convert_f32_bf16")
    _count(1)
    return out


def dense_tc_bf16_eligible(f1, f2, n):
    """shapes cbrs_dense_tc_bf16 takes: source widths multiples of 64 (one 128-byte swizzle row of bf16), n <= 256"""
    return f1 > 0 and f1 % 64 == 0 and f2 % 64 == 0 and 0 < n <= 256


def dense_tc_bf16(x1, w, b=None, act=None, x2=None, idx1=None, idx2=None, out=None, image=None, out_dtype=torch.float32):
    """cbrs_dense_tc over bf16-STORED sources, fed by TMA (tile::gather4 for indexed rows):
    act([x1[idx1] || x2[idx2]] @ bf16(w) + b), fp32 accumulate; the output is fp32 or bf16 (`out_dtype` / `out`)."""
    lib = L.load()
    if x1.dtype != torch.bfloat16 or (x2 is not None and x2.dtype != torch.bfloat16):
        raise L.CbrsError("dense_tc_bf16: sources must be stored as bf16 (ops.to_bf16)")

    def _bf16_rows(x):
        if x.dim() != 2 or x.stride(1) != 1 or not x.is_cuda:
            raise L.CbrsError("dense_tc_bf16: sources must be row-major CUDA matrices")
        return x, (x.stride(0) if x.shape[0] > 1 else x.shape[1])

    x1, ld1 = _bf16_rows(x1)
    f1, f2, ld2, rows2 = x1.shape[1], 0, 0, 0
    if x2 is not None:
        x2, ld2 = _bf16_rows(x2)
        f2, rows2 = x2.shape[1], x2.shape[0]
    m = idx1.numel() if idx1 is not None else x1.shape[0]
    if w.dim() != 2 or w.shape[0] != f1 + f2 or not w.is_contiguous():
        raise L.CbrsError("dense_tc_bf16: kernel must be contiguous [{}, n], got {}".format(f1 + f2, tuple(w.shape)))
    n = w.shape[1]
    if image is None:
        image = dense_tc_image(w)
    if out is None:
        out = torch.empty(m, n, dtype=out_dtype, device=x1.device)
    if out.dtype not in (torch.float32, torch.bfloat16) or out.dim() != 2 or out.stride(1) != 1 or tuple(out.shape) != (m, n):
        raise L.CbrsError("dense_tc_bf16: out must be a row-major fp32 or bf16 [{}, {}]".format(m, n))
    ldo = out.stride(0) if m > 1 else n
    code = act if isinstance(act, int) else L.ACTS[act]
    L.check(lib.cbrs_dense_tc_bf16(_ptr(x1, torch.bfloat16), ld1, x1.shape[0], _ptr(idx1, torch.int64), f1,
                                   _ptr(x2, torch.bfloat16), ld2, rows2, _ptr(idx2, torch.int64), f2, _ptr(image),
                                   _ptr(b, torch.float32), m, n, code, _ptr(out, out.dtype), ldo,
                                   L.DTYPE_BF16 if out.dtype == torch.bfloat16 else L.DTYPE_F32, _stream()), "cbrs_dense_tc_bf16")
    _count(1)
    return out


def dense_tc_image(w):
    """bf16 tensor-core operand image of a Keras kernel [k, n] (cbrs_dense_tc_prepare)"""
    lib = L.load()
    k, n = w.shape
    image = torch.empty(lib.cbrs_dense_tc_image_bytes(k, n), dtype=torch.uint8, device=w.device)
    L.check(lib.cbrs_dense_tc_prepare(_ptr(w, torch.float32), k, n, _ptr(image), _stream()), "cbrs_dense_tc_prepare")
    _count(1)
    return image


def reduce_layers(hs, coefs=None, divide_by=1.0, out=None):
    lib = L.load()
    n_rows, d = hs[0].shape
    if out is None:
        out = torch.empty(n_rows, d, dtype=torch.float32, device=hs[0].device)
    out, ldo = _rowmajor(out)
    n = len(hs)
    ptrs = (ctypes.c_void_p * n)(*[h.data_ptr() for h in hs])
    lds = (ctypes.c_int64 * n)(*[_rowmajor(h)[1] for h in hs])
    cf = (ctypes.c_float * n)(*[float(c) for c in coefs]) if coefs is not None else None
    L.check(lib.cbrs_reduce_layers(ptrs, lds, n, cf, float(divide_by), n_rows, d, _ptr(out), ldo, _stream()),
            "cbrs_reduce_layers")
    _count(1)
    return out


def gather_rows(x, idx, out=None):
    lib = L.load()
    x, ldx = _rowmajor(x)
    m, d = idx.numel(), x.shape[1]
    if out is None:
        out = torch.empty(m, d, dtype=torch.float32, device=x.device)
    out, ldo = _rowmajor(out)
    L.check(lib.cbrs_gather_rows(_ptr(x), ldx, _ptr(idx, torch.int64), m, d, _ptr(out), ldo, _stream()),
            "cbrs_gather_rows")
    _count(1)
    return out


def push_rows(view, buf):
    """Store the finished row block `view` (a view into the local copy of the SymmetricBuffer `buf`) into every rank's copy:
    one coalesced pass to the NVSwitch multicast mapping when the buffer has one, else one per peer (cbrs_push_rows).
    An empty block stores nothing (torch gives it no address inside the buffer)."""
    if view.numel() == 0:
        return
    lib = L.load()
    v = view if view.dim() == 2 else view.reshape(-1, 1)
    v, ld = _rowmajor(v)
    m, w = v.shape
    mc = buf.mc_addr(view)
    targets = [mc] if mc else buf.peer_addrs(view)
    if PROFILE_ON:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    for addr in targets:
        L.check(lib.cbrs_push_rows(_ptr(v), ld, ctypes.c_void_p(addr), ld, m, w, _stream()), "cbrs_push_rows")
    _count(len(targets))
    if PROFILE_ON:
        e1.record()
        PROFILE.append(("push", e0, e1, m * w * 4))


# ------------------------------------------------------------------ top-k
def topk_rows(scores, k):
    lib = L.load()
    scores, ld = _rowmajor(scores)
    n_users, n_items = scores.shape
    ids = torch.empty(n_users, k, dtype=torch.int32, device=scores.device)
    vals = torch.empty(n_users, k, dtype=torch.float32, device=scores.device)
    L.check(lib.cbrs_topk_rows(_ptr(scores), ld, n_users, n_items, k, _ptr(ids), _ptr(vals), _stream()),
            "cbrs_topk_rows")
    _count(1)
    return ids, vals


def _exclusion(exclude, n_rows):
    """(rowptr, items) pointers of per-row exclusion lists (include/cbrs_b200.h, above cbrs_score_catalog_topk_ex), or
    (None, None).  rowptr: CUDA int64 with at least n_rows + 1 entries (row r = the r-th scored row); items: CUDA int32."""
    if exclude is None:
        return None, None
    rowptr, items = exclude
    if rowptr.dim() != 1 or rowptr.numel() < n_rows + 1 or (rowptr.numel() > 1 and rowptr.stride(0) != 1):
        raise L.CbrsError("exclusion rowptr must be a contiguous 1-D tensor of at least n_rows + 1 = {} entries".format(n_rows + 1))
    if items.dim() != 1 or (items.numel() > 1 and items.stride(0) != 1):
        raise L.CbrsError("exclusion items must be a contiguous 1-D tensor")
    if items.numel() == 0:   # an empty tensor has no address; every row is empty, so any valid pointer will do
        items = torch.zeros(1, dtype=torch.int32, device=rowptr.device)
    return _ptr(rowptr, torch.int64), _ptr(items, torch.int32)


def exclude_cols(scores, col_base, exclude):
    """Overwrite with -inf, in place, the listed items of each row of the score block scores [n_rows, n_cols] whose
    columns are catalog items col_base .. col_base + n_cols - 1 (cbrs_exclude_cols).  exclude = (rowptr, items)."""
    lib = L.load()
    scores, ld = _rowmajor(scores)
    n_rows, n_cols = scores.shape
    rp, it = _exclusion(exclude, n_rows)
    L.check(lib.cbrs_exclude_cols(_ptr(scores), ld, n_rows, n_cols, col_base, rp, it, _stream()), "cbrs_exclude_cols")
    _count(1)
    return scores


RANK_METRICS = ("precision", "recall", "hit_rate", "mrr", "ndcg", "map")   # the per-user columns of cbrs_rank_metrics


def rank_metrics_cutoffs(ids, cutoffs):
    """The cutoffs as a list of ints, or CbrsError (before any device work) unless ids is a 2-D int32 tensor with unit
    column stride and cutoffs are 1..8 strictly ascending values in [1, k]."""
    if not torch.is_tensor(ids) or ids.dim() != 2 or ids.dtype != torch.int32 or (ids.shape[1] > 1 and ids.stride(1) != 1):
        raise L.CbrsError("rank_metrics: ids must be a 2-D int32 tensor with unit column stride")
    k = ids.shape[1]
    cutoffs = [int(c) for c in cutoffs]
    if not cutoffs or len(cutoffs) > 8 or k > 128 or any(c < 1 or c > k for c in cutoffs) \
            or any(b <= a for a, b in zip(cutoffs, cutoffs[1:])):
        raise L.CbrsError("rank_metrics: cutoffs {} must be 1..8 strictly ascending values in [1, k = {}], k <= 128".format(
            cutoffs, k))
    return cutoffs


def rank_metrics(ids, rel, users, cutoffs, per_user=False, n_items=None):
    """Ranking metrics of top-k lists against per-user relevance lists (cbrs_rank_metrics), on the device.
    ids [n_rows, k] int32 (row r = the list of users[r], or of user r when users is None; -1 = empty slot);
    rel = (rowptr, items): CSR over global user ids, sorted distinct catalog indices per row; n_items: ids at or past it
    never hit (default: no bound beyond the lists).  cutoffs: strictly ascending, each in [1, k], at most 8.
    Returns (sums fp64 [n_cutoffs, 7] on the device: columns RANK_METRICS summed over the scored users with at least one
    relevant item, then their count; per_user fp64 [n_rows, n_cutoffs, 6] (NaN for rows without one) or None)."""
    cutoffs = rank_metrics_cutoffs(ids, cutoffs)
    lib = L.load()
    n_rows, k = ids.shape
    ld = ids.stride(0) if n_rows > 1 else k
    rowptr, items = rel
    n_users = rowptr.numel() - 1
    rp, it = _exclusion(rel, n_users)
    if users is not None:
        users = users.to(ids.device, torch.int64).contiguous()
        if users.numel() != n_rows:
            raise L.CbrsError("rank_metrics: {} users for {} lists".format(users.numel(), n_rows))
    nc = len(cutoffs)
    sums = torch.empty(nc, 7, dtype=torch.float64, device=ids.device)
    pu = torch.empty(n_rows, nc, 6, dtype=torch.float64, device=ids.device) if per_user else None
    ws = _ws(lib.cbrs_rank_metrics_workspace_bytes(n_rows, nc), ids.device)
    L.check(lib.cbrs_rank_metrics(_ptr(ids), ld, n_rows, k, (1 << 31) - 1 if n_items is None else int(n_items),
                                  _ptr(users, torch.int64), n_users, rp, it, (ctypes.c_int32 * nc)(*cutoffs), nc,
                                  _ptr(sums), _ptr(pu), _ptr(ws), ws.numel(), _stream()), "cbrs_rank_metrics")
    _count(2)
    return sums, pu


def topk_pairs(users, scores, n_users, k):
    """Rows of the pair list kept by the reference's per-user head(k), in (user asc, score desc) order."""
    lib = L.load()
    n = users.numel()
    order = torch.empty(n, dtype=torch.int32, device=users.device)
    rank = torch.empty(n, dtype=torch.int32, device=users.device)
    ws = _ws(lib.cbrs_topk_pairs_workspace_bytes(n), users.device)
    L.check(lib.cbrs_topk_pairs(_ptr(users, torch.int64), _ptr(scores.reshape(-1), torch.float32), n, n_users,
                                _ptr(order), _ptr(rank), _ptr(ws), ws.numel(), _stream()), "cbrs_topk_pairs")
    return order[rank < k].to(torch.int64)


def score_catalog_topk(P, Q, w2, b2, w3, b3, k, precision="fp32", exclude=None):
    """Fused BasicRS catalog scorer: P [U,c1] (bias folded in), Q [I,c1] -> (ids int32 [U,k], scores [U,k]).
    precision 'fp32' = fp32-accurate (1e-5 parity): the 3xTF32 tensor-core kernel for the shapes it takes (c1 in {32, 64},
    c2 <= 64: the reference's grids), the FFMA kernel otherwise; 'fp32-ffma' forces the FFMA kernel;
    'bf16' = bf16 operands on the tensor cores.
    exclude = (rowptr, items): per-row lists of catalog items kept out of row r's top-k (row r = row r of P)."""
    lib = L.load()
    rp, it = _exclusion(exclude, P.shape[0])
    if precision not in ("fp32", "fp32-ffma", "bf16"):
        raise L.CbrsError("score_catalog_topk: precision must be 'fp32', 'fp32-ffma' or 'bf16'")
    P, ldp = _rowmajor(P)
    Q, ldq = _rowmajor(Q)
    n_users, c1 = P.shape
    n_items = Q.shape[0]
    c2 = w2.shape[1]
    # entry point, workspace bytes (None: takes no workspace), launches
    if precision == "fp32" and lib.cbrs_score_catalog_topk_tf32x3_eligible(c1, c2):
        name, ws_bytes, launches = "cbrs_score_catalog_topk_tf32x3", lib.cbrs_score_catalog_topk_tf32x3_workspace_bytes(c1, c2), 2
    elif precision == "bf16":
        name, ws_bytes, launches = ("cbrs_score_catalog_topk_bf16",
                                    lib.cbrs_score_catalog_topk_bf16_workspace_bytes(n_items, c1, c2),
                                    4 if (c1 <= 64 and c2 <= 64) else (3 if c1 <= 64 and c2 <= 128 else 2))
    else:
        name, ws_bytes, launches = "cbrs_score_catalog_topk", None, 1
    ids = torch.empty(n_users, k, dtype=torch.int32, device=P.device)
    vals = torch.empty(n_users, k, dtype=torch.float32, device=P.device)
    args = [_ptr(P), ldp, _ptr(Q), ldq, n_users, n_items, c1, _ptr(w2, torch.float32), _ptr(b2, torch.float32), c2,
            _ptr(w3, torch.float32), _ptr(b3, torch.float32), k, _ptr(ids), _ptr(vals), rp, it]
    if ws_bytes is not None:
        ws = _ws(ws_bytes, P.device)
        args += [_ptr(ws), ws.numel()]
    L.check(getattr(lib, name + "_ex")(*args, _stream()), name)
    _count(launches)
    return ids, vals


# ------------------------------------------------------------------ misc
def _score_hybrid_topk(fn, name, ws_bytes, launches, tensors, k, exclude):
    """Body of the two hybrid catalog scorers: entry point fn (reported as name), its workspace bytes and launch count;
    tensors = (P1, Q1, P2, Q2, w3a2, ..., bc3) as in score_hybrid_topk_bf16."""
    ts = [t.contiguous() for t in tensors]
    n_users, c = ts[0].shape
    rp, it = _exclusion(exclude, n_users)
    n_items = ts[1].shape[0]
    dev = ts[0].device
    ids = torch.empty(n_users, k, dtype=torch.int32, device=dev)
    vals = torch.empty(n_users, k, dtype=torch.float32, device=dev)
    ws = _ws(ws_bytes, dev)
    L.check(fn(_ptr(ts[0], torch.float32), _ptr(ts[1], torch.float32), _ptr(ts[2], torch.float32), _ptr(ts[3], torch.float32),
               n_users, n_items, c, *[_ptr(t, torch.float32) for t in ts[4:]], k, _ptr(ids), _ptr(vals), rp, it, _ptr(ws),
               ws.numel(), _stream()), name)
    _count(launches)
    return ids, vals


def score_hybrid_topk_bf16(P1, Q1, P2, Q2, w3a2, b3a2, w3b2, b3b2, wc1, bc1, wc2, bc2, wc3, bc3, k, exclude=None):
    """Feature-based hybrid scorer over the whole catalog + per-user top-k, chained tcgen05 kernel
    (cbrs_score_hybrid_topk_bf16).  Returns (item index int32 [U, k], score float32 [U, k]).
    exclude = (rowptr, items) as in score_catalog_topk."""
    lib = L.load()
    return _score_hybrid_topk(lib.cbrs_score_hybrid_topk_bf16_ex, "cbrs_score_hybrid_topk_bf16",
                              lib.cbrs_score_hybrid_topk_bf16_workspace_bytes(), 2,
                              (P1, Q1, P2, Q2, w3a2, b3a2, w3b2, b3b2, wc1, bc1, wc2, bc2, wc3, bc3), k, exclude)


def score_hybrid_topk_tf32x3(P1, Q1, P2, Q2, w3a2, b3a2, w3b2, b3b2, wc1, bc1, wc2, bc2, wc3, bc3, k, exclude=None):
    """The scorer of score_hybrid_topk_bf16 at fp32 accuracy (1e-5): the five 64 x 64 products as 3xTF32 on the tensor
    cores (cbrs_score_hybrid_topk_tf32x3).  Same arguments and return value as score_hybrid_topk_bf16."""
    lib = L.load()
    return _score_hybrid_topk(lib.cbrs_score_hybrid_topk_tf32x3, "cbrs_score_hybrid_topk_tf32x3",
                              lib.cbrs_score_hybrid_topk_tf32x3_workspace_bytes(), 6,
                              (P1, Q1, P2, Q2, w3a2, b3a2, w3b2, b3b2, wc1, bc1, wc2, bc2, wc3, bc3), k, exclude)


def synth_bipartite(n_users, n_items, n_edges, seed, device, scatter_items=True):
    lib = L.load()
    row = torch.empty(2 * n_edges, dtype=torch.int32, device=device)
    col = torch.empty(2 * n_edges, dtype=torch.int32, device=device)
    L.check(lib.cbrs_synth_bipartite_ex(n_users, n_items, n_edges, seed, 1 if scatter_items else 0, _ptr(row), _ptr(col),
                                        _stream()), "cbrs_synth_bipartite_ex")
    return row, col


def synth_bipartite_range(n_users, n_items, n_edges, seed, edge_lo, edge_hi, device, scatter_items=True, out=None):
    """The entries of edges [edge_lo, edge_hi) of synth_bipartite(n_users, n_items, n_edges, seed): (row, col) of
    2 * (edge_hi - edge_lo) entries, the forward ones first, then their reverses.  out: (row, col) int32 buffers of
    at least that length to write into (views of them are returned)."""
    lib = L.load()
    m = max(int(edge_hi) - int(edge_lo), 0)     # an inverted range is refused by the library
    if out is None:
        out = (torch.empty(2 * m, dtype=torch.int32, device=device), torch.empty(2 * m, dtype=torch.int32, device=device))
    row, col = out[0][:2 * m], out[1][:2 * m]
    L.check(lib.cbrs_synth_bipartite_range(n_users, n_items, n_edges, seed, 1 if scatter_items else 0, int(edge_lo),
                                           int(edge_hi), _ptr(row, torch.int32), _ptr(col, torch.int32), _stream()),
            "cbrs_synth_bipartite_range")
    return row, col


def sort_pairs_u64(keys, payload, key_bits):
    """In-place stable ascending sort (keys: int64 tensor holding uint64 bit patterns; payload int32)."""
    lib = L.load()
    n = keys.numel()
    ws = _ws(lib.cbrs_sort_workspace_bytes(n), keys.device)
    L.check(lib.cbrs_sort_pairs_u64(_ptr(keys, torch.int64), _ptr(payload, torch.int32), n, key_bits, _ptr(ws),
                                    ws.numel(), _stream()), "cbrs_sort_pairs_u64")
    return keys, payload


# ------------------------------------------------------------------ training step (scope row (f)-1)
def act_grad(dout, out, act):
    """dPre = dOut * act'(out)"""
    lib = L.load()
    dout, ldd = _rowmajor(dout)
    out, ldo = _rowmajor(out)
    rows, d = out.shape
    dpre = torch.empty(rows, d, dtype=torch.float32, device=out.device)
    code = act if isinstance(act, int) else L.ACTS[act]
    L.check(lib.cbrs_act_grad(_ptr(dout), ldd, _ptr(out), ldo, rows, d, code, _ptr(dpre), d, _stream()), "cbrs_act_grad")
    _count(1)
    return dpre


def dense_grad_w(x1, dpre, x2=None, idx1=None, idx2=None, want_bias=True):
    """(dW [f1+f2, n], db [n] or None) of out = [x1[idx1] || x2[idx2]] @ W + b given dPre [m, n]"""
    lib = L.load()
    x1, ld1 = _rowmajor(x1)
    f1, f2, ld2 = x1.shape[1], 0, 0
    if x2 is not None:
        x2, ld2 = _rowmajor(x2)
        f2 = x2.shape[1]
    dpre, ldd = _rowmajor(dpre)
    m, n = dpre.shape
    dw = torch.empty(f1 + f2, n, dtype=torch.float32, device=dpre.device)
    db = torch.empty(n, dtype=torch.float32, device=dpre.device) if want_bias else None
    ws = _ws(lib.cbrs_dense_grad_w_workspace_bytes(m, f1 + f2, n), dpre.device)
    L.check(lib.cbrs_dense_grad_w(_ptr(x1), ld1, _ptr(idx1, torch.int64), f1, _ptr(x2), ld2, _ptr(idx2, torch.int64), f2,
                                  _ptr(dpre), ldd, m, n, _ptr(dw), _ptr(db), _ptr(ws), ws.numel(), _stream()),
            "cbrs_dense_grad_w")
    _count(3 if want_bias else 2)
    return dw, db


def colsum(x):
    """column sums of a [m, n] matrix in the fixed slab order of cbrs_dense_grad_w (its db output)"""
    _, db = dense_grad_w(x[:, :1], x, want_bias=True)
    return db


def transpose(w):
    lib = L.load()
    if w.dim() != 2 or not w.is_contiguous():
        raise L.CbrsError("transpose: expected a contiguous 2-D tensor")
    out = torch.empty(w.shape[1], w.shape[0], dtype=torch.float32, device=w.device)
    L.check(lib.cbrs_transpose_f32(_ptr(w, torch.float32), w.shape[0], w.shape[1], _ptr(out), _stream()),
            "cbrs_transpose_f32")
    _count(1)
    return out


def scatter_add_rows(src, idx, dst):
    """dst[idx[m]] += src[m] (duplicates added in ascending m)"""
    lib = L.load()
    src, lds = _rowmajor(src)
    dst, ldd = _rowmajor(dst)
    m, d = src.shape
    ws = _ws(lib.cbrs_scatter_add_rows_workspace_bytes(m), src.device)
    L.check(lib.cbrs_scatter_add_rows(_ptr(src), lds, _ptr(idx, torch.int64), m, d, dst.shape[0], _ptr(dst), ldd,
                                      _ptr(ws), ws.numel(), _stream()), "cbrs_scatter_add_rows")
    _count(4)
    return dst


def l2norm_act(v, relu=True, out=None):
    lib = L.load()
    v, ldv = _rowmajor(v)
    rows, d = v.shape
    if out is None:
        out = torch.empty(rows, d, dtype=torch.float32, device=v.device)
    out, ldo = _rowmajor(out)
    L.check(lib.cbrs_l2norm_act(_ptr(v), ldv, rows, d, 1 if relu else 0, _ptr(out), ldo, _stream()), "cbrs_l2norm_act")
    _count(1)
    return out


def l2norm_relu_grad(v, dout, relu=True):
    lib = L.load()
    v, ldv = _rowmajor(v)
    dout, ldd = _rowmajor(dout)
    rows, d = v.shape
    dv = torch.empty(rows, d, dtype=torch.float32, device=v.device)
    L.check(lib.cbrs_l2norm_relu_grad(_ptr(v), ldv, _ptr(dout), ldd, rows, d, 1 if relu else 0, _ptr(dv), d, _stream()),
            "cbrs_l2norm_relu_grad")
    _count(1)
    return dv


def scale_rows_inv_degree(x, rowptr):
    lib = L.load()
    x, ldx = _rowmajor(x)
    rows, d = x.shape
    out = torch.empty(rows, d, dtype=torch.float32, device=x.device)
    L.check(lib.cbrs_scale_rows_inv_degree(_ptr(x), ldx, _ptr(rowptr, torch.int64), rows, d, _ptr(out), d, _stream()),
            "cbrs_scale_rows_inv_degree")
    _count(1)
    return out


def axpby(a, ca=1.0, b=None, cb=1.0, out=None):
    """out = ca*a + cb*b on 2-D (possibly strided) views"""
    lib = L.load()
    a, lda = _rowmajor(a)
    ldb = 0
    if b is not None:
        b, ldb = _rowmajor(b)
    rows, d = a.shape
    if out is None:
        out = torch.empty(rows, d, dtype=torch.float32, device=a.device)
    out, ldo = _rowmajor(out)
    L.check(lib.cbrs_axpby2d(_ptr(a), lda, float(ca), _ptr(b), ldb, float(cb), rows, d, _ptr(out), ldo, _stream()),
            "cbrs_axpby2d")
    _count(1)
    return out


def bce(p, y, want_grad=True):
    """Keras binary cross-entropy of probabilities p vs labels y (float32 [n]):
    (loss [1], dLoss/dp [n] or None, correct-count [1])"""
    lib = L.load()
    p = p.reshape(-1)
    n = p.numel()
    loss = torch.empty(1, dtype=torch.float32, device=p.device)
    correct = torch.empty(1, dtype=torch.float32, device=p.device)
    dp = torch.empty(n, dtype=torch.float32, device=p.device) if want_grad else None
    L.check(lib.cbrs_bce(_ptr(p, torch.float32), _ptr(y, torch.float32), n, _ptr(loss), _ptr(dp), _ptr(correct),
                         _stream()), "cbrs_bce")
    _count(1)
    return loss, dp, correct


def sum_squares(w, scale, out, accumulate=True):
    lib = L.load()
    ws = _ws(lib.cbrs_sum_squares_workspace_bytes(), w.device)
    L.check(lib.cbrs_sum_squares(_ptr(w, torch.float32), w.numel(), float(scale), _ptr(out, torch.float32),
                                 1 if accumulate else 0, _ptr(ws), ws.numel(), _stream()), "cbrs_sum_squares")
    _count(2)
    return out


def adam_step(w, g, m, v, lr_t, beta1, beta2, eps, l2=0.0, lr_t_dev=None):
    lib = L.load()
    if not (w.is_contiguous() and g.is_contiguous()):
        raise L.CbrsError("adam_step: weight and gradient must be contiguous")
    L.check(lib.cbrs_adam_step(_ptr(w, torch.float32), _ptr(g, torch.float32), _ptr(m, torch.float32),
                               _ptr(v, torch.float32), w.numel(), float(lr_t), _ptr(lr_t_dev, torch.float32), float(beta1),
                               float(beta2), float(eps), float(l2), _stream()), "cbrs_adam_step")
    _count(1)


def adam_step_multi(ws, gs, ms, vs, l2s, lr_t, beta1, beta2, eps, lr_t_dev=None):
    """cbrs_adam_step for every weight tensor of a model in one launch"""
    lib = L.load()
    k = len(ws)
    for w, g in zip(ws, gs):
        if not (w.is_contiguous() and g.is_contiguous()) or w.dtype != torch.float32 or g.dtype != torch.float32:
            raise L.CbrsError("adam_step_multi: weights and gradients must be contiguous float32")
    arr = lambda ts: (ctypes.c_void_p * k)(*[t.data_ptr() for t in ts])
    L.check(lib.cbrs_adam_step_multi(k, arr(ws), arr(gs), arr(ms), arr(vs), (ctypes.c_int64 * k)(*[w.numel() for w in ws]),
                                     (ctypes.c_float * k)(*[float(c) for c in l2s]), float(lr_t),
                                     _ptr(lr_t_dev, torch.float32), float(beta1), float(beta2), float(eps), _stream()),
            "cbrs_adam_step_multi")
    _count((k + 47) // 48)


def gat_backward(csr, z, p, q, y, bias, d_o, a_self, a_neigh):
    """(dz [N,h] incl. the dp/dq rank-1 terms, dp [N], dq [N]) of the fused GAT layer"""
    lib = L.load()
    z, ldz = _rowmajor(z)
    y, ldy = _rowmajor(y)
    d_o, ldo = _rowmajor(d_o)
    n, h = z.shape
    dz = torch.empty(n, h, dtype=torch.float32, device=z.device)
    dp = torch.empty(n, dtype=torch.float32, device=z.device)
    dq = torch.empty(n, dtype=torch.float32, device=z.device)
    ws = _ws(lib.cbrs_gat_backward_workspace_bytes(n), z.device)
    L.check(lib.cbrs_gat_backward(ctypes.byref(csr.desc), _ptr(z), ldz, _ptr(p, torch.float32), _ptr(q, torch.float32),
                                  _ptr(y), ldy, _ptr(bias, torch.float32), _ptr(d_o), ldo, h,
                                  _ptr(a_self, torch.float32), _ptr(a_neigh, torch.float32), _ptr(dz), h, _ptr(dp),
                                  _ptr(dq), _ptr(ws), ws.numel(), _stream()), "cbrs_gat_backward")
    _count(3)
    return dz, dp, dq


def _out_targets(out, targets, what):
    """(address the kernel stores `out` to, host array of peer addresses, peer count) for one output of a row-slice
    kernel: targets = None / {} (local only), {"peers": [addresses]} or {"mc": multicast address}"""
    targets = targets or {}
    if targets.get("mc"):
        return ctypes.c_void_p(int(targets["mc"])), None, 0
    peers = targets.get("peers") or []
    if len(peers) >= L.MAX_PEERS:
        raise L.CbrsError("{}: {} peer copies (at most {})".format(what, len(peers), L.MAX_PEERS - 1))
    return _ptr(out), (_ptr_array(peers) if peers else None), len(peers)


def gat_backward_stats_rows(csr, p, q, y, bias, d_o, stats, peers=None, mc=None):
    """Phase 1 of gat_backward on the row slice `csr` (rows csr.row_offset + [0, n_rows)): (m, S, t) of its rows into
    `stats` ([n_rows, 3] view) and into the peers' copies (or once, to the multicast address `mc`) - cbrs_gat_backward_stats_rows.
    p, q [N], y, d_o [N, h] are whole-graph tensors."""
    lib = L.load()
    y, ldy = _rowmajor(y)
    d_o, ldo = _rowmajor(d_o)
    stats, _ = _rowmajor(stats)
    if tuple(stats.shape) != (csr.n_rows, 3) or not stats.is_contiguous():
        raise L.CbrsError("gat_backward_stats_rows: stats must be a contiguous [{}, 3] view".format(csr.n_rows))
    dst, arr, n_peers = _out_targets(stats, {"peers": peers, "mc": mc}, "gat_backward_stats_rows")
    L.check(lib.cbrs_gat_backward_stats_rows(ctypes.byref(csr.desc), csr.row_offset, _ptr(p, torch.float32),
                                             _ptr(q, torch.float32), _ptr(y), ldy, _ptr(bias, torch.float32), _ptr(d_o),
                                             ldo, y.shape[1], dst, arr, n_peers, _stream()),
            "cbrs_gat_backward_stats_rows")
    _count(1)
    return stats


def gat_backward_grad_rows(csr, z, p, q, d_o, stats, a_self, a_neigh, dz, dp, dq, targets=None):
    """Phase 2 of gat_backward on the row slice `csr`: dz ([n_rows, h] view, the dp/dq terms included), dp, dq
    ([n_rows, 1] views) of its rows - cbrs_gat_backward_grad_rows.  `stats` is the whole [N, 3] array of phase 1.
    targets: None, or one dict per output (dz, dp, dq) as for _out_targets; every output takes the same kind."""
    lib = L.load()
    z, ldz = _rowmajor(z)
    d_o, ldo = _rowmajor(d_o)
    dz, lddz = _rowmajor(dz)
    h = z.shape[1]
    if dz.shape[1] != h or not all(t.shape[0] == csr.n_rows and t.numel() == csr.n_rows for t in (dp, dq)):
        raise L.CbrsError("gat_backward_grad_rows: outputs do not match the slice's {} rows".format(csr.n_rows))
    targets = list(targets) if targets else [None] * 3
    outs = [_out_targets(t, tg, "gat_backward_grad_rows") for t, tg in zip((dz, dp, dq), targets)]
    if len({o[2] for o in outs}) != 1:
        raise L.CbrsError("gat_backward_grad_rows: dz, dp and dq need the same number of peer copies")
    L.check(lib.cbrs_gat_backward_grad_rows(ctypes.byref(csr.desc), csr.row_offset, _ptr(z), ldz, _ptr(p, torch.float32),
                                            _ptr(q, torch.float32), _ptr(d_o), ldo, h, _ptr(stats, torch.float32),
                                            _ptr(a_self, torch.float32), _ptr(a_neigh, torch.float32), outs[0][0], lddz,
                                            outs[1][0], outs[2][0], outs[0][1], outs[1][1], outs[2][1], outs[0][2],
                                            _stream()), "cbrs_gat_backward_grad_rows")
    _count(1)
    return dz, dp, dq


# ------------------------------------------------------------------ id compaction (rows G0 / (f)-2)
def compact_ids(ids):
    """np.unique(ids, return_inverse=True) on device: (sorted uniques int64 [k], inverse int64 [n])"""
    lib = L.load()
    n = ids.numel()
    uniques = torch.empty(n, dtype=torch.int64, device=ids.device)
    inverse = torch.empty(n, dtype=torch.int64, device=ids.device)
    count = torch.zeros(1, dtype=torch.int64, device=ids.device)
    ws = _ws(lib.cbrs_compact_ids_workspace_bytes(n), ids.device)
    L.check(lib.cbrs_compact_ids(_ptr(ids, torch.int64), n, _ptr(uniques), _ptr(inverse), _ptr(count), _ptr(ws),
                                 ws.numel(), _stream()), "cbrs_compact_ids")
    return uniques[:int(count.item())], inverse


def lookup_ids(vocab_sorted, ids):
    """index of each id in the sorted vocabulary (int64), -1 where absent"""
    lib = L.load()
    out = torch.empty(ids.numel(), dtype=torch.int64, device=ids.device)
    L.check(lib.cbrs_lookup_ids(_ptr(vocab_sorted, torch.int64), vocab_sorted.numel(), _ptr(ids, torch.int64),
                                ids.numel(), _ptr(out), _stream()), "cbrs_lookup_ids")
    return out


# ------------------------------------------------------------------ DGCF operator build (scope row (f)-3)
def spgemm_products(left, right):
    """COO (row int32, col int32, val float32) of the elementary products of left @ right (both graph.CsrSlice);
    duplicates are NOT summed here - cbrs_graph_build_csr does that."""
    lib = L.load()
    dev = left.rowptr.device
    offsets = torch.empty(left.n_rows, dtype=torch.int64, device=dev)
    total = torch.zeros(1, dtype=torch.int64, device=dev)
    ws = _ws(lib.cbrs_spgemm_workspace_bytes(left.n_rows), dev)
    L.check(lib.cbrs_spgemm_count(ctypes.byref(left.desc), ctypes.byref(right.desc), _ptr(offsets), _ptr(total), _ptr(ws),
                                  ws.numel(), _stream()), "cbrs_spgemm_count")
    n = int(total.item())
    row = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
    col = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
    val = torch.empty(max(n, 1), dtype=torch.float32, device=dev)
    L.check(lib.cbrs_spgemm_expand(ctypes.byref(left.desc), ctypes.byref(right.desc), _ptr(offsets), _ptr(row), _ptr(col),
                                   _ptr(val), _stream()), "cbrs_spgemm_expand")
    return row[:n], col[:n], val[:n]


def count_above(vals, eps_list):
    """[#(vals > eps) for eps in eps_list] (python ints)"""
    lib = L.load()
    k = len(eps_list)
    counts = torch.zeros(k, dtype=torch.int64, device=vals.device)
    L.check(lib.cbrs_count_above(_ptr(vals, torch.float32), vals.numel(), (ctypes.c_float * k)(*[float(e) for e in eps_list]),
                                 k, _ptr(counts), _stream()), "cbrs_count_above")
    return [int(c) for c in counts.tolist()]


def csr_filter_above(csr, eps, count):
    """COO of the entries of `csr` (with values) greater than eps; `count` from count_above"""
    lib = L.load()
    dev = csr.rowptr.device
    row = torch.empty(max(count, 1), dtype=torch.int32, device=dev)
    col = torch.empty(max(count, 1), dtype=torch.int32, device=dev)
    val = torch.empty(max(count, 1), dtype=torch.float32, device=dev)
    ws = _ws(lib.cbrs_csr_filter_above_workspace_bytes(csr.nnz), dev)
    L.check(lib.cbrs_csr_filter_above(ctypes.byref(csr.desc), float(eps), _ptr(row), _ptr(col), _ptr(val), _ptr(ws),
                                      ws.numel(), _stream()), "cbrs_csr_filter_above")
    return row[:count], col[:count], val[:count]


def row_gate(x, w, out=None):
    """x * sigmoid(w) with w [N] or [N,1] (LocalityAdaptive, dgcf_conv.py:101-102)"""
    lib = L.load()
    x, ldx = _rowmajor(x)
    rows, d = x.shape
    if out is None:
        out = torch.empty(rows, d, dtype=torch.float32, device=x.device)
    out, ldo = _rowmajor(out)
    L.check(lib.cbrs_row_gate(_ptr(x), ldx, _ptr(w.reshape(-1), torch.float32), rows, d, _ptr(out), ldo, _stream()),
            "cbrs_row_gate")
    _count(1)
    return out


def row_gate_grad(g, x, w):
    """(dx [N,d], dw [N]) of out = x * sigmoid(w)"""
    lib = L.load()
    g, ldg = _rowmajor(g)
    x, ldx = _rowmajor(x)
    rows, d = x.shape
    dx = torch.empty(rows, d, dtype=torch.float32, device=x.device)
    dw = torch.empty(rows, dtype=torch.float32, device=x.device)
    L.check(lib.cbrs_row_gate_grad(_ptr(g), ldg, _ptr(x), ldx, _ptr(w.reshape(-1), torch.float32), rows, d, _ptr(dx), d,
                                   _ptr(dw), _stream()), "cbrs_row_gate_grad")
    _count(1)
    return dx, dw


# ------------------------------------------------------------------ hybrid tweaks grid (scope row (f)-3)
def attn_fuse(a, b, ta, tb):
    """softmax over the two sources, per feature: (e^ta a + e^tb b) / (e^ta + e^tb)"""
    lib = L.load()
    a, lda = _rowmajor(a)
    b, ldb = _rowmajor(b)
    rows, d = a.shape
    out = torch.empty(rows, d, dtype=torch.float32, device=a.device)
    L.check(lib.cbrs_attn_fuse(_ptr(a), lda, _ptr(b), ldb, _ptr(ta.contiguous(), torch.float32),
                               _ptr(tb.contiguous(), torch.float32), rows, d, _ptr(out), d, _stream()), "cbrs_attn_fuse")
    _count(1)
    return out


def attn_fuse_grad(g, a, b, ta, tb):
    """(da, db, dta, dtb) of attn_fuse"""
    lib = L.load()
    g, ldg = _rowmajor(g)
    a, lda = _rowmajor(a)
    b, ldb = _rowmajor(b)
    rows, d = a.shape
    outs = [torch.empty(rows, d, dtype=torch.float32, device=a.device) for _ in range(4)]
    L.check(lib.cbrs_attn_fuse_grad(_ptr(g), ldg, _ptr(a), lda, _ptr(b), ldb, _ptr(ta.contiguous(), torch.float32),
                                    _ptr(tb.contiguous(), torch.float32), rows, d, _ptr(outs[0]), _ptr(outs[1]),
                                    _ptr(outs[2]), _ptr(outs[3]), _stream()), "cbrs_attn_fuse_grad")
    _count(1)
    return outs


def add3_act(a, b, c, act=None):
    """act(a + b + c)"""
    lib = L.load()
    a, lda = _rowmajor(a)
    b, ldb = _rowmajor(b)
    c, ldc = _rowmajor(c)
    rows, d = a.shape
    out = torch.empty(rows, d, dtype=torch.float32, device=a.device)
    code = act if isinstance(act, int) else L.ACTS[act]
    L.check(lib.cbrs_add3_act(_ptr(a), lda, _ptr(b), ldb, _ptr(c), ldc, rows, d, code, _ptr(out), d, _stream()),
            "cbrs_add3_act")
    _count(1)
    return out
