"""Device-resident graph: the adjacency the reference hands to its layers as a
tf.SparseTensor (/root/reference/src/models/gnn.py:49, src/utilities/math.py:37-56),
kept in HBM as CSR + a chunk decomposition.

Two views are built on demand from the same COO entries:
  * norm: duplicates summed, self loops added, D^-1/2 (A+I) D^-1/2  -> GCN, LightGCN
          (what GCNConv.preprocess / LightGCNConv.preprocess return, gnn.py:283,380)
  * raw : row-major sorted, duplicates kept, values ignored          -> GraphSAGE, GAT
          (gnn.py:298-319,331-352 pass the adjacency through untouched)
"""
import os

import numpy as np
import torch

from . import _lib as L
from . import ops

DEFAULT_CHUNK_EDGES = 1024

# Column-blocked schedule (cbrs_chunks_blocked_*): used when the gathered operand table cannot stay in L2.  The
# policy is a function of the GLOBAL column count only, so every rank of a row partition and the single-GPU run
# cut a row at the same places (bit-identical results).  CBRS_BLOCK_COLS / CBRS_BLOCK_MIN_LEN override it
# (0 disables); tuned on config 5 (profiles/r02_tune_blocked.log).
BLOCK_COLS = 98304          # operand rows per window: 48 MB at D = 128 fp32 (L2: 126 MB, two dies)
BLOCK_MIN_LEN = 1024        # rows shorter than this stay row-major (a partial per segment would cost more than it saves)
BLOCK_MIN_COLS = 1 << 19    # tables below 2^19 rows (256 MB at D = 128) are left to the L2's own replacement


FORCED_BLOCKING = None      # (block_cols, block_min_len): tests and the multi-GPU self-check block small graphs with it


def blocking_policy(n_cols):
    """(block_cols, block_min_len) for a graph with n_cols columns; (0, 0) = row-major schedule."""
    if FORCED_BLOCKING is not None:
        return tuple(FORCED_BLOCKING)
    cols = int(os.environ.get("CBRS_BLOCK_COLS", BLOCK_COLS))
    min_len = int(os.environ.get("CBRS_BLOCK_MIN_LEN", BLOCK_MIN_LEN))
    min_cols = int(os.environ.get("CBRS_BLOCK_MIN_COLS", BLOCK_MIN_COLS))
    if cols <= 0 or min_len <= 0 or n_cols < min_cols:
        return 0, 0
    return cols, min_len


# Per-batch model call: a GCN / LightGCN stack whose layers are concatenated is read by the scorer only at the batch's
# rows, so its LAST layer's sparse product may run on those rows alone (graph.CsrSubset).  Layers before it stay full:
# their outputs feed the last layer at every neighbour.  The subset costs a few passes over the chunk list and one
# small device-to-host copy per call; on graphs of at least this many rows that is far below the rows it skips
# (config 5, 1.1e7 rows: ~3.5 % of the last layer's edges are needed by a 65,536-pair batch).  The MovieLens-1M-sized
# graphs (~1e4 rows, a batch needs ~40 % of them) stay on the full product, and their launch count.
SUBSET_MIN_ROWS = 1 << 20
FORCED_SUBSET = None        # True / False: tests decide the size condition with it


def last_layer_subset_policy(n_rows, partitioned, concatenated, last_layer_gcn):
    """True when the per-batch call computes the last layer's sparse product only at the rows its batch scores.
    Never under a row partition, for other reductions or layer families, or while a CUDA graph is being captured (a
    replay must stay valid for any ids)."""
    if partitioned or not concatenated or not last_layer_gcn:
        return False
    large = bool(FORCED_SUBSET) if FORCED_SUBSET is not None else n_rows >= SUBSET_MIN_ROWS
    return large and not torch.cuda.is_current_stream_capturing()


class CsrSlice:
    """Rows [row_offset, row_offset + n_rows) of a CSR matrix plus its work decomposition."""

    def __init__(self, rowptr, colidx, vals, n_cols, chunk_edges=DEFAULT_CHUNK_EDGES, row_offset=0, blocking=None):
        self.rowptr, self.colidx, self.vals = rowptr, colidx, vals
        self.n_rows = rowptr.numel() - 1
        self.n_cols = n_cols
        self.nnz = colidx.numel()
        self.row_offset = row_offset
        self.chunk_edges = chunk_edges
        self.blocking = blocking_policy(n_cols) if blocking is None else tuple(blocking)
        self.chunks = ops.build_chunks(rowptr, chunk_edges, colidx, n_cols, *self.blocking)
        self.desc = _desc(self, self.chunks)

    def row_slice(self, r0, r1, chunk_edges=None):
        """Rows [r0, r1) with global column ids (1-D row partition, SURVEY 8e)."""
        b, e = int(self.rowptr[r0].item()), int(self.rowptr[r1].item())
        rowptr = (self.rowptr[r0:r1 + 1] - b).contiguous()
        vals = self.vals[b:e].contiguous() if self.vals is not None else None
        return CsrSlice(rowptr, self.colidx[b:e].contiguous(), vals, self.n_cols,
                        chunk_edges or self.chunk_edges, self.row_offset + r0, blocking=self.blocking)

    def row_subset(self, ids):
        """The rows `ids` of this slice as a CsrSubset (int64 device ids, local row numbers)."""
        return CsrSubset(self, ids)

    def coo_rows(self):
        """row id of every stored entry (int32 [nnz])"""
        lens = self.rowptr[1:] - self.rowptr[:-1]
        return torch.repeat_interleave(torch.arange(self.n_rows, dtype=torch.int32, device=self.rowptr.device), lens)

    def transposed(self):
        """The transpose as a CsrSlice ([n_cols, n_rows], entries of a row in ascending column order, duplicates
        kept): what the backward of a sparse layer multiplies by when the adjacency is not symmetric, and, for the
        relational operator's stacked [N, R*N] layout, the matrix whose one product yields every relation's dZ."""
        if getattr(self, "_t", None) is None:
            m = max(self.n_rows, self.n_cols)
            rowptr, colidx, vals = ops.graph_build_csr(self.colidx, self.coo_rows(), self.vals, m, 0)
            rowptr = rowptr[:self.n_cols + 1].contiguous()
            self._t = CsrSlice(rowptr, colidx.contiguous(), vals.contiguous() if self.vals is not None else None,
                               self.n_rows, self.chunk_edges, blocking=self.blocking)
        return self._t

    def to_scipy(self):
        from scipy import sparse
        vals = (self.vals if self.vals is not None else torch.ones_like(self.colidx, dtype=torch.float32)).cpu().numpy()
        return sparse.csr_matrix((vals, self.colidx.cpu().numpy(), self.rowptr.cpu().numpy()),
                                 shape=(self.n_rows, self.n_cols))


def _desc(csr, c):
    """cbrs_csr_t of the matrix held by `csr` under the chunk decomposition `c` (ops.build_chunks / ops.csr_subset)"""
    d = L.CsrDesc()
    d.n_rows, d.nnz = csr.n_rows, csr.colidx.numel()
    d.rowptr, d.colidx = csr.rowptr.data_ptr(), csr.colidx.data_ptr()
    d.vals = csr.vals.data_ptr() if csr.vals is not None else None
    d.chunk_edges, d.n_chunks = csr.chunk_edges, c["n_chunks"]
    d.chunk_row, d.chunk_begin, d.chunk_slot = (c["chunk_row"].data_ptr(), c["chunk_begin"].data_ptr(),
                                                c["chunk_slot"].data_ptr())
    d.n_heavy, d.n_slots = c["n_heavy"], c["n_slots"]
    d.heavy_row = c["heavy_row"].data_ptr() if c["n_heavy"] else None
    d.heavy_slot_ptr = c["heavy_slot_ptr"].data_ptr()
    d.chunk_len = c["chunk_len"].data_ptr() if c["chunk_len"] is not None else None
    return d


class CsrSubset:
    """Some rows of a CsrSlice: the same matrix, with only those rows' chunks, in their original order, and their
    partial slots renumbered in order (cbrs_csr_subset_*).  A propagation launch on it writes exactly those rows of its
    [n_rows, D] output, each with the bits the full launch gives it, and leaves every other row as it was."""

    def __init__(self, full, ids):
        self.full = full    # keeps the shared rowptr / colidx / vals alive
        self.rowptr, self.colidx, self.vals = full.rowptr, full.colidx, full.vals
        self.n_rows, self.n_cols, self.row_offset = full.n_rows, full.n_cols, full.row_offset
        self.chunk_edges, self.blocking = full.chunk_edges, full.blocking
        self.chunks = ops.csr_subset(full, ids)
        self.n_needed = self.chunks["rows"]     # distinct rows a launch computes
        self.nnz = self.chunks["edges"]         # the edges it gathers
        self.desc = _desc(self, self.chunks)


class DeviceGraph:
    def __init__(self, row, col, val, n_nodes, chunk_edges=DEFAULT_CHUNK_EDGES, rel=None, n_rel=1):
        ops.check_device()
        self.row, self.col, self.val, self.rel = row, col, val, rel
        self.n_nodes, self.n_rel = int(n_nodes), int(n_rel)
        self.chunk_edges = chunk_edges
        self.shape = (self.n_nodes, self.n_nodes)
        self._views = {}

    @classmethod
    def from_scipy(cls, adj, device=None, chunk_edges=DEFAULT_CHUNK_EDGES, relational=False):
        """scipy sparse (any format; COO entry order is preserved) -> device COO.  relational=True keeps the edge types
        of a data.preprocess.RelationalAdjacency (RGCN); every other layer family sees the untyped graph."""
        if isinstance(adj, DeviceGraph):
            return adj
        device = torch.device(device or "cuda")
        coo = adj.tocoo()
        row = torch.from_numpy(np.ascontiguousarray(coo.row, dtype=np.int32)).to(device)
        col = torch.from_numpy(np.ascontiguousarray(coo.col, dtype=np.int32)).to(device)
        val = torch.from_numpy(np.ascontiguousarray(coo.data, dtype=np.float32)).to(device)
        if relational and hasattr(adj, "rel") and hasattr(adj, "n_rel"):   # typed edges (row R)
            rel = torch.from_numpy(np.ascontiguousarray(adj.rel, dtype=np.int32)).to(device)
            return cls(row, col, val, coo.shape[0], chunk_edges, rel=rel, n_rel=adj.n_rel)
        return cls(row, col, val, coo.shape[0], chunk_edges)

    def _view(self, name, flags, keep_vals, self_rel=0):
        if name not in self._views:
            rowptr, colidx, vals = ops.graph_build_csr(self.row, self.col, self.val, self.n_nodes, flags,
                                                       rel=self.rel, n_rel=self.n_rel, self_rel=self_rel)
            self._views[name] = CsrSlice(rowptr, colidx.contiguous(), vals.contiguous() if keep_vals else None,
                                         self.n_nodes * self.n_rel, self.chunk_edges)
        return self._views[name]

    def release_coo(self):
        """Drop the COO entries once the needed views exist (frees 12 B per entry)."""
        self.row = self.col = self.val = self.rel = None

    @property
    def symmetric(self):
        """True when the entries (row, col[, rel], value) and (col, row[, rel], value) form the same multiset, i.e.
        A == A^T with duplicates.  The explicit backward of the sparse layers multiplies by the FORWARD operator only
        in that case (training.py); the loaders build such graphs for `symmetric_adjacency: True`
        (/root/reference/src/data/preprocess.py:83-84), which every grid of the reference uses."""
        if getattr(self, "_symmetric", None) is None:
            if self.row is not None:
                row, col, val, rel = self.row.long(), self.col.long(), self.val, self.rel
            else:
                v = next(iter(self._views.values()))
                row, col, val, rel = v.coo_rows().long(), v.colidx.long() % self.n_nodes, v.vals, v.colidx.long() // self.n_nodes
                if self.n_rel == 1:
                    rel = None
            n = self.n_nodes
            r = rel.long() * n * n if rel is not None else 0
            a, b = r + row * n + col, r + col * n + row

            def canon(k):
                if val is None:
                    return torch.sort(k)[0], None
                o1 = torch.sort(val, stable=True)[1]
                o2 = torch.sort(k[o1], stable=True)[1]
                o = o1[o2]
                return k[o], val[o]
            (ka, va), (kb, vb) = canon(a), canon(b)
            self._symmetric = bool(torch.equal(ka, kb) and (va is None or torch.equal(va, vb)))
        return self._symmetric

    @property
    def norm(self):
        return self._view("norm", L.GRAPH_DEDUP_SUM | L.GRAPH_ADD_SELF_LOOPS | L.GRAPH_SYM_NORM, True)

    @property
    def raw(self):
        return self._view("raw", 0, False)

    @property
    def plain(self):
        """duplicates summed, values kept, nothing else: scipy's A.tocsr()"""
        return self._view("plain", L.GRAPH_DEDUP_SUM, True)

    DGCF_EPSILONS = (1e-1, 1e-2, 1e-3, 5e-4)  # dgcf_conv.py:60

    @property
    def dgcf(self):
        """DGCFConv.preprocess on device (/root/reference/src/layers/dgcf_conv.py:38-80):
        gcn_filter(A) + high_pass(gcn_filter(A.A)) + I as one CSR."""
        if "dgcf" not in self._views:
            n = self.n_nodes
            a = self.plain
            r, c, v = ops.spgemm_products(a, a)                                   # crosshop = a.dot(a)
            flags = L.GRAPH_DEDUP_SUM | L.GRAPH_ADD_SELF_LOOPS | L.GRAPH_SYM_NORM
            cross = CsrSlice(*[t.contiguous() for t in ops.graph_build_csr(r, c, v, n, flags)], n, self.chunk_edges)
            del r, c, v
            a_hat = self.norm                                                      # gcn_filter(a)
            counts = ops.count_above(cross.vals, self.DGCF_EPSILONS)
            edges = a_hat.nnz
            ratios = [float("inf") if k == 0 else (edges / k if edges > k else k / edges) for k in counts]
            best = min(range(len(ratios)), key=lambda j: (ratios[j], j))           # argmin, first on ties
            self.dgcf_info = dict(edges=edges, cross_edges=counts, ratios=ratios, epsilon=self.DGCF_EPSILONS[best])
            fr, fc, fv = ops.csr_filter_above(cross, self.DGCF_EPSILONS[best], counts[best])
            ar, ac, av = ops.csr_filter_above(a_hat, float("-inf"), a_hat.nnz)     # A_hat as COO
            eye = torch.arange(n, dtype=torch.int32, device=fr.device)
            row = torch.cat([ar, fr, eye])
            col = torch.cat([ac, fc, eye])
            val = torch.cat([av, fv, torch.ones(n, dtype=torch.float32, device=fr.device)])
            rowptr, colidx, vals = ops.graph_build_csr(row, col, val, n, L.GRAPH_DEDUP_SUM)  # (a + crosshop) + I
            self._views["dgcf"] = CsrSlice(rowptr, colidx.contiguous(), vals.contiguous(), n, self.chunk_edges)
        return self._views["dgcf"]
