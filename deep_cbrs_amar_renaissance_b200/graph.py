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


# ------------------------------------------------------------------ partitioned build (one rank's row blocks only)
# A rank of a row partition builds the CSR rows of its own blocks and never holds the other ranks' COO entries or the
# whole graph's sort workspace (DESIGN.md section 3).  The COO is streamed twice from a source: pass 1 counts the
# entries of every row (cuts, exact buffer sizes), pass 2 selects the rank's entries in their input order.  Each block
# is then built by the kernels of the whole build with a row offset (cbrs_graph_build_block); the normalised view
# needs every column's degree, so the blocks' degrees are gathered between its two phases (`gather_degrees`).  Every
# slice equals DeviceGraph(...).<view>.row_slice(a, b) bit for bit: rowptr, colidx, vals and chunk decomposition.
PIECE_EDGES = 1 << 25       # edges per generated piece of a synthetic source (2^26 entries, 512 MB of int32 pairs)
PIECE_ENTRIES = 1 << 26     # entries per uploaded piece of a host COO source

# view name -> (cbrs_graph_build flags, values kept): DeviceGraph.norm and DeviceGraph.raw
BLOCK_VIEWS = {"norm": (L.GRAPH_DEDUP_SUM | L.GRAPH_ADD_SELF_LOOPS | L.GRAPH_SYM_NORM, True), "raw": (0, False)}


class SyntheticSource:
    """The graph ops.synth_bipartite(n_users, n_items, n_edges, seed, scatter_items) generates, produced in pieces of
    `piece_edges` edges (cbrs_synth_bipartite_range) instead of all 2 * n_edges entries at once."""

    def __init__(self, n_users, n_items, n_edges, seed, scatter_items=True, piece_edges=None):
        self.n_users, self.n_items, self.n_edges = int(n_users), int(n_items), int(n_edges)
        self.seed, self.scatter_items = int(seed), bool(scatter_items)
        self.n_nodes = self.n_users + self.n_items
        self.piece_edges = int(piece_edges or PIECE_EDGES)

    def pieces(self, device):
        """(row, col, val=None) pieces whose concatenation is the whole COO in its order: the forward entries of every
        edge range, then their reverses.  A piece is valid until the next one is requested (stream order)."""
        pe = min(self.piece_edges, max(self.n_edges, 1))
        buf = (torch.empty(2 * pe, dtype=torch.int32, device=device), torch.empty(2 * pe, dtype=torch.int32, device=device))
        for half in (0, 1):
            for lo in range(0, self.n_edges, pe):
                hi = min(lo + pe, self.n_edges)
                m = hi - lo
                row, col = ops.synth_bipartite_range(self.n_users, self.n_items, self.n_edges, self.seed, lo, hi, device,
                                                     self.scatter_items, out=buf)
                yield row[half * m:(half + 1) * m], col[half * m:(half + 1) * m], None


class CooSource:
    """A host COO matrix (scipy, any format; the COO entry order is kept, as DeviceGraph.from_scipy keeps it), uploaded
    in pieces of `piece_entries` entries."""

    def __init__(self, adj, piece_entries=None):
        coo = adj.tocoo()
        self.row = np.ascontiguousarray(coo.row, dtype=np.int32)
        self.col = np.ascontiguousarray(coo.col, dtype=np.int32)
        self.val = np.ascontiguousarray(coo.data, dtype=np.float32)
        self.n_nodes = int(coo.shape[0])
        self.piece_entries = int(piece_entries or PIECE_ENTRIES)

    def pieces(self, device):
        for lo in range(0, self.row.shape[0], self.piece_entries):
            hi = min(lo + self.piece_entries, self.row.shape[0])
            yield tuple(torch.from_numpy(a[lo:hi]).to(device) for a in (self.row, self.col, self.val))


def as_source(src):
    """a SyntheticSource / CooSource, or a scipy matrix wrapped as a CooSource"""
    return src if hasattr(src, "pieces") else CooSource(src)


def row_histogram(source, device):
    """Pass 1: the number of COO entries of every row (int64 [n_nodes], on `device`)."""
    source = as_source(source)
    counts = torch.zeros(source.n_nodes, dtype=torch.int64, device=device)
    for row, _, _ in source.pieces(device):
        ops.coo_row_histogram(row, source.n_nodes, counts)
    return counts


def estimated_rowptr(hist, self_loops=True):
    """[N+1] row pointer of the normalised view as far as the histogram tells it: every entry plus a self loop per row.
    Duplicates make it an upper bound; RowPartition(balance_rowptr=...) cuts by it, and the cuts only have to be the
    same on every rank (results do not depend on them)."""
    lens = hist + 1 if self_loops else hist
    return torch.cat([torch.zeros(1, dtype=torch.int64, device=hist.device), torch.cumsum(lens, 0)])


def _select_blocks(source, blocks, hist, device):
    """Pass 2: every block's COO entries (global row ids) in their input order, in exactly sized buffers."""
    caps = [int(hist[a:b].sum().item()) for a, b in blocks]
    sel = []
    for cap in caps:
        sel.append([torch.empty(cap, dtype=torch.int32, device=device), torch.empty(cap, dtype=torch.int32, device=device),
                    None, torch.zeros(1, dtype=torch.int64, device=device)])
    for row, col, val in source.pieces(device):
        for (a, b), s in zip(blocks, sel):
            if val is not None and s[2] is None:
                s[2] = torch.empty(s[0].numel(), dtype=torch.float32, device=device)
            ops.coo_select_rows(row, col, val, a, b, s[0], s[1], s[2], s[3])
    got = [int(s[3].item()) for s in sel]
    if got != caps:
        raise L.CbrsError("partitioned build: selected {} entries where the histogram counted {}".format(got, caps))
    return [(r, c, v) for r, c, v, _ in sel]


def build_row_blocks(source, blocks, gather_degrees, views=("norm",), hist=None, chunk_edges=DEFAULT_CHUNK_EDGES,
                     device=None):
    """This rank's rows of the graph views `views` ("norm", "raw"): {view: [CsrSlice of rows [a, b) per block]}, each
    equal to DeviceGraph(...).<view>.row_slice(a, b) bit for bit.

    source: a SyntheticSource, CooSource or scipy matrix.  blocks: [(a, b)] non-empty row ranges.  hist: pass 1's
    row_histogram when the caller already has it.  gather_degrees(local) -> full d: called once, for the normalised
    view, with local = [(a, b, d of rows a..b)] of this rank; returns every node's degree (float32 [n_nodes] on the
    device): an all-gather over the ranks (distributed.RowPartition.build_graph), or LoopbackDegrees in one process."""
    source = as_source(source)
    n = source.n_nodes
    blocks = [(int(a), int(b)) for a, b in blocks]
    if any(b <= a or a < 0 or b > n for a, b in blocks):
        raise ValueError("partitioned build: row blocks {} of a {}-node graph (each non-empty)".format(blocks, n))
    unknown = [v for v in views if v not in BLOCK_VIEWS]
    if unknown:
        raise ValueError("partitioned build: views {} (built: {})".format(unknown, sorted(BLOCK_VIEWS)))
    device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    if hist is None:
        hist = row_histogram(source, device)
    coo = _select_blocks(source, blocks, hist, device)
    built = {}
    for view in views:
        flags, _ = BLOCK_VIEWS[view]
        built[view] = [ops.graph_build_block(r, c, v if flags & L.GRAPH_DEDUP_SUM else None, a, b, n, flags)
                       for (a, b), (r, c, v) in zip(blocks, coo)]
    del coo
    if "norm" in built:
        d = gather_degrees([(a, b, blk[3]) for (a, b), blk in zip(blocks, built["norm"])])
        for (a, _), (rowptr, colidx, vals, _) in zip(blocks, built["norm"]):
            ops.graph_block_scale(rowptr, colidx, vals, a, n, d)
        del d
    blocking = blocking_policy(n)
    return {view: [CsrSlice(rowptr, colidx.contiguous(), vals.contiguous() if BLOCK_VIEWS[view][1] else None, n,
                            chunk_edges, row_offset=a, blocking=blocking)
                   for (a, _), (rowptr, colidx, vals, _) in zip(blocks, built[view])]
            for view in views}


class LoopbackDegrees:
    """gather_degrees for the ranks of a partition emulated one after the other in one process: the full degree vector
    is assembled from every rank's blocks, each built in turn (phase 1 of the normalised view, only its degrees kept).
    A call checks that the calling rank's own degrees are the ones assembled, bit for bit."""

    def __init__(self, source, ranges, hist=None, device=None):
        source = as_source(source)
        device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        hist = row_histogram(source, device) if hist is None else hist
        flags = BLOCK_VIEWS["norm"][0]
        self.d = torch.empty(source.n_nodes, dtype=torch.float32, device=device)
        for rank_blocks in ranges:
            blocks = [(a, b) for a, b in rank_blocks if b > a]
            for (a, b), (r, c, v) in zip(blocks, _select_blocks(source, blocks, hist, device)):
                self.d[a:b].copy_(ops.graph_build_block(r, c, v, a, b, source.n_nodes, flags)[3])
                del r, c, v

    def __call__(self, local):
        for a, b, d in local:
            if not torch.equal(d, self.d[a:b]):
                raise L.CbrsError("loopback degrees: rows [{}, {}) differ from the assembled vector".format(a, b))
        return self.d


class PartitionedGraph(DeviceGraph):
    """What a model sees of a partitioned build (distributed.RowPartition.build_graph): the graph's shape and node
    count only.  The rows exist on the ranks that own them, as the partition's csr_slices; whole-graph access raises,
    so no code path can pick up a partial matrix in place of the whole one."""

    def __init__(self, n_nodes, views, chunk_edges=DEFAULT_CHUNK_EDGES):
        self.n_nodes, self.n_rel = int(n_nodes), 1
        self.shape = (self.n_nodes, self.n_nodes)
        self.views = tuple(views)
        self.chunk_edges = chunk_edges
        self.row = self.col = self.val = self.rel = None
        self._views = {}

    def _whole(self, what):
        raise NotImplementedError(
            "{} of a partitioned graph build: each rank holds only its own row blocks (views {}), as "
            "RowPartition.csr_slices; build a DeviceGraph for whole-graph access".format(what, ", ".join(self.views)))

    def _view(self, name, flags, keep_vals, self_rel=0):
        self._whole("the '%s' view" % name)

    @property
    def symmetric(self):
        self._whole("the symmetry test")

    @property
    def dgcf(self):
        self._whole("the 'dgcf' view")

    def transposed(self):
        self._whole("the transpose")

    def row_subset(self, ids):
        self._whole("a row subset")

    def release_coo(self):
        pass


def refuse_partitioned(graphs, what):
    """NotImplementedError when one of `graphs` is a PartitionedGraph: `what` has no partitioned build."""
    if any(isinstance(g, PartitionedGraph) for g in graphs):
        raise NotImplementedError("{} on a partitioned graph build (it has no partitioned form; build a DeviceGraph)"
                                  .format(what))
