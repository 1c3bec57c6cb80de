"""Row-partitioned propagation over several GPUs of one box (SURVEY.md 8e).

One process per GPU (torch.distributed, NCCL over NVLink/NVSwitch).  Output rows of a layer
are independent given all input rows, so rank r owns a block of user rows and a block of item
(+property) rows - interleaving the two node types balances edges, because user rows are
short and item rows long - computes them with the same kernels on CSR row slices (global
column ids), and the layer outputs are exchanged with an all-gather.  Every row's reduction
order is rank-independent (ascending columns, fixed chunk tree), so the G-rank result equals
the 1-rank result bit for bit.  Scoring is sharded by user with items replicated: no
collective.

Two exchange mechanisms (RowPartition(exchange=...)):
  "peer" (default on GPUs): the operand buffers are symmetric peer-mapped allocations
         (PeerHeap, CUDA IPC over NVLink/NVSwitch) and the kernel that PRODUCES an operand
         stores every finished row into all ranks' copies (cbrs_dense_bcast /
         cbrs_spmm_csr_bcast / cbrs_gat_csr_bcast); a one-CTA flag barrier
         (cbrs_peer_barrier) is the only thing between producer and consumer.  No NCCL call
         on the data path.
  "nccl": producer kernel, then an all-gather (the baseline; also what the gloo CPU tests
         exercise).
"""
import ctypes
import os

import torch
import torch.distributed as dist


def block_ranges(n_rows_by_type, world_size):
    """[[(r0, r1) per node type] per rank]; each type's rows are cut into world_size blocks of
    ceil(n/world_size) rows (the last may be short or empty).  `n_rows_by_type` lists the
    sizes of the consecutive id ranges (users, items[, properties])."""
    out = [[] for _ in range(world_size)]
    base = 0
    for n in n_rows_by_type:
        blk = -(-n // world_size)
        for r in range(world_size):
            lo = min(r * blk, n)
            hi = min(lo + blk, n)
            out[r].append((base + lo, base + hi))
        base += n
    return out


# Relative cost of one edge of a row that is NOT column-blocked (graph.blocking_policy) on a graph whose operand table
# exceeds L2: its gathers stream from HBM, a blocked row's come out of the L2 window.  Calibrated on the unscattered
# config-5 graph over 4 GPUs (profiles/r02_bench_c5_n4_unscattered*.json): with 1.4 the rank holding the hottest items
# finished its item rows in 26.7 ms against 48-54 ms for the ranks holding the cold tail, i.e. a streamed edge costs
# about 2.5 blocked ones.  CBRS_COLD_EDGE_COST overrides.
COLD_EDGE_COST = float(os.environ.get("CBRS_COLD_EDGE_COST", "2.4"))


def edge_cost_prefix(rowptr, n_rows_by_type, block_min_len=0, cold_cost=COLD_EDGE_COST):
    """[N+1] prefix sums of a per-row cost for balanced_ranges: the row's edge count, times `cold_cost` for rows of
    node types that contain column-blocked rows (>= block_min_len edges) but are themselves below the threshold.
    block_min_len == 0 (row-major schedule): plain edge counts, i.e. rowptr itself."""
    if not block_min_len:
        return rowptr
    lens = (rowptr[1:] - rowptr[:-1]).to(torch.float64)
    cost = lens.clone()
    base = 0
    for n in n_rows_by_type:
        seg = lens[base:base + n]
        if n and bool((seg >= block_min_len).any()):
            cost[base:base + n] = torch.where(seg >= block_min_len, seg, seg * cold_cost)
        base += n
    return torch.cat([torch.zeros(1, dtype=torch.float64, device=rowptr.device), torch.cumsum(cost, 0)])


def balanced_ranges(n_rows_by_type, world_size, rowptr):
    """block_ranges with each node type cut at (about) equal EDGE count (or edge COST, when `rowptr` is an
    edge_cost_prefix) instead of equal row count: block r of a type ends at the first row whose prefix reaches r/world
    of the type's total (SURVEY 8e).  `rowptr` is the [N+1] row pointer of the CSR view the sparse kernel runs on (host
    or device tensor); every rank computes the same cuts from it.  Real ids come out of np.unique in id order, so
    popular items may sit next to each other; equal row counts would then give one rank most of the edges."""
    out = [[] for _ in range(world_size)]
    base = 0
    for n in n_rows_by_type:
        rp = rowptr[base:base + n + 1]
        cuts = [0] * (world_size + 1)
        cuts[world_size] = n
        if n > 0:
            lo, hi = rp[0].item(), rp[-1].item()
            targets = torch.tensor([lo + (hi - lo) * k / world_size for k in range(1, world_size)], device=rp.device).to(rp.dtype)
            mids = torch.searchsorted(rp.contiguous(), targets).tolist() if world_size > 1 else []
            for k, m in enumerate(mids):
                cuts[k + 1] = min(max(int(m), cuts[k]), n)
        for r in range(world_size):
            out[r].append((base + cuts[r], base + max(cuts[r + 1], cuts[r])))
        base += n
    return out


def exchange_rows(x, ranges, group=None):
    """All ranks end up with every row block of x (each block is authored by its owner).

    Even blocks take one all_gather_into_tensor per node type (in place: the owner's block is
    already where the gathered tensor wants it); ragged blocks fall back to one broadcast per
    owner.  x must be row-contiguous [N, H]."""
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    n_types = len(ranges[0])
    for t in range(n_types):
        sizes = [ranges[r][t][1] - ranges[r][t][0] for r in range(world)]
        lo = ranges[0][t][0]
        if len(set(sizes)) == 1 and sizes[0] > 0 and x.is_contiguous():
            span = x[lo:lo + world * sizes[0]]
            mine = x[ranges[rank][t][0]:ranges[rank][t][1]]
            dist.all_gather_into_tensor(span, mine, group=group)
        else:
            for r in range(world):
                a, b = ranges[r][t]
                if b > a:
                    dist.broadcast(x[a:b], src=dist.get_global_rank(group, r) if group is not None else r, group=group)
    return x


def gather_degrees_dist(ranges, n_nodes, group=None):
    """gather_degrees for graph.build_row_blocks in a real run: every rank contributes its blocks' degrees and gets the
    whole vector (float32 [n_nodes]), one broadcast per block: the blocks are ragged, and gloo groups take it too."""
    def gather(local):
        d = torch.zeros(n_nodes, dtype=torch.float32, device=local[0][2].device if local else "cuda")
        for a, b, v in local:
            d[a:b].copy_(v)
        for r, blocks in enumerate(ranges):
            src = dist.get_global_rank(group, r) if group is not None else r
            for a, b in blocks:
                if b > a:
                    dist.broadcast(d[a:b], src=src, group=group)
        return d
    return gather


class SymmetricBuffer:
    """One allocation of a PeerHeap: the same number of bytes on every rank, all copies mapped here."""

    def __init__(self, heap, nbytes, ptrs, mc_ptr=0, keep=None):
        self.heap, self.nbytes, self.ptrs = heap, nbytes, ptrs  # ptrs[r] = address of rank r's copy
        self.mc_ptr = int(mc_ptr or 0)   # NVSwitch multicast mapping of all copies (0: none); a store there lands in every copy
        self._keep = keep                # the torch symmetric-memory tensor + handle that own the mapping ("symm" backend)
        self.local = ptrs[heap.rank]
        self._iface = type("_Raw", (), {})()
        self._iface.__cuda_array_interface__ = {"shape": (nbytes // 4,), "typestr": "<f4",
                                                "data": (self.local, False), "version": 2}
        self.flat = torch.as_tensor(self._iface, device=torch.device("cuda", torch.cuda.current_device()))
        if self.flat.data_ptr() != self.local:
            raise RuntimeError("torch copied the symmetric buffer instead of viewing it")

    def matrix(self, n, w, dtype=torch.float32):
        """[n, w] view of the local copy (float32 or bfloat16)"""
        if dtype == torch.bfloat16:
            return self.flat.view(torch.bfloat16)[:n * w].view(n, w)
        return self.flat[:n * w].view(n, w)

    def peer_addrs(self, view):
        """addresses, in every OTHER rank's copy, of `view` (a view into the local copy)"""
        off = view.data_ptr() - self.local
        if off < 0 or off >= self.nbytes:
            raise ValueError("view does not live in this symmetric buffer")
        return [p + off for r, p in enumerate(self.ptrs) if r != self.heap.rank]

    def mc_addr(self, view):
        """address of `view` in the multicast mapping, or None when the buffer has none"""
        if not self.mc_ptr:
            return None
        off = view.data_ptr() - self.local
        if off < 0 or off >= self.nbytes:
            raise ValueError("view does not live in this symmetric buffer")
        return self.mc_ptr + off


class PeerHeap:
    """Symmetric peer-mapped allocations for the ranks of one box + the flag barrier.
    alloc() is collective: every rank calls it in the same order with the same size."""

    def __init__(self, group=None, backend=None):
        """backend: "ipc" = cudaMalloc + CUDA IPC handles (cbrs_peer_*); "symm" = torch.distributed symmetric memory
        (plumbing only: allocation + rendezvous), which also maps the buffers through an NVSwitch MULTICAST object when
        the fabric supports it (NCCL calls the same facility NVLS) - SymmetricBuffer.mc_ptr.  Default: CBRS_PEER_BACKEND
        or "symm", falling back to "ipc" together on every rank if symmetric memory cannot be set up."""
        from . import _lib as L
        self.group = group
        self.world = dist.get_world_size(group)
        self.rank = dist.get_rank(group)
        self.backend = backend or os.environ.get("CBRS_PEER_BACKEND", "symm")
        if self.backend not in ("ipc", "symm"):
            raise ValueError("peer backend must be 'ipc' or 'symm'")
        if self.backend == "symm":
            ok = 1
            try:
                import torch.distributed._symmetric_memory as symm_mem   # noqa: F401
                probe = self._alloc_symm(256)
                del probe
            except Exception as e:  # noqa: BLE001
                ok, self._symm_error = 0, e
            flag = torch.tensor([ok], dtype=torch.int32, device="cuda")
            dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)
            if int(flag.item()) != 1:
                self.backend = "ipc"
        if self.world > L.MAX_PEERS:
            raise L.CbrsError("peer exchange supports up to {} ranks (one NVSwitch box)".format(L.MAX_PEERS))
        self._lib = L.load()
        self._owned, self._opened = [], []
        self._open_error = None
        self.flags = self.alloc(L.MAX_PEERS * 8)
        self.status = torch.zeros(1, dtype=torch.int32, device="cuda")
        self.epoch = 0
        ok = torch.tensor([0 if self._open_error else 1], dtype=torch.int32, device="cuda")
        dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=group)
        if int(ok.item()) != 1:  # every rank raises together (nobody is left spinning in the flag barrier)
            raise L.CbrsError("peer mapping failed: {}".format(self._open_error or "on another rank"))
        self.barrier()
        self.check()

    def _alloc_symm(self, nbytes):
        import torch.distributed._symmetric_memory as symm_mem
        t = symm_mem.empty(nbytes // 4, dtype=torch.float32, device=torch.device("cuda", torch.cuda.current_device()))
        hdl = symm_mem.rendezvous(t, self.group if self.group is not None else dist.group.WORLD)
        t.zero_()
        torch.cuda.synchronize()
        ptrs = [int(a) for a in hdl.buffer_ptrs]
        ptrs[self.rank] = t.data_ptr()
        mc = int(hdl.multicast_ptr) if getattr(hdl, "has_multicast_support", lambda *_: True) and hdl.multicast_ptr else 0
        if os.environ.get("CBRS_MULTICAST", "1") == "0":
            mc = 0
        return SymmetricBuffer(self, nbytes, ptrs, mc_ptr=mc, keep=(t, hdl))

    def alloc(self, nbytes):
        from . import _lib as L
        nbytes = (int(nbytes) + 255) // 256 * 256
        if self.backend == "symm":
            sb = self._alloc_symm(nbytes)
            dist.barrier(group=self.group)   # every rank zeroed its copy before anybody stores into it
            return sb
        ptr = ctypes.c_void_p()
        handle = (ctypes.c_ubyte * L.IPC_HANDLE_BYTES)()
        # a local failure (cudaMalloc out of memory, export error) must not skip the collective below: the other
        # ranks would wait in it forever.  Every rank sends (size, handle or None, error) and all decide together.
        local_error = None
        try:
            L.check(self._lib.cbrs_peer_alloc(nbytes, ctypes.byref(ptr)), "cbrs_peer_alloc")
            self._owned.append(ptr.value)
            L.check(self._lib.cbrs_peer_export(ptr, handle), "cbrs_peer_export")
        except L.CbrsError as e:
            local_error = str(e)
        handles = [None] * self.world
        dist.all_gather_object(handles, (nbytes, None if local_error else bytes(handle), local_error), group=self.group)
        failed = [(r, err) for r, (_, _, err) in enumerate(handles) if err]
        if failed:
            raise L.CbrsError("symmetric allocation of {} bytes failed on rank {}: {}".format(nbytes, *failed[0]))
        ptrs = []
        for r, (nb, h, _) in enumerate(handles):
            if nb != nbytes:
                raise L.CbrsError("symmetric allocation sizes differ: rank {} asked for {} bytes, rank {} for {}"
                                  .format(self.rank, nbytes, r, nb))
            if r == self.rank:
                ptrs.append(ptr.value)
                continue
            q = ctypes.c_void_p()
            try:
                L.check(self._lib.cbrs_peer_open((ctypes.c_ubyte * L.IPC_HANDLE_BYTES).from_buffer_copy(h),
                                                 ctypes.byref(q)), "cbrs_peer_open")
            except L.CbrsError as e:
                if getattr(self, "status", None) is not None:
                    raise  # after construction every rank already knows P2P works; a later failure is fatal
                self._open_error = e
                ptrs.append(0)
                continue
            self._opened.append(q.value)
            ptrs.append(q.value)
        return SymmetricBuffer(self, nbytes, ptrs)

    def barrier(self):
        """Stream-ordered rendezvous of all ranks (cbrs_peer_barrier) on torch's current stream."""
        from . import _lib as L
        from . import ops
        self.epoch += 1
        arr = (ctypes.c_void_p * self.world)(*self.flags.ptrs)
        if ops.PROFILE_ON:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        L.check(self._lib.cbrs_peer_barrier(arr, self.world, self.rank, self.epoch,
                                            ctypes.c_void_p(self.status.data_ptr()), 30.0,
                                            ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)),
                "cbrs_peer_barrier")
        ops._count(1)
        if ops.PROFILE_ON:
            e1.record()
            ops.PROFILE.append(("barrier", e0, e1, None))

    def check(self):
        """Synchronises; raises if any barrier so far timed out.  (A timed-out barrier kernel also traps, so the
        stream is already dead and this read itself raises a CUDA error: either way the failure is loud.)"""
        from . import _lib as L
        if int(self.status.item()) != 0:
            raise L.CbrsError("peer barrier timed out: a rank did not arrive within 30 s")

    def close(self):
        torch.cuda.synchronize()
        self.check()
        dist.barrier(group=self.group)
        self.flags = None   # "symm" backend: the mappings go with the tensors
        for q in self._opened:
            self._lib.cbrs_peer_close(ctypes.c_void_p(q))
        self._opened = []
        dist.barrier(group=self.group)
        for q in self._owned:
            self._lib.cbrs_peer_free(ctypes.c_void_p(q))
        self._owned = []


class RowPartition:
    """Attach to a SequentialGNN to run its layer loop on this rank's row blocks.

    What travels per layer:
      GCN        : under the peer exchange, the layer OUTPUT: every rank computes the whole transform
                   Z = X W from a layer input that is complete on every rank; under "nccl", Z for OWN
                   rows only, all-gathered, then A_hat Z on own rows;
      RGCN       : the stacked Z = [X W_r] for OWN rows only, all-gathered, then A_hat Z on own rows;
      GAT        : z = X W, q = z.a_neigh for own rows, all-gathered; p stays local;
      GraphSage / LightGCN : the layer INPUT X^(l) is all-gathered (layer 0 reads the
                   replicated embedding table).
    After the last layer only the node types in `final_types` (default: everything but users)
    are exchanged, because scoring is sharded by user."""

    # the peer exchange's one GCN schedule: every rank transforms all rows, only layer outputs travel (DESIGN.md section 5).
    # Nothing in the package reads it; bench.py and tools/scale_families.py report it in their output.
    pipeline = "replicate"

    def __init__(self, n_rows_by_type, group=None, final_types=None, exchange=None, balance_rowptr=None,
                 balance_min_len=0):
        self.group = group
        exchange = exchange or os.environ.get("CBRS_EXCHANGE") or ("peer" if torch.cuda.is_available() else "nccl")
        if exchange not in ("peer", "nccl"):
            raise ValueError("exchange must be 'peer' or 'nccl'")
        self.exchange = exchange
        self.heap = None
        if exchange == "peer":
            # mapping a peer's memory can fail on boxes without P2P between some GPU pair; the ranks agree on the
            # outcome (the handle exchange inside PeerHeap is collective, so every rank gets this far) and fall back to
            # the NCCL all-gather together rather than one of them raising while the others wait
            heap, ok = None, 1
            try:
                heap = PeerHeap(group)
            except Exception as e:  # noqa: BLE001
                ok, why = 0, e
            flag = torch.tensor([ok], dtype=torch.int32, device="cuda")
            dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)
            if int(flag.item()) == 1:
                self.heap = heap
            else:
                import warnings
                warnings.warn("peer-memory exchange unavailable ({}); using the NCCL all-gather".format(
                    why if not ok else "another rank could not map its peers"))
                self.exchange = "nccl"
        self._sym = {}
        self.n_rows_by_type = list(n_rows_by_type)
        self.world = dist.get_world_size(group)
        self.rank = dist.get_rank(group)
        # balance_rowptr: the CSR row pointer to balance EDGES by (balanced_ranges); None = equal row counts.
        # balance_min_len: the graph's column-blocking threshold (CsrSlice.blocking[1]) - rows below it in a node type
        # that has blocked rows cost COLD_EDGE_COST per edge (edge_cost_prefix)
        self.ranges = (block_ranges(n_rows_by_type, self.world) if balance_rowptr is None
                       else balanced_ranges(n_rows_by_type, self.world,
                                            edge_cost_prefix(balance_rowptr, n_rows_by_type, balance_min_len)))
        self.mine = [rg for rg in self.ranges[self.rank] if rg[1] > rg[0]]
        self.final_types = list(range(1, len(n_rows_by_type))) if final_types is None else list(final_types)
        self._slices = {}
        self._bufs = {}

    def attach(self, seq_gnn):
        seq_gnn.partition = self
        return self

    def close(self):
        """Unmap and free the symmetric buffers (collective)."""
        self._sym.clear()
        if self.heap is not None:
            self.heap.close()
            self.heap = None

    def csr_slices(self, view_name, graph):
        """This rank's rows of a CSR view: one slice per owned node-type block."""
        if view_name not in self._slices:
            full = getattr(graph, view_name)
            self._slices[view_name] = [full.row_slice(a, b) for a, b in self.mine]
        return self._slices[view_name]

    def build_graph(self, source, views=("norm",), gather_degrees=None, hist=None, chunk_edges=None):
        """Partitioned build: this rank builds only its own row blocks of the graph `views` ("norm" for GCN / LightGCN,
        "raw" for GraphSage / GAT) from `source` (graph.SyntheticSource, graph.CooSource or a scipy matrix), streamed
        twice, and puts them in the csr_slices cache.  Each slice equals the whole build's row_slice bit for bit.
        Returns a graph.PartitionedGraph for the model constructors (BasicGCN(graph, ...)); it has no whole-graph
        views.  gather_degrees: graph.build_row_blocks; default gather_degrees_dist over this partition's group.
        hist: graph.row_histogram(source) when the caller already has it (e.g. to cut the partition with
        balance_rowptr=graph.estimated_rowptr(hist))."""
        from . import graph as G
        source = G.as_source(source)
        n = sum(self.n_rows_by_type)
        if source.n_nodes != n:
            raise ValueError("partitioned build: the source has {} nodes, the partition {}".format(source.n_nodes, n))
        chunk_edges = chunk_edges or G.DEFAULT_CHUNK_EDGES
        gather = gather_degrees or gather_degrees_dist(self.ranges, n, self.group)
        for view, slices in G.build_row_blocks(source, self.mine, gather, views, hist, chunk_edges).items():
            self._slices[view] = slices
        return G.PartitionedGraph(n, views, chunk_edges)

    def release_full_views(self, graph):
        """Keep only this rank's row slices in HBM."""
        graph._views.clear()
        graph.release_coo()

    def local_edges(self, view_name):
        return sum(s.nnz for s in self._slices.get(view_name, []))

    def _buf(self, key, n, w, device, dtype=torch.float32):
        key = key + (str(dtype),)
        if key not in self._bufs:
            self._bufs[key] = torch.empty(n, w, dtype=dtype, device=device)
        return self._bufs[key]

    def _exchange(self, x, types=None):
        from . import ops
        ranges = self.ranges if types is None else [[rg[t] for t in types] for rg in self.ranges]
        if ops.PROFILE_ON:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            exchange_rows(x, ranges, self.group)
            e1.record()
            ops.PROFILE.append(("exchange", e0, e1, x.numel() * 4))
            return x
        return exchange_rows(x, ranges, self.group)

    # ------------------------------------------------------------------ peer exchange
    def _symbuf(self, key, n, w, dtype=torch.float32):
        """symmetric [n, w] buffer -> (SymmetricBuffer, local matrix view)"""
        key = key + (str(dtype),)
        if key not in self._sym:
            sb = self.heap.alloc(n * w * (2 if dtype == torch.bfloat16 else 4))
            self._sym[key] = (sb, sb.matrix(n, w, dtype))
        return self._sym[key]

    @staticmethod
    def _targets(sb, view):
        """keyword arguments for the sparse kernels that make their stores of `view` reach every rank's copy of the
        SymmetricBuffer `sb`: one store to the multicast mapping when the buffer has one, else a store per peer copy"""
        mc = sb.mc_addr(view)
        return {"mc": mc} if mc else {"peers": sb.peer_addrs(view)}

    # ------------------------------------------------------------------ training (row-split sparse products)
    def buffer(self, key, rows, w):
        """[rows, w] float32 output buffer for sparse_rows, kept across steps: symmetric under the peer exchange"""
        if self.heap is not None:
            return self._symbuf(("train",) + tuple(key), rows, w)[1]
        return self._buf(("train",) + tuple(key), rows, w, torch.device("cuda", torch.cuda.current_device()))

    def _owner(self, view):
        for sb, _ in self._sym.values():
            if sb.local <= view.data_ptr() < sb.local + sb.nbytes:
                return sb
        raise ValueError("sparse_rows: output is not a view of a RowPartition.buffer")

    def sparse_rows(self, csr, outs, launch):
        """Run a sparse product on this rank's rows of the operator `csr` and leave every output complete on every rank.

        csr: a whole operator (a graph view or its transpose) of G*N rows, N = the partitioned node count; the stacked
        transpose of the relational operator has one group of N rows per relation, and this rank owns its row blocks of
        every group.  outs: [G*N, w] views of RowPartition.buffer tensors, one per kernel output.
        launch(sl, views, targets) launches the kernel on the row slice `sl` (global column ids, sl.row_offset = its
        first row) with views[k] = outs[k][its rows] and targets[k] = the keyword arguments (peers= / mc=) that make
        output k's stores reach the other ranks.  Under the peer exchange those stores are the exchange: a flag barrier
        before (no rank still reads a copy from an earlier use of the buffers) and one after (every row has landed).
        Under "nccl" the kernel writes own rows and exchange_rows moves them.  Row results do not depend on the
        slicing, so every output equals the single-GPU product bit for bit."""
        n = sum(self.n_rows_by_type)
        if csr.n_rows % n or any(o.shape[0] != csr.n_rows for o in outs):
            raise ValueError("sparse_rows: operator of {} rows, outputs of {} rows, {} nodes".format(
                csr.n_rows, [o.shape[0] for o in outs], n))
        key = ("rows", id(csr))
        if key not in self._slices:
            self._slices[key] = (csr, [csr.row_slice(g * n + a, g * n + b)
                                       for g in range(csr.n_rows // n) for a, b in self.mine])
        slices = self._slices[key][1]
        peer = self.heap is not None
        owners = [self._owner(o) for o in outs] if peer else None
        if peer:
            self.heap.barrier()
        for sl in slices:
            a, b = sl.row_offset, sl.row_offset + sl.n_rows
            views = [o[a:b] for o in outs]
            launch(sl, views, [self._targets(sb, v) for sb, v in zip(owners, views)] if peer else [{}] * len(outs))
        if peer:
            self.heap.barrier()
            return outs
        for o in outs:
            for g in range(csr.n_rows // n):
                blk = o[g * n:(g + 1) * n]
                if blk.is_contiguous():
                    self._exchange(blk)
                else:   # a column slice (the 'concatenation' buffer): the collectives move contiguous rows
                    tmp = blk.contiguous()
                    self._exchange(tmp)
                    blk.copy_(tmp)
        return outs

    def _type_of(self, a):
        base = 0
        for t, cnt in enumerate(self.n_rows_by_type):
            if base <= a < base + cnt or (cnt == 0 and a == base):
                return t
            base += cnt
        return len(self.n_rows_by_type) - 1

    def _propagate_peer(self, seq):
        """The layer loop with the all-gather fused into the producing kernels (module docstring).

        Who needs what: the sparse kernel of a layer gathers rows of its operand from ANY rank, so
        the operand's producer stores its rows everywhere; a layer OUTPUT is needed remotely only on
        the rows of `final_types` (scoring is sharded by user, items are replicated), so the kernel
        that finishes those rows stores them everywhere too.  One flag barrier separates producers
        from consumers; the first one also keeps a fast rank from overwriting buffers a slow rank is
        still reading from the previous call."""
        from . import _lib as L
        from . import ops
        from .layers import GATConv, GCNConv, GraphSageConv, LightGCNConv, RGCNConv
        heap = self.heap
        emb = seq.embeddings
        n = emb.shape[0]
        widths = seq._widths()
        graph = seq.adj_matrix
        layers = seq.seq_layers
        concat = seq.final_node == 'concatenation'
        final = set(self.final_types)
        type_lo = [sum(self.n_rows_by_type[:t]) for t in range(len(self.n_rows_by_type))]

        def is_final(a):
            return self._type_of(a) in final

        heap.barrier()
        if concat:
            csb, cbuf = self._symbuf(("concat",), n, sum(widths))
        # layer 0 input: the replicated embedding table; valid on every row of every rank
        h0 = cbuf[:, :widths[0]] if concat else emb
        if concat:
            for a, b in self.mine:
                cbuf[a:b, :widths[0]].copy_(emb[a:b])
            for t in final:
                cbuf[type_lo[t]:type_lo[t] + self.n_rows_by_type[t], :widths[0]].copy_(
                    emb[type_lo[t]:type_lo[t] + self.n_rows_by_type[t]])
        x_full, hs = emb, [h0]
        off = widths[0]
        for l, layer in enumerate(layers):
            if not layer.built:
                layer.build([(n, widths[l]), None])
                layer.built = True
            if concat:
                osb, out = csb, cbuf[:, off:off + widths[l + 1]]
                off += widths[l + 1]
            else:
                osb, out = self._symbuf(("h", l), n, widths[l + 1])
            relu = getattr(layer, "activation", None) == "relu"
            nxt = layers[l + 1] if l + 1 < len(layers) else None
            # the next layer's sparse kernel gathers from this output directly -> every row travels
            everywhere = isinstance(nxt, (GCNConv, GraphSageConv, LightGCNConv))

            def out_peers(view, a):
                return osb.peer_addrs(view) if (everywhere or is_final(a)) else None

            def out_targets(view, a):
                return self._targets(osb, view) if (everywhere or is_final(a)) else {}

            if isinstance(layer, GCNConv):
                # Every rank computes the WHOLE transform Z = X W itself (2.5 ms for 1.1e7 x 128 x 128 on the tensor
                # cores) from a layer input that is complete on every rank: layer 0 reads the replicated embedding
                # table, later layers read the previous output, whose rows the sparse kernel's epilogue stored into
                # every rank's copy while it ran.  So the only inter-GPU traffic of a layer is spread over its sparse
                # kernel, nothing NVLink-bound is ever exposed, and there is no second exchange for the final rows.
                if l > 0:
                    heap.barrier()   # the previous output's remote rows have landed
                zdt = torch.bfloat16 if getattr(layer, "feature_dtype", "fp32") == "bf16" else torch.float32
                z = self._buf(("zrep", layer.channels), n, layer.channels, emb.device, zdt)
                ops.gcn_transform(x_full, layer.kernel, n, out=z)
                for sl in self.csr_slices("norm", graph):
                    a, b = sl.row_offset, sl.row_offset + sl.n_rows
                    ov = out[a:b]
                    ops.spmm(sl, z, ov, bias=layer.bias, relu=relu, **out_targets(ov, a))
            elif isinstance(layer, RGCNConv):
                # own rows of every relation's transform, stored into every rank's copy of the stacked operand
                n_rel = len(layer.kernels)
                zsb, z = self._symbuf(("z", l), n_rel * n, layer.channels)
                for a, b in self.mine:
                    zv = z[a:(n_rel - 1) * n + b]
                    ops.dense_grouped(x_full[a:b], layer.kernels, zv, n, peers=zsb.peer_addrs(zv))
                heap.barrier()
                for sl in self.csr_slices("norm", graph):
                    ov = out[sl.row_offset:sl.row_offset + sl.n_rows]
                    ops.spmm(sl, z, ov, bias=layer.bias, relu=relu, **out_targets(ov, sl.row_offset))
            elif isinstance(layer, GATConv):
                zsb, z = self._symbuf(("z", l), n, layer.channels)
                qsb, q = self._symbuf(("q", l), n, 1)
                p = self._buf(("p", l), n, 1, emb.device)
                for a, b in self.mine:
                    zv, qv = z[a:b], q[a:b, 0]
                    # the transform stores its rows locally; the finished block is pushed to the other ranks in one
                    # coalesced pass (multicast when the fabric has it).  The tensor-core kernel's epilogue writes one row
                    # per thread - 32-byte pieces of 32 different rows per instruction, which the fabric carries badly:
                    # with 7 peers GAT ran at 54.9 G edges/s on 8 GPUs that way (profiles/r02_scale_families_n8.jsonl)
                    _, pp, _ = ops.gat_transform(x_full[a:b], layer.kernel.reshape(widths[l], layer.channels),
                                                 layer.attn_kernel_self.reshape(-1), layer.attn_kernel_neighs.reshape(-1), n,
                                                 out=zv, q_out=qv)
                    ops.push_rows(zv, zsb)
                    ops.push_rows(q[a:b], qsb)
                    p[a:b, 0].copy_(pp)
                heap.barrier()
                for sl in self.csr_slices("raw", graph):
                    ov = out[sl.row_offset:sl.row_offset + sl.n_rows]
                    ops.gat(sl, z, p.reshape(-1), q.reshape(-1), ov, bias=layer.bias, relu=relu,
                            row_offset=sl.row_offset, peers=out_peers(ov, sl.row_offset))
            elif isinstance(layer, LightGCNConv):
                if l > 0:
                    heap.barrier()  # x_full = previous output, pushed everywhere by its producer
                for sl in self.csr_slices("norm", graph):
                    ov = out[sl.row_offset:sl.row_offset + sl.n_rows]
                    ops.spmm(sl, x_full, ov, **out_targets(ov, sl.row_offset))
            elif isinstance(layer, GraphSageConv):
                if l > 0:
                    heap.barrier()
                for sl in self.csr_slices("raw", graph):
                    a, b = sl.row_offset, sl.row_offset + sl.n_rows
                    agg = self._buf(("agg", l, a), sl.n_rows, widths[l], emb.device)
                    ops.spmm(sl, x_full, agg, agg=L.AGG_MEAN if layer.aggregate == "mean" else L.AGG_SUM)
                    ov = out[a:b]
                    ops.sage_dense(x_full[a:b], agg, layer.kernel, layer.bias, layer.activation, x_full.shape[0], out=ov)
                    if out_peers(ov, a) is not None:   # finished block -> every rank's copy, one coalesced pass (see GAT)
                        ops.push_rows(ov, osb)
            else:
                raise NotImplementedError("no partitioned form for {}".format(type(layer).__name__))
            x_full = out
            hs.append(out)
        heap.barrier()  # the final-type rows stored by the other ranks have landed
        return cbuf if concat else seq.reduce(hs)

    def propagate(self, seq):
        """SequentialGNN.call on the partition.  Returns [N, D_out]; rows of other ranks' users
        are NOT valid unless final_types covers type 0."""
        if self.heap is not None:
            return self._propagate_peer(seq)
        from . import _lib as L
        from . import ops
        from .layers import GATConv, GCNConv, GraphSageConv, LightGCNConv, RGCNConv
        emb = seq.embeddings
        n, dev = emb.shape[0], emb.device
        widths = seq._widths()
        graph = seq.adj_matrix
        x_full, x_full_valid = emb, True   # the layer input; valid on all rows?
        hs = [emb]
        # with 'concatenation' and layers that exchange their own operand (GCN/RGCN/GAT) the outputs go
        # straight into column slices of one [N, D_out] buffer, as on a single GPU
        concat = seq.final_node == 'concatenation' and all(isinstance(ly, (GCNConv, RGCNConv, GATConv))
                                                           for ly in seq.seq_layers)
        if concat:
            cbuf = self._buf(("concat",), n, sum(widths), dev)
            for a, b in self.mine:
                cbuf[a:b, :widths[0]].copy_(emb[a:b])
            off = widths[0]
        for l, layer in enumerate(seq.seq_layers):
            if not layer.built:
                layer.build([(n, widths[l]), None])
                layer.built = True
            if concat:
                out = cbuf[:, off:off + widths[l + 1]]
                off += widths[l + 1]
            else:
                out = self._buf(("h", l), n, widths[l + 1], dev)  # own rows valid
            relu = getattr(layer, "activation", None) == "relu"
            if isinstance(layer, (GCNConv, RGCNConv)):
                kernels = layer.kernels if isinstance(layer, RGCNConv) else [layer.kernel]
                zdt = torch.bfloat16 if getattr(layer, "feature_dtype", "fp32") == "bf16" else torch.float32
                z = self._buf(("z", l), len(kernels) * n, layer.channels, dev, zdt)
                for a, b in self.mine:   # the transform each layer type runs on one GPU (GCNConv.call, RGCNConv.call)
                    if isinstance(layer, RGCNConv):
                        ops.dense_grouped(x_full[a:b], kernels, z[a:(len(kernels) - 1) * n + b], n)
                    else:
                        ops.gcn_transform(x_full[a:b], kernels[0], n, out=z[a:b])
                for r in range(len(kernels)):
                    self._exchange(z[r * n:(r + 1) * n])
                for sl in self.csr_slices("norm", graph):
                    ops.spmm(sl, z, out[sl.row_offset:sl.row_offset + sl.n_rows], bias=layer.bias, relu=relu)
            elif isinstance(layer, GATConv):
                z = self._buf(("z", l), n, layer.channels, dev)
                p = self._buf(("p", l), n, 1, dev)
                q = self._buf(("q", l), n, 1, dev)
                for a, b in self.mine:
                    _, pp, qq = ops.gat_transform(x_full[a:b], layer.kernel.reshape(widths[l], layer.channels),
                                                  layer.attn_kernel_self.reshape(-1), layer.attn_kernel_neighs.reshape(-1), n,
                                                  out=z[a:b])
                    p[a:b, 0].copy_(pp)
                    q[a:b, 0].copy_(qq)
                self._exchange(z)
                self._exchange(q)
                for sl in self.csr_slices("raw", graph):
                    ops.gat(sl, z, p.reshape(-1), q.reshape(-1), out[sl.row_offset:sl.row_offset + sl.n_rows],
                            bias=layer.bias, relu=relu, row_offset=sl.row_offset)
            elif isinstance(layer, (GraphSageConv, LightGCNConv)):
                if not x_full_valid:
                    self._exchange(x_full)
                view = "raw" if isinstance(layer, GraphSageConv) else "norm"
                for sl in self.csr_slices(view, graph):
                    layer([x_full, graph], out=out[sl.row_offset:sl.row_offset + sl.n_rows], csr=sl)
            else:
                raise NotImplementedError("no partitioned form for {}".format(type(layer).__name__))
            x_full, x_full_valid = out, False
            hs.append(out)
        red = cbuf if concat else seq.reduce(hs)
        if self.final_types:
            red = red if red.is_contiguous() else red.contiguous()
            self._exchange(red, self.final_types)
        return red
