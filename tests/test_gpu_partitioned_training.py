"""Training under the row partition, tested on one GPU.

Under a RowPartition the training tape splits only its sparse products by rows (RowPartition.sparse_rows) and runs
everything dense on all rows on every rank, so every weight, the embedding table, the Adam moments and the loss must be
bit-identical to the single-GPU step.

A. The row-slice GAT backward (cbrs_gat_backward_stats_rows / cbrs_gat_backward_grad_rows): slices that start or end at
   a heavy row give the bits of cbrs_gat_backward, under the row-major and the column-blocked schedule; 0, 1 and 7
   stand-in peer copies and a multicast target receive exactly those bits; bad arguments are refused before any write.
B. A loopback of the peer exchange: 2 and 3 ranks emulated in one process.  The tape runs as rank 0; each of its sparse
   products runs every emulated rank's row slices in turn (RowPartition.sparse_rows, peer path), each storing into its
   own copy and the others' copies.  Every copy must equal rank 0's after every product, and three optimiser steps must
   equal the unpartitioned ones bit for bit.  The flag barrier is replaced by a counter: one process runs every rank,
   so there is nothing to wait for.
C. Two processes on the same GPU with a gloo group and exchange="nccl": train_on_batch steps and a fit epoch,
   partitioned and unpartitioned in each process, both schedules.
D. What has no partitioned form is refused before any launch."""
import json
import os
import types
import zlib

import numpy as np
import pytest
import torch

from tests.test_gpu_peer_stores import F32, MAX_COPIES, SENT, Arena, _heavy_row, _randn, _stub, check_peer_stores, same_bits

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    from deep_cbrs_amar_renaissance_b200 import ops
    ops.check_device()
    return torch.device("cuda", 0)


@pytest.fixture(scope="module")
def sym_adj():
    from deep_cbrs_amar_renaissance_b200.selfcheck import small_graph
    return small_graph(301, 199, 6000, seed=5, n_props=51, n_links=600, dup_links=40), (301, 199, 51)


# --------------------------------------------------------------------------------------- A. row-slice GAT backward
def _gat_inputs(n, h, dev):
    z = _randn((n, h), dev, 1)
    p, q = _randn((n,), dev, 2, 0.7), _randn((n,), dev, 3, 0.7)
    y = _randn((n, h), dev, 4)
    d_o = _randn((n, h), dev, 5)
    d_o[::7, ::3] = 0.0                       # the stats kernel skips zero gradients
    return z, p, q, y, _randn((h,), dev, 6, 0.1), d_o, _randn((h,), dev, 7), _randn((h,), dev, 8)


@pytest.mark.parametrize("h", [64, 18])     # float4 row dots, scalar row dots
@pytest.mark.parametrize("blocking", [None, (97, 25)], ids=["row-major", "blocked"])
def test_gat_backward_rows_match_the_whole_graph_call(dev, sym_adj, monkeypatch, blocking, h):
    from deep_cbrs_amar_renaissance_b200 import graph as G
    from deep_cbrs_amar_renaissance_b200 import ops
    monkeypatch.setattr(G, "FORCED_BLOCKING", blocking)
    adj, _ = sym_adj
    g = G.DeviceGraph.from_scipy(adj, dev, chunk_edges=16)
    raw = g.raw
    assert raw.blocking == (blocking or (0, 0))
    n = raw.n_rows
    z, p, q, y, bias, d_o, a_s, a_n = _gat_inputs(n, h, dev)
    dz_ref, dp_ref, dq_ref = ops.gat_backward(raw, z, p, q, y, bias, d_o, a_s, a_n)
    stats_ref = torch.full((n, 3), SENT, device=dev)
    ops.gat_backward_stats_rows(raw, p, q, y, bias, d_o, stats_ref)
    hv = _heavy_row(raw)
    for cuts in ([0, hv, n], [0, 37, hv + 1, n]):
        slices = [raw.row_slice(a, b) for a, b in zip(cuts[:-1], cuts[1:])]
        stats = torch.full((n, 3), SENT, device=dev)
        for sl in slices:
            ops.gat_backward_stats_rows(sl, p, q, y, bias, d_o, stats[sl.row_offset:sl.row_offset + sl.n_rows])
        assert same_bits(stats, stats_ref), cuts
        dz, dp, dq = (torch.full(s, SENT, device=dev) for s in ((n, h), (n, 1), (n, 1)))
        for sl in slices:
            a, b = sl.row_offset, sl.row_offset + sl.n_rows
            ops.gat_backward_grad_rows(sl, z, p, q, d_o, stats, a_s, a_n, dz[a:b], dp[a:b], dq[a:b])
        torch.cuda.synchronize()
        assert same_bits(dz, dz_ref) and same_bits(dp.reshape(-1), dp_ref) and same_bits(dq.reshape(-1), dq_ref), cuts

    # peer copies of one slice that starts at the heavy row
    sl = raw.row_slice(hv, n)
    m = sl.n_rows
    check_peer_stores(dev, [(m, 3, 3, F32, 0)],
                      lambda v, peers: ops.gat_backward_stats_rows(sl, p, q, y, bias, d_o, v[0],
                                                                   peers=peers[0] if peers else None),
                      "gat_backward_stats_rows", counts=(1, MAX_COPIES))
    _, local = check_peer_stores(
        dev, [(m, h, h, F32, 0), (m, 1, 1, F32, 0), (m, 1, 1, F32, 0)],
        lambda v, peers: ops.gat_backward_grad_rows(sl, z, p, q, d_o, stats_ref, a_s, a_n, *v,
                                                    targets=[{"peers": pl} for pl in peers] if peers else None),
        "gat_backward_grad_rows", counts=(1, MAX_COPIES))
    assert same_bits(local[0], dz_ref[hv:]) and same_bits(local[1].reshape(-1), dp_ref[hv:])
    assert same_bits(local[2].reshape(-1), dq_ref[hv:])
    # a multicast target: the only store goes there, the local view is not written
    outs = [torch.full(s, SENT, device=dev) for s in ((m, h), (m, 1), (m, 1))]
    mcs = [torch.full(s, SENT, device=dev) for s in ((m, h), (m, 1), (m, 1))]
    ops.gat_backward_grad_rows(sl, z, p, q, d_o, stats_ref, a_s, a_n, *outs,
                               targets=[{"mc": t.data_ptr()} for t in mcs])
    torch.cuda.synchronize()
    assert same_bits(mcs[0], dz_ref[hv:]) and same_bits(mcs[1].reshape(-1), dp_ref[hv:])
    assert all(bool((o == SENT).all()) for o in outs)


def test_gat_backward_rows_refuse_bad_arguments_before_any_write(dev, sym_adj):
    import ctypes
    from deep_cbrs_amar_renaissance_b200 import _lib as L
    from deep_cbrs_amar_renaissance_b200.graph import DeviceGraph
    lib = L.load()
    adj, _ = sym_adj
    raw = DeviceGraph.from_scipy(adj, dev, chunk_edges=16).raw
    n, h = raw.n_rows, 32
    z, p, q, y, bias, d_o, a_s, a_n = _gat_inputs(n, h, dev)
    a = Arena(dev, 2 * 1024 + 4 * (n * h + 2048) + 8 * 2048)
    stats, dz, dp, dq = a.take(n, 3, mark=False), a.take(n, h, mark=False), a.take(n, 1, mark=False), a.take(n, 1, mark=False)
    peer = a.take(n, h, mark=False)
    P = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None  # noqa: E731
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    d = ctypes.byref(raw.desc)
    arr = lambda ts: (ctypes.c_void_p * max(len(ts), 1))(*[t.data_ptr() if t is not None else None for t in ts])  # noqa: E731

    def stats_call(off=0, ldy=h, hh=h, out=stats, peers=(), n_peers=None):
        return lib.cbrs_gat_backward_stats_rows(d, off, P(p), P(q), P(y), ldy, P(bias), P(d_o), h, hh, P(out),
                                                arr(list(peers)), len(peers) if n_peers is None else n_peers, st)

    def grad_call(off=0, hh=h, lddz=h, out=dz, peers=(), n_peers=None):
        pl = arr(list(peers))
        return lib.cbrs_gat_backward_grad_rows(d, off, P(z), h, P(p), P(q), P(d_o), h, hh, P(stats), P(a_s), P(a_n),
                                               P(out), lddz, P(dp), P(dq), pl, pl, pl,
                                               len(peers) if n_peers is None else n_peers, st)

    bad = [("stats: null output", lambda: stats_call(out=None)),
           ("stats: ldy < h", lambda: stats_call(ldy=h - 1)),
           ("stats: h = 0", lambda: stats_call(hh=0)),
           ("stats: negative row offset", lambda: stats_call(off=-1)),
           ("stats: 8 peer copies", lambda: stats_call(peers=[peer] * 8)),
           ("stats: a null peer copy", lambda: stats_call(peers=[peer, None])),
           ("stats: peers counted but no list", lambda: lib.cbrs_gat_backward_stats_rows(
               d, 0, P(p), P(q), P(y), h, P(bias), P(d_o), h, h, P(stats), None, 2, st)),
           ("grad: null dz", lambda: grad_call(out=None)),
           ("grad: h = 257", lambda: grad_call(hh=257)),
           ("grad: lddz < h", lambda: grad_call(lddz=h - 1)),
           ("grad: negative row offset", lambda: grad_call(off=-3)),
           ("grad: 8 peer copies", lambda: grad_call(peers=[peer] * 8)),
           ("grad: a null peer copy", lambda: grad_call(peers=[None]))]
    for what, call in bad:
        assert call() == -1, what
        torch.cuda.synchronize()
        assert bool((a.buf == SENT).all()), what + ": refused, but something was written"


# ----------------------------------------------------------------------------- B. loopback of the peer exchange
class _CountingHeap:
    """stands in for PeerHeap: every emulated rank runs in this one process, one after the other, so a flag barrier
    would find every flag already set; it only counts"""

    def __init__(self):
        self.barriers = 0

    def barrier(self):
        self.barriers += 1


class LoopbackPartition:
    """What the training tape sees of a RowPartition, for `world` ranks emulated in one process: buffer() allocates
    one copy per rank (a SymmetricBuffer of each rank over all copies), sparse_rows() runs every rank's
    RowPartition.sparse_rows in turn and checks that every copy ends up equal to rank 0's, which it returns."""

    def __init__(self, sizes, cuts, dev):
        from deep_cbrs_amar_renaissance_b200.distributed import RowPartition, SymmetricBuffer
        self.SymmetricBuffer, self.dev = SymmetricBuffer, dev
        self.world = len(cuts) - 1
        self.ranks = []
        for r in range(self.world):
            p = RowPartition.__new__(RowPartition)
            p.n_rows_by_type, p.world, p.rank = list(sizes), self.world, r
            p.mine = [(cuts[r], cuts[r + 1])]
            p.heap, p._slices, p._sym, p._bufs = _CountingHeap(), {}, {}, {}
            self.ranks.append(p)
        self.copies = {}
        self.calls = 0

    def buffer(self, key, rows, w):
        if key not in self.copies:
            copies = [torch.full((rows, w), -3.0e38, device=self.dev) for _ in range(self.world)]
            ptrs = [c.data_ptr() for c in copies]
            for r, p in enumerate(self.ranks):
                p._sym[key] = (self.SymmetricBuffer(_stub(r), rows * w * 4, ptrs), copies[r])
            self.copies[key] = copies
        return self.copies[key][0]

    def _copies_of(self, view):
        for copies in self.copies.values():
            base = copies[0]
            if base.data_ptr() <= view.data_ptr() < base.data_ptr() + base.numel() * 4:
                return [c.as_strided(view.shape, view.stride(), view.storage_offset()) for c in copies]
        raise AssertionError("output is not a LoopbackPartition.buffer view")

    def sparse_rows(self, csr, outs, launch):
        per_out = [self._copies_of(o) for o in outs]
        for r, p in enumerate(self.ranks):
            before = p.heap.barriers
            p.sparse_rows(csr, [cs[r] for cs in per_out], launch)
            assert p.heap.barriers == before + 2      # one before the stores, one after
        torch.cuda.synchronize()
        for k, cs in enumerate(per_out):
            for r in range(1, self.world):
                assert same_bits(cs[r], cs[0]), "output %d: copy of rank %d differs from rank 0's" % (k, r)
        self.calls += 1
        return outs


def _rgcn_graph(adj, nu, ni, dev):
    from deep_cbrs_amar_renaissance_b200.graph import DeviceGraph
    rel = ((adj.row >= nu + ni) | (adj.col >= nu + ni)).astype(np.int32)
    t = lambda v, dt: torch.from_numpy(np.ascontiguousarray(v, dt)).to(dev)  # noqa: E731
    return DeviceGraph(t(adj.row, np.int32), t(adj.col, np.int32), t(adj.data, np.float32), adj.shape[0], 16,
                       rel=t(rel, np.int32), n_rel=2)


FAMILIES = ["BasicGCN", "BasicRGCN", "BasicLightGCN", "BasicGraphSage", "BasicGAT", "HybridBertGCN"]
CONTENT = 24


def _model(name, adj, sizes, dev, final_node="concatenation"):
    from deep_cbrs_amar_renaissance_b200.keras_like import set_seed
    from deep_cbrs_amar_renaissance_b200.models import basic, hybrid
    set_seed(31)
    kw = dict(embedding_dim=16, final_node=final_node)
    if name == "HybridBertGCN":
        m = hybrid.HybridBertGCN(adj, n_hiddens=[16, 16], dense_units=[[48, 48], [32, 32], [32, 32]], clf_units=[16, 16],
                                 **kw)
        m.build_weights(CONTENT)
    else:
        if name == "BasicRGCN":
            adj = _rgcn_graph(adj, sizes[0], sizes[1], dev)
        if name == "BasicLightGCN":
            m = basic.BasicLightGCN(adj, n_layers=2, dense_units=[32, 16], clf_units=[16, 16], **kw)
        else:
            m = getattr(basic, name)(adj, n_hiddens=[16, 16], dense_units=[32, 16], clf_units=[16, 16], **kw)
        m.build_weights()
    with torch.no_grad():     # non-zero biases so that the bias gradients and epilogues are exercised
        for nm, w in m.named_weights():
            if nm.endswith("bias"):
                w.copy_(_randn(w.shape, dev, zlib.crc32(nm.encode()) % 1000, 0.05))
    m.compile(loss="binary_crossentropy", optimizer={"learning_rate": 1e-2})
    return m


def _batches(sizes, n_batches, bs, seed):
    rng = np.random.RandomState(seed)
    out = []
    for _ in range(n_batches):
        u = rng.randint(0, sizes[0], size=bs)
        i = rng.randint(0, sizes[1], size=bs) + sizes[0]
        y = (rng.rand(bs) < 0.5).astype(np.float32)
        out.append((u, i, y))
    return out


def _inputs(name, u, i, seed, dev):
    if name != "HybridBertGCN":
        return (u, i)
    return (u, i, _randn((len(u), CONTENT), dev, seed), _randn((len(u), CONTENT), dev, seed + 1))


def _train(model, name, batches, dev):
    """three train_on_batch steps -> (losses, weights, Adam m, Adam v) on the host"""
    losses = []
    for k, (u, i, y) in enumerate(batches):
        loss, _ = model.train_on_batch(_inputs(name, u, i, 100 + k, dev), y)
        losses.append(loss.clone())
    torch.cuda.synchronize()
    st = model._adam._state
    ws = list(model.weights)
    return ([x.cpu() for x in losses], [w.detach().cpu().clone() for w in ws],
            [st[id(w)][0].cpu() if id(w) in st else None for w in ws],
            [st[id(w)][1].cpu() if id(w) in st else None for w in ws])


def _same_run(a, b):
    for what, xs, ys in zip(("loss", "weight", "adam m", "adam v"), a, b):
        assert len(xs) == len(ys)
        for k, (x, y) in enumerate(zip(xs, ys)):
            assert (x is None and y is None) or torch.equal(x, y), "%s %d differs from the single-GPU step" % (what, k)


@pytest.mark.parametrize("final_node", ["concatenation", "mean"])
@pytest.mark.parametrize("blocking", [None, (97, 25)], ids=["row-major", "blocked"])
@pytest.mark.parametrize("name", FAMILIES)
def test_peer_exchange_loopback_trains_bit_identically(dev, sym_adj, monkeypatch, name, blocking, final_node):
    from deep_cbrs_amar_renaissance_b200 import graph as G
    monkeypatch.setattr(G, "FORCED_BLOCKING", blocking)
    adj, sizes = sym_adj
    n = sum(sizes)
    batches = _batches(sizes, 3, 256, 7)
    want = _train(_model(name, adj, sizes, dev, final_node), name, batches, dev)
    model = _model(name, adj, sizes, dev, final_node)
    hv = _heavy_row(model.gnn.gnn_layers.adj_matrix.raw)
    for cuts in ([0, hv, n], [0, 37, hv + 1, n]):      # a rank starts, or ends, at a heavy row
        model = _model(name, adj, sizes, dev, final_node)
        part = LoopbackPartition(sizes, cuts, dev)
        model.gnn.gnn_layers.partition = part
        got = _train(model, name, batches, dev)
        n_layers = 2
        sparse_per_step = n_layers * (3 if name == "BasicGAT" else 2)
        assert part.calls == 3 * sparse_per_step
        _same_run(got, want)


# ------------------------------------------------------------------- C. two processes, one GPU, the "nccl" exchange
class _Seq:
    """a minimal keras Sequence of (inputs, labels) batches"""

    def __init__(self, name, batches, dev):
        self.items = [(_inputs(name, u, i, 200 + k, dev), y) for k, (u, i, y) in enumerate(batches)]

    def __len__(self):
        return len(self.items)

    def __getitem__(self, k):
        return self.items[k]


def _worker(rank, world, init, out_dir, sizes):
    import torch.distributed as dist
    from deep_cbrs_amar_renaissance_b200 import graph as G
    from deep_cbrs_amar_renaissance_b200.distributed import RowPartition
    from deep_cbrs_amar_renaissance_b200.selfcheck import small_graph
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", init_method=init, rank=rank, world_size=world)
    dev = torch.device("cuda", 0)
    adj = small_graph(sizes[0], sizes[1], 6000, seed=5, n_props=sizes[2], n_links=600, dup_links=40)
    failures, cases = [], 0
    try:
        for blocking in (None, (97, 25)):
            G.FORCED_BLOCKING = blocking
            for name in FAMILIES:
                batches = _batches(sizes, 3, 256, 11)
                for balanced in (False, True):
                    tag = "%s %s %s" % (name, "blocked" if blocking else "row-major", "edge-balanced" if balanced else "even")
                    want = _train(_model(name, adj, sizes, dev), name, batches, dev)
                    ref = _model(name, adj, sizes, dev)
                    ref.fit(_Seq(name, batches, dev), epochs=1)
                    model = _model(name, adj, sizes, dev)
                    seq = model.gnn.gnn_layers
                    rp = seq.adj_matrix.norm.rowptr if balanced else None
                    RowPartition(sizes, exchange="nccl", balance_rowptr=rp).attach(seq)
                    got = _train(model, name, batches, dev)
                    fitted = _model(name, adj, sizes, dev)
                    RowPartition(sizes, exchange="nccl", balance_rowptr=rp).attach(fitted.gnn.gnn_layers)
                    fitted.fit(_Seq(name, batches, dev), epochs=1)
                    torch.cuda.synchronize()
                    for what, run in (("train_on_batch", lambda: _same_run(got, want)),
                                      ("fit", lambda: _same_run(
                                          ([], [w.cpu() for w in fitted.weights], [], []),
                                          ([], [w.cpu() for w in ref.weights], [], [])))):
                        cases += 1
                        try:
                            run()
                        except AssertionError as e:
                            failures.append("%s %s: %s" % (tag, what, e))
    finally:
        G.FORCED_BLOCKING = None
        with open(os.path.join(out_dir, "rank%d.json" % rank), "w") as f:
            json.dump({"cases": cases, "failures": failures}, f)
        dist.destroy_process_group()


def test_two_processes_on_one_gpu_train_bit_identically(dev, tmp_path):
    """Both ranks share cuda:0 and a gloo group.  Every node type has an odd row count, so the even cut is ragged too
    and exchange_rows moves the rows by broadcast, which gloo runs on CUDA tensors (its all_gather_into_tensor is not
    relied on)."""
    import torch.multiprocessing as mp
    sizes = (301, 199, 51)
    assert all(s % 2 for s in sizes)
    mp.spawn(_worker, args=(2, "file://" + str(tmp_path / "store"), str(tmp_path), sizes), nprocs=2, join=True)
    for r in range(2):
        res = json.load(open(tmp_path / ("rank%d.json" % r)))
        assert res["cases"] == 2 * 2 * len(FAMILIES) * 2 and not res["failures"], res["failures"]


# ------------------------------------------------------------------------------------------------ D. refusals
def _refused(model, call, match):
    from deep_cbrs_amar_renaissance_b200 import ops
    torch.cuda.synchronize()
    launches = ops.LAUNCHES
    with pytest.raises(NotImplementedError, match=match):
        call()
    assert ops.LAUNCHES == launches


def test_what_has_no_partitioned_form_is_refused_before_any_launch(dev, sym_adj):
    from deep_cbrs_amar_renaissance_b200.models import basic
    adj, (nu, ni, _) = sym_adj
    part = types.SimpleNamespace()      # never used: the refusal comes first
    u, i = np.arange(8), np.arange(8) + nu
    y = np.ones(8, np.float32)
    m = basic.BasicDGCF(adj, embedding_dim=8, n_layers=2, dense_units=[16], clf_units=[8])
    m.build_weights()
    m.compile()
    m.gnn.gnn_layers.partition = part
    _refused(m, lambda: m.train_on_batch((u, i), y), "DGCFConv")
    from deep_cbrs_amar_renaissance_b200.selfcheck import small_graph
    n_props = 20
    ui, ip, up = small_graph(nu, ni, 3000, seed=1), small_graph(ni, n_props, 300, seed=2), small_graph(nu, n_props, 300, seed=3)
    for m in (basic.BasicTSGCN(nu, ni, (ui, ip), n_hiddens=[8, 8], embedding_dim=8, dense_units=[16], clf_units=[8]),
              basic.BasicTWGCN(nu, ni, (ui, ip, up), n_hiddens=[8, 8], embedding_dim=8, dense_units=[16], clf_units=[8])):
        m.gnn.step_two_gnn_layers.partition = part
        _refused(m, lambda: m.train_on_batch((u, i), y), "TwoStepGCN|TwoWayGCN")
    m = basic.BasicGCN(adj, n_hiddens=[8, 8], embedding_dim=8, dense_units=[16], clf_units=[8])
    m.build_weights()
    m.compile()
    m.gnn.gnn_layers.partition = part
    _refused(m, lambda: m.make_graphed_train_step(8), "CUDA-graphed")
    batches = [((u, i), y), ((u, i), y)]
    seq = type("S", (), {"__len__": lambda s: 2, "__getitem__": lambda s, k: batches[k]})()
    _refused(m, lambda: m.fit(seq, epochs=1, cuda_graph=True), "CUDA-graphed")
