"""Multi-GPU self-check: the row-partitioned propagation must equal the single-GPU one BIT FOR BIT (SURVEY 8e,
"Determinism": every row's reduction order is rank-independent and the exchange is a pure copy).

Called by bench.py before timing whenever WORLD_SIZE > 1 (the JSON line carries the outcome as "partition_parity")
and by tests/multi_gpu_check.py.  Every rank builds the same small graph and weights, runs each layer family once
unpartitioned and then partitioned - ragged and even blocks, peer stores and the NCCL all-gather, both GCN transform
kernels, the column-blocked schedule - and compares with torch.equal.
Nothing here is timed; the graphs are MovieLens-sized so the whole check takes a few seconds."""
import numpy as np
import torch
import torch.distributed as dist
from scipy import sparse

from . import graph as G
from .distributed import RowPartition
from .keras_like import set_seed
from .models import basic


def small_graph(n_users, n_items, n_pos, seed=0, n_props=0, n_links=0, dup_links=0):
    """Symmetrised COO adjacency in the reference's entry order (preprocess.py:68-86,149-168 + math.py:13-20):
    unique (user, item) pairs, optional item-property links with duplicates kept."""
    rng = np.random.RandomState(seed)
    keys = np.unique(rng.randint(0, n_users * n_items, size=n_pos))
    rng.shuffle(keys)
    r, c = keys // n_items, keys % n_items + n_users
    n = n_users + n_items + n_props
    if n_props:
        ii = rng.randint(0, n_items, size=n_links) + n_users
        pp = rng.randint(0, n_props, size=n_links) + n_users + n_items
        pick = rng.randint(0, n_links, size=dup_links)
        r = np.concatenate([r, ii, ii[pick]])
        c = np.concatenate([c, pp, pp[pick]])
    rows = np.concatenate([r, c]).astype(np.int32)
    cols = np.concatenate([c, r]).astype(np.int32)
    return sparse.coo_matrix((np.ones(len(rows), np.float32), (rows, cols)), shape=(n, n), dtype=np.float32)


def _pad(adj, n_users, n_items, n_props, sizes):
    """Re-index nodes so each type has the padded size (extra nodes are isolated)."""
    def remap(x):
        x = x.astype(np.int64)
        out = x.copy()
        out[x >= n_users] += sizes[0] - n_users
        out[x >= n_users + n_items] += sizes[1] - n_items
        return out.astype(np.int32)
    n = sum(sizes)
    return sparse.coo_matrix((adj.data, (remap(adj.row), remap(adj.col))), shape=(n, n), dtype=np.float32)


def partition_parity(group=None, log=None, families=("BasicGCN", "BasicGraphSage", "BasicGAT", "BasicLightGCN")):
    """Collective.  Returns {"bit_identical": bool, "cases": n, "failures": [names]} (the same on every rank)."""
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    gpu = torch.cuda.is_available()
    failures, cases = [], 0

    def check(ok, name):
        nonlocal cases
        cases += 1
        if not ok:
            failures.append(name)

    def say(msg):
        if log is not None and rank == 0:
            log(msg)

    n_users, n_items, n_props = 3001, 1999, 500
    adj = small_graph(n_users, n_items, 150000, seed=21, n_props=n_props, n_links=4000, dup_links=300)
    u = np.arange(512) % n_users
    i = np.arange(512) % n_items + n_users
    exchanges = ("peer", "nccl") if gpu else ("nccl",)
    for blocking in (None, (257, 40)):          # row-major schedule, then the column-blocked one on the same graph
        G.FORCED_BLOCKING = blocking
        try:
            for name in families:
                for even in (False, True):
                    if blocking is not None and even:
                        continue
                    set_seed(7)
                    sizes = [n_users, n_items, n_props]
                    if even:  # a node count every type divides by the world size -> all_gather path
                        sizes = [n_users + (-n_users) % world, n_items + (-n_items) % world, n_props + (-n_props) % world]
                    model = getattr(basic, name)(adj if not even else _pad(adj, n_users, n_items, n_props, sizes),
                                                 n_hiddens=[16, 16], n_layers=2, embedding_dim=16, dense_units=[48, 48],
                                                 clf_units=[64, 64])
                    seq = model.gnn.gnn_layers
                    model((u, i))
                    full = model.gnn(None).clone()
                    for exchange in exchanges:
                        tag = "%s %s %s%s" % (name, "even" if even else "ragged", exchange, " blocked" if blocking else "")
                        part = RowPartition(sizes, group=group, final_types=[0, 1, 2], exchange=exchange).attach(seq)
                        for rep in range(3):  # repeated calls reuse the symmetric buffers
                            got = model.gnn(None)
                            if gpu:
                                torch.cuda.synchronize()
                            check(torch.equal(got, full), tag + " rep %d" % rep)
                        part.close()
                        seq.partition = None
                        # items only: user rows of other ranks are not exchanged, own rows and item rows must match
                        part = RowPartition(sizes, group=group, final_types=[1], exchange=exchange).attach(seq)
                        got = model.gnn(None)
                        if gpu:
                            torch.cuda.synchronize()
                        lo, hi = sizes[0], sizes[0] + sizes[1]
                        ok = torch.equal(got[lo:hi], full[lo:hi])
                        for a, b in part.mine:
                            ok = ok and torch.equal(got[a:b], full[a:b])
                        check(ok, tag + " items-only")
                        part.close()
                        seq.partition = None
                    say("partition parity: %s %s%s done" % (name, "even" if even else "ragged", " blocked" if blocking else ""))
            if gpu:
                # 128-wide GCN stack under the peer exchange, once with each transform kernel: the FFMA kernel and the
                # tensor-core one (forced here: the graph is below its automatic threshold).  Both must equal the
                # single-GPU result bit for bit.
                from . import ops
                saved = ops.GCN_TRANSFORM
                try:
                    for transform in ("ffma", "tf32x3"):
                        ops.GCN_TRANSFORM = transform
                        set_seed(11)
                        model = basic.BasicGCN(adj, n_hiddens=[128, 128, 128], embedding_dim=128, dense_units=[48, 48],
                                               clf_units=[64, 64], final_node="concatenation")
                        seq = model.gnn.gnn_layers
                        model((u, i))
                        full = model.gnn(None).clone()
                        part = RowPartition([n_users, n_items, n_props], group=group, final_types=[0, 1, 2],
                                            exchange="peer").attach(seq)
                        for rep in range(2):
                            got = model.gnn(None)
                            torch.cuda.synchronize()
                            check(torch.equal(got, full), "128-wide GCN %s%s rep %d" % (
                                transform, " blocked" if blocking else "", rep))
                        part.close()
                        seq.partition = None
                        if transform == "tf32x3":   # the GAT transform (z, p, q) on the tensor-core kernel, partitioned
                            set_seed(13)
                            model = basic.BasicGAT(adj, n_hiddens=[64, 64], embedding_dim=64, dense_units=[48, 48],
                                                   clf_units=[64, 64])
                            seq = model.gnn.gnn_layers
                            model((u, i))
                            full = model.gnn(None).clone()
                            part = RowPartition([n_users, n_items, n_props], group=group, final_types=[0, 1, 2],
                                                exchange="peer").attach(seq)
                            got = model.gnn(None)
                            torch.cuda.synchronize()
                            check(torch.equal(got, full), "64-wide GAT tf32x3%s" % (" blocked" if blocking else ""))
                            part.close()
                            seq.partition = None
                            # GraphSage with its dense part as two tensor-core products (ops.sage_dense), partitioned
                            set_seed(17)
                            model = basic.BasicGraphSage(adj, n_hiddens=[64, 64], embedding_dim=64, dense_units=[48, 48],
                                                         clf_units=[64, 64])
                            seq = model.gnn.gnn_layers
                            model((u, i))
                            full = model.gnn(None).clone()
                            part = RowPartition([n_users, n_items, n_props], group=group, final_types=[0, 1, 2],
                                                exchange="peer").attach(seq)
                            got = model.gnn(None)
                            torch.cuda.synchronize()
                            check(torch.equal(got, full), "64-wide GraphSage tf32x3%s" % (" blocked" if blocking else ""))
                            part.close()
                            seq.partition = None
                finally:
                    ops.GCN_TRANSFORM = saved
                say("partition parity: 128-wide GCN (FFMA / tensor-core transform)%s done" % (" blocked" if blocking else ""))
        finally:
            G.FORCED_BLOCKING = None
    if gpu:
        # user-sharded catalog top-k: each rank ranks its own users with replicated item rows
        set_seed(7)
        adj2 = small_graph(n_users, n_items, 150000, seed=22)
        model = basic.BasicGCN(adj2, n_hiddens=[16, 16], embedding_dim=16, dense_units=[48, 48], clf_units=[64, 64])
        model((u, i))
        model.cache_propagation = True
        ids_full, vals_full = model.recommend_top_k(n_users, n_items, 10)
        model.invalidate()
        part = RowPartition([n_users, n_items], group=group, final_types=[1]).attach(model.gnn.gnn_layers)
        a, b = part.ranges[rank][0]
        mine = torch.arange(a, b, device="cuda")
        ids, vals = model.recommend_top_k(n_users, n_items, 10, users=mine)
        check(torch.equal(ids, ids_full[a:b]) and torch.equal(vals, vals_full[a:b]), "user-sharded top-k")
        part.close()
        model.gnn.gnn_layers.partition = None
    # every rank must agree on the outcome
    flag = torch.tensor([0 if failures else 1], dtype=torch.int32, device="cuda" if gpu else "cpu")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)
    gathered = [None] * world
    dist.all_gather_object(gathered, failures, group=group)
    all_failures = sorted({f for fl in gathered for f in fl})
    return {"bit_identical": bool(int(flag.item()) == 1), "cases": cases, "failures": all_failures}


def _train_model(name, adj, sizes, relational):
    """a small model of family `name` with fixed weights (non-zero biases) and a compiled Adam"""
    import zlib
    from .models import hybrid
    set_seed(31)
    kw = dict(embedding_dim=16, final_node="concatenation")
    if name == "HybridBertGCN":
        m = hybrid.HybridBertGCN(adj, n_hiddens=[16, 16], dense_units=[[48, 48], [32, 32], [32, 32]], clf_units=[16, 16],
                                 **kw)
        m.build_weights(24)
    else:
        if name == "BasicLightGCN":
            m = basic.BasicLightGCN(adj, n_layers=2, dense_units=[32, 16], clf_units=[16, 16], **kw)
        else:
            m = getattr(basic, name)(relational if name == "BasicRGCN" else adj, n_hiddens=[16, 16],
                                     dense_units=[32, 16], clf_units=[16, 16], **kw)
        m.build_weights()
    with torch.no_grad():
        for nm, w in m.named_weights():
            if nm.endswith("bias"):
                g = torch.Generator(w.device).manual_seed(zlib.crc32(nm.encode()) % 1000)
                w.copy_(torch.randn(w.shape, device=w.device, generator=g) * 0.05)
    m.compile(loss="binary_crossentropy", optimizer={"learning_rate": 1e-2})
    return m


def _train_steps(model, name, sizes, steps=3):
    """`steps` train_on_batch calls on the same seeded batches on every rank -> host copies of (losses, weights,
    Adam m, Adam v)"""
    rng = np.random.RandomState(11)
    losses = []
    for k in range(steps):
        u = rng.randint(0, sizes[0], size=256)
        i = rng.randint(0, sizes[1], size=256) + sizes[0]
        y = (rng.rand(256) < 0.5).astype(np.float32)
        x = (u, i)
        if name == "HybridBertGCN":
            g = torch.Generator("cuda").manual_seed(100 + k)
            x = (u, i, torch.randn(256, 24, device="cuda", generator=g), torch.randn(256, 24, device="cuda", generator=g))
        loss, _ = model.train_on_batch(x, y)
        losses.append(loss.clone())
    torch.cuda.synchronize()
    st = model._adam._state
    ws = list(model.weights)
    return ([t.cpu() for t in losses], [w.detach().cpu().clone() for w in ws],
            [st[id(w)][0].cpu() for w in ws if id(w) in st], [st[id(w)][1].cpu() for w in ws if id(w) in st])


def training_parity(group=None, log=None, families=("BasicGCN", "BasicRGCN", "BasicLightGCN", "BasicGraphSage",
                                                    "BasicGAT", "HybridBertGCN")):
    """Collective.  The row-partitioned training step must equal the single-GPU step BIT FOR BIT: for each family,
    three optimiser steps unpartitioned and then partitioned - peer stores and the NCCL all-gather, even and
    edge-balanced cuts, the row-major and the column-blocked schedule - compared with torch.equal on the losses, every
    weight (the embedding table included) and the Adam moments.  Returns {"bit_identical", "cases", "failures"} (the
    same on every rank)."""
    from .graph import DeviceGraph
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    failures, cases = [], 0

    def say(msg):
        if log is not None and rank == 0:
            log(msg)

    n_users, n_items, n_props = 3001, 1999, 500
    adj = small_graph(n_users, n_items, 60000, seed=23, n_props=n_props, n_links=4000, dup_links=300)
    dev = torch.device("cuda", torch.cuda.current_device())
    rel = ((adj.row >= n_users + n_items) | (adj.col >= n_users + n_items)).astype(np.int32)
    t = lambda v, dt: torch.from_numpy(np.ascontiguousarray(v, dt)).to(dev)  # noqa: E731
    sizes = [n_users, n_items, n_props]
    for blocking in (None, (257, 40)):
        G.FORCED_BLOCKING = blocking
        try:
            for name in families:
                relational = DeviceGraph(t(adj.row, np.int32), t(adj.col, np.int32), t(adj.data, np.float32),
                                         adj.shape[0], rel=t(rel, np.int32), n_rel=2)
                want = _train_steps(_train_model(name, adj, sizes, relational), name, sizes)
                for exchange in ("peer", "nccl"):
                    for balanced in (False, True):
                        model = _train_model(name, adj, sizes, relational)
                        seq = model.gnn.gnn_layers
                        part = RowPartition(sizes, group=group, exchange=exchange,
                                            balance_rowptr=seq.adj_matrix.norm.rowptr if balanced else None).attach(seq)
                        got = _train_steps(model, name, sizes)
                        part.close()
                        seq.partition = None
                        cases += 1
                        ok = all(len(a) == len(b) and all(torch.equal(x, y) for x, y in zip(a, b))
                                 for a, b in zip(got, want))
                        if not ok:
                            failures.append("%s %s %s%s" % (name, exchange, "edge-balanced" if balanced else "even",
                                                            " blocked" if blocking else ""))
                say("training parity: %s%s done" % (name, " blocked" if blocking else ""))
        finally:
            G.FORCED_BLOCKING = None
    flag = torch.tensor([0 if failures else 1], dtype=torch.int32, device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)
    gathered = [None] * world
    dist.all_gather_object(gathered, failures, group=group)
    return {"bit_identical": bool(int(flag.item()) == 1), "cases": cases,
            "failures": sorted({f for fl in gathered for f in fl})}
