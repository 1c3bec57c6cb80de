"""GPU parity of the training backward where the model tests do not reach: the GAT backward kernel on its own,
model gradients at hot-path widths on hub-heavy graphs (row-major and column-blocked schedules), one-directional
adjacencies (the transposed backward operator), the training forward against the tensor-core inference forward,
and a width sweep of the warp-per-row helpers.  Every reference is float64 torch autograd (oracle/train.py for
whole models).

Tolerance: gradients 2e-4 relative to the largest entry of the same tensor (tests/test_gpu_training.py),
probabilities 2e-5, forward values of the element-wise helpers 1e-5."""
import functools
import time

import numpy as np
import pytest
import torch
from scipy import sparse

from oracle import train as ot
from tests.helpers import assert_close, export_weights
from tests.test_gpu_models import KINDS, _build, _oracle_graph, _randomise
from tests.test_gpu_training import TRAINABLE, _batch, _named_grads, _oracle_names, assert_grad_close

pytestmark = pytest.mark.gpu

F64 = torch.float64


@pytest.fixture(scope="module", autouse=True)
def _device():
    from deep_cbrs_amar_renaissance_b200 import ops
    ops.check_device()
    torch.cuda.set_device(0)


def _cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a, np.float32)).cuda()


def _in_wide(a, lead, width):
    """a [rows, d] copied into columns [lead, lead + d) of a zero [rows, width] buffer: a strided column view"""
    buf = torch.zeros(a.shape[0], width, dtype=torch.float32, device="cuda")
    view = buf[:, lead:lead + a.shape[1]]
    view.copy_(torch.as_tensor(a, dtype=torch.float32))
    return view


# ================================================================== 1. cbrs_gat_backward, kernel level
GAT_N = 8000
GAT_HUB_DEGREE = 5200
GAT_BORDER_ROWS = {30: 5201, 31: 5202, 32: 5203, 33: 5204}   # degree -> row: n_edges = degree + 1 crosses 32


@functools.lru_cache(maxsize=1)
def _gat_graph():
    """A symmetric multiset of edges (the contract of gat_bwd.cu) with: one hub row of 5,200 edges, rows of degree
    30-33, duplicate edges, explicit self loops, and isolated nodes 7000..7999 (only the added self edge).
    Returns (raw device CSR, oracle GAT edge list (rows, cols) as int64 tensors)."""
    from oracle import graph as og
    from deep_cbrs_amar_renaissance_b200.graph import DeviceGraph
    rng = np.random.RandomState(11)
    hub_nb = np.arange(1, GAT_HUB_DEGREE + 1)
    pairs = [np.stack([np.zeros_like(hub_nb), hub_nb], 1)]
    for d, r in GAT_BORDER_ROWS.items():
        pairs.append(np.stack([np.full(d, r), rng.choice(np.arange(6000, 7000), size=d, replace=False)], 1))
    pool = np.concatenate([np.arange(1, GAT_HUB_DEGREE + 1), np.arange(6000, 7000)])
    bg = pool[rng.randint(0, len(pool), size=(12000, 2))]
    bg = bg[bg[:, 0] != bg[:, 1]]
    pairs += [bg, bg[rng.randint(0, len(bg), size=300)]]          # duplicates
    pairs = np.concatenate(pairs)
    loops = rng.choice(pool, size=200, replace=False)            # explicit self loops (replaced by the added one)
    rows = np.concatenate([pairs[:, 0], pairs[:, 1], loops]).astype(np.int32)
    cols = np.concatenate([pairs[:, 1], pairs[:, 0], loops]).astype(np.int32)
    adj = sparse.coo_matrix((np.ones(len(rows), np.float32), (rows, cols)), shape=(GAT_N, GAT_N))
    g = DeviceGraph.from_scipy(adj)
    assert g.symmetric
    csr = g.raw
    ptr, idx, _ = og.reorder_raw(adj)
    deg = np.diff(ptr)
    assert deg[0] == GAT_HUB_DEGREE and (deg[7000:] == 0).all()
    for d, r in GAT_BORDER_ROWS.items():
        assert deg[r] == d
    assert np.array_equal(csr.rowptr.cpu().numpy(), ptr)
    gptr, gcols = og.gat_edges(ptr, idx)
    return csr, (torch.from_numpy(np.repeat(np.arange(GAT_N), np.diff(gptr))), torch.from_numpy(gcols.astype(np.int64)))


def _gat_case(h, relu, with_bias, seed=0):
    """numpy inputs and the float64 autograd reference of one GAT layer on _gat_graph():
    y = act(o + b), loss = sum(dY * y); z is the leaf, p = z.a_self and q = z.a_neigh retained non-leaves."""
    _, (g_rows, g_cols) = _gat_graph()
    rng = np.random.RandomState(100 + h + seed)
    z = rng.standard_normal((GAT_N, h)).astype(np.float32)
    a_s = (rng.standard_normal(h) / np.sqrt(h)).astype(np.float32)
    a_n = (rng.standard_normal(h) / np.sqrt(h)).astype(np.float32)
    b = (rng.standard_normal(h) * 0.3).astype(np.float32) if with_bias else None
    dy = rng.standard_normal((GAT_N, h)).astype(np.float32)
    zt = torch.tensor(z, dtype=F64, requires_grad=True)
    p = zt @ torch.tensor(a_s, dtype=F64)
    q = zt @ torch.tensor(a_n, dtype=F64)
    p.retain_grad()
    q.retain_grad()
    s = p[g_rows] + q[g_cols]
    e = torch.nn.functional.leaky_relu(s, 0.2)
    mx = torch.full((GAT_N,), -float("inf"), dtype=F64).scatter_reduce(0, g_rows, e, reduce="amax")
    w = torch.exp(e - mx[g_rows])
    ssum = torch.zeros(GAT_N, dtype=F64).index_add(0, g_rows, w)
    alpha = w / (ssum[g_rows] + 1e-9)
    o = torch.zeros(GAT_N, h, dtype=F64).index_add(0, g_rows, alpha[:, None] * zt[g_cols])
    pre = o + torch.tensor(b, dtype=F64) if b is not None else o
    y = torch.relu(pre) if relu else pre
    (torch.tensor(dy, dtype=F64) * y).sum().backward()
    assert (s > 0).any() and (s < 0).any()        # both leaky-relu slopes carry gradient
    if relu:
        assert (pre < 0).any() and (pre > 0).any()
    y32 = y.detach().numpy().astype(np.float32)
    d_o = (dy * (y32 > 0)) if relu else dy
    inputs = dict(z=z, p=p.detach().numpy().astype(np.float32), q=q.detach().numpy().astype(np.float32), y=y32, b=b,
                  d_o=d_o.astype(np.float32), a_s=a_s, a_n=a_n)
    want = dict(dz=zt.grad.numpy(), dp=p.grad.numpy(), dq=q.grad.numpy())
    return inputs, want


def _run_gat_backward(inp, z=None, y=None, d_o=None):
    from deep_cbrs_amar_renaissance_b200 import ops
    csr, _ = _gat_graph()
    dz, dp, dq = ops.gat_backward(csr, _cuda(inp["z"]) if z is None else z, _cuda(inp["p"]), _cuda(inp["q"]),
                                  _cuda(inp["y"]) if y is None else y, None if inp["b"] is None else _cuda(inp["b"]),
                                  _cuda(inp["d_o"]) if d_o is None else d_o, _cuda(inp["a_s"]), _cuda(inp["a_n"]))
    torch.cuda.synchronize()
    return dz, dp, dq


def _check_gat(got, want, what):
    for name, g in zip(("dz", "dp", "dq"), got):
        assert_grad_close(g.cpu().numpy(), want[name], "%s %s" % (what, name))


@pytest.mark.parametrize("with_bias", [True, False], ids=["bias", "nobias"])
@pytest.mark.parametrize("relu", [True, False], ids=["relu", "linear"])
@pytest.mark.parametrize("h", [1, 3, 20, 32, 33, 64, 128, 255, 256])
def test_gat_backward_matches_float64_autograd(h, relu, with_bias):
    inp, want = _gat_case(h, relu, with_bias)
    got = _run_gat_backward(inp)
    _check_gat(got, want, "gat_backward h=%d" % h)
    # the rows the kernel treats specially, each against its own scale (the hub dominates the tensor maxima)
    dz = got[0].cpu().numpy()
    for r in [0] + list(GAT_BORDER_ROWS.values()) + [7000, 7999]:
        assert_grad_close(dz[r], want["dz"][r], "gat_backward h=%d dz row %d" % (h, r))


@pytest.mark.parametrize("h", [3, 33, 128])
def test_gat_backward_on_column_slices_of_wider_buffers(h):
    """y and d_o handed over as column slices (ld != h), as the concatenation reduction does"""
    inp, want = _gat_case(h, True, True, seed=1)
    y = _in_wide(inp["y"], 8, h + 24)
    d_o = _in_wide(inp["d_o"], 16, h + 40)
    _check_gat(_run_gat_backward(inp, y=y, d_o=d_o), want, "gat_backward strided h=%d" % h)


@pytest.mark.parametrize("h", [20, 128])
def test_gat_backward_scalar_row_dot_on_a_misaligned_z(h):
    """z one float off a 16-byte boundary (ld a multiple of 4, h % 4 == 0): only the alignment turns the float4 dot
    products off, so the scalar branch runs on a shape the vector branch also takes"""
    inp, want = _gat_case(h, True, True, seed=2)
    z = _in_wide(inp["z"], 1, h + 4)
    assert z.data_ptr() % 16 != 0 and z.stride(0) % 4 == 0
    got = _run_gat_backward(inp, z=z)
    _check_gat(got, want, "gat_backward misaligned z h=%d" % h)
    aligned = _run_gat_backward(inp)
    for name, a, b in zip(("dz", "dp", "dq"), got, aligned):
        assert_grad_close(a.cpu().numpy(), b.cpu().numpy().astype(np.float64), "misaligned vs aligned %s" % name)


def test_gat_backward_is_deterministic():
    inp, _ = _gat_case(128, True, True, seed=3)
    first = _run_gat_backward(inp)
    second = _run_gat_backward(inp)
    for a, b in zip(first, second):
        assert torch.equal(a, b)


def test_gat_backward_refuses_h_above_256():
    from deep_cbrs_amar_renaissance_b200 import _lib as L
    from deep_cbrs_amar_renaissance_b200 import ops
    csr, _ = _gat_graph()
    h = 257
    z = torch.zeros(GAT_N, h, device="cuda")
    vec = torch.zeros(GAT_N, device="cuda")
    a = torch.zeros(h, device="cuda")
    with pytest.raises(L.CbrsError, match="max 256"):
        ops.gat_backward(csr, z, vec, vec, z, None, z, a, a)


# ================================================================== 2. models at width 128 on hub graphs
HOT_GRID = (128, [128, 128, 128], [64, 64], [64, 64])


@functools.lru_cache(maxsize=1)
def _hub_graph():
    """oracle.synth.synth_bipartite (the device generator's numpy twin): 3,000 users, 1,000 items, 60,000 edges;
    its Zipf head gives item rows of up to ~6,000 edges"""
    from oracle.synth import synth_bipartite
    row, col = synth_bipartite(3000, 1000, 60000, 7)
    adj = sparse.coo_matrix((np.ones(len(row), np.float32), (row, col)), shape=(4000, 4000))
    assert np.bincount(row, minlength=4000).max() > 5000
    return adj


def _view_of(kind):
    return {"gcn": "norm", "lightgcn": "norm", "dgcf": "dgcf"}.get(kind, "raw")


def _attention_of_both_signs(model):
    """a_neigh = -a_self + noise, so that s_ij = p_i + q_j ~ p_i - p_j takes both signs on the symmetric edge set.
    Past the first layer the rows of x are alike and, with independent attention vectors, every score of a layer
    shares one sign: the softmax then cancels dp exactly, attn_kernel_self's gradient is analytically zero, and
    the comparison would check nothing but rounding noise."""
    rng = np.random.RandomState(12)
    ws = dict(model.named_weights())
    with torch.no_grad():
        for name, a_s in ws.items():
            if name.endswith("/attn_kernel_self"):
                a_n = ws[name[:-len("self")] + "neigh"]
                noise = torch.from_numpy(rng.standard_normal(tuple(a_n.shape)).astype(np.float32)).cuda()
                a_n.copy_(-a_s + 0.1 * a_s.abs().mean() * noise)
    if hasattr(model, "invalidate"):
        model.invalidate()


def _check_model_gradients(model, kind, adj, n_users, n_items, what, aggregate="mean", batch_seed=3):
    """test_gradients_match_autograd_oracle on an arbitrary model / graph: probabilities, loss, accuracy count and
    every gradient against oracle.train.gradients"""
    from deep_cbrs_amar_renaissance_b200 import training
    u, i, y = _batch(n_users, n_items, 1024, batch_seed)
    model((u, i))
    _randomise(model, seed=5)
    if kind == "gat":
        _attention_of_both_signs(model)
    w = export_weights(model)
    tape, loss, correct, probs = training.forward_backward(model, (u, i), y)
    torch.cuda.synchronize()
    fn = "mean" if kind in ("lightgcn", "dgcf") else "concatenation"
    want, want_loss, want_p = ot.gradients(kind, w, _oracle_graph(kind, adj), (u, i), y, final_node=fn,
                                           aggregate=aggregate)
    assert_close(probs.cpu().numpy().reshape(-1), want_p, rtol=2e-5, what=what + " probabilities")
    assert abs(float(loss.item()) - want_loss) <= 1e-5 * max(1.0, abs(want_loss))
    assert int(correct.item()) == int(((want_p > 0.5) == (y > 0.5)).sum())
    got = _named_grads(model, tape)
    assert set(got) == set(want), (sorted(got), sorted(want))
    for k in sorted(want):
        assert_grad_close(got[k], want[k], "%s grad %s" % (what, k))
    return (u, i, y), probs


def _hot_model(name, monkeypatch, schedule, **extra):
    from deep_cbrs_amar_renaissance_b200 import graph
    if schedule == "blocked":
        # 256-column windows, rows of >= 64 edges: every item row of the Zipf head is cut into several blocked chunks
        # and merged through heavy-row slots, in the forward and in the backward SpMM
        monkeypatch.setattr(graph, "FORCED_BLOCKING", (256, 64))
    adj = _hub_graph()
    model = _build(name, adj, HOT_GRID, **extra)
    return adj, model


def _assert_schedule(model, kind, schedule):
    csr = getattr(model.gnn.gnn_layers.adj_matrix, _view_of(kind))
    if schedule == "blocked":
        assert csr.blocking != (0, 0) and csr.chunks["n_heavy"] > 0 and csr.chunks["chunk_len"] is not None
    else:
        assert csr.blocking == (0, 0)


@pytest.mark.parametrize("schedule", ["rowmajor", "blocked"])
@pytest.mark.parametrize("name", TRAINABLE)
def test_hot_width_gradients_on_a_hub_graph(name, schedule, monkeypatch):
    adj, model = _hot_model(name, monkeypatch, schedule)
    kind = KINDS[name]
    _check_model_gradients(model, kind, adj, 3000, 1000, "%s %s" % (name, schedule))
    _assert_schedule(model, kind, schedule)


@pytest.mark.parametrize("schedule", ["rowmajor", "blocked"])
def test_hot_width_graphsage_sum_gradients(schedule, monkeypatch):
    adj, model = _hot_model("BasicGraphSage", monkeypatch, schedule)
    for layer in model.gnn.gnn_layers.seq_layers:
        layer.aggregate = "sum"
    _check_model_gradients(model, "sage", adj, 3000, 1000, "GraphSage-sum " + schedule, aggregate="sum")
    _assert_schedule(model, "sage", schedule)


def test_gat_wider_than_the_attention_epilogue_is_refused():
    """the attention row-op of cbrs_dense keeps a row's 128 outputs in one tile: a 160-wide GAT layer must fail at its
    first forward with the kernel's message, not train on a truncated transform"""
    from deep_cbrs_amar_renaissance_b200 import _lib as L
    from deep_cbrs_amar_renaissance_b200 import training
    adj = _hub_graph()
    model = _build("BasicGAT", adj, (128, [160], [64], [64]))
    u, i, y = _batch(3000, 1000, 64, 0)
    with pytest.raises(L.CbrsError, match="n <= 128"):
        model((u, i))
    with pytest.raises(L.CbrsError, match="n <= 128"):
        training.forward_backward(model, (u, i), y)


# ================================================================== 3. one-directional adjacency
DIR_USERS, DIR_ITEMS = 300, 200
DIR_GRID = (32, [32, 32], [48, 48], [64, 64])


@functools.lru_cache(maxsize=2)
def _directed_graph(form):
    """symmetric_adjacency: False (user -> item entries only) from seeded ratings; 'partial' adds the reverse of a
    random 20 % of them so that A.A is not empty and DGCF has a crosshop, 'pure' leaves A.A empty"""
    from deep_cbrs_amar_renaissance_b200.data.preprocess import build_adjacency_matrix
    rng = np.random.RandomState(4)
    uu = rng.randint(0, DIR_USERS, 5000)
    ii = rng.randint(0, DIR_ITEMS, 5000) + DIR_USERS
    ratings = np.unique(np.stack([uu, ii, rng.randint(0, 2, 5000)], 1), axis=0)
    adj = build_adjacency_matrix(ratings, np.arange(DIR_USERS), np.arange(DIR_ITEMS), symmetric_adjacency=False)
    assert (adj.row < DIR_USERS).all() and (adj.col >= DIR_USERS).all()
    if form == "partial":
        pick = rng.rand(adj.nnz) < 0.2
        adj = sparse.coo_matrix((np.concatenate([adj.data, adj.data[pick]]),
                                 (np.concatenate([adj.row, adj.col[pick]]), np.concatenate([adj.col, adj.row[pick]]))),
                                shape=adj.shape)
    a = adj.tocsr()
    assert ((a @ a).nnz > 0) == (form == "partial")
    return adj


def _directed_model(name, form, grid=DIR_GRID):
    model = _build(name, _directed_graph(form), grid)
    assert model.gnn.gnn_layers.adj_matrix.symmetric is False
    return model


@pytest.mark.parametrize("schedule", ["rowmajor", "blocked"])
@pytest.mark.parametrize("form", ["partial", "pure"])
@pytest.mark.parametrize("name", ["BasicGCN", "BasicLightGCN", "BasicGraphSage", "BasicGraphSage-sum", "BasicDGCF"])
def test_one_directional_gradients(name, form, schedule, monkeypatch):
    """the backward multiplies by the transposed operator (training._bwd_csr) when the adjacency is not symmetric; on
    the blocked schedule the transpose inherits the forward CSR's column blocking"""
    from deep_cbrs_amar_renaissance_b200 import graph
    base = name.split("-")[0]
    kind = KINDS[base]
    if schedule == "blocked":
        monkeypatch.setattr(graph, "FORCED_BLOCKING", (64, 8))   # rows of >= 8 edges cut at 64-column windows
    model = _directed_model(base, form)
    aggregate = "sum" if name.endswith("-sum") else "mean"
    if aggregate == "sum":
        for layer in model.gnn.gnn_layers.seq_layers:
            layer.aggregate = "sum"
    adj = _directed_graph(form)
    _check_model_gradients(model, kind, adj, DIR_USERS, DIR_ITEMS, "%s %s %s" % (name, form, schedule),
                           aggregate=aggregate)
    fwd = getattr(model.gnn.gnn_layers.adj_matrix, _view_of(kind))
    bwd = fwd.transposed()
    assert bwd.n_rows == fwd.n_cols and bwd.nnz == fwd.nnz and bwd.blocking == fwd.blocking
    if schedule == "blocked":
        assert fwd.blocking != (0, 0) and fwd.chunks["n_heavy"] > 0 and bwd.chunks["n_heavy"] > 0
    if kind == "dgcf":
        from oracle import layers as ol
        g = model.gnn.gnn_layers.adj_matrix
        _, info = ol.dgcf_preprocess(adj)
        assert g.dgcf_info["cross_edges"] == info["cross_edges"] and g.dgcf_info["epsilon"] == info["epsilon"]
        if form == "pure":
            # A.A is empty: the filtered crosshop is gcn_filter's diagonal alone, every threshold keeps all n of its
            # entries, and the tie goes to the first threshold
            assert info["cross_edges"] == [DIR_USERS + DIR_ITEMS] * 4 and info["epsilon"] == g.DGCF_EPSILONS[0]


@pytest.mark.parametrize("name", ["BasicGCN", "BasicLightGCN", "BasicGraphSage", "BasicDGCF"])
def test_one_directional_adam_step(name):
    """one step of test_three_adam_steps_match_oracle on the partial one-directional graph: loss with the l2 penalty,
    every gradient, and the Adam update against the written-out Keras formula"""
    from deep_cbrs_amar_renaissance_b200 import ops, training
    kind = KINDS[name]
    model = _directed_model(name, "partial", (8, [8, 8], [24, 24], [48, 48]))
    u, i, y = _batch(DIR_USERS, DIR_ITEMS, 512, 10)
    model((u, i))
    _randomise(model, seed=8)
    adam = training.Adam(learning_rate=1e-2)
    l2 = training.l2_coefficients(model)
    w = export_weights(model)
    tape, loss, _, _ = training.forward_backward(model, (u, i), y)
    ws = [x for x in model.trainable_weights if id(x) in tape.wgrads]
    for x in ws:
        if l2.get(id(x)):
            ops.sum_squares(x, l2[id(x)], loss, accumulate=True)
    fn = "mean" if kind in ("lightgcn", "dgcf") else "concatenation"
    want, want_loss, _ = ot.gradients(kind, w, _oracle_graph(kind, _directed_graph("partial")), (u, i), y, l2=1e-4,
                                      final_node=fn)
    assert abs(float(loss.item()) - want_loss) <= 2e-5 * max(1.0, abs(want_loss))
    before = {n: x.detach().cpu().numpy().astype(np.float64) for n, x in model.named_weights()}
    names = dict(zip([n for n, _ in model.named_weights()], _oracle_names(model)))
    full = {}
    for n, x in model.named_weights():
        full[n] = tape.wgrads[id(x)].detach().cpu().numpy().astype(np.float64) + 2 * l2.get(id(x), 0.0) * before[n]
        assert_grad_close(full[n], want[names[n]].reshape(full[n].shape), "%s grad %s" % (name, n))
    adam.apply(ws, [tape.wgrads[id(x)] for x in ws], [l2.get(id(x), 0.0) for x in ws])
    torch.cuda.synchronize()
    for n, x in model.named_weights():
        new, _, _ = ot.adam_update(before[n], full[n], np.zeros_like(full[n]), np.zeros_like(full[n]), 1, lr=1e-2)
        assert_close(x.detach().cpu().numpy(), new, atol=2e-6, what="%s adam %s" % (name, n))


def test_one_directional_gat_forward_matches_and_training_is_refused():
    from oracle import layers as ol
    from deep_cbrs_amar_renaissance_b200 import training
    adj = _directed_graph("partial")
    model = _directed_model("BasicGAT", "partial")
    u, i, y = _batch(DIR_USERS, DIR_ITEMS, 256, 1)
    model((u, i))
    _randomise(model, seed=2)
    w = export_weights(model)
    emb = ol.propagate("gat", w["embeddings"], _oracle_graph("gat", adj), w["layers"])
    assert_close(model.gnn(None).cpu().numpy(), emb, what="one-directional GAT embeddings")
    with pytest.raises(NotImplementedError, match="symmetric"):
        training.forward_backward(model, (u, i), y)


# ================================================================== 4. training vs inference forward at tensor-core size
@pytest.mark.parametrize("name", ["BasicGCN", "BasicGraphSage"])
def test_training_forward_agrees_with_the_tensor_core_inference_forward(name):
    """From TF32X3_MIN_ROWS nodes inference runs the 3xTF32 tensor-core transform, the training tape the FFMA kernels:
    a model trained with one is served with the other, so both forwards and the gradients are held to the oracle"""
    from deep_cbrs_amar_renaissance_b200 import ops, training
    from oracle.synth import synth_bipartite
    n_users, n_items = 60000, 12000
    row, col = synth_bipartite(n_users, n_items, 300000, 21)
    n = n_users + n_items
    assert n > ops.TF32X3_MIN_ROWS
    adj = sparse.coo_matrix((np.ones(len(row), np.float32), (row, col)), shape=(n, n))
    model = _build(name, adj, (64, [64, 64], [64, 64], [64, 64]))
    assert ops.tf32x3_chosen(n, 64, 64)
    u, i, y = _batch(n_users, n_items, 1024, 6)
    model((u, i))
    _randomise(model, seed=4)
    served = model((u, i)).cpu().numpy().reshape(-1)
    w = export_weights(model)
    tape, loss, _, probs = training.forward_backward(model, (u, i), y)
    probs = probs.cpu().numpy().reshape(-1)
    assert_close(probs, served, rtol=2e-5, what=name + " training vs inference probabilities")
    kind = KINDS[name]
    t0 = time.perf_counter()
    want, want_loss, want_p = ot.gradients(kind, w, _oracle_graph(kind, adj), (u, i), y)
    print("%s float64 oracle at %d nodes: %.1f s" % (name, n, time.perf_counter() - t0))
    assert_close(served, want_p, rtol=2e-5, what=name + " inference probabilities")
    assert_close(probs, want_p, rtol=2e-5, what=name + " training probabilities")
    got = _named_grads(model, tape)
    assert set(got) == set(want)
    for k in sorted(want):
        assert_grad_close(got[k], want[k], "%s grad %s" % (name, k))


# ================================================================== 5. warp-per-row helpers, width sweep
def _layout(a, strided, lead):
    return _in_wide(a, lead, a.shape[1] + lead + 5) if strided else _cuda(a)


@pytest.mark.parametrize("strided", [False, True], ids=["contiguous", "strided"])
@pytest.mark.parametrize("relu", [True, False], ids=["relu", "linear"])
@pytest.mark.parametrize("d", [1, 31, 33, 128, 256])
def test_l2norm_act_and_grad_width_sweep(d, relu, strided):
    from deep_cbrs_amar_renaissance_b200 import ops
    rng = np.random.RandomState(d)
    rows = 300
    v = rng.standard_normal((rows, d)).astype(np.float32)
    v[0] = -np.abs(v[0]) - 0.1                  # all negative: the relu mask of the row is all zero
    v[1] = (rng.standard_normal(d) * 1e-8).astype(np.float32)    # sum v^2 < 1e-12: the floored row
    v[2] = np.abs(v[2]) + 0.1
    dout = rng.standard_normal((rows, d)).astype(np.float32)
    vt = torch.tensor(v, dtype=F64, requires_grad=True)
    nrm = vt / torch.sqrt(torch.clamp((vt * vt).sum(1, keepdim=True), min=1e-12))
    out = torch.relu(nrm) if relu else nrm
    (torch.tensor(dout, dtype=F64) * out).sum().backward()
    want_dv = vt.grad.numpy()
    dst = _layout(np.zeros((rows, d), np.float32), strided, 3) if strided else None
    got = ops.l2norm_act(_layout(v, strided, 2), relu=relu, out=dst)
    assert_close(got.cpu().numpy(), out.detach().numpy(), what="l2norm_act d=%d" % d)
    if strided:
        assert got.data_ptr() == dst.data_ptr()
    dv = ops.l2norm_relu_grad(_layout(v, strided, 2), _layout(dout, strided, 1), relu=relu).cpu().numpy()
    # the floored row's gradient is 1e6 times the others: each kind of row against its own scale
    assert_grad_close(dv[1], want_dv[1], "l2norm_relu_grad d=%d floored row" % d)
    keep = np.arange(rows) != 1
    if d > 1:
        assert_grad_close(dv[keep], want_dv[keep], "l2norm_relu_grad d=%d" % d)
    else:
        # one column: n = +-1 whatever v is, so dv = (g - n^2 g) / s vanishes analytically and the kernel returns the
        # float32 rounding of that difference; it is held to 2e-4 of the terms it cancels, g / s
        terms = np.abs(dout[keep] / v[keep]).max()
        assert_close(dv[keep], want_dv[keep], atol=2e-4 * terms, what="l2norm_relu_grad d=1")
    if relu:
        assert (dv[0] == 0).all()


@pytest.mark.parametrize("strided", [False, True], ids=["contiguous", "strided"])
@pytest.mark.parametrize("d", [1, 33, 128])
def test_row_gate_and_grad_width_sweep(d, strided):
    from deep_cbrs_amar_renaissance_b200 import ops
    rng = np.random.RandomState(7 + d)
    rows = 400
    x = rng.standard_normal((rows, d)).astype(np.float32)
    w = rng.standard_normal(rows).astype(np.float32)
    w[:50], w[50:100] = 30.0, -30.0                 # saturated sigmoid on both sides
    g = rng.standard_normal((rows, d)).astype(np.float32)
    xt = torch.tensor(x, dtype=F64, requires_grad=True)
    wt = torch.tensor(w, dtype=F64, requires_grad=True)
    out = xt * torch.sigmoid(wt)[:, None]
    (torch.tensor(g, dtype=F64) * out).sum().backward()
    wd = _cuda(w.reshape(-1, 1))
    got = ops.row_gate(_layout(x, strided, 2), wd).cpu().numpy()
    assert_close(got, out.detach().numpy(), what="row_gate d=%d" % d)
    dx, dw = ops.row_gate_grad(_layout(g, strided, 1), _layout(x, strided, 2), wd)
    dx, dw = dx.cpu().numpy(), dw.cpu().numpy()
    assert_grad_close(dx, xt.grad.numpy(), "row_gate_grad dx d=%d" % d)
    assert_grad_close(dw, wt.grad.numpy(), "row_gate_grad dw d=%d" % d)
    # the w = -30 rows: gate ~9.4e-14, gradients relative to their own scale
    assert_close(got[50:100], out.detach().numpy()[50:100], what="row_gate d=%d at w=-30" % d)
    assert_close(dx[50:100], xt.grad.numpy()[50:100], what="row_gate_grad dx d=%d at w=-30" % d)
    assert_close(dw[50:100], wt.grad.numpy()[50:100], what="row_gate_grad dw d=%d at w=-30" % d)


@pytest.mark.parametrize("strided", [False, True], ids=["contiguous", "strided"])
@pytest.mark.parametrize("d", [1, 33, 128])
def test_attn_fuse_and_grad_width_sweep(d, strided):
    from deep_cbrs_amar_renaissance_b200 import ops
    rng = np.random.RandomState(30 + d)
    rows = 300
    a, b, g = (rng.standard_normal((rows, d)).astype(np.float32) for _ in range(3))
    ta, tb = (np.tanh(rng.standard_normal((rows, d)) * 2).astype(np.float32) for _ in range(2))
    leaves = [torch.tensor(t, dtype=F64, requires_grad=True) for t in (a, b, ta, tb)]
    at, bt, tat, tbt = leaves
    att = torch.softmax(torch.stack([tat, tbt], 1), dim=1)
    out = (att * torch.stack([at, bt], 1)).sum(1)
    (torch.tensor(g, dtype=F64) * out).sum().backward()
    got = ops.attn_fuse(_layout(a, strided, 2), _layout(b, strided, 3), _cuda(ta), _cuda(tb)).cpu().numpy()
    assert_close(got, out.detach().numpy(), what="attn_fuse d=%d" % d)
    grads = ops.attn_fuse_grad(_layout(g, strided, 1), _layout(a, strided, 2), _layout(b, strided, 3), _cuda(ta), _cuda(tb))
    for name, gg, leaf in zip(("da", "db", "dta", "dtb"), grads, leaves):
        assert_grad_close(gg.cpu().numpy(), leaf.grad.numpy(), "attn_fuse_grad %s d=%d" % (name, d))


@pytest.mark.parametrize("strided", [False, True], ids=["contiguous", "strided"])
@pytest.mark.parametrize("act", [None, "relu", "sigmoid", "tanh"])
def test_add3_act_every_activation(act, strided):
    from deep_cbrs_amar_renaissance_b200 import ops
    rng = np.random.RandomState(5)
    a, b, c = (rng.standard_normal((200, 65)).astype(np.float32) for _ in range(3))
    s = torch.tensor(a, dtype=F64) + torch.tensor(b, dtype=F64) + torch.tensor(c, dtype=F64)
    want = {None: s, "relu": torch.relu(s), "sigmoid": torch.sigmoid(s), "tanh": torch.tanh(s)}[act].numpy()
    got = ops.add3_act(_layout(a, strided, 1), _layout(b, strided, 2), _layout(c, strided, 3), act).cpu().numpy()
    assert_close(got, want, what="add3_act %s" % act)
