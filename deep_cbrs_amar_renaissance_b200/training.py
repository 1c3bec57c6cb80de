"""The training step of the hot path (scope row (f)-1): forward with saved activations,
explicit backward through scorer, lookup, reduction and GNN layers, loss, l2 penalty, Adam.

The reference trains through Keras `fit` (/root/reference/src/experiment.py:155-188):
`model.compile(loss='binary_crossentropy', optimizer=Adam(...))`, one `model(batch)` per batch
with TensorFlow autograd behind it, the l2 penalties registered at src/models/gnn.py:239-246
and :293-294 added to the loss.  Here the same derivatives are spelled out as kernel calls
(csrc/train.cu for the new ones; the sparse backward is the forward SpMM because every
adjacency is symmetric, and dX = dPre W^T is the forward dense kernel on W^T).

A tiny tape keeps the order: every forward helper appends a closure that, given the gradient
of its output, accumulates the gradients of its inputs (`Node.grad`) and of its weights
(`Tape.wgrads`).  Nothing here touches torch.autograd.
"""
import math

import numpy as np
import torch

from . import _lib as L
from . import ops
from .layers import DGCFConv, GATConv, GCNConv, GraphSageConv, LightGCNConv, RGCNConv


class Node:
    """A value on the tape: matrix `x` (optionally seen through the row index `idx`, i.e. the
    value is x[idx]) and the gradient w.r.t. that value once backward has reached it."""
    __slots__ = ("x", "idx", "grad", "needs_grad")

    def __init__(self, x, idx=None, needs_grad=True):
        self.x, self.idx, self.grad, self.needs_grad = x, idx, None, needs_grad

    def add_grad(self, g):
        if not self.needs_grad:
            return
        self.grad = g if self.grad is None else ops.axpby(self.grad, 1.0, g, 1.0)


class Tape:
    def __init__(self):
        self.ops = []
        self.wgrads = {}   # id(weight) -> gradient tensor (same shape, contiguous)
        self.weights = {}  # id(weight) -> weight

    def wgrad(self, w, g):
        if w is None or g is None:
            return
        g = g.reshape(w.shape)
        k = id(w)
        self.weights[k] = w
        self.wgrads[k] = g if k not in self.wgrads else ops.axpby(self.wgrads[k].reshape(g.shape[0], -1), 1.0,
                                                                   g.reshape(g.shape[0], -1), 1.0).reshape(w.shape)

    def backward(self):
        for fn in reversed(self.ops):
            fn()


# ------------------------------------------------------------------ Dense stacks
def dense_train(tape, layer, srcs):
    """Keras Dense on one or two (possibly row-indexed) sources, recorded on the tape."""
    s1 = srcs[0]
    s2 = srcs[1] if len(srcs) > 1 else None
    f1 = s1.x.shape[1]
    layer.build_for(f1 + (s2.x.shape[1] if s2 is not None else 0))
    out = ops.dense(s1.x, layer.kernel, layer.bias, layer.activation, x2=s2.x if s2 is not None else None,
                    idx1=s1.idx, idx2=s2.idx if s2 is not None else None)
    node = Node(out)

    def bwd():
        if node.grad is None:
            return
        dpre = ops.act_grad(node.grad, out, layer.activation)
        dw, db = ops.dense_grad_w(s1.x, dpre, x2=s2.x if s2 is not None else None, idx1=s1.idx,
                                  idx2=s2.idx if s2 is not None else None, want_bias=layer.bias is not None)
        tape.wgrad(layer.kernel, dw)
        tape.wgrad(layer.bias, db)
        if s1.needs_grad or (s2 is not None and s2.needs_grad):
            da = ops.dense(dpre, ops.transpose(layer.kernel))
            s1.add_grad(da[:, :f1])
            if s2 is not None:
                s2.add_grad(da[:, f1:])

    tape.ops.append(bwd)
    return node


def stack_train(tape, stack, srcs):
    """DenseStack (models.Sequential of Dense) -> list of output nodes (the inputs themselves when
    the stack is empty, as in BasicRS with dense_units=[])."""
    if not stack.layers:
        return list(srcs)
    node = dense_train(tape, stack.layers[0], srcs)
    for layer in stack.layers[1:]:
        node = dense_train(tape, layer, [node])
    return [node]


def basic_rs_train(tape, rs, u_src, i_src):
    """BasicRS.call (/root/reference/src/models/basic.py:31-37)"""
    u = stack_train(tape, rs.unet, [u_src])
    i = stack_train(tape, rs.inet, [i_src])
    return stack_train(tape, rs.clf, u + i)[0]


class _Linear:
    """Dense-like view of a bare weight (FusionLayer's projection / attention matrices) for dense_train."""

    def __init__(self, kernel, activation=None):
        self.kernel, self.bias, self.activation = kernel, None, activation

    def build_for(self, in_features):
        return self.kernel.shape[1]


def fuse_train(tape, layer, a, b):
    """FusionLayer (/root/reference/src/layers/fusion.py:49-68) on the tape -> the node list the next Dense consumes."""
    if layer.method == 'concatenate':
        return [a, b]
    layer.build_for(a.x.shape[1], b.x.shape[1])
    if layer.proj_first is not None:
        if layer.proj_first:
            a = dense_train(tape, _Linear(layer.proj_weight), [a])
        else:
            b = dense_train(tape, _Linear(layer.proj_weight), [b])
    ta = dense_train(tape, _Linear(layer.att_weight, "tanh"), [a])
    tb = dense_train(tape, _Linear(layer.att_weight, "tanh"), [b])
    node = Node(ops.attn_fuse(a.x, b.x, ta.x, tb.x))

    def bwd():
        if node.grad is None:
            return
        da, db, dta, dtb = ops.attn_fuse_grad(node.grad, a.x, b.x, ta.x, tb.x)
        a.add_grad(da)
        b.add_grad(db)
        ta.add_grad(dta)
        tb.add_grad(dtb)

    tape.ops.append(bwd)
    return [node]


def hybrid_rs_train(tape, rs, ug, ig, ub, ib):
    """HybridCBRS.call (/root/reference/src/models/hybrid.py:72-89): towers, fusion ('concatenate' or 'attention'),
    classifier or residual classifier"""
    for name in ("dense1a", "dense1b", "dense2a", "dense2b", "dense3a", "dense3b"):
        if not getattr(rs, name).layers:
            raise NotImplementedError("training a HybridCBRS with an empty '%s' stack" % name)
    ug = stack_train(tape, rs.dense1a, [ug])[0]
    ig = stack_train(tape, rs.dense1b, [ig])[0]
    ub = stack_train(tape, rs.dense2a, [ub])[0]
    ib = stack_train(tape, rs.dense2b, [ib])[0]
    if rs.feature_based:
        x1 = stack_train(tape, rs.dense3a, fuse_train(tape, rs.fuse1a, ug, ig))[0]
        x2 = stack_train(tape, rs.dense3b, fuse_train(tape, rs.fuse1b, ub, ib))[0]
    else:
        x1 = stack_train(tape, rs.dense3a, fuse_train(tape, rs.fuse1a, ug, ub))[0]
        x2 = stack_train(tape, rs.dense3b, fuse_train(tape, rs.fuse1b, ig, ib))[0]
    x = fuse_train(tape, rs.fuse2, x1, x2)
    if rs.residual is None:
        return stack_train(tape, rs.clf, x)[0]
    r = stack_train(tape, rs.residual, x)[0]
    h = Node(ops.add3_act(r.x, x1.x, x2.x, rs.activation))

    def bwd():
        if h.grad is None:
            return
        ds = ops.act_grad(h.grad, h.x, rs.activation)
        r.add_grad(ds)
        x1.add_grad(ds)
        x2.add_grad(ds)

    tape.ops.append(bwd)
    return stack_train(tape, rs.clf, [h])[0]


# ------------------------------------------------------------------ GNN layers
def _bwd_csr(graph, view):
    """The operator the backward of a sparse layer multiplies by: the forward CSR when the adjacency is symmetric
    (A^T = A as a multiset of entries, DeviceGraph.symmetric), its transpose otherwise."""
    csr = getattr(graph, view)
    return csr if graph.symmetric else csr.transposed()


def _gcn_train(tape, layer, x_node, graph, out, part=None):
    """GCNConv / RGCNConv: y = act(A_hat (x W) + b).  Backward: dPre = dY*act'(y); db = colsum dPre;
    dZ = A_hat^T dPre (= A_hat dPre on a symmetric graph); dW = x^T dZ; dx = dZ W^T.
    Relational operator (stacked layout [N, R*N]: column r*N + j carries relation r): ONE product with the transposed
    stacked operator gives every relation's dZ_r at once (rows r*N .. (r+1)*N of the result), whatever the symmetry of
    the individual relation blocks.
    part: a RowPartition; the sparse products then run on this rank's rows (RowPartition.sparse_rows), everything else
    as on one GPU."""
    x = x_node.x
    csr = graph.norm
    n = x.shape[0]
    relational = isinstance(layer, RGCNConv)
    kernels = layer.kernels if relational else [layer.kernel]
    relu = layer.activation == "relu"
    z = torch.empty(len(kernels) * n, layer.channels, dtype=torch.float32, device=x.device)
    ops.dense_grouped(x, kernels, z, n)
    if part is None:
        y = ops.spmm(csr, z, out, bias=layer.bias, relu=relu)
    else:
        y, = part.sparse_rows(csr, [out], lambda sl, v, t: ops.spmm(sl, z, v[0], bias=layer.bias, relu=relu, **t[0]))
    node = Node(y)

    def bwd():
        if node.grad is None:
            return
        dpre = ops.act_grad(node.grad, y, layer.activation)
        if layer.bias is not None:
            tape.wgrad(layer.bias, ops.colsum(dpre))
        if not relational:
            if part is None:
                dz = torch.empty(n, layer.channels, dtype=torch.float32, device=x.device)
                ops.spmm(_bwd_csr(graph, "norm"), dpre, dz)
            else:
                dz, = part.sparse_rows(_bwd_csr(graph, "norm"), [part.buffer(("gcn_dz", id(layer)), n, layer.channels)],
                                       lambda sl, v, t: ops.spmm(sl, dpre, v[0], **t[0]))
            dw, _ = ops.dense_grad_w(x, dz, want_bias=False)
            tape.wgrad(layer.kernel, dw)
            x_node.add_grad(ops.dense(dz, ops.transpose(layer.kernel)))
            return
        if part is None:
            dz_all = torch.empty(len(kernels) * n, layer.channels, dtype=torch.float32, device=x.device)
            ops.spmm(csr.transposed(), dpre, dz_all)
        else:
            dz_all, = part.sparse_rows(csr.transposed(),
                                       [part.buffer(("rgcn_dz", id(layer)), len(kernels) * n, layer.channels)],
                                       lambda sl, v, t: ops.spmm(sl, dpre, v[0], **t[0]))
        dx = None
        for r, w in enumerate(kernels):
            dz = dz_all[r * n:(r + 1) * n]
            dw, _ = ops.dense_grad_w(x, dz, want_bias=False)
            tape.wgrad(w, dw)
            t = ops.dense(dz, ops.transpose(w))
            dx = t if dx is None else ops.axpby(dx, 1.0, t, 1.0)
        x_node.add_grad(dx)

    tape.ops.append(bwd)
    return node


def _lightgcn_train(tape, layer, x_node, graph, out, part=None):
    csr = graph.norm
    x = x_node.x
    if part is None:
        y = ops.spmm(csr, x, out)
    else:
        y, = part.sparse_rows(csr, [out], lambda sl, v, t: ops.spmm(sl, x, v[0], **t[0]))
    node = Node(y)

    def bwd():
        if node.grad is None:
            return
        g = node.grad if node.grad.stride(1) == 1 else node.grad.contiguous()
        if part is None:
            dx = torch.empty_like(y) if y.is_contiguous() else torch.empty(y.shape, dtype=torch.float32, device=y.device)
            ops.spmm(_bwd_csr(graph, "norm"), g, dx)
        else:
            dx, = part.sparse_rows(_bwd_csr(graph, "norm"), [part.buffer(("lightgcn_dx", id(layer)), *y.shape)],
                                   lambda sl, v, t: ops.spmm(sl, g, v[0], **t[0]))
        x_node.add_grad(dx)

    tape.ops.append(bwd)
    return node


def _dgcf_train(tape, layer, x_node, graph, out):
    """DGCFConv: y = M (x * sigmoid(w)); dGated = M^T dY (M is a sum of symmetric pieces when A is symmetric)."""
    csr = graph.dgcf
    x = x_node.x
    w = layer.locality_adaptive.w
    gated = ops.row_gate(x, w)
    y = ops.spmm(csr, gated, out)
    node = Node(y)

    def bwd():
        if node.grad is None:
            return
        dg = torch.empty(csr.n_rows, x.shape[1], dtype=torch.float32, device=x.device)
        ops.spmm(_bwd_csr(graph, "dgcf"), node.grad, dg)
        dx, dw = ops.row_gate_grad(dg, x, w)
        tape.wgrad(w, dw)
        x_node.add_grad(dx)

    tape.ops.append(bwd)
    return node


def _sage_train(tape, layer, x_node, graph, out, part=None):
    """GraphSageConv: agg = mean/sum over the raw edge list; v = [x || agg] W + b; out = relu(v / |v|).
    Training keeps v (the fused inference epilogue does not), so the epilogue is its own kernel."""
    x = x_node.x
    csr = graph.raw
    f = x.shape[1]
    mean = layer.aggregate == "mean"
    if part is None:
        agg = torch.empty(csr.n_rows, f, dtype=torch.float32, device=x.device)
        ops.spmm(csr, x, agg, agg=L.AGG_MEAN if mean else L.AGG_SUM)
    else:
        agg, = part.sparse_rows(csr, [part.buffer(("sage_agg", id(layer)), csr.n_rows, f)],
                                lambda sl, v, t: ops.spmm(sl, x, v[0], agg=L.AGG_MEAN if mean else L.AGG_SUM, **t[0]))
    v = ops.dense(x, layer.kernel, layer.bias, None, x2=agg)
    relu = layer.activation == "relu"
    y = ops.l2norm_act(v, relu=relu, out=out)
    node = Node(y)

    def bwd():
        if node.grad is None:
            return
        dv = ops.l2norm_relu_grad(v, node.grad, relu=relu)
        dw, db = ops.dense_grad_w(x, dv, x2=agg, want_bias=layer.bias is not None)
        tape.wgrad(layer.kernel, dw)
        tape.wgrad(layer.bias, db)
        da = ops.dense(dv, ops.transpose(layer.kernel))
        dagg = da[:, f:]
        t = ops.scale_rows_inv_degree(dagg, csr.rowptr) if mean else dagg.contiguous()
        # A^T = A on a symmetric graph (the raw edge list holds both directions of every edge); else the transpose
        if part is None:
            dxa = torch.empty(csr.n_rows, f, dtype=torch.float32, device=x.device)
            ops.spmm(_bwd_csr(graph, "raw"), t, dxa, agg=L.AGG_SUM)
        else:
            dxa, = part.sparse_rows(_bwd_csr(graph, "raw"), [part.buffer(("sage_dxa", id(layer)), csr.n_rows, f)],
                                    lambda sl, v, tg: ops.spmm(sl, t, v[0], agg=L.AGG_SUM, **tg[0]))
        x_node.add_grad(ops.axpby(da[:, :f], 1.0, dxa, 1.0))

    tape.ops.append(bwd)
    return node


def _gat_train(tape, layer, x_node, graph, out, part=None):
    """GATConv: z = x W, p = z.a_self, q = z.a_neigh, fused edge softmax + aggregate (csrc/gat.cu);
    backward = csrc/gat_bwd.cu, then the dense pieces."""
    x = x_node.x
    csr = graph.raw
    if not graph.symmetric:
        # gat_bwd.cu reads the edges ENDING in j from row j, which holds them only when the structure is symmetric
        raise NotImplementedError("GAT training needs a symmetric adjacency (symmetric_adjacency: True, as in every "
                                  "grid of the reference); the forward pass has no such restriction")
    f = x.shape[1]
    w2 = layer.kernel.reshape(f, layer.channels)
    a_s, a_n = layer.attn_kernel_self.reshape(-1), layer.attn_kernel_neighs.reshape(-1)
    z, p, q = ops.dense(x, w2, rowop=L.ROWOP_ATTN, a_self=a_s, a_neigh=a_n)
    relu = layer.activation == "relu"
    if part is None:
        y = ops.gat(csr, z, p, q, out, bias=layer.bias, relu=relu)
    else:
        y, = part.sparse_rows(csr, [out], lambda sl, v, t: ops.gat(sl, z, p, q, v[0], bias=layer.bias, relu=relu,
                                                                   row_offset=sl.row_offset, **t[0]))
    node = Node(y)

    def bwd():
        if node.grad is None:
            return
        d_o = ops.act_grad(node.grad, y, layer.activation)
        if layer.bias is not None:
            tape.wgrad(layer.bias, ops.colsum(d_o))
        if part is None:
            dz, dp, dq = ops.gat_backward(csr, z, p, q, y, layer.bias, d_o, a_s, a_n)
        else:
            # two row-split phases: every rank needs the softmax stats of its rows' neighbours before the gradients
            n, h = z.shape
            stats, = part.sparse_rows(csr, [part.buffer(("gat_stats", id(layer)), n, 3)],
                                      lambda sl, v, t: ops.gat_backward_stats_rows(sl, p, q, y, layer.bias, d_o, v[0],
                                                                                   **t[0]))
            dz, dp, dq = part.sparse_rows(
                csr, [part.buffer(("gat_dz", id(layer)), n, h), part.buffer(("gat_dp", id(layer)), n, 1),
                      part.buffer(("gat_dq", id(layer)), n, 1)],
                lambda sl, v, t: ops.gat_backward_grad_rows(sl, z, p, q, d_o, stats, a_s, a_n, *v, targets=t))
        da_s, _ = ops.dense_grad_w(z, dp.reshape(-1, 1), want_bias=False)
        da_n, _ = ops.dense_grad_w(z, dq.reshape(-1, 1), want_bias=False)
        tape.wgrad(layer.attn_kernel_self, da_s)
        tape.wgrad(layer.attn_kernel_neighs, da_n)
        dw, _ = ops.dense_grad_w(x, dz, want_bias=False)
        tape.wgrad(layer.kernel, dw)
        x_node.add_grad(ops.dense(dz, ops.transpose(w2)))

    tape.ops.append(bwd)
    return node


def embeddings_train(tape, emb):
    """A learnable table as a tape value; its gradient is handed to the optimiser once every consumer recorded
    after this point has run its backward (the sink sits before them on the tape)."""
    node = Node(emb)

    def bwd():
        if node.grad is not None:
            g = node.grad
            tape.wgrad(emb, g if g.is_contiguous() else g.contiguous())

    tape.ops.append(bwd)
    return node


def head_rows_train(tape, node, n):
    """x[:n] (tsgnn.py:94, twgnn.py:96-99): the rows past n get no gradient from this consumer"""
    out = Node(node.x[:n])

    def bwd():
        if out.grad is None:
            return
        g = torch.zeros(node.x.shape, dtype=torch.float32, device=node.x.device)
        g[:n].copy_(out.grad)
        node.add_grad(g)

    tape.ops.append(bwd)
    return out


def concat_rows_train(tape, nodes):
    """tf.concat(..., axis=0) of node-row blocks (gnn.py:137, twgnn.py:96-99)"""
    out = Node(torch.cat([nd.x for nd in nodes], dim=0))

    def bwd():
        if out.grad is None:
            return
        o = 0
        for nd in nodes:
            r = nd.x.shape[0]
            nd.add_grad(out.grad[o:o + r])
            o += r

    tape.ops.append(bwd)
    return out


PARTITIONED_LAYERS = (GCNConv, RGCNConv, LightGCNConv, GraphSageConv, GATConv)


def check_not_partitioned_build(model):
    """Raises NotImplementedError, before any device work, when a GNN stack of `model` runs on a partitioned graph
    build: the partitioned tape multiplies by row slices of the whole operator and of its transpose, which no rank of
    such a build holds."""
    from .graph import PartitionedGraph
    from .models.gnn import SequentialGNN
    gnn = getattr(model, "gnn", None)
    for s in (vars(gnn).values() if gnn is not None else ()):
        if isinstance(s, SequentialGNN) and isinstance(s.adj_matrix, PartitionedGraph):
            raise NotImplementedError("training on a partitioned graph build (RowPartition.build_graph holds only each "
                                      "rank's row blocks; train on a DeviceGraph)")


def check_partitioned_training(seq):
    """Raises NotImplementedError, before any device work, for a partitioned stack the row-split tape does not cover."""
    for layer in seq.seq_layers:
        if not isinstance(layer, PARTITIONED_LAYERS):
            raise NotImplementedError("training {} layers under a RowPartition (no partitioned form; train them on one "
                                      "GPU)".format(type(layer).__name__))


def gnn_train(tape, seq, x_node=None):
    """SequentialGNN.call (/root/reference/src/models/gnn.py:74-84) on the tape -> Node of [N, D_out].
    x_node: the initial node features when they are not the GNN's own embeddings alone
    (HalfInputSequentialGNN / FullInputSequentialGNN, gnn.py:136-147,198-207)."""
    if x_node is None:
        x_node = embeddings_train(tape, seq.embeddings)
    emb = x_node.x
    n = emb.shape[0]
    widths = seq._widths()
    graph = seq.adj_matrix
    part = seq.partition
    if part is not None:
        check_partitioned_training(seq)
    concat = seq.final_node == 'concatenation'
    if seq.final_node not in ('concatenation', 'mean', 'sum', 'last'):
        raise NotImplementedError("training with final_node='%s'" % seq.final_node)
    if part is None:
        buf = torch.empty(n, sum(widths), dtype=torch.float32, device=emb.device) if concat else None
    else:
        buf = part.buffer(("concat",), n, sum(widths)) if concat else None
    nodes = [x_node]
    off = widths[0]
    if concat:
        buf[:, :widths[0]].copy_(emb)
    for layer, w in zip(seq.seq_layers, widths[1:]):
        if not layer.built:
            layer.build([(n, x_node.x.shape[1]), None])
            layer.built = True
        if concat:
            out = buf[:, off:off + w]
        elif part is None:
            out = torch.empty(n, w, dtype=torch.float32, device=emb.device)
        else:
            out = part.buffer(("h", id(layer)), n, w)
        off += w
        if isinstance(layer, (GCNConv, RGCNConv)):
            x_node = _gcn_train(tape, layer, x_node, graph, out, part)
        elif isinstance(layer, LightGCNConv):
            x_node = _lightgcn_train(tape, layer, x_node, graph, out, part)
        elif isinstance(layer, GraphSageConv):
            x_node = _sage_train(tape, layer, x_node, graph, out, part)
        elif isinstance(layer, GATConv):
            x_node = _gat_train(tape, layer, x_node, graph, out, part)
        elif isinstance(layer, DGCFConv):
            x_node = _dgcf_train(tape, layer, x_node, graph, out)
        else:
            raise NotImplementedError("no training form for {}".format(type(layer).__name__))
        nodes.append(x_node)
    k1 = len(nodes)
    if concat:
        red = buf
    elif seq.final_node == 'last':
        red = nodes[-1].x
    else:
        red = ops.reduce_layers([nd.x for nd in nodes], divide_by=float(k1) if seq.final_node == 'mean' else 1.0)
    red_node = Node(red)

    def bwd_reduce():
        g = red_node.grad
        if g is None:
            return
        if concat:
            o = 0
            for nd, w in zip(nodes, widths):
                nd.add_grad(g[:, o:o + w])
                o += w
        elif seq.final_node == 'last':
            nodes[-1].add_grad(g)
        else:
            gs = ops.axpby(g, 1.0 / k1) if seq.final_node == 'mean' else g
            for nd in nodes:
                nd.add_grad(gs)

    # order on the tape: the embeddings sink (appended by embeddings_train before the layers, so it runs after
    # them), the layers in forward order, then the reduction (runs first)
    tape.ops.append(bwd_reduce)
    return red_node


def model_gnn_train(tape, gnn):
    """model.gnn(None) on the tape for every family: GNN (gnn.py:262-264), TwoStepGNN (tsgnn.py:92-94),
    TwoWayGNN (twgnn.py:93-100)."""
    from .models.tsgnn import TwoStepGNN
    from .models.twgnn import TwoWayGNN
    if isinstance(gnn, (TwoStepGNN, TwoWayGNN)):
        stacks = [getattr(gnn, k) for k in ("step_one_gnn_layers", "way_one_gnn_layers", "way_two_gnn_layers",
                                            "step_two_gnn_layers") if hasattr(gnn, k)]
        if any(getattr(s, "partition", None) is not None for s in stacks):
            raise NotImplementedError("training a {} under a RowPartition (no partitioned form; train it on one GPU)"
                                      .format(type(gnn).__name__))
    if isinstance(gnn, TwoStepGNN):
        items = head_rows_train(tape, gnn_train(tape, gnn.step_one_gnn_layers), gnn.n_embeddings)
        two = gnn.step_two_gnn_layers
        x = concat_rows_train(tape, [embeddings_train(tape, two.embeddings), items])
        return gnn_train(tape, two, x)
    if isinstance(gnn, TwoWayGNN):
        users = head_rows_train(tape, gnn_train(tape, gnn.way_one_gnn_layers), gnn.n_users)
        items = head_rows_train(tape, gnn_train(tape, gnn.way_two_gnn_layers), gnn.n_items)
        return gnn_train(tape, gnn.step_two_gnn_layers, concat_rows_train(tape, [users, items]))
    return gnn_train(tape, gnn.gnn_layers)


def lookup_train(tape, table_node, ids_list):
    """tf.nn.embedding_lookup of the propagated table for each id vector
    (/root/reference/src/models/basic.py:72-75) -> one indexed Node per id vector."""
    srcs = [Node(table_node.x, idx) for idx in ids_list]

    def bwd():
        g = None
        for s in srcs:
            if s.grad is None:
                continue
            if g is None:
                g = torch.zeros(table_node.x.shape, dtype=torch.float32, device=table_node.x.device)
            ops.scatter_add_rows(s.grad, s.idx, g)
        if g is not None:
            table_node.add_grad(g)

    tape.ops.append(bwd)
    return srcs


# ------------------------------------------------------------------ optimiser
class Adam:
    """keras.optimizers.Adam(learning_rate=1e-3, beta_1=0.9, beta_2=0.999, epsilon=1e-7)
    (/root/reference/config.yaml:52-56; Keras defaults for what the file leaves out)."""

    def __init__(self, learning_rate=1e-3, beta_1=0.9, beta_2=0.999, epsilon=1e-7, **kwargs):
        self.learning_rate, self.beta_1, self.beta_2, self.epsilon = (float(learning_rate), float(beta_1),
                                                                      float(beta_2), float(epsilon))
        self.iterations = 0
        self._state = {}
        self.lr_t_dev = None  # set by GraphedTrainStep: the captured Adam kernels read the rate from here

    @classmethod
    def from_config(cls, cfg):
        if isinstance(cfg, Adam):
            return cfg
        if cfg is None or isinstance(cfg, str):
            if cfg not in (None, "adam", "Adam"):
                raise NotImplementedError("optimizer '%s' (the reference's configs use Adam)" % cfg)
            return cls()
        if isinstance(cfg, dict):
            cfg = dict(cfg)
            cfg.pop("name", None)
            return cls(**cfg)
        get = lambda k, d: float(getattr(cfg, k, d))  # a keras-like optimizer object
        return cls(get("learning_rate", 1e-3), get("beta_1", 0.9), get("beta_2", 0.999), get("epsilon", 1e-7))

    HYPER_PARAMETERS = ("learning_rate", "beta_1", "beta_2", "epsilon")

    def rate(self, t):
        return self.learning_rate * math.sqrt(1.0 - self.beta_2 ** t) / (1.0 - self.beta_1 ** t)

    def state_dict(self, model):
        """{'iterations', the hyper-parameters, 'm': {weight path: first moment}, 'v': {...: second moment}} for the
        weights of `model` that have moments (a weight gets them at its first update).  The moments are the slot
        tensors themselves, not copies."""
        out = {"iterations": int(self.iterations), "m": {}, "v": {}}
        out.update({k: getattr(self, k) for k in self.HYPER_PARAMETERS})
        for path, w in model.named_weights():
            st = self._state.get(id(w))
            if st is not None:
                out["m"][path], out["v"][path] = st
        return out

    def load_state_dict(self, model, state):
        """Put back what state_dict returned (moments as tensors, ndarrays or anything np.asarray reads).  Refuses,
        before any write, hyper-parameters that differ from this optimiser's and moments whose path, shape or dtype
        does not match a weight of `model`.  Existing slots are filled in place (a captured GraphedTrainStep keeps
        reading them); missing ones are created; a slot the state has no moments for is zeroed, as a weight that was
        never updated."""
        from . import checkpoint
        for k in self.HYPER_PARAMETERS:
            if float(state[k]) != getattr(self, k):
                raise ValueError("Adam state: {} = {!r}, this optimiser has {!r}".format(k, float(state[k]),
                                                                                           getattr(self, k)))
        weights = dict(model.named_weights())
        m, v = state["m"], state["v"]
        want = [(p, tuple(w.shape), "float32") for p, w in model.named_weights() if p in m or p in v]
        checkpoint.check_arrays("Adam first moments", want, m)
        checkpoint.check_arrays("Adam second moments", want, v)
        for path, w in weights.items():
            st = self._state.get(id(w))
            if path not in m:
                if st is not None:
                    st[0].zero_()
                    st[1].zero_()
                continue
            if st is None:
                st = self._state[id(w)] = (torch.empty_like(w), torch.empty_like(w))
            for slot, a in zip(st, (m[path], v[path])):
                slot.copy_(a if isinstance(a, torch.Tensor) else torch.from_numpy(np.asarray(a)))
        self.iterations = int(state["iterations"])

    def apply(self, weights, grads, l2s, capturing=False):
        if not capturing:
            self.iterations += 1
        lr_t = self.rate(max(self.iterations, 1))
        ms, vs = [], []
        for w in weights:
            st = self._state.get(id(w))
            if st is None:
                st = self._state[id(w)] = (torch.zeros_like(w), torch.zeros_like(w))
            ms.append(st[0])
            vs.append(st[1])
        grads = [g if g.is_contiguous() else g.contiguous() for g in grads]
        ops.adam_step_multi(weights, grads, ms, vs, l2s, lr_t, self.beta_1, self.beta_2, self.epsilon,
                            lr_t_dev=self.lr_t_dev if capturing else None)


# ------------------------------------------------------------------ one step
def forward_backward(model, inputs, y):
    """Forward with saved activations, loss, backward.  Returns (tape, loss [1], correct [1], probs)."""
    from .models.basic import BasicGNN, BasicRS, _ids, _rows
    from .models.hybrid import HybridBertGNN, HybridCBRS
    tape = Tape()
    const = lambda rows: Node(_rows(rows), None, needs_grad=False)  # noqa: E731  (a batch input, not differentiated)
    if isinstance(model, BasicRS):  # the scorer alone over pre-computed embedding rows (config.yaml:6)
        u, i = const(inputs[0]), const(inputs[1])
        model.build_for(u.x.shape[1])
        p = basic_rs_train(tape, model, u, i)
    elif isinstance(model, HybridCBRS):
        ug, ig, ub, ib = (const(t) for t in inputs)
        model.build_for(ug.x.shape[1], ub.x.shape[1])
        p = hybrid_rs_train(tape, model, ug, ig, ub, ib)
    elif isinstance(model, BasicGNN):
        red = model_gnn_train(tape, model.gnn)
        u, i = _ids(inputs[0]), _ids(inputs[1])
        model.rs.build_for(red.x.shape[1])
        us, is_ = lookup_train(tape, red, [u, i])
        p = basic_rs_train(tape, model.rs, us, is_)
    elif isinstance(model, HybridBertGNN):
        red = model_gnn_train(tape, model.gnn)
        if len(inputs) == 2:
            if model.content_table is None:
                raise ValueError("ids-only call needs set_content_table(...) first")
            u, i = _ids(inputs[0]), _ids(inputs[1])
            ub, ib = Node(model.content_table, u, needs_grad=False), Node(model.content_table, i, needs_grad=False)
        else:
            u, i = _ids(inputs[0]), _ids(inputs[1])
            ub, ib = const(inputs[2]), const(inputs[3])
        model.rs.build_for(red.x.shape[1], ub.x.shape[1])
        us, is_ = lookup_train(tape, red, [u, i])
        p = hybrid_rs_train(tape, model.rs, us, is_, ub, ib)
    else:
        raise NotImplementedError("no training form for {}".format(type(model).__name__))
    yt = y if isinstance(y, torch.Tensor) else torch.as_tensor(y)
    yt = yt.to(device=p.x.device, dtype=torch.float32).reshape(-1)
    loss, dp, correct = ops.bce(p.x, yt)
    p.grad = dp.reshape(-1, 1)
    tape.backward()
    return tape, loss, correct, p.x


def l2_coefficients(model):
    """id(weight) -> l2 coefficient, from the regularisers attached at add_weight time."""
    out = {}

    def walk(layer):
        for name, w in layer._weights.items():
            reg = layer._regularizers.get(name)
            if reg is not None:
                out[id(w)] = reg.l2
        for _, sub in layer._sublayers():
            walk(sub)

    walk(model)
    return out


def train_step(model, optimizer, inputs, y, capturing=False):
    """One optimiser step on one batch.  Returns device scalars (loss incl. the l2 penalty, #correct)."""
    check_not_partitioned_build(model)
    tape, loss, correct, _ = forward_backward(model, inputs, y)
    l2 = l2_coefficients(model)
    ws = [w for w in model.trainable_weights if id(w) in tape.wgrads]
    for w in ws:
        c = l2.get(id(w), 0.0)
        if c:
            ops.sum_squares(w, c, loss, accumulate=True)
    optimizer.apply(ws, [tape.wgrads[id(w)] for w in ws], [l2.get(id(w), 0.0) for w in ws], capturing=capturing)
    if hasattr(model, "invalidate"):
        model.invalidate()
    return loss, correct


class GraphedTrainStep:
    """The whole optimiser step (forward, backward, loss, Adam: ~100 kernels) captured once into a CUDA
    graph over static batch buffers and replayed per batch.  At MovieLens-1M shape the step is bound by
    launch latency and host dispatch, not by the kernels; replay leaves three small H2D copies, one
    fill of the step's Adam rate and one graph launch on the host side.  Results are the eager step's:
    same kernels, same order."""

    def __init__(self, model, optimizer, batch_size, content_dim=None):
        import numpy as np
        from .models.gnn import SequentialGNN
        check_not_partitioned_build(model)
        gnn = getattr(model, "gnn", None)
        stacks = [s for s in vars(gnn).values() if isinstance(s, SequentialGNN)] if gnn is not None else []
        if any(s.partition is not None for s in stacks):
            # the flag barrier of the peer exchange takes a new epoch per call, which a replayed graph cannot
            raise NotImplementedError("a CUDA-graphed training step under a RowPartition (train eagerly: "
                                      "train_on_batch / fit(cuda_graph=False))")
        self.model, self.optimizer, self.batch_size = model, optimizer, int(batch_size)
        dev = torch.device("cuda", torch.cuda.current_device())
        self.u = torch.zeros(self.batch_size, dtype=torch.int64, device=dev)
        self.i = torch.zeros(self.batch_size, dtype=torch.int64, device=dev)
        self.y = torch.zeros(self.batch_size, dtype=torch.float32, device=dev)
        self.inputs = (self.u, self.i)
        if content_dim:
            self.ub = torch.zeros(self.batch_size, content_dim, dtype=torch.float32, device=dev)
            self.ib = torch.zeros(self.batch_size, content_dim, dtype=torch.float32, device=dev)
            self.inputs = (self.u, self.i, self.ub, self.ib)
        optimizer.lr_t_dev = torch.zeros(1, dtype=torch.float32, device=dev)
        # warm-up off the capture (sizes workspaces, creates the Adam slots), then put everything back
        if content_dim:
            model.build_weights(content_dim)
        else:
            model.build_weights()
        saved_w = [w.clone() for w in model.weights]
        saved_it = optimizer.iterations
        saved_s = {k: (m.clone(), v.clone()) for k, (m, v) in optimizer._state.items()}
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):
                train_step(model, optimizer, self.inputs, self.y)
            for w, s0 in zip(model.weights, saved_w):
                w.copy_(s0)
            for k, (m, v) in optimizer._state.items():
                if k in saved_s:
                    m.copy_(saved_s[k][0])
                    v.copy_(saved_s[k][1])
                else:
                    m.zero_()
                    v.zero_()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        optimizer.iterations = saved_it
        self._np = np
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.loss, self.correct = train_step(model, optimizer, self.inputs, self.y, capturing=True)

    def __call__(self, inputs, y):
        np = self._np
        n = len(y)
        if n != self.batch_size:
            raise ValueError("captured for batches of {}, got {}".format(self.batch_size, n))
        for dst, src in zip(self.inputs + (self.y,), tuple(inputs) + (y,)):
            t = src if isinstance(src, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(src))
            dst.copy_(t.to(dst.dtype), non_blocking=True)
        self.optimizer.iterations += 1
        self.optimizer.lr_t_dev.fill_(self.optimizer.rate(self.optimizer.iterations))
        self.graph.replay()
        if hasattr(self.model, "invalidate"):
            self.model.invalidate()  # a propagated table cached by evaluate / predict is stale after this update
        return self.loss.clone(), self.correct.clone()
