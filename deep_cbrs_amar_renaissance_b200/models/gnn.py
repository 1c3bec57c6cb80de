"""GNN builders (mirror of /root/reference/src/models/gnn.py:13-84,210-415).

Same class names, constructor keywords and call convention as the reference:
`GCN(adj, n_hiddens=..., embedding_dim=..., final_node=..., l2_regularizer=..., **ignored)`,
`model(None) -> [N, D_out]`.  The adjacency is uploaded once and lives in HBM as a
DeviceGraph; every layer output is written straight into its column slice of one
[N, D_out] buffer, so the 'concatenation' reduction is free.
"""
import abc

import torch

from .. import graph
from ..graph import DeviceGraph
from ..keras_like import L2, Model, default_device
from ..layers import DGCFConv, GATConv, GCNConv, GraphSageConv, LightGCNConv, ReductionLayer, RGCNConv
from ..utilities.math import convert_to_tensor


class SequentialGNN(Model):
    def __init__(self, adj_matrix, seq_layers, embedding_dim=8, final_node='concatenation', dropout=None,
                 regularizer=None, cache_neighbours=False):
        super().__init__("sequential_gnn")
        if cache_neighbours:
            raise NotImplementedError("Multi-hops neighbours caching is not yet completely supported!")
        if dropout:
            raise NotImplementedError("layer dropout is None in every reference grid (forward path only)")
        self.cache_neighbours = cache_neighbours
        self.embedding_dim = int(embedding_dim)
        self.embeddings = self.add_weight('embeddings', (adj_matrix.shape[0], embedding_dim), 'glorot_uniform',
                                          regularizer)
        self._finish_init(adj_matrix, seq_layers, final_node)

    def _finish_init(self, adj_matrix, seq_layers, final_node):
        if type(self) is not SequentialGNN:
            graph.refuse_partitioned([adj_matrix], "a Two-Step / Two-Way GNN stack")
        for layer in seq_layers:
            if not isinstance(layer, (GCNConv, LightGCNConv, GraphSageConv, GATConv)):
                graph.refuse_partitioned([adj_matrix], type(layer).__name__)
        self.adj_matrix = convert_to_tensor(adj_matrix, device=default_device())
        self.n_nodes = int(adj_matrix.shape[0])
        self.dropout = None
        self.final_node = final_node
        self.reduce = ReductionLayer(final_node)
        self.seq_layers = list(seq_layers)
        self._buf = None
        self.partition = None  # set by distributed.RowPartition.attach
        self.built = True

    def set_feature_dtype(self, dtype):
        """'fp32' (the reference's arithmetic, default) or 'bf16': GCN layers store the transform Z = X W that the
        sparse kernel gathers as bf16 (fp32 products and sums; stated tolerance in tests/test_gpu_bf16.py)."""
        if dtype not in ("fp32", "bf16"):
            raise ValueError("feature dtype must be 'fp32' or 'bf16'")
        for layer in self.seq_layers:
            if dtype == "bf16" and not isinstance(layer, GCNConv):
                raise NotImplementedError("bf16 operand storage is built for GCNConv stacks")
            layer.feature_dtype = dtype

    @property
    def n_hops(self):
        return len(self.seq_layers)

    def __len__(self):
        return self.n_hops

    def build_layers(self):
        """Create every layer's weights without running a kernel (Keras does it on the first call)."""
        f = self.embedding_dim
        for layer in self.seq_layers:
            if not layer.built:
                layer.build([(self.n_nodes, f), None])
                layer.built = True
            f = getattr(layer, "channels", f)

    @property
    def out_dim(self):
        w = self._widths()
        return sum(w) if self.final_node == 'concatenation' else w[-1]

    def _widths(self):
        return [self.embedding_dim] + [getattr(layer, "channels", self.embedding_dim) for layer in self.seq_layers]

    def call(self, inputs, **kwargs):
        if self.partition is not None:
            return self.partition.propagate(self)
        return self._run(self.embeddings)

    def last_layer_subset(self):
        """True when a call that only reads the output at some rows may run the last layer's sparse product on those
        rows alone (graph.last_layer_subset_policy)."""
        last = self.seq_layers[-1] if self.seq_layers else None
        return graph.last_layer_subset_policy(self.n_nodes, self.partition is not None,
                                              self.final_node == 'concatenation',
                                              isinstance(last, (GCNConv, LightGCNConv)))

    def _run(self, x, rows=None):
        """the layer loop + reduction of gnn.py:74-84 on the initial node features x.
        rows (int64 device ids; only when last_layer_subset() holds): the last layer's output is computed at these
        rows only - every other row of its slice is left unfilled, so the result must not leave the caller."""
        n = x.shape[0]
        if self.final_node == 'concatenation':
            # the subset is built before layer 1 is enqueued: its one device-to-host copy exposes only a launch gap
            last_csr = self.adj_matrix.norm.row_subset(rows) if rows is not None else None
            widths = self._widths()
            if self._buf is None or self._buf.shape != (n, sum(widths)):
                self._buf = torch.empty(n, sum(widths), dtype=torch.float32, device=x.device)
            buf = self._buf
            buf[:, :widths[0]].copy_(x)
            hs = [buf[:, :widths[0]]]
            off = widths[0]
            for k, (layer, w) in enumerate(zip(self.seq_layers, widths[1:])):
                out = buf[:, off:off + w]
                if last_csr is not None and k == len(self.seq_layers) - 1:
                    x = layer([x, self.adj_matrix], out=out, csr=last_csr)
                else:
                    x = layer([x, self.adj_matrix], out=out)
                hs.append(out)
                off += w
            for h in hs:
                h._cbrs_concat_buf = buf
            return self.reduce(hs)
        hs = [x]
        for layer in self.seq_layers:
            x = layer([x, self.adj_matrix])
            hs.append(x)
        return self.reduce(hs)


class HalfInputSequentialGNN(SequentialGNN):
    """gnn.py:87-147: the first `n_random_embeddings` node rows are learnable embeddings, the remaining rows come in
    as the call's input (the item rows produced by the first step of a Two-Step model)."""

    def __init__(self, adj_matrix, seq_layers, n_random_embeddings, final_node='concatenation', dropout=None,
                 embedding_dim=8, regularizer=None, cache_neighbours=False):
        Model.__init__(self, "half_input_sequential_gnn")
        if cache_neighbours:
            raise NotImplementedError("Multi-hops neighbours caching is not yet completely supported!")
        if dropout:
            raise NotImplementedError("layer dropout is None in every reference grid (forward path only)")
        self.cache_neighbours = cache_neighbours
        self.embedding_dim = int(embedding_dim)
        self.embeddings = self.add_weight('embeddings', (n_random_embeddings, embedding_dim), 'glorot_uniform', regularizer)
        self._finish_init(adj_matrix, seq_layers, final_node)

    def call(self, inputs, **kwargs):
        if inputs.shape[1] != self.embedding_dim:
            raise ValueError("input rows are {} wide, the embeddings {}".format(inputs.shape[1], self.embedding_dim))
        x = torch.cat([self.embeddings, inputs], dim=0)
        if x.shape[0] != self.n_nodes:
            raise ValueError("{} embedding rows + {} input rows != {} graph nodes".format(
                self.embeddings.shape[0], inputs.shape[0], self.n_nodes))
        return self._run(x)


class FullInputSequentialGNN(SequentialGNN):
    """gnn.py:150-207: no embeddings of its own; every node row comes in as the call's input (the user rows and item
    rows the two ways of a Two-Way model produce).  `embedding_dim` is the width of that input: the reference learns
    it at the first call, here the owner states it so that the weights can be created before any kernel runs."""

    def __init__(self, adj_matrix, seq_layers, final_node='concatenation', dropout=None, cache_neighbours=False,
                 embedding_dim=None):
        Model.__init__(self, "full_input_sequential_gnn")
        if cache_neighbours:
            raise NotImplementedError("Multi-hops neighbours caching is not yet completely supported!")
        if dropout:
            raise NotImplementedError("layer dropout is None in every reference grid (forward path only)")
        self.cache_neighbours = cache_neighbours
        self.embedding_dim = int(embedding_dim) if embedding_dim is not None else None
        self.embeddings = None
        self._finish_init(adj_matrix, seq_layers, final_node)

    def build_layers(self):
        if self.embedding_dim is None:
            raise ValueError("the input width is unknown before the first call; pass embedding_dim")
        super().build_layers()

    def call(self, inputs, **kwargs):
        if self.embedding_dim is None:
            self.embedding_dim = int(inputs.shape[1])
        if inputs.shape != (self.n_nodes, self.embedding_dim):
            raise ValueError("input is {}, the graph has {} nodes of width {}".format(
                tuple(inputs.shape), self.n_nodes, self.embedding_dim))
        return self._run(inputs if inputs.is_contiguous() else inputs.contiguous())


class GNN(Model, abc.ABC):
    def __init__(self, adj_matrix, n_hops, embedding_dim=8, final_node="concatenation", dropout=None,
                 l2_regularizer=None, cache_neighbours=False, **kwargs):
        super().__init__(type(self).__name__.lower())
        regularizer = L2(l2_regularizer) if l2_regularizer is not None else None
        gnn_layers = [self.build_gnn_layer(i, regularizer=regularizer) for i in range(n_hops)]
        self.gnn_layers = SequentialGNN(adj_matrix, gnn_layers, embedding_dim=embedding_dim, final_node=final_node,
                                        dropout=dropout, regularizer=regularizer, cache_neighbours=cache_neighbours)
        self.built = True

    @abc.abstractmethod
    def build_gnn_layer(self, i, **kwargs):
        pass

    def build_layers(self):
        self.gnn_layers.build_layers()

    @property
    def out_dim(self):
        return self.gnn_layers.out_dim

    def call(self, inputs, **kwargs):
        return self.gnn_layers(None)


class GCN(GNN):
    def __init__(self, adj_matrix, n_hiddens=(8, 8, 8), **kwargs):
        self.n_hiddens = n_hiddens
        adj_matrix = GCNConv.preprocess(adj_matrix)
        super().__init__(adj_matrix, len(n_hiddens), **kwargs)

    def build_gnn_layer(self, i, regularizer=None, **kwargs):
        return GCNConv(self.n_hiddens[i], activation='relu', kernel_regularizer=regularizer,
                       bias_regularizer=regularizer)


class GAT(GNN):
    def __init__(self, adj_matrix, n_hiddens=(8, 8, 8), dropout_rate=0.0, **kwargs):
        self.n_hiddens = n_hiddens
        self.dropout_rate = dropout_rate
        super().__init__(adj_matrix, len(n_hiddens), **kwargs)

    def build_gnn_layer(self, i, regularizer=None, **kwargs):
        return GATConv(self.n_hiddens[i], dropout_rate=self.dropout_rate, activation='relu',
                       kernel_regularizer=regularizer, bias_regularizer=regularizer)


class GraphSage(GNN):
    def __init__(self, adj_matrix, n_hiddens=(8, 8, 8), aggregate='mean', **kwargs):
        self.n_hiddens = n_hiddens
        self.aggregate = aggregate
        super().__init__(adj_matrix, len(n_hiddens), **kwargs)

    def build_gnn_layer(self, i, regularizer=None, **kwargs):
        return GraphSageConv(self.n_hiddens[i], activation='relu', aggregate=self.aggregate,
                             kernel_regularizer=regularizer, bias_regularizer=regularizer)


class LightGCN(GNN):
    def __init__(self, adj_matrix, n_layers=3, **kwargs):
        kwargs['final_node'] = 'mean'  # gnn.py:378
        adj_matrix = LightGCNConv.preprocess(adj_matrix)
        super().__init__(adj_matrix, n_layers, **kwargs)

    def build_gnn_layer(self, i, **kwargs):
        return LightGCNConv()


class DGCF(GNN):
    """gnn.py:391-415: final_node forced to 'mean', adjacency replaced by the crosshop operator."""

    def __init__(self, adj_matrix, n_layers=3, **kwargs):
        kwargs['final_node'] = 'mean'
        adj_matrix = DGCFConv.preprocess(adj_matrix)
        super().__init__(adj_matrix, n_layers, **kwargs)

    def build_gnn_layer(self, i, regularizer=None, **kwargs):
        return DGCFConv(regularizer)


class RGCN(GNN):
    """Relational extension (scope row R): `adj_matrix` is what `load_user_item_graph(..., relations=...)` returns
    (data.preprocess.RelationalAdjacency) or a DeviceGraph carrying relation ids (graph.DeviceGraph(..., rel=, n_rel=));
    with one relation - e.g. a plain scipy matrix - it equals GCN."""

    def __init__(self, adj_matrix, n_hiddens=(8, 8, 8), **kwargs):
        graph.refuse_partitioned([adj_matrix], "RGCN")
        if not isinstance(adj_matrix, DeviceGraph):
            adj_matrix = DeviceGraph.from_scipy(adj_matrix, relational=True)   # keeps RelationalAdjacency's edge types
        self.n_hiddens = n_hiddens
        self.n_rel = adj_matrix.n_rel
        super().__init__(adj_matrix, len(n_hiddens), **kwargs)

    def build_gnn_layer(self, i, regularizer=None, **kwargs):
        return RGCNConv(self.n_hiddens[i], self.n_rel, activation='relu', kernel_regularizer=regularizer,
                        bias_regularizer=regularizer)
