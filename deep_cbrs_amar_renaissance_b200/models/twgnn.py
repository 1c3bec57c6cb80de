"""Two-Way GNNs (mirror of /root/reference/src/models/twgnn.py:12-285, scope row (f)-4): one GNN propagates over the
user-property graph [U+P], another over the item-property graph [I+P]; the user rows of the first and the item rows of
the second, stacked, are the input of a third GNN over the user-item graph [U+I], which has no embeddings of its own.
Host wiring only: all three run on the same kernels as the one-step models.
`adj_matrices` = (user-item, item-property, user-property), what load_user_item_graph(type_adjacency='unary-kg',
user_properties=True) puts in `trainset.adj_matrix` (loaders.py:319-322); constructor call as in experiment.py:142-146:
cls(len(users), len(items), trainset.adj_matrix, **config.model)."""
import abc

import torch

from .. import graph
from ..keras_like import L2, Model
from ..layers import DGCFConv, GATConv, GCNConv, GraphSageConv, LightGCNConv
from .gnn import FullInputSequentialGNN, SequentialGNN


class TwoWayGNN(Model, abc.ABC):
    def __init__(self, n_users, n_items, adj_matrices, n_hops, embedding_dim=8, user_item_node="mean",
                 final_node="concatenation", dropout=None, l2_regularizer=None, cache_neighbours=False, **kwargs):
        super().__init__(type(self).__name__.lower())
        regularizer = L2(l2_regularizer) if l2_regularizer is not None else None
        if len(adj_matrices) != 3:
            raise ValueError('Exactly three adjacency matrix are needed!')
        graph.refuse_partitioned(adj_matrices, type(self).__name__)
        adj_ui_matrix, adj_ip_matrix, adj_up_matrix = adj_matrices
        way_one = [self.build_gnn_layer(i, regularizer=regularizer) for i in range(n_hops)]
        self.way_one_gnn_layers = SequentialGNN(adj_up_matrix, way_one, embedding_dim=embedding_dim, final_node=user_item_node,
                                                dropout=dropout, regularizer=regularizer, cache_neighbours=cache_neighbours)
        way_two = [self.build_gnn_layer(i, regularizer=regularizer) for i in range(n_hops)]
        self.way_two_gnn_layers = SequentialGNN(adj_ip_matrix, way_two, embedding_dim=embedding_dim, final_node=user_item_node,
                                                dropout=dropout, regularizer=regularizer, cache_neighbours=cache_neighbours)
        self.n_items = n_items
        self.n_users = n_users
        # widths of the third GNN (twgnn.py:70-77); extension made on a copy, see tsgnn.py
        if hasattr(self, 'n_hiddens'):
            self.n_hiddens = list(self.n_hiddens)
            if n_hops == len(self.n_hiddens):
                if user_item_node == 'concatenation':
                    self.n_hiddens.extend([embedding_dim * (n_hops + 1) for _ in range(n_hops)])
                else:
                    self.n_hiddens.extend([embedding_dim for _ in range(n_hops)])
        step_two = [self.build_gnn_layer(i + n_hops, regularizer=regularizer) for i in range(n_hops)]
        if self.way_one_gnn_layers.out_dim != self.way_two_gnn_layers.out_dim:
            raise ValueError("the two ways produce rows of different widths")
        self.step_two_gnn_layers = FullInputSequentialGNN(adj_ui_matrix, step_two, final_node=final_node, dropout=dropout,
                                                          cache_neighbours=cache_neighbours,
                                                          embedding_dim=self.way_one_gnn_layers.out_dim)
        self.built = True

    @abc.abstractmethod
    def build_gnn_layer(self, i, **kwargs):
        pass

    def build_layers(self):
        self.way_one_gnn_layers.build_layers()
        self.way_two_gnn_layers.build_layers()
        self.step_two_gnn_layers.build_layers()

    @property
    def out_dim(self):
        return self.step_two_gnn_layers.out_dim

    def call(self, inputs, **kwargs):
        users = self.way_one_gnn_layers(None)
        items = self.way_two_gnn_layers(None)
        return self.step_two_gnn_layers(torch.cat([users[:self.n_users], items[:self.n_items]], dim=0))


class TwoWayGCN(TwoWayGNN):
    def __init__(self, n_users, n_items, adj_matrices, n_hiddens=(8, 8, 8), **kwargs):
        self.n_hiddens = list(n_hiddens)
        adj_matrices = [GCNConv.preprocess(m) for m in adj_matrices]
        super().__init__(n_users, n_items, adj_matrices, len(n_hiddens), **kwargs)

    def build_gnn_layer(self, i, regularizer=None, **kwargs):
        return GCNConv(self.n_hiddens[i], activation='relu', kernel_regularizer=regularizer, bias_regularizer=regularizer)


class TwoWayGraphSage(TwoWayGNN):
    def __init__(self, n_users, n_items, adj_matrices, n_hiddens=(8, 8, 8), aggregate='mean', **kwargs):
        self.n_hiddens = list(n_hiddens)
        self.aggregate = aggregate
        super().__init__(n_users, n_items, adj_matrices, len(n_hiddens), **kwargs)

    def build_gnn_layer(self, i, regularizer=None, **kwargs):
        return GraphSageConv(self.n_hiddens[i], activation='relu', aggregate=self.aggregate,
                             kernel_regularizer=regularizer, bias_regularizer=regularizer)


class TwoWayGAT(TwoWayGNN):
    def __init__(self, n_users, n_items, adj_matrix, n_hiddens=(8, 8, 8), dropout_rate=0.0, **kwargs):
        self.n_hiddens = list(n_hiddens)
        self.dropout_rate = dropout_rate
        super().__init__(n_users, n_items, adj_matrix, len(n_hiddens), **kwargs)

    def build_gnn_layer(self, i, regularizer=None, **kwargs):
        return GATConv(self.n_hiddens[i], dropout_rate=self.dropout_rate, activation='relu',
                       kernel_regularizer=regularizer, bias_regularizer=regularizer)


class TwoWayLightGCN(TwoWayGNN):
    def __init__(self, n_users, n_items, adj_matrix, n_layers=3, **kwargs):
        kwargs['final_node'] = 'mean'  # twgnn.py:238 (user_item_node keeps its own default, 'mean')
        adj_matrix = [LightGCNConv.preprocess(m) for m in adj_matrix]
        super().__init__(n_users, n_items, adj_matrix, n_layers, **kwargs)

    def build_gnn_layer(self, i, **kwargs):
        return LightGCNConv()


class TwoWayDGCF(TwoWayGNN):
    def __init__(self, n_users, n_items, adj_matrix, n_layers=3, **kwargs):
        kwargs['final_node'] = 'mean'
        adj_matrix = [DGCFConv.preprocess(m) for m in adj_matrix]
        super().__init__(n_users, n_items, adj_matrix, n_layers, **kwargs)

    def build_gnn_layer(self, i, regularizer=None, **kwargs):
        return DGCFConv(regularizer)
