"""Two-Step GNNs (mirror of /root/reference/src/models/tsgnn.py:11-265, scope row (f)-4): a first GNN propagates over
the item-property graph [I+P], its item rows become - next to fresh user embeddings - the input of a second GNN over
the user-item graph [U+I].  Host wiring only: both steps run on the same kernels as the one-step models.
`adj_matrices` = (user-item adjacency, item-property adjacency), what load_user_item_graph(type_adjacency='unary-kg')
puts in `trainset.adj_matrix`; constructor call as in experiment.py:142-146:
cls(len(users), len(items), trainset.adj_matrix, **config.model)."""
import abc

from .. import graph
from ..keras_like import L2, Model
from ..layers import DGCFConv, GATConv, GCNConv, GraphSageConv, LightGCNConv
from .gnn import HalfInputSequentialGNN, SequentialGNN


class TwoStepGNN(Model, abc.ABC):
    def __init__(self, n_users, n_items, adj_matrices, n_hops, embedding_dim=8, item_node="mean",
                 final_node="concatenation", dropout=None, l2_regularizer=None, cache_neighbours=False, **kwargs):
        super().__init__(type(self).__name__.lower())
        regularizer = L2(l2_regularizer) if l2_regularizer is not None else None
        if len(adj_matrices) != 2:
            raise ValueError('Exactly two adjacency matrix are needed!')
        graph.refuse_partitioned(adj_matrices, type(self).__name__)
        adj_ui_matrix, adj_kg_matrix = adj_matrices
        step_one = [self.build_gnn_layer(i, regularizer=regularizer) for i in range(n_hops)]
        self.step_one_gnn_layers = SequentialGNN(adj_kg_matrix, step_one, embedding_dim=embedding_dim, final_node=item_node,
                                                 dropout=dropout, regularizer=regularizer, cache_neighbours=cache_neighbours)
        self.n_embeddings = n_items
        # widths of the second step (tsgnn.py:66-77).  The reference EXTENDS the caller's n_hiddens list in place
        # (config.model.n_hiddens grows from K to 2K entries); here the extension is made on a copy.
        if hasattr(self, 'n_hiddens'):
            self.n_hiddens = list(self.n_hiddens)
            if n_hops == len(self.n_hiddens):
                if item_node == 'concatenation':
                    second_embedding_dim = embedding_dim * (n_hops + 1)
                    self.n_hiddens.extend([second_embedding_dim for _ in range(n_hops)])
                else:
                    self.n_hiddens.extend([embedding_dim for _ in range(n_hops)])
                    second_embedding_dim = embedding_dim
            else:  # the reference leaves second_embedding_dim unbound here and fails with a NameError
                raise ValueError("n_hiddens must list exactly one width per hop of the first step")
        else:
            second_embedding_dim = embedding_dim
        step_two = [self.build_gnn_layer(i + n_hops, regularizer=regularizer) for i in range(n_hops)]
        self.step_two_gnn_layers = HalfInputSequentialGNN(adj_ui_matrix, step_two, n_users, embedding_dim=second_embedding_dim,
                                                          final_node=final_node, dropout=dropout,
                                                          cache_neighbours=cache_neighbours)
        self.built = True

    @abc.abstractmethod
    def build_gnn_layer(self, i, **kwargs):
        pass

    def build_layers(self):
        self.step_one_gnn_layers.build_layers()
        self.step_two_gnn_layers.build_layers()

    @property
    def out_dim(self):
        return self.step_two_gnn_layers.out_dim

    def call(self, inputs, **kwargs):
        x = self.step_one_gnn_layers(None)
        return self.step_two_gnn_layers(x[:self.n_embeddings])


class TwoStepGCN(TwoStepGNN):
    def __init__(self, n_users, n_items, adj_matrices, n_hiddens=(8, 8, 8), **kwargs):
        self.n_hiddens = list(n_hiddens)
        adj_matrices = [GCNConv.preprocess(m) for m in adj_matrices]
        super().__init__(n_users, n_items, adj_matrices, len(n_hiddens), **kwargs)

    def build_gnn_layer(self, i, regularizer=None, **kwargs):
        return GCNConv(self.n_hiddens[i], activation='relu', kernel_regularizer=regularizer, bias_regularizer=regularizer)


class TwoStepGraphSage(TwoStepGNN):
    def __init__(self, n_users, n_items, adj_matrices, n_hiddens=(8, 8, 8), aggregate='mean', **kwargs):
        self.n_hiddens = list(n_hiddens)
        self.aggregate = aggregate
        super().__init__(n_users, n_items, adj_matrices, len(n_hiddens), **kwargs)

    def build_gnn_layer(self, i, regularizer=None, **kwargs):
        return GraphSageConv(self.n_hiddens[i], activation='relu', aggregate=self.aggregate,
                             kernel_regularizer=regularizer, bias_regularizer=regularizer)


class TwoStepGAT(TwoStepGNN):
    def __init__(self, n_users, n_items, adj_matrix, n_hiddens=(8, 8, 8), dropout_rate=0.0, **kwargs):
        self.n_hiddens = list(n_hiddens)
        self.dropout_rate = dropout_rate
        super().__init__(n_users, n_items, adj_matrix, len(n_hiddens), **kwargs)

    def build_gnn_layer(self, i, regularizer=None, **kwargs):
        return GATConv(self.n_hiddens[i], dropout_rate=self.dropout_rate, activation='relu',
                       kernel_regularizer=regularizer, bias_regularizer=regularizer)


class TwoStepLightGCN(TwoStepGNN):
    def __init__(self, n_users, n_items, adj_matrix, n_layers=3, **kwargs):
        kwargs['final_node'] = 'mean'  # tsgnn.py:222 (item_node keeps its own default, 'mean')
        adj_matrix = [LightGCNConv.preprocess(m) for m in adj_matrix]
        super().__init__(n_users, n_items, adj_matrix, n_layers, **kwargs)

    def build_gnn_layer(self, i, **kwargs):
        return LightGCNConv()


class TwoStepDGCF(TwoStepGNN):
    def __init__(self, n_users, n_items, adj_matrix, n_layers=3, **kwargs):
        kwargs['final_node'] = 'mean'
        adj_matrix = [DGCFConv.preprocess(m) for m in adj_matrix]
        super().__init__(n_users, n_items, adj_matrix, n_layers, **kwargs)

    def build_gnn_layer(self, i, regularizer=None, **kwargs):
        return DGCFConv(regularizer)
