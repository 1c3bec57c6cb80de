"""BasicRS scorer and the BasicGNN family (mirror of /root/reference/src/models/basic.py:11-120).

`BasicGCN(adj, **config.model)` / `model((u_ids, i_ids)) -> [B,1]` exactly as
experiment.py:150-151,166 calls them.  Unknown keyword arguments are swallowed, as the
reference's constructors do.  The embedding lookup, the concatenation and the first
Dense of every stack run as one kernel (cbrs_dense with row indices)."""
import abc

import numpy as np
import torch

from ..keras_like import Model, default_device
from .dense import build_dense_classifier, build_dense_network
from .gnn import GAT, GCN, DGCF, GNN, RGCN, GraphSage, LightGCN
from .tsgnn import TwoStepDGCF, TwoStepGAT, TwoStepGCN, TwoStepGraphSage, TwoStepLightGCN
from .twgnn import TwoWayDGCF, TwoWayGAT, TwoWayGCN, TwoWayGraphSage, TwoWayLightGCN


def _ids(x):
    """int64 ids (numpy from the Sequence, or tensors) -> CUDA int64 tensor (the per-batch H2D copy)."""
    if isinstance(x, torch.Tensor):
        return x.to(device=default_device(), dtype=torch.int64, non_blocking=True)
    return torch.from_numpy(np.ascontiguousarray(x, dtype=np.int64)).to(default_device(), non_blocking=True)


def _rows(x):
    """float rows (numpy from the Sequence, or tensors) -> CUDA float32 tensor (the per-batch H2D copy)"""
    if isinstance(x, torch.Tensor):
        return x.to(device=default_device(), dtype=torch.float32, non_blocking=True)
    return torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).to(default_device(), non_blocking=True)


class BasicRS(Model):
    def __init__(self, dense_units=(512, 256, 128), clf_units=(64, 64), activation='relu', **kwargs):
        super().__init__("basic_rs")
        self.unet = build_dense_network(dense_units, activation=activation)
        self.inet = build_dense_network(dense_units, activation=activation)
        self.clf = build_dense_classifier(clf_units, n_classes=1, activation=activation)
        self.built = True

    def build_for(self, d):
        du = self.unet.build_for(d)
        di = self.inet.build_for(d)
        self.clf.build_for(du + di)

    def build_from_shapes(self, shapes):
        """the input width from a weight file: the first tower kernel's rows (half the classifier's without towers)"""
        key = "unet/layers.0/kernel" if self.unet.layers else "clf/layers.0/kernel"
        if key in shapes:
            self.build_for(shapes[key][0] if self.unet.layers else shapes[key][0] // 2)

    def call(self, inputs, **kwargs):
        """as a model of its own (config.yaml:6, experiment.py:152): inputs = the (user rows, item rows) batches of
        data.datasets.UserItemEmbeddings"""
        u, i = inputs
        return self.call_sources((_rows(u), None), (_rows(i), None))

    def call_sources(self, u_src, i_src):
        u = self.unet.call_sources([u_src])
        i = self.inet.call_sources([i_src])
        if not self.unet.layers:  # identity towers: keep the gather fused into the classifier
            return self.clf.call_sources([u_src, i_src])
        return self.clf.call_sources([(u, None), (i, None)])


class BasicGNN(Model, abc.ABC):
    def __init__(self, dense_units=(32, 16), clf_units=(16, 16), activation='relu', **kwargs):
        super().__init__(type(self).__name__.lower())
        self.rs = BasicRS(dense_units, clf_units, activation=activation)
        self.cache_propagation = False  # inference-only option: propagate once, score many batches
        self._cached = None
        self.built = True

    def build_weights(self):
        """Create all weights (what the reference's first `model(batch)` does, experiment.py:166)."""
        self.gnn.build_layers()
        self.rs.build_for(self.gnn.out_dim)
        return self

    def propagate(self):
        if self.cache_propagation and self._cached is not None:
            return self._cached
        emb = self.gnn(None)
        if self.cache_propagation:
            self._cached = emb
        return emb

    def invalidate(self):
        self._cached = None

    def set_scorer_precision(self, precision):
        """'bf16': the scorer's Dense layers run on the tensor cores (bf16 operands, fp32 accumulate; inference only,
        tolerance in tests/test_zz_gpu_dense_tc.py); 'fp32' (default): the reference's arithmetic."""
        from ..layers.dense import set_scorer_precision
        set_scorer_precision(self.rs, precision)
        return self

    def call(self, inputs, **kwargs):
        seq = getattr(self.gnn, "gnn_layers", None)
        if not self.cache_propagation and isinstance(self.gnn, GNN) and seq.last_layer_subset():
            # the scorer reads the table at the batch's rows only: the last layer is computed there alone.  The
            # partly filled table never leaves this call (nor stays cached)
            u, i = inputs
            u, i = _ids(u), _ids(i)
            self._cached = None
            emb = seq._run(seq.embeddings, rows=torch.cat([u, i]))
            return self.rs.call_sources((emb, u), (emb, i))
        updated_embeddings = self.propagate()
        return self.embed_recommend(updated_embeddings, inputs)

    def embed_recommend(self, embeddings, inputs):
        u, i = inputs
        return self.rs.call_sources((embeddings, _ids(u)), (embeddings, _ids(i)))

    # -- full-catalog scoring + per-user top-k (new capability, scope row T) ----------------
    def recommend_top_k(self, n_users, n_items, k=10, users=None, user_block=None, fused=True, precision="fp32",
                        exclude=None):
        """Top-k items for every user (or `users`) over the whole catalog.

        Returns (item_index int32 [U,k] in [0, n_items), score float32 [U,k]); ties go to
        the lower item index, which equals "score every pair with the reference scorer,
        stable-sort descending".  exclude: a scoring.ItemLists (e.g. ItemLists.from_ratings of
        the training ratings) whose items are kept out of each user's list; slots past the
        number of eligible items hold -1 / -inf.

        precision (fused=True): 'fp32' (fp32 accuracy, 1e-5) runs the 3xTF32 tensor-core kernel
        (cbrs_score_catalog_topk_tf32x3) for classifier widths c1 in {32, 64}, c2 <= 64, and the
        FFMA kernel otherwise; 'fp32-ffma' always the FFMA kernel; 'bf16' the bf16 tensor-core
        kernel.  fused=False runs the generic blocked pair pipeline."""
        from ..scoring import catalog_top_k
        return catalog_top_k(self, self.propagate(), n_users, n_items, k, users, user_block, fused, precision, exclude)


class BasicTSGNN(BasicGNN):
    pass


class BasicTWGNN(BasicGNN):
    pass


class BasicKnowledgeGCN(BasicGNN):
    pass


def BasicGNNFactory(name, Parent, GNN):
    def __init__(self, *args, **kwargs):
        Parent.__init__(self, **kwargs)
        self.gnn = self.gnn_class(*args, **kwargs)

    return type(name, (Parent,), {"gnn_class": GNN, "__init__": __init__})


BASIC_GNNS = [(BasicGNN, [GCN, GAT, GraphSage, LightGCN, DGCF, RGCN], None),
              (BasicTSGNN, [TwoStepGCN, TwoStepGraphSage, TwoStepGAT, TwoStepLightGCN, TwoStepDGCF],
               lambda name: 'BasicTS' + name[7:]),
              (BasicTWGNN, [TwoWayGCN, TwoWayGraphSage, TwoWayGAT, TwoWayLightGCN, TwoWayDGCF],
               lambda name: 'BasicTW' + name[6:])]


def generate_basics():
    for parent, gnns, name_getter in BASIC_GNNS:
        for gnn in gnns:
            name = name_getter(gnn.__name__) if name_getter is not None else 'Basic' + gnn.__name__
            globals()[name] = BasicGNNFactory(name, parent, gnn)


generate_basics()
