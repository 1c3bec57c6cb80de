"""HybridCBRS scorer and the HybridBertGNN family (mirror of
/root/reference/src/models/hybrid.py:13-181).

`HybridBertGCN(adj, **config.model)` / `model((u_ids, i_ids, u_bert, i_bert)) -> [B,1]`.
The reference gathers the 768-d content rows on the host per batch
(src/data/datasets.py:65-66) and ships 2 x [B,768] floats over PCIe; that call form is
kept, and `set_content_table` adds the B200 form: the [N,768] table is uploaded once
and the rows are gathered inside the first Dense kernel from the ids alone."""
import abc

from ..keras_like import Model
from ..layers.fusion import FusionLayer
from .basic import _ids, _rows
from .. import ops
from ..layers.dense import materialize
from .dense import build_dense_classifier, build_dense_network, build_residual_dense_network
from .gnn import GAT, GCN, DGCF, RGCN, GraphSage, LightGCN
from .tsgnn import TwoStepDGCF, TwoStepGAT, TwoStepGCN, TwoStepGraphSage, TwoStepLightGCN
from .twgnn import TwoWayDGCF, TwoWayGAT, TwoWayGCN, TwoWayGraphSage, TwoWayLightGCN


class HybridCBRS(Model):
    def __init__(self, feature_based=True, dense_units=((512, 256, 128), (512, 256, 128), (64, 64)),
                 clf_units=(64, 64), activation='relu', fusion_method='concatenate', residual=False, **kwargs):
        super().__init__("hybrid_cbrs")
        self.feature_based = feature_based
        if feature_based:
            self.fuse1a, self.fuse1b, self.fuse2 = FusionLayer('concatenate'), FusionLayer('concatenate'), FusionLayer(fusion_method)
        else:
            self.fuse1a, self.fuse1b, self.fuse2 = FusionLayer(fusion_method), FusionLayer(fusion_method), FusionLayer('concatenate')
        self.dense1a = build_dense_network(dense_units[0], activation=activation)
        self.dense1b = build_dense_network(dense_units[0], activation=activation)
        self.dense2a = build_dense_network(dense_units[1], activation=activation)
        self.dense2b = build_dense_network(dense_units[1], activation=activation)
        self.dense3a = build_dense_network(dense_units[2], activation=activation)
        self.dense3b = build_dense_network(dense_units[2], activation=activation)
        if residual:
            if dense_units[2][-1] != clf_units[-1]:
                raise ValueError("The last dense units before the last fusion layer "
                                 "must be equal to the last classifier units for residual connections")
            self.residual = build_residual_dense_network(clf_units, activation=activation)
            self.activation = activation
            self.clf = build_dense_classifier([], n_classes=1)
        else:
            self.residual = self.activation = None
            self.clf = build_dense_classifier(clf_units, n_classes=1, activation=activation)
        self.built = True

    def build_for(self, d_graph, d_content):
        g = self.dense1a.build_for(d_graph)
        self.dense1b.build_for(d_graph)
        c = self.dense2a.build_for(d_content)
        self.dense2b.build_for(d_content)
        if self.feature_based:
            o1 = self.dense3a.build_for(self.fuse1a.build_for(g, g))
            o2 = self.dense3b.build_for(self.fuse1b.build_for(c, c))
        else:
            o1 = self.dense3a.build_for(self.fuse1a.build_for(g, c))
            o2 = self.dense3b.build_for(self.fuse1b.build_for(g, c))
        x = self.fuse2.build_for(o1, o2)
        if self.residual is not None:
            self.clf.build_for(self.residual.build_for(x))
        else:
            self.clf.build_for(x)

    def build_from_shapes(self, shapes):
        """the graph and content widths from a weight file: the rows of the first graph and content tower kernels"""
        g, c = shapes.get("dense1a/layers.0/kernel"), shapes.get("dense2a/layers.0/kernel")
        if g is not None and c is not None:
            self.build_for(g[0], c[0])

    def call(self, inputs, **kwargs):
        ug, ig, ub, ib = inputs
        return self.call_sources((_rows(ug), None), (_rows(ig), None), (_rows(ub), None), (_rows(ib), None))

    def call_sources(self, ug_src, ig_src, ub_src, ib_src):
        ug = (self.dense1a.call_sources([ug_src]), None)
        ig = (self.dense1b.call_sources([ig_src]), None)
        ub = (self.dense2a.call_sources([ub_src]), None)
        ib = (self.dense2b.call_sources([ib_src]), None)
        return self.tail(ug, ig, ub, ib)

    @staticmethod
    def _fuse(layer, a_src, b_src):
        """FusionLayer on two (matrix, row index) sources -> the source list the next Dense consumes:
        both sources for 'concatenate' (the kernel concatenates on the fly), the fused matrix for 'attention'."""
        if layer.method == 'concatenate':
            return [a_src, b_src]
        return [(layer([materialize([a_src]), materialize([b_src])]), None)]

    def tail(self, ug, ig, ub, ib):
        """Everything after the four per-entity towers (hybrid.py:79-89); arguments are (matrix, row index) sources."""
        if self.feature_based:
            x1 = self.dense3a.call_sources(self._fuse(self.fuse1a, ug, ig))
            x2 = self.dense3b.call_sources(self._fuse(self.fuse1b, ub, ib))
        else:
            x1 = self.dense3a.call_sources(self._fuse(self.fuse1a, ug, ub))
            x2 = self.dense3b.call_sources(self._fuse(self.fuse1b, ig, ib))
        x = self._fuse(self.fuse2, (x1, None), (x2, None))
        if self.residual is None:
            return self.clf.call_sources(x)
        r = self.residual.call_sources(x)
        return self.clf.call_sources([(ops.add3_act(r, x1, x2, self.activation), None)])


class HybridBertGNN(Model, abc.ABC):
    def __init__(self, dense_units=(32, 16), clf_units=(16, 16), feature_based=False, activation='relu',
                 fusion_method='concatenate', residual=False, **kwargs):
        super().__init__(type(self).__name__.lower())
        self.rs = HybridCBRS(feature_based=feature_based, dense_units=dense_units, clf_units=clf_units,
                             activation=activation, fusion_method=fusion_method, residual=residual)
        self.content_table = None
        self.cache_propagation = False
        self._cached = None
        self.built = True

    def build_weights(self, content_dim=768):
        self.gnn.build_layers()
        self.rs.build_for(self.gnn.out_dim, content_dim)
        return self

    def build_from_shapes(self, shapes):
        """the content width from a weight file: the rows of the first content tower kernel"""
        c = shapes.get("rs/dense2a/layers.0/kernel")
        if c is not None:
            self.build_weights(c[0])

    def set_content_table(self, table, dtype="fp32"):
        """Upload the [N, 768] content embeddings once (rows ordered like node ids).  dtype='bf16' keeps the table
        rounded to bf16 (round to nearest even - what the tensor-core scorer does to every row it reads anyway) and
        feeds the towers by TMA (cbrs_dense_tc_bf16); needs set_scorer_precision('bf16')."""
        if dtype not in ("fp32", "bf16"):
            raise ValueError("dtype must be 'fp32' or 'bf16'")
        table = _rows(table).contiguous()
        if dtype == "bf16":
            from .. import ops
            table = ops.to_bf16(table)
        self.content_table = table

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
        updated_embeddings = self.propagate()
        return self.embed_recommend(updated_embeddings, inputs)

    def embed_recommend(self, embeddings, inputs):
        if len(inputs) == 2:
            if self.content_table is None:
                raise ValueError("ids-only call needs set_content_table(...) first")
            u, i = _ids(inputs[0]), _ids(inputs[1])
            return self.rs.call_sources((embeddings, u), (embeddings, i), (self.content_table, u),
                                        (self.content_table, i))
        ug, ig, ub, ib = inputs
        return self.rs.call_sources((embeddings, _ids(ug)), (embeddings, _ids(ig)), (_rows(ub), None),
                                    (_rows(ib), None))

    def recommend_top_k(self, n_users, n_items, k=10, users=None, user_block=None, fused=True, precision="fp32",
                        exclude=None):
        """Top-k items for every user (or `users`) over the whole catalog; returns, ties and `exclude` as
        BasicGNN.recommend_top_k.  Which kernel runs:
          * feature-based scorer with the reference grids' shapes (dense3a / dense3b two 64-wide relu layers,
            classifier 64 -> 64 -> 1, plain concatenation, no residual, content table set, k <= 128):
            precision 'fp32' the chained 3xTF32 tensor-core kernel (cbrs_score_hybrid_topk_tf32x3, fp32 accuracy,
            1e-5), 'bf16' the chained bf16 kernel (cbrs_score_hybrid_topk_bf16), both when k <= n_items;
            'fp32-ffma' and k > n_items the generic pair pipeline;
          * entity-based scorer with plain concatenation: the fused BasicRS kernels, as BasicGNN.recommend_top_k;
          * any other shape, and fused=False: the generic blocked pair pipeline (HybridCBRS.tail over item blocks)."""
        from ..scoring import catalog_top_k
        return catalog_top_k(self, self.propagate(), n_users, n_items, k, users, user_block, fused, precision, exclude)


def BasicGNNFactory(name, Parent, GNN):
    def __init__(self, *args, **kwargs):
        Parent.__init__(self, **kwargs)
        self.gnn = self.gnn_class(*args, **kwargs)

    return type(name, (Parent,), {"gnn_class": GNN, "__init__": __init__})


class HybridBertTSGNN(HybridBertGNN):
    pass


class HybridBertTWGNN(HybridBertGNN):
    pass


HYBRID_GNNS = [(HybridBertGNN, [GCN, GAT, GraphSage, LightGCN, DGCF, RGCN], None),
               (HybridBertTSGNN, [TwoStepGCN, TwoStepGraphSage, TwoStepGAT, TwoStepLightGCN, TwoStepDGCF],
                lambda name: 'HybridBertTS' + name[7:]),
               (HybridBertTWGNN, [TwoWayGCN, TwoWayGraphSage, TwoWayGAT, TwoWayLightGCN, TwoWayDGCF],
                lambda name: 'HybridBertTW' + name[6:])]


def generate_hybrids():
    for parent, gnns, name_getter in HYBRID_GNNS:
        for gnn in gnns:
            name = name_getter(gnn.__name__) if name_getter is not None else 'HybridBert' + gnn.__name__
            globals()[name] = BasicGNNFactory(name, parent, gnn)


generate_hybrids()
