"""``GraphSAGE`` -- constructor and forward of the reference's ``stag.zoo.GraphSAGE``
(stag/zoo/graph_sage.py:7-119, a ``dgl.nn.SAGEConv`` subclass), 'mean', 'gcn' and 'pool'
aggregators on the fused kernels:

* mean (:70-75,107): ``fc_self(h_v) + fc_neigh( sum_e w*h_u / clamp(indeg,1) )``
* gcn  (:76-91):     ``fc_neigh( (sum_e w*h_u + h_v) / (indeg + 1) )``
* pool (SAGEConv):   ``fc_self(h_v) + fc_neigh( max_e w * relu(fc_pool(h_u)) )``  (max aggregation kernels)

'lstm' is a sequential recurrence over the neighbours, not a segmented reduction: rejected.
"""
import torch
from torch import nn

from .. import ops
from ..graph import as_graph


class GraphSAGE(nn.Module):
    accepts_noise_spec = True
    accepts_sample_batch = True   # [S,N,D] features with one sample-batched NoiseSpec (StagModel._can_batch)

    def __init__(self, in_features, out_features, activation=None, aggregator_type="mean"):
        super().__init__()
        if aggregator_type not in ("mean", "gcn", "pool", "lstm"):
            raise KeyError("Aggregator type {} not recognized.".format(aggregator_type))
        if aggregator_type == "lstm":
            raise NotImplementedError(
                "stag_b200.zoo.GraphSAGE: aggregator_type='lstm' is a sequential recurrence over the neighbours, "
                "not a segmented reduction; it has no fused kernel")
        self._in_src_feats = self._in_dst_feats = in_features
        self._out_feats = out_features
        self._aggre_type = aggregator_type
        self.norm = None
        self.feat_drop = nn.Dropout(0.0)
        self.activation = activation
        if aggregator_type == "pool":
            self.fc_pool = nn.Linear(in_features, in_features)
        if aggregator_type != "gcn":
            self.fc_self = nn.Linear(in_features, out_features, bias=False)
        self.fc_neigh = nn.Linear(in_features, out_features, bias=False)
        self.bias = nn.Parameter(torch.zeros(out_features))
        self.reset_parameters()

    def reset_parameters(self):
        gain = nn.init.calculate_gain("relu")
        if self._aggre_type == "pool":
            nn.init.xavier_uniform_(self.fc_pool.weight, gain=gain)
        if self._aggre_type != "gcn":
            nn.init.xavier_uniform_(self.fc_self.weight, gain=gain)
        nn.init.xavier_uniform_(self.fc_neigh.weight, gain=gain)

    def forward(self, graph, feat, edge_weight=None):
        g = as_graph(graph)
        st = g._s
        feat = self.feat_drop(feat)
        n_samples = ops.spec_samples(edge_weight, feat)
        if self._aggre_type == "mean":
            h_neigh = ops.stochastic_aggregate(g, feat, edge_weight, reduce="mean", n_samples=n_samples)
            rst = ops.dense_transform(feat, self.fc_self.weight, transposed=True) + \
                ops.dense_transform(h_neigh, self.fc_neigh.weight, transposed=True)
        elif self._aggre_type == "pool":
            pooled = ops.dense_transform(feat, self.fc_pool.weight, bias=self.fc_pool.bias, relu=True, transposed=True)
            h_neigh = ops.stochastic_aggregate(g, pooled, edge_weight, reduce="max", n_samples=n_samples)
            rst = ops.dense_transform(feat, self.fc_self.weight, transposed=True) + \
                ops.dense_transform(h_neigh, self.fc_neigh.weight, transposed=True)
        else:  # gcn
            neigh = ops.stochastic_aggregate(g, feat, edge_weight, reduce="sum", n_samples=n_samples)
            inv1 = st.scale(True, "inv1").unsqueeze(-1)
            rst = ops.dense_transform((neigh + feat) * inv1, self.fc_neigh.weight, transposed=True)
        if self.bias is not None:
            rst = rst + self.bias
        if self.activation is not None:
            rst = self.activation(rst)
        if self.norm is not None:
            rst = self.norm(rst)
        return rst
