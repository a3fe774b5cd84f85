"""``GIN`` -- the reference's ``stag.zoo.GIN`` (stag/zoo/gin.py:1-11): ``dgl.nn.GINConv``
with a Linear ``apply_func``; ``rst = apply_func((1 + eps) * h_v + agg_e w * h_u)``, agg = sum, mean or max."""
import torch
from torch import nn

from .. import ops
from ..graph import as_graph


class GIN(nn.Module):
    accepts_noise_spec = True
    accepts_sample_batch = True   # [S,N,D] features with one sample-batched NoiseSpec (StagModel._can_batch)

    def __init__(self, in_features, out_features, aggregator_type="sum", init_eps=0, learn_eps=False,
                 activation=None):
        super().__init__()
        if aggregator_type not in ("sum", "mean", "max"):
            raise NotImplementedError("stag_b200.zoo.GIN: aggregator_type=%r" % aggregator_type)
        self.apply_func = nn.Linear(in_features, out_features)
        self._aggregator_type = aggregator_type
        self.activation = activation
        if learn_eps:
            self.eps = nn.Parameter(torch.FloatTensor([init_eps]))
        else:
            self.register_buffer("eps", torch.FloatTensor([init_eps]))

    def forward(self, graph, feat, edge_weight=None):
        g = as_graph(graph)
        n_samples = ops.spec_samples(edge_weight, feat)
        neigh = ops.stochastic_aggregate(g, feat, edge_weight, reduce=self._aggregator_type,
                                         n_samples=n_samples)
        rst = (1 + self.eps) * feat + neigh
        rst = self.apply_func(rst)
        if self.activation is not None:
            rst = self.activation(rst)
        return rst
