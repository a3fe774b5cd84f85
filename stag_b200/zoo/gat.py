"""``GAT`` -- constructor and forward of the reference's ``stag.zoo.GAT`` (stag/zoo/gat.py:7-149).
The noise ``[E,H]`` multiplies the pre-softmax logits (:117-119).  Attention: the logits
``edge_weight * leaky_relu(el[u] + er[v])`` are computed INSIDE the segmented softmax over the in-edges of each node
(``stag_attention_softmax``, forward and a deterministic backward, csrc/edge_softmax.cu: no ``[E,H]`` logits, no atomics).
With a :class:`~stag_b200.ops.NoiseSpec` in ``edge_weight=`` (``accepts_noise_spec``) the kernel draws the logit noise
itself and runs S Monte-Carlo samples per launch (``accepts_sample_batch``: ``[S,N,D]`` features, or shared ``[N,D]``
ones with a sample-batched spec); in-norm specs go through the materialised noise tensor.
The weighted aggregation ``update_all(u_mul_e('ft','a'), sum)`` (:125-126) runs on ``stag_spmm_fwd`` with the attention as
external weights: all heads in one launch with expanded ``[(S,) E, H*F]`` weights on small (launch-bound) graphs
(<= 4 MB), else ``ops.heads_aggregate`` -- one launch per head over every sample, each head reading / writing its F
columns in place.
"""
import torch
from torch import nn

from .. import ops
from ..graph import as_graph


class GAT(nn.Module):
    accepts_noise_spec = True
    accepts_sample_batch = True

    def __init__(self, in_feats, out_feats, last=False, num_heads=4, feat_drop=0.0, attn_drop=0.0,
                 negative_slope=0.2, residual=False, activation=None, allow_zero_in_degree=False, bias=True):
        super().__init__()
        self._num_heads = num_heads
        self._in_src_feats = self._in_dst_feats = in_feats
        self._out_feats = out_feats
        self._allow_zero_in_degree = allow_zero_in_degree
        self.fc = nn.Linear(in_feats, out_feats * num_heads, bias=False)
        self.attn_l = nn.Parameter(torch.empty(1, num_heads, out_feats))
        self.attn_r = nn.Parameter(torch.empty(1, num_heads, out_feats))
        self.feat_drop = nn.Dropout(feat_drop)
        self.attn_drop = nn.Dropout(attn_drop)
        self.leaky_relu = nn.LeakyReLU(negative_slope)
        if bias:
            self.bias = nn.Parameter(torch.empty(num_heads * out_feats))
        else:
            self.register_buffer("bias", None)
        if residual:
            if in_feats != out_feats * num_heads:
                self.res_fc = nn.Linear(in_feats, num_heads * out_feats, bias=False)
            else:
                self.res_fc = nn.Identity()
        else:
            self.register_buffer("res_fc", None)
        self.activation = activation
        self.last = last
        self.sample_dimension = num_heads
        self.reset_parameters()

    def reset_parameters(self):
        gain = nn.init.calculate_gain("relu")
        nn.init.xavier_uniform_(self.fc.weight, gain=gain)
        nn.init.xavier_uniform_(self.attn_l, gain=gain)
        nn.init.xavier_uniform_(self.attn_r, gain=gain)
        if self.bias is not None:
            nn.init.constant_(self.bias, 0)
        if isinstance(self.res_fc, nn.Linear):
            nn.init.xavier_uniform_(self.res_fc.weight, gain=gain)

    def forward(self, graph, feat, get_attention=False, edge_weight=None):
        g = as_graph(graph)
        H, F = self._num_heads, self._out_feats
        E = g.number_of_edges()
        # S Monte-Carlo samples: [S,N,D] features, or shared [N,D] ones with a sample-batched NoiseSpec
        S = feat.shape[0] if feat.dim() == 3 else ops.spec_samples(edge_weight, feat)
        if S is not None and feat.dim() == 2 and self.training and self.feat_drop.p > 0:
            # one dropout mask per sample, as S sequential passes draw them
            feat = feat.unsqueeze(0).expand((S,) + tuple(feat.shape))
        h = self.feat_drop(feat)
        ft = self.fc(h).view(tuple(h.shape[:-1]) + (H, F))                        # [(S,) N, H, F]
        el = (ft * self.attn_l).sum(dim=-1)
        er = (ft * self.attn_r).sum(dim=-1)
        # attention: softmax over the in-edges of  edge_weight * leaky_relu(el[u] + er[v])  in one fused pass per direction
        # (stag_attention_softmax: the [E,H] logits and their autograd graph never exist; a NoiseSpec is drawn inside)
        a = self.attn_drop(ops.attention_softmax(g, el, er, edge_weight, self.leaky_relu.negative_slope,
                                                 n_samples=S))                    # [(S,) E, H]
        lead = tuple(ft.shape[:-3])                                                # (S,) for per-sample features
        if (1 if S is None else S) * E * H * F * 4 <= (4 << 20):
            # small graphs are launch-bound: ONE fused launch over the H*F channels, the attention of head k expanded to the
            # weight of channels k*F .. (k+1)*F - 1 (external per-channel weights [(S,) E, H*F], at most 4 MB; autograd sums
            # the SDDMM gradient back over the F channels of a head)
            aw = a.unsqueeze(-1).expand(tuple(a.shape) + (F,)).reshape(tuple(a.shape[:-1]) + (H * F,))
            rst = ops.stochastic_aggregate(g, ft.reshape(lead + (ft.shape[-3], H * F)), aw, n_samples=S)
            rst = rst.view(tuple(rst.shape[:-1]) + (H, F))
        else:
            # one launch per head on the per-edge-weight kernel, every head reading / writing its F columns in place (row
            # stride H*F): no [E, H*F] expansion, no per-head copies
            rst = ops.heads_aggregate(g, ft, a)
        if self.res_fc is not None:
            rst = rst + self.res_fc(h).view(tuple(h.shape[:-1]) + (-1, F))
        if self.bias is not None:
            rst = rst + self.bias.view(1, H, F)
        rst = rst.mean(-2) if self.last else rst.flatten(-2, -1)
        if self.activation:
            rst = self.activation(rst)
        if get_attention:
            return rst, a.unsqueeze(-1)
        return rst
