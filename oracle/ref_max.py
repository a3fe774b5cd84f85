"""TEST INFRASTRUCTURE ONLY -- CPU restatement of the max aggregation (DGL's ``update_all(u_mul_e, fn.max)`` as
SAGEConv 'pool' and GINConv 'max' use it), next to the sum restatement of ref_spmm.py.  torch CPU ops only;
autograd on these functions is the gradient oracle.

Tie rule (include/stag_b200.h, stag_spmm_max_fwd): the first edge in edge-id order that reaches the maximum wins and
alone receives the gradient; rows without in-edges are 0 with arg -1.  That is why the gradient here flows through an
explicit gather at ``arg`` and not through ``scatter_reduce('amax')``, which splits the gradient of a tie evenly (as
the DGL shim's fn.max does).
"""
import torch


def u_mul_e_max(src, dst, num_nodes, x, w=None):
    """-> (out [N, ...], arg [N, ...] int64 original edge ids) of max over the in-edges e = (u -> v) of w[e] * x[u]
    (w broadcast over trailing dims, product first, then compare)."""
    m = x[src]
    if w is not None:
        ww = w
        while ww.dim() < m.dim():
            ww = ww.unsqueeze(-1)
        m = m * ww
    E = m.shape[0]
    md = m.detach()
    idx = dst.reshape((-1,) + (1,) * (md.dim() - 1)).expand_as(md)
    mx = torch.full((num_nodes,) + md.shape[1:], float("-inf"), dtype=md.dtype).scatter_reduce(
        0, idx, md, reduce="amax", include_self=True)
    # the first edge reaching the maximum: the smallest edge id among the edges equal to it
    eids = torch.arange(E).reshape((-1,) + (1,) * (md.dim() - 1)).expand_as(md)
    cand = torch.where(md == mx[dst], eids, torch.full_like(eids, E))
    arg = torch.full((num_nodes,) + md.shape[1:], E, dtype=torch.int64).scatter_reduce(
        0, idx, cand, reduce="amin", include_self=True)
    empty = arg == E
    arg = torch.where(empty, torch.full_like(arg, -1), arg)
    if E == 0:
        return torch.zeros_like(mx), arg
    out = torch.gather(m, 0, arg.clamp(min=0))
    return torch.where(empty, torch.zeros_like(out), out), arg


def u_mul_e_min(src, dst, num_nodes, x, w=None):
    """fn.min as -max(-message): ties go to the first minimum."""
    out, arg = u_mul_e_max(src, dst, num_nodes, -x, w)
    return -out, arg


def sage_pool_forward(src, dst, num_nodes, feat, edge_weight, fc_pool_w, fc_pool_b, fc_self_w, fc_neigh_w, bias,
                      activation=None):
    """DGL SAGEConv 'pool' (the reference's GraphSAGE passes aggregator_type through):
    fc_self(h_v) + fc_neigh(max_e w * relu(fc_pool(h_u))) + bias.  Linear weights in torch.nn.Linear layout."""
    pooled = torch.relu(feat @ fc_pool_w.t() + fc_pool_b)
    h_neigh, _ = u_mul_e_max(src, dst, num_nodes, pooled, edge_weight)
    rst = feat @ fc_self_w.t() + h_neigh @ fc_neigh_w.t()
    if bias is not None:
        rst = rst + bias
    if activation is not None:
        rst = activation(rst)
    return rst


def gin_max_forward(src, dst, num_nodes, feat, edge_weight, apply_w, apply_b, eps=0.0):
    """GINConv with aggregator_type='max': apply_func((1 + eps) h_v + max_e w h_u)."""
    neigh, _ = u_mul_e_max(src, dst, num_nodes, feat, edge_weight)
    return ((1 + eps) * feat + neigh) @ apply_w.t() + apply_b
