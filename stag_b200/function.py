"""DGL-style builtin message / reduce functions, executed by the fused CUDA kernels.

Covers the builtins the reference uses: ``fn.u_mul_e`` / ``fn.copy_src`` (copy_u) /
``fn.copy_edge`` (copy_e) with ``fn.sum`` / ``fn.mean`` (stag/layers.py:12-15;
stag/zoo/gcn.py:59,63,95; stag/zoo/graph_sage.py:53,57,72,86; stag/zoo/gated_gcn.py:30-42),
``fn.max`` / ``fn.min`` (SAGEConv 'pool', GINConv 'max'; ties go to the first edge in edge-id order)
and ``fn.u_add_v`` for ``apply_edges`` (stag/zoo/gat.py:114).
"""
import torch


class Message:
    def __init__(self, kind, a, b, out):
        self.kind, self.a, self.b, self.out = kind, a, b, out

    def edgewise(self, g):
        src, dst = g.edges()
        if self.kind == "u_add_v":
            return g.ndata[self.a][src] + g.ndata[self.b][dst]
        if self.kind == "copy_u":
            return g.ndata[self.a][src]
        if self.kind == "copy_e":
            return g.edata[self.a]
        if self.kind == "u_mul_e":
            u, e = g.ndata[self.a][src], g.edata[self.b]
            while e.dim() < u.dim():
                e = e.unsqueeze(-1)
            return u * e
        raise NotImplementedError(self.kind)


class Reduce:
    def __init__(self, kind, msg, out):
        self.kind, self.msg, self.out = kind, msg, out


def copy_u(u, out):
    return Message("copy_u", u, None, out)


copy_src = copy_u


def copy_e(e, out):
    return Message("copy_e", e, None, out)


copy_edge = copy_e


def u_mul_e(u, e, out):
    return Message("u_mul_e", u, e, out)


def u_add_v(u, v, out):
    return Message("u_add_v", u, v, out)


def sum(msg, out):  # noqa: A001
    return Reduce("sum", msg, out)


def mean(msg, out):
    return Reduce("mean", msg, out)


def max(msg, out):  # noqa: A001
    return Reduce("max", msg, out)


def min(msg, out):  # noqa: A001
    return Reduce("min", msg, out)


def run(g, message, reduce):
    """update_all(message, reduce) on the CUDA kernels."""
    from . import ops
    if reduce.kind not in ("sum", "mean", "max", "min"):
        raise NotImplementedError("reduce %r" % reduce.kind)
    if message.kind == "copy_u":
        x = g.ndata[message.a]
        lead = x.shape[1:]
        out = ops.stochastic_aggregate(g, x.reshape(x.shape[0], -1), None, reduce=reduce.kind)
        return out.reshape((x.shape[0],) + tuple(lead))
    if message.kind == "u_mul_e":
        x, w = g.ndata[message.a], g.edata[message.b]
        lead = x.shape[1:]
        x2 = x.reshape(x.shape[0], -1)
        if w.dim() > 1 and w.numel() == w.shape[0] * x2.shape[1]:
            w2 = w.reshape(w.shape[0], -1)
        elif w.numel() == w.shape[0]:
            w2 = w.reshape(-1, 1)
        else:  # broadcast over trailing dims, e.g. (E,H,1) x (N,H,F)
            w2 = w.expand((w.shape[0],) + tuple(lead)).reshape(w.shape[0], -1)
        out = ops.stochastic_aggregate(g, x2, w2, reduce=reduce.kind)
        return out.reshape((x.shape[0],) + tuple(lead))
    if message.kind == "copy_e":
        w = g.edata[message.a]
        lead = w.shape[1:]
        w2 = w.reshape(w.shape[0], -1)
        ones = torch.ones((g.number_of_nodes(), w2.shape[1]), dtype=torch.float32, device=w.device)
        out = ops.stochastic_aggregate(g, ones, w2, reduce=reduce.kind)
        return out.reshape((g.number_of_nodes(),) + tuple(lead))
    raise NotImplementedError("message %r" % message.kind)
