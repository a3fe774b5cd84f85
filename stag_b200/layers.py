"""``StagLayer`` and glue layers -- same constructors, forward signatures, attributes and
``state_dict`` keys as the reference's ``stag.layers`` (stag/layers.py:39-178).

What changed underneath: the reference draws an ``[E,K]`` noise tensor with
``q_a.expand([E,K]).rsample()`` (stag/layers.py:115-129), optionally applies relu and
``_in_norm`` (:98-105, :8-36) and hands the tensor to ``base_layer.forward(edge_weight=)``
(:109-113).  Here ``forward`` hands fused-capable base layers (everything in
``stag_b200.zoo``) a lazy :class:`~stag_b200.ops.NoiseSpec` in the same
``edge_weight=`` slot (GAT included: its attention kernel draws the logit noise); the CUDA kernel generates,
transforms, normalises and consumes the noise in one pass and regenerates it in the backward.  Base layers that are not
fused, and the vi+norm combination, receive a real tensor emitted from the same Philox
stream (``stag_noise_emit``), so both routes see identical noise.
"""
import weakref
from typing import Union

import torch

from . import ops
from .distributions import Distribution, ParametrizedDistribution
from .graph import as_graph, sum_nodes, mean_nodes


def _in_norm(graph, edge_weight_sample):
    """Rescale edge weights so that each node's in-edge weights sum to its in-degree
    (stag/layers.py:8-36); nodes whose weights sum to zero keep scale 1."""
    from . import function as fn
    graph = as_graph(graph).local_var()
    graph.edata["h_a"] = edge_weight_sample
    graph.update_all(fn.copy_e("h_a", "m_a"), fn.sum("m_a", "h_a"))
    current_sum = graph.ndata["h_a"]
    desired_sum = graph.in_degrees().unsqueeze(-1)
    node_scaling = torch.where(
        torch.ne(current_sum, 0.0), desired_sum / current_sum, torch.ones_like(current_sum))
    _, dst = graph.edges()
    return edge_weight_sample * node_scaling[dst]


class _GraphRef:
    """Weak reference to the STRUCTURE of the last forward's graph (the local_var view itself dies with the call)."""

    def __init__(self, graph):
        self._ref = weakref.ref(graph._s)

    def __call__(self):
        from .graph import Graph
        s = self._ref()
        return None if s is None else Graph(_structure=s)


class StagLayer(torch.nn.Module):
    """Make a graph-convolution layer stochastic (stag/layers.py:39-145).

    Parameters
    ----------
    base_layer : a ``stag_b200.zoo`` layer (or any module with
        ``forward(graph=, feat=, edge_weight=)``)
    q_a : posterior over the multiplicative edge noise
    p_a : prior (registered as a sub-module as in the reference, so with ``vi=True`` its
        parameters are trainable too)
    norm, relu, vi : as in the reference
    """

    def __init__(
        self,
        base_layer: torch.nn.Module,
        q_a: Union[Distribution, torch.distributions.Distribution] = torch.distributions.Normal(1.0, 1.0),
        p_a: Union[None, Distribution, torch.distributions.Distribution] = torch.distributions.Normal(1.0, 1.0),
        norm: bool = False,
        relu: bool = False,
        vi: bool = False,
    ) -> None:
        super().__init__()
        self.base_layer = base_layer
        if isinstance(q_a, torch.distributions.Distribution):
            q_a = ParametrizedDistribution(q_a, vi=vi)
        if isinstance(p_a, torch.distributions.MixtureSameFamily):
            p_a.base_distribution = p_a
        elif isinstance(p_a, torch.distributions.Distribution):
            p_a = ParametrizedDistribution(p_a, vi=vi)
        elif p_a is None:
            p_a = ParametrizedDistribution(q_a, vi=vi)
        self.add_module("q_a", q_a)
        self.p_a = p_a
        self.norm = norm
        self.relu = relu
        self.vi = vi
        self._noise_spec = None
        self._noise_tensor = None
        self._graph_ref = None

    # transient per-forward state (last graph, lazy noise) is not part of the module: it holds device structure
    # (ctypes structs with pointers) and [E,K] tensors, so it is dropped on pickling / deepcopy
    def __getstate__(self):
        state = dict(self.__dict__)
        state["_noise_spec"] = state["_noise_tensor"] = state["_graph_ref"] = None
        return state

    @property
    def _last_graph(self):
        return None if self._graph_ref is None else self._graph_ref()

    # the sample of the last forward, materialised on demand (stag/layers.py:107)
    @property
    def _edge_weight_sample(self):
        if self._noise_tensor is None and self._noise_spec is not None:
            spec = self._noise_spec
            w = spec.materialize()
            if spec.in_norm:
                g = self._last_graph
                if g is None:
                    raise RuntimeError("the graph of the last forward is gone: _edge_weight_sample with norm=True "
                                       "must be read while that graph is alive")
                w = _in_norm(g, w)
            self._noise_tensor = w
        return self._noise_tensor

    @_edge_weight_sample.setter
    def _edge_weight_sample(self, value):
        self._noise_tensor = value

    def _sample_dimension(self, feat):
        if hasattr(self.base_layer, "sample_dimension"):
            return self.base_layer.sample_dimension
        return feat.shape[-1]

    def noise_spec(self, graph, sample_dimension, n_samples=1, sample_base=0, batched=False):
        """Describe this forward's noise for the fused kernels; None when the posterior is
        not one of Normal / Uniform / Bernoulli."""
        fused = self.q_a.fused_parameters()
        if fused is None:
            return None
        kind, p0, p1 = fused
        if not self.vi:
            p0 = p0.detach()
            p1 = None if p1 is None else p1.detach()
        dev = as_graph(graph).device
        p0 = p0.to(dev)
        p1 = None if p1 is None else p1.to(dev)
        return ops.NoiseSpec(kind, p0, p1, sample_dimension, as_graph(graph).number_of_edges(),
                             relu=self.relu, in_norm=self.norm, n_samples=n_samples,
                             sample_base=sample_base, batched=batched)

    def forward(self, graph, feat, n_samples=None, sample_base=0):
        """Forward pass (stag/layers.py:84-113).  ``n_samples`` / ``sample_base`` are
        extensions used by the sample-batched ``StagModel``: with ``n_samples=S`` the layer
        draws S independent noise samples in one kernel launch and returns ``[S,N,D_out]``."""
        graph = as_graph(graph).local_var()
        self.q_a.condition(graph, feat)
        sample_dimension = self._sample_dimension(feat)
        S = 1 if n_samples is None else int(n_samples)
        spec = self.noise_spec(graph, sample_dimension, n_samples=S, sample_base=sample_base,
                               batched=n_samples is not None)
        self._graph_ref = _GraphRef(graph)
        self._noise_tensor = None
        self._noise_spec = spec

        overridden = "rsample_noise" in self.__dict__ or type(self).rsample_noise is not StagLayer.rsample_noise
        fused_ok = (
            spec is not None
            and not overridden
            and getattr(self.base_layer, "accepts_noise_spec", False)
            and not (self.norm and spec.requires_grad)
            and feat.dim() == (2 if n_samples is None else feat.dim())
        )
        if fused_ok:
            return self.base_layer.forward(graph=graph, feat=feat, edge_weight=spec)
        if n_samples is not None:
            raise NotImplementedError("sample-batched forward needs a fused base layer")
        if overridden:  # the reference's seam for externally supplied noise (stag/layers.py:96)
            edge_weight_sample = self.rsample_noise(graph, sample_dimension)
            self._noise_spec = None
        else:
            edge_weight_sample = self.rsample_noise(graph, sample_dimension, _spec=spec)
        if self.relu:
            edge_weight_sample = edge_weight_sample.relu()
        if self.norm:
            edge_weight_sample = _in_norm(graph, edge_weight_sample)
        self._noise_tensor = edge_weight_sample
        return self.base_layer.forward(graph=graph, feat=feat, edge_weight=edge_weight_sample)

    def rsample_noise(self, graph, sample_dimension, _spec=None):
        """Noise tensor ``[E, sample_dimension]`` (stag/layers.py:115-129): reparameterised when
        ``vi`` is set, a plain sample otherwise.  Drawn from the library's Philox stream for
        Normal / Uniform / Bernoulli, from torch.distributions for anything else."""
        spec = _spec if _spec is not None else self.noise_spec(graph, sample_dimension)
        if spec is not None:
            spec_plain = spec.with_samples(1, spec.sample_base)
            spec_plain.relu = False
            w = spec_plain.materialize()
            return w if self.vi else w.detach()
        dist = self.q_a.expand([as_graph(graph).number_of_edges(), sample_dimension])
        if self.vi:
            return dist.rsample()
        with torch.no_grad():
            return dist.sample()

    def kl_divergence(self):
        """KL(q_a || p_a) averaged over the parameter shape, with the reference's sample-based
        fallback when no analytic KL is registered (stag/layers.py:132-145)."""
        if not self.vi:
            return 0.0
        try:
            return torch.distributions.kl_divergence(
                self.q_a.base_distribution, self.p_a.base_distribution).mean()
        except Exception:
            # no analytic KL (a mixture prior): the reference evaluates both log-probs on the stored [E,K] sample
            # (stag/layers.py:141-143).  When the forward was fused that sample was never stored: stag_noise_kl
            # regenerates it from the forward's (seed, offset) and reduces the two sums on the fly.
            spec = self._noise_spec
            if spec is not None and self._noise_tensor is None and spec.kind in ("normal", "uniform") \
                    and not spec.in_norm and spec.p0.is_cuda and spec.lib_kind != ops._lib.NOISE_NORMAL_HADAMARD:
                prior = ops.describe_prior(self.p_a)
                if prior is not None:
                    return ops.fused_kl_fallback(spec, prior)
            w = self._edge_weight_sample
            return self.q_a.log_prob(w).sum(dim=-1).mean() - self.p_a.log_prob(w).sum(dim=-1).mean()


class FeatOnlyLayer(torch.nn.Module):
    """Apply a plain torch module to the node features (stag/layers.py:147-154)."""
    vi = False

    def __init__(self, layer):
        super().__init__()
        self.layer = layer

    def forward(self, graph, feat):
        return self.layer(feat)


class SumNodes(torch.nn.Module):
    """Per-graph sum readout (stag/layers.py:156-166)."""
    vi = False

    def __init__(self, name="to_sum"):
        super().__init__()
        self.name = name

    def forward(self, graph, feat):
        graph = as_graph(graph).local_var()
        graph.ndata[self.name] = feat
        return sum_nodes(graph, self.name)


class MeanNodes(torch.nn.Module):
    """Per-graph mean readout (stag/layers.py:168-178)."""
    vi = False

    def __init__(self, name="to_mean"):
        super().__init__()
        self.name = name

    def forward(self, graph, feat):
        graph = as_graph(graph).local_var()
        graph.ndata[self.name] = feat
        return mean_nodes(graph, self.name)
