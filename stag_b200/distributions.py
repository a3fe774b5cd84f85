"""nn.Module wrappers around torch.distributions -- same interface as the reference's
``stag.distributions`` (stag/distributions.py:6-243): ``Distribution``,
``DeltaDistribution``, ``ParametrizedDistribution`` (parameters as buffers, or with
``vi=True`` as trainable ``nn.Parameter``s with positive ones stored as ``log_<name>``;
state_dict keys ``loc`` / ``scale`` | ``log_scale`` ...) and ``AmortizedDistribution``
(edge MLP producing per-edge parameters).

New here: :meth:`Distribution.fused_parameters` tells the fused CUDA path which law to
draw from and hands it the parameters in natural units, so the ``[E,K]`` expand +
rsample of stag/layers.py:117-127 never has to be materialised.
"""
from functools import partial
from typing import Callable, Union

import torch
from torch.distributions import constraints

_FUSABLE = {
    torch.distributions.Normal: ("normal", "loc", "scale"),
    torch.distributions.Uniform: ("uniform", "low", "high"),
    torch.distributions.Bernoulli: ("bernoulli", "probs", None),
}


class Distribution(torch.nn.Module):
    """Facade: every query is forwarded to ``self.base_distribution``."""

    def __init__(self):
        super().__init__()

    @property
    def batch_shape(self):
        return self.base_distribution.batch_shape

    @property
    def mean(self):
        return self.base_distribution.mean

    @property
    def stddev(self):
        return self.base_distribution.stddev

    @property
    def variance(self):
        return self.base_distribution.variance

    def expand(self, *args, **kwargs):
        return self.base_distribution.expand(*args, **kwargs)

    def rsample(self, *args, **kwargs):
        return self.base_distribution.rsample(*args, **kwargs)

    def sample(self, *args, **kwargs):
        return self.base_distribution.sample(*args, **kwargs)

    def log_prob(self, *args, **kwargs):
        return self.base_distribution.log_prob(*args, **kwargs)

    def cdf(self, *args, **kwargs):
        return self.base_distribution.cdf(*args, **kwargs)

    def icdf(self, *args, **kwargs):
        return self.base_distribution.icdf(*args, **kwargs)

    def entropy(self, *args, **kwargs):
        return self.base_distribution.entropy(*args, **kwargs)

    def condition(self, *args, **kwargs):
        return self

    def fused_parameters(self):
        """(kind, p0, p1) for Normal / Uniform / Bernoulli, else None (-> emitted-noise path
        is not possible either and the torch sampler is used)."""
        base = self.base_distribution
        spec = _FUSABLE.get(type(base))
        if spec is None:
            return None
        kind, n0, n1 = spec
        return kind, getattr(base, n0), (getattr(base, n1) if n1 else None)


class DeltaDistribution(Distribution):
    """Point mass (stag/distributions.py:50-91)."""

    def __init__(self, value=0.0):
        super().__init__()
        self.register_buffer("value", torch.tensor(value))

    @property
    def batch_shape(self):
        return self.value.shape

    @property
    def mean(self):
        return self.value

    @property
    def stddev(self):
        return torch.zeros_like(self.value)

    @property
    def variance(self):
        return torch.zeros_like(self.value)

    def rsample(self, *args, **kwargs):
        return self.value

    def sample(self, *args, **kwargs):
        return self.value

    def _unsupported(self, *args, **kwargs):
        raise NotImplementedError

    expand = log_prob = cdf = icdf = entropy = _unsupported

    def fused_parameters(self):
        return None


def _as_tensor(value):
    if isinstance(value, torch.Tensor):
        return value.detach().clone()
    return torch.tensor(value)


class ParametrizedDistribution(Distribution):
    """Holds the parameters of a torch distribution as module state
    (stag/distributions.py:93-144)."""

    def __init__(self, base_distribution: torch.distributions.Distribution, vi: bool = False):
        super().__init__()
        cls = base_distribution.__class__
        # read from the instance: some families (Uniform) define arg_constraints as a property
        arg_constraints = base_distribution.arg_constraints
        names = [k for k in arg_constraints.keys() if k != "logits"]
        stored = []
        for name in names:
            value = _as_tensor(getattr(base_distribution, name))
            if vi and arg_constraints[name] == constraints.positive:
                setattr(self, "log_" + name, torch.nn.Parameter(torch.log(value)))
                stored.append("log_" + name)
            elif vi:
                setattr(self, name, torch.nn.Parameter(value))
                stored.append(name)
            else:
                self.register_buffer(name, value)
                stored.append(name)
        self.base_distribution_class = partial(cls, validate_args=False)
        self.new_parameter_names = stored

    def __repr__(self):
        return repr(self.base_distribution)

    @property
    def base_distribution(self):
        kwargs = {}
        for key in self.new_parameter_names:
            value = getattr(self, key)
            if "log_" in key:
                kwargs[key.replace("log_", "")] = value.exp()
            else:
                kwargs[key] = value
        return self.base_distribution_class(**kwargs)


class AmortizedDistribution(Distribution):
    """Per-edge parameters from an MLP on cat(h_src, h_dst)
    (stag/distributions.py:146-242).  The MLP is dense torch; its ``[E,out]`` outputs are
    what the fused kernel consumes as EDGE / EDGE_CHANNEL parameters."""

    def __init__(
        self,
        in_features: int,
        out_features: int,
        hidden_features: Union[None, int] = None,
        activation: Callable = torch.nn.SiLU(),
        base_distribution_class: type = torch.distributions.Normal,
        init_like: Union[None, torch.distributions.Distribution, Distribution] = None,
    ):
        super().__init__()
        if hidden_features is None:
            hidden_features = out_features
        names = []
        for name, cons in base_distribution_class.arg_constraints.items():
            positive = cons == constraints.positive or (
                hasattr(cons, "base_constraint") and cons.base_constraint == constraints.positive)
            names.append("log_" + name if positive else name)
        self.new_parameter_names = names
        self.embedding_mlp = torch.nn.Sequential(
            torch.nn.Linear(2 * in_features, hidden_features),
            activation,
        )
        self.parameters_mlp = torch.nn.ModuleDict(
            {key: torch.nn.Linear(hidden_features, out_features) for key in names})
        self.base_distribution_class = base_distribution_class
        self.out_features = out_features
        if init_like is not None:
            self._init_like(init_like)

    def _init_like(self, init_like):
        if isinstance(init_like, Distribution):
            init_like = init_like.base_distribution
        for key in self.new_parameter_names:
            if "log_" in key:
                target = torch.log(getattr(init_like, key.replace("log_", ""))).mean()
            else:
                target = getattr(init_like, key).mean()
            torch.nn.init.constant_(self.parameters_mlp[key].bias, float(target))

    def condition(self, graph, feat):
        """Per-edge parameters (stag/distributions.py:221-233).  The reference gathers ``cat(h_u, h_v)`` into an
        ``[E, 2 D]`` tensor and runs the first Linear on E rows; here that Linear is split into its source and
        destination halves and applied to the N NODE rows first,
            W1 cat(h_u, h_v) + b1  =  (h W1[:, :D]^T)[u] + (h W1[:, D:]^T + b1)[v],
        so that only ``[E, hidden]`` is ever gathered (hidden = 1 for the ``re`` posteriors of scripts/arxiv_rec:
        two matrix-vector products and scalar work per edge instead of a 1.2 GB concat) and the matrix product
        shrinks by E / N.  Same function, other summation order: parity against the reference's golden vectors
        in tests/test_gpu_layers.py (amortised cases)."""
        from .graph import as_graph
        src, dst = as_graph(graph).edges()
        first = self.embedding_mlp[0]
        D = feat.shape[-1]
        if isinstance(first, torch.nn.Linear) and first.in_features == 2 * D:
            w = first.weight
            pa = torch.nn.functional.linear(feat, w[:, :D])
            pb = torch.nn.functional.linear(feat, w[:, D:], first.bias)
            h = pa.index_select(-2, src) + pb.index_select(-2, dst)
            for layer in list(self.embedding_mlp)[1:]:
                h = layer(h)
        else:  # a user-replaced embedding: the reference's literal form
            h = self.embedding_mlp(torch.cat([feat.index_select(-2, src), feat.index_select(-2, dst)], dim=-1))
        self.new_parameters = {key: self.parameters_mlp[key](h) for key in self.new_parameter_names}
        return self

    @property
    def base_distribution(self):
        kwargs = {}
        for key in self.new_parameter_names:
            value = self.new_parameters[key]
            if "log_" in key:
                kwargs[key.replace("log_", "")] = value.exp()
            else:
                kwargs[key] = value
        return self.base_distribution_class(**kwargs)
