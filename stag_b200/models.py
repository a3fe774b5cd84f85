"""``StagModel`` -- same constructor and method signatures as the reference's
``stag.models`` (stag/models.py:27-89, 92-144).

The reference runs the Monte-Carlo samples as ``n_samples`` sequential passes
(stag/models.py:47-51, :67-68).  With ``batch_samples=True`` (default when every
stochastic layer is fused) the S samples travel through the layers together as
``[S,N,D]`` tensors: one kernel launch per layer draws S independent noise samples
(Philox sample index = s) and, in the first layer, reads the shared input features
once.  Feature-only layers (BatchNorm / Dropout ...) are still applied per sample, in
sample order, so their semantics (batch statistics, running averages) are unchanged.
"""
from typing import List

import torch

from .layers import StagLayer
from .likelihoods import Likelihood, CategoricalLikelihood
from .graph import as_graph


def nll_contrastive(q_a, graph, feat):
    """Contrastive edge objective for amortised posteriors (stag/models.py:7-25)."""
    graph = as_graph(graph)
    n, e = graph.number_of_nodes(), graph.number_of_edges()
    fake_src = torch.randint(high=n, size=[e], device=feat.device)
    fake_dst = torch.randint(high=n, size=[e], device=feat.device)
    h_fake = q_a.embedding_mlp(torch.cat([feat[fake_src], feat[fake_dst]], dim=-1))
    fake = {key: q_a.parameters_mlp[key](h_fake) for key in q_a.new_parameter_names}
    q_a_negative = q_a.base_distribution_class(**{
        key.replace("log_", ""): fake[key].exp() if "log_" in key else fake[key]
        for key in q_a.new_parameter_names})
    nll = -q_a.log_prob(torch.tensor(1.0, device=feat.device)) \
        - q_a_negative.log_prob(torch.tensor(0.0, device=feat.device))
    return nll.sum(dim=-1).mean()


class StagModel(torch.nn.Module):
    def __init__(self, layers: List[StagLayer], likelihood: Likelihood = CategoricalLikelihood(),
                 kl_scaling=1.0, batch_samples=True):
        super().__init__()
        self.layers = layers
        self.likelihood = likelihood
        self.kl_scaling = kl_scaling
        self.batch_samples = batch_samples

    # --- one stochastic pass ------------------------------------------------------------
    def _forward(self, graph, feat):
        graph = as_graph(graph).local_var()
        for layer in self.layers:
            feat = layer(graph, feat)
        return feat

    # --- S passes at once ---------------------------------------------------------------
    def _can_batch(self):
        if not self.batch_samples:
            return False
        for layer in self.layers:
            if isinstance(layer, StagLayer):
                if not getattr(layer.base_layer, "accepts_noise_spec", False):
                    return False
                # a base layer must say that it takes [S,N,D] features with a sample-batched NoiseSpec: GCN, SAGE, GIN and
                # GAT do (GAT's attention kernel draws the logit noise of all S samples in one launch); GatedGCN takes a
                # NoiseSpec but runs its BatchNorm per pass: sequential passes, as the reference
                if not getattr(layer.base_layer, "accepts_sample_batch", False):
                    return False
                # an amortised posterior conditions on the [N,D] features of one pass, not on [S,N,D] ones
                if layer.q_a.__class__.__name__ == "AmortizedDistribution":
                    return False
                if layer.q_a.fused_parameters() is None or (layer.norm and layer.vi):
                    return False
            elif getattr(layer, "vi", False):
                return False
        return True

    def _forward_samples(self, graph, feat, n_samples, sample_base=0):
        """[S, N, C] outputs of S Monte-Carlo passes (sample s uses Philox sample index
        ``sample_base + s``)."""
        batched = self._can_batch() and feat.device.type == "cuda"
        if sample_base != 0 and not batched:
            # sequential passes take a fresh Philox call counter each and always draw sample index 0: ranks sharing a
            # seed would all draw the SAME noise
            raise NotImplementedError("sample_base (Monte-Carlo samples sharded over ranks) needs the sample-batched "
                                      "path: fused base layers on a CUDA device")
        if (n_samples == 1 and sample_base == 0) or not batched:
            return torch.stack([self._forward(graph, feat) for _ in range(n_samples)], dim=0)
        graph = as_graph(graph).local_var()
        h = feat  # [N,D] shared by all samples until the first stochastic layer
        for layer in self.layers:
            if isinstance(layer, StagLayer):
                h = layer(graph, h, n_samples=n_samples, sample_base=sample_base)
            elif h.dim() == feat.dim():
                h = layer(graph, h)  # still sample-independent
            else:
                # unbind, not h[s]: the backward of S selects is S zero-filled [S,N,D] tensors and S adds
                h = torch.stack([layer(graph, hs) for hs in h.unbind(0)], dim=0)
        if h.dim() == feat.dim():
            h = h.unsqueeze(0).expand((n_samples,) + tuple(h.shape))
        return h

    def forward(self, graph, feat, n_samples=1, return_parameters=False, sample_base=0):
        """Monte-Carlo predictive: mean of the outputs of ``n_samples`` stochastic passes,
        then (unless ``return_parameters``) a sample from the likelihood (stag/models.py:45-61).
        ``sample_base`` (extension): global index of this call's first Monte-Carlo sample -- ranks that shard the S
        samples of one predictive pass ``sample_base = parallel.shard_samples(S, rank, world)[0]`` and a common seed."""
        feat = self._forward_samples(graph, feat, n_samples, sample_base=sample_base).mean(dim=0)
        if return_parameters is True:
            return feat
        return self.likelihood.condition(feat).sample()

    def loss_terms(self, graph, feat, y, mask=None, n_samples=1, kl_scaling=None, sample_base=0):
        """(mean NLL, kl_scaling * mean KL) over ``n_samples`` passes (stag/models.py:63-84)."""
        if kl_scaling is None:
            kl_scaling = self.kl_scaling
        outs = self._forward_samples(graph, feat, n_samples, sample_base=sample_base)
        if hasattr(self.likelihood, "nll_samples"):
            # all samples in one fused pass on CUDA (stag_nll), torch.distributions otherwise
            total_nll = self.likelihood.nll_samples(outs, y, mask).sum()
        else:
            total_nll = 0.0
            for out_s in outs.unbind(0):
                nll = -self.likelihood.log_prob(out_s, y)
                if mask is not None:
                    nll = nll[mask]
                total_nll = total_nll + nll.mean()
        reg = 0.0
        for layer in self.layers:
            if layer.vi:
                reg = reg + layer.kl_divergence()
        # the reference re-evaluates the (sample-independent, analytic) KL once per pass and
        # averages: the mean of n identical terms
        total_nll = total_nll / n_samples
        total_reg = reg * kl_scaling
        return total_nll, total_reg

    def loss(self, graph, feat, y, mask=None, n_samples=1, kl_scaling=None, sample_base=0):
        nll, reg = self.loss_terms(graph, feat, y, mask=mask, n_samples=n_samples, kl_scaling=kl_scaling,
                                   sample_base=sample_base)
        return nll + reg


class StagModelContrastive(StagModel):
    """Adds the contrastive edge term of the last amortised layer (stag/models.py:92-144)."""

    def _forward(self, graph, feat):
        graph = as_graph(graph).local_var()
        _nll_contrastive = 0.0
        for layer in self.layers:
            _feat = layer(graph, feat)
            if hasattr(layer, "q_a"):
                _nll_contrastive = nll_contrastive(layer.q_a, graph, feat)
            else:
                _nll_contrastive = 0.0
            feat = _feat
        return feat, _nll_contrastive

    def loss_terms(self, graph, feat, y, mask=None, n_samples=1, kl_scaling=None):
        if kl_scaling is None:
            kl_scaling = self.kl_scaling
        total_nll = 0.0
        total_reg = 0.0
        for _ in range(n_samples):
            _feat, reg = self._forward(graph, feat)
            nll = -self.likelihood.log_prob(_feat, y)
            if mask is not None:
                nll = nll[mask]
            for layer in self.layers:
                if layer.vi:
                    reg = reg + layer.kl_divergence()
            total_nll = total_nll + nll.mean()
            total_reg = total_reg + reg
        return total_nll / n_samples, total_reg / n_samples * kl_scaling

    def forward(self, graph, feat, n_samples=1, return_parameters=False):
        feat = torch.stack([self._forward(graph, feat)[0] for _ in range(n_samples)], dim=0).mean(dim=0)
        if return_parameters is True:
            return feat
        return self.likelihood.condition(feat).sample()
