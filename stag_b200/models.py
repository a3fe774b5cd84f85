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
from typing import List, NamedTuple, Optional

import torch
import torch.distributed as dist

from . import calibration as _calibration, ops, parallel, random as _random
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


class Predictive(NamedTuple):
    """Monte-Carlo predictive of ``n_samples`` stochastic passes, per node: the mean output (what
    ``forward(..., return_parameters=True)`` returns), the entropy of the predictive distribution (total uncertainty),
    the mean entropy of the per-sample distributions (aleatoric), their difference (mutual information between the
    label and the noise: epistemic) and the log-likelihood of the labels under the mean (None without labels)."""
    mean: torch.Tensor
    entropy: torch.Tensor
    expected_entropy: torch.Tensor
    mutual_information: torch.Tensor
    log_likelihood: Optional[torch.Tensor]
    n_samples: int


def mc_predictive(chunks, n_samples, kind, y=None, group=None, accumulate=None, finalize=None):
    """:class:`Predictive` of ``n_samples`` Monte-Carlo outputs, of which ``chunks`` yields this rank's as ``[s,N,C]``
    tensors in sample order.  Each chunk is added to two float64 accumulators and dropped, so memory does not grow with
    the number of samples.  With ``group`` the accumulators of the ranks are views of one flat buffer, summed by one
    all-reduce before the statistics are taken: every rank returns the statistics of all ``n_samples``.
    ``accumulate`` / ``finalize`` default to the CUDA kernels (:func:`ops.mc_accumulate`, :func:`ops.mc_finalize`)."""
    accumulate = accumulate or ops.mc_accumulate
    finalize = finalize or ops.mc_finalize
    flat = acc_sum = acc_ent = None
    for out in chunks:
        if out.dim() != 3:
            raise ValueError("Monte-Carlo predictive: the model output must be [N, C], got %s per sample"
                             % (tuple(out.shape[1:]),))
        if flat is None:
            N, C = out.shape[1:]
            flat = torch.zeros(N * C + N, dtype=torch.float64, device=out.device)
            acc_sum, acc_ent = flat[: N * C].view(N, C), flat[N * C:]
        accumulate(out, acc_sum, acc_ent, kind)
        del out   # before the next chunk is computed: only one chunk of outputs is alive at a time
    if flat is None:
        raise ValueError("Monte-Carlo predictive: no samples")
    if group is not None and dist.get_world_size(group) > 1:
        dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
    return Predictive(*finalize(acc_sum, acc_ent, n_samples, kind, y), n_samples=int(n_samples))


class LossTerms(NamedTuple):
    """Detached values of the two terms of ``loss_terms``: the mean NLL over the samples and ``kl_scaling`` times the
    KL."""
    nll: torch.Tensor
    reg: torch.Tensor


def mc_loss_backward(chunks, n_samples, kl_scaling, group=None, backward=None):
    """Add to the parameters' ``.grad`` the gradient of the Monte-Carlo objective over ``n_samples`` samples, of which
    ``chunks`` yields this rank's, in sample order, as ``(c, nll_c, reg_c)``: the chunk's sample count, the sum of its
    per-sample NLLs and the sum of the vi layers' KL taken right after its forward.  Each chunk's objective
        ``nll_c / n_samples + (c / n_samples) * kl_scaling * reg_c``
    is backpropagated and dropped before the next chunk is computed, so memory is that of one chunk.  The KL weights sum
    to one over the chunks of all ranks: a sample-independent (analytic) KL counts once, and a sample-based one (the
    fallback of :func:`ops.fused_kl_fallback`, a mean over the chunk's samples) becomes the mean over all samples.
    With one chunk the expression is the one ``loss_terms`` builds, so the gradients are those of ``loss().backward()``
    bit for bit.  Returns the :class:`LossTerms` of all samples; with ``group`` the ranks' values are summed by one
    all-reduce.  ``backward`` (default ``torch.autograd.backward``) is called once per chunk with its objective."""
    backward = backward or torch.autograd.backward
    nll_total = reg_total = None
    for item in chunks:
        c, nll_c, reg_c = item
        del item
        nll = nll_c / n_samples
        reg = reg_c * (kl_scaling * (c / n_samples))
        backward(nll + reg)
        nll = nll.detach()
        reg = (reg.detach() if torch.is_tensor(reg) else torch.tensor(float(reg))).to(nll)
        nll_total = nll if nll_total is None else nll_total + nll
        reg_total = reg if reg_total is None else reg_total + reg
        del nll_c, reg_c, nll, reg   # before the next chunk is computed: the chunk's graph goes with them
    if nll_total is None:
        raise ValueError("Monte-Carlo loss: no samples")
    values = torch.stack([nll_total, reg_total])
    if group is not None and dist.get_world_size(group) > 1:
        dist.all_reduce(values, op=dist.ReduceOp.SUM, group=group)
    return LossTerms(values[0], values[1])


def _shard(what, n_samples, group, batched):
    """(sample_base, n_local) of this rank's share of ``n_samples``; all of them without ``group``."""
    if group is None:
        return 0, n_samples
    if not batched:
        raise NotImplementedError("%s: sharding the samples over ranks needs the sample-batched path (sample_base); this "
                                  "model runs its samples as sequential passes" % what)
    world = dist.get_world_size(group)
    if n_samples < world:
        raise ValueError("%s: %d samples cannot be sharded over %d ranks" % (what, n_samples, world))
    return parallel.shard_samples(n_samples, dist.get_rank(group), world)


def _sample_counts(what, n_samples, chunk_samples):
    n_samples = int(n_samples)
    chunk = n_samples if chunk_samples is None else int(chunk_samples)
    if n_samples < 1 or chunk < 1:
        raise ValueError("%s: n_samples and chunk_samples must be positive" % what)
    return n_samples, chunk


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

    def predictive(self, graph, feat, n_samples, chunk_samples=None, y=None, group=None):
        """Monte-Carlo predictive of ``n_samples`` stochastic passes with per-node uncertainty (:class:`Predictive`),
        in memory that does not grow with ``n_samples``: the samples run ``chunk_samples`` at a time (all at once
        when None) and each chunk's outputs are reduced into float64 accumulators by one kernel and dropped.
        Models that run their samples as sequential passes (GatedGCN, amortised posteriors) accumulate one pass at a
        time.  The samples drawn are those of ``forward(n_samples=n_samples)`` from the same Philox state, whatever the
        chunk size, and the state is left where that call would leave it.  ``y``: labels for the log-likelihood.
        ``group``: a ``torch.distributed`` group whose ranks shard the samples (``parallel.shard_samples``, common
        seed); every rank returns the statistics of all ``n_samples``.  No autograd."""
        kind = getattr(self.likelihood, "fused_kind", None)
        if kind is None:
            raise NotImplementedError("predictive: Categorical and Bernoulli likelihoods only, got %s"
                                      % type(self.likelihood).__name__)
        n_samples, chunk = _sample_counts("predictive", n_samples, chunk_samples)
        batched = self._can_batch() and feat.device.type == "cuda"
        base, n_local = _shard("predictive", n_samples, group, batched)
        # sequential passes accumulate one at a time
        chunks = self._sample_chunks(base, n_local, chunk if batched else 1, batched,
                                     lambda c, b: self._forward_samples(graph, feat, c, sample_base=b))
        with torch.no_grad():
            return mc_predictive(chunks, n_samples, kind, y=y, group=group)

    def calibration(self, probs, y, mask=None, n_bins=15):
        """:class:`stag_b200.calibration.Calibration` of the predictions ``probs [N,C]`` against the labels ``y``
        (``y [N]`` class indices for a Categorical likelihood, ``[N,C]`` label values for a Bernoulli one) over the rows
        where ``mask`` is set, in ``n_bins`` equal-width bins: ECE, reliability diagram, Brier score and accuracy /
        micro-F1, e.g. ``model.calibration(model.predictive(g, x, 256, 32).mean, y, mask=test_mask)``.  The table adds
        over minibatches (``+``) and ranks (``all_reduce``) exactly."""
        kind = getattr(self.likelihood, "fused_kind", None)
        if kind is None:
            raise NotImplementedError("calibration: Categorical and Bernoulli likelihoods only, got %s"
                                      % type(self.likelihood).__name__)
        return _calibration.calibration(probs, y, kind, n_bins=n_bins, mask=mask)

    def _sample_chunks(self, base, n, chunk, batched, run):
        """``run(c, sample_base)`` for consecutive chunks of at most ``chunk`` of this call's ``n`` samples, in sample
        order, from the Philox state at entry."""
        if not batched:
            # sequential passes reserve fresh offsets per pass and always draw sample index 0: the chunks continue the
            # stream as the passes of one call would
            for s0 in range(0, n, chunk):
                yield run(min(chunk, n - s0), 0)
            return
        # a batched pass reserves the same Philox offsets whatever its sample count, and sample s draws with index
        # sample_base + s: every chunk starts from the entry state, and after the last one the state is where one
        # forward(n_samples=n) leaves it
        seed, offset = _random.get_state()
        for s0 in range(0, n, chunk):
            _random._rewind(seed, offset)
            yield run(min(chunk, n - s0), base + s0)

    def _sample_terms(self, graph, feat, y, mask, n_samples, sample_base):
        """(sum of the per-sample NLLs, sum of the vi layers' KL after the forward) of ``n_samples`` passes."""
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
        return total_nll, reg

    def loss_terms(self, graph, feat, y, mask=None, n_samples=1, kl_scaling=None, sample_base=0):
        """(mean NLL, kl_scaling * mean KL) over ``n_samples`` passes (stag/models.py:63-84)."""
        if kl_scaling is None:
            kl_scaling = self.kl_scaling
        total_nll, reg = self._sample_terms(graph, feat, y, mask, n_samples, sample_base)
        # the reference re-evaluates the (sample-independent, analytic) KL once per pass and
        # averages: the mean of n identical terms
        total_nll = total_nll / n_samples
        total_reg = reg * kl_scaling
        return total_nll, total_reg

    def _loss_chunks(self, graph, feat, y, mask, base, n, chunk, batched):
        return self._sample_chunks(base, n, chunk, batched,
                                   lambda c, b: (c,) + self._sample_terms(graph, feat, y, mask, c, b))

    def loss_backward(self, graph, feat, y, mask=None, n_samples=1, chunk_samples=None, kl_scaling=None, group=None):
        """Add to every parameter's ``.grad`` the gradient that ``loss(graph, feat, y, mask, n_samples,
        kl_scaling).backward()`` adds, running the samples ``chunk_samples`` at a time (all at once when None): each
        chunk is backpropagated and freed before the next one runs, so peak memory is that of one chunk whatever
        ``n_samples``.  Returns the detached :class:`LossTerms` ``(nll, reg)`` that ``loss_terms`` returns.

        * The samples are those of ``loss(n_samples=n_samples)`` from the same Philox state, and the state is left
          where that call and its backward leave it (as in :meth:`predictive`).  Chunks agree with the whole batch to
          rounding, not bit for bit (the dense transform picks its split-K from the row count); with one chunk the
          gradients are bitwise those of ``loss().backward()``.
        * Chunk objective: ``nll_c / n_samples + (c / n_samples) * kl_scaling * reg_c`` (:func:`mc_loss_backward`).
        * Feature-only layers see each layer's samples in sample order, so BatchNorm running statistics end where
          ``loss()`` leaves them.  Dropout masks come from torch's RNG, whose draws are ordered by chunk: with dropout
          the gradients agree with those of ``loss()`` in distribution only.
        * Models that run their samples as sequential passes (GatedGCN, amortised posteriors, vi with norm,
          ``batch_samples=False``) run ``chunk_samples`` passes per chunk; ``chunk_samples=1`` holds one pass.  Where
          the KL depends on the pass (an amortised posterior conditioned on stochastic features), each chunk weights
          the KL of its last pass: with ``chunk_samples=1`` that is the per-pass mean the reference's loop takes,
          with one chunk it is the KL of the last pass, as ``loss_terms`` takes it.
        * ``group``: rank r runs ``parallel.shard_samples(n_samples, r, world)`` (common seed) and scales its terms by
          the global ``n_samples``, so the SUM of the ranks' gradients is the full gradient: finish the step with one
          ``parallel.GradBucket.allreduce(average=False)``.  The returned values are summed over the ranks by one
          all-reduce.  Sequential-pass models cannot shard and raise ``NotImplementedError``."""
        n_samples, chunk = _sample_counts("loss_backward", n_samples, chunk_samples)
        if kl_scaling is None:
            kl_scaling = self.kl_scaling
        batched = self._can_batch() and feat.device.type == "cuda"
        base, n_local = _shard("loss_backward", n_samples, group, batched)
        return mc_loss_backward(self._loss_chunks(graph, feat, y, mask, base, n_local, chunk, batched), n_samples,
                                kl_scaling, group=group)

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

    def loss_backward(self, *args, **kwargs):
        raise NotImplementedError("StagModelContrastive.loss_backward: the passes return (output, contrastive term) "
                                  "tuples; use loss().backward()")

    def forward(self, graph, feat, n_samples=1, return_parameters=False):
        feat = torch.stack([self._forward(graph, feat)[0] for _ in range(n_samples)], dim=0).mean(dim=0)
        if return_parameters is True:
            return feat
        return self.likelihood.condition(feat).sample()
