"""float64 restatement of the Monte-Carlo predictive statistics (stag_mc_accumulate / stag_mc_finalize,
csrc/mc_predictive.cu) with the probability semantics of torch.distributions:

* Categorical(probs=p): q = p / sum(p), entropy = -sum_c q_c log(clamp(q_c, eps, 1 - eps)), log_prob(y) = log(clamp(q_y))
* Bernoulli(probs=p):   entropy = -(p log pc + (1 - p) log(1 - pc)), pc = clamp(p, eps, 1 - eps), summed over the labels;
                        log_prob(y) = y log pc + (1 - y) log(1 - pc), summed over the labels

with eps = torch.finfo(float32).eps (the network output is float32).  A NaN stays NaN through the clamp, as in torch;
an out-of-range Categorical label gives NaN (torch raises).  ``accumulate`` / ``finalize`` take the arguments of
``stag_b200.ops.mc_accumulate`` / ``mc_finalize``, so tests can inject them in their place.
"""
import torch

EPS = float(torch.finfo(torch.float32).eps)
KINDS = {"categorical": 0, "bernoulli": 1}


def _clamp(q):
    return q.clamp(EPS, 1.0 - EPS)      # torch.clamp propagates NaN


def entropy(p, kind):
    """Per-row entropy [..., N] of outputs p [..., N, C] (any float dtype; computed in float64)."""
    p = p.to(torch.float64)
    if KINDS.get(kind, kind) == 0:
        q = p / p.sum(-1, keepdim=True)
        return -(q * torch.log(_clamp(q))).sum(-1)
    pc = _clamp(p)
    return -(p * torch.log(pc) + (1.0 - p) * torch.log1p(-pc)).sum(-1)


def log_prob(p, y, kind):
    """Row log-likelihood [N] of labels y under the distribution with parameters p [N, C]."""
    p = p.to(torch.float64)
    if KINDS.get(kind, kind) == 0:
        C = p.shape[-1]
        q = p / p.sum(-1, keepdim=True)
        y = y.to(torch.int64)
        bad = (y < 0) | (y >= C)
        ll = torch.log(_clamp(q.gather(-1, y.clamp(0, C - 1).unsqueeze(-1)).squeeze(-1)))
        return torch.where(bad, torch.full_like(ll, float("nan")), ll)
    pc, yy = _clamp(p), y.to(torch.float64)
    return (yy * torch.log(pc) + (1.0 - yy) * torch.log1p(-pc)).sum(-1)


def accumulate(probs, acc_sum, acc_ent, kind="categorical"):
    """acc_sum [N,C] += p_s and acc_ent [N] += H(p_s) for each sample of probs [S,N,C], in sample order."""
    for p in probs.unbind(0):
        acc_sum += p.to(torch.float64)
        acc_ent += entropy(p, kind)
    return acc_sum, acc_ent


def finalize(acc_sum, acc_ent, n_samples, kind="categorical", y=None):
    """(mean, pred_entropy, exp_entropy, mutual_info, loglik or None) from the accumulators of n_samples samples."""
    mean = acc_sum / float(n_samples)
    pred = entropy(mean, kind)
    expd = acc_ent / float(n_samples)
    ll = None if y is None else log_prob(mean, y, kind)
    return mean, pred, expd, pred - expd, ll


def predictive(probs, kind="categorical", y=None):
    """The statistics of a whole [S,N,C] stack at once."""
    S, N, C = probs.shape
    acc_sum = torch.zeros((N, C), dtype=torch.float64)
    acc_ent = torch.zeros(N, dtype=torch.float64)
    accumulate(probs.cpu(), acc_sum, acc_ent, kind)
    return finalize(acc_sum, acc_ent, S, kind, None if y is None else y.cpu())
