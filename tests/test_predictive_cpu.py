"""CPU: the float64 oracle of the Monte-Carlo predictive statistics against torch.distributions on hand-made rows,
the sample-sharded host logic of ``StagModel.predictive`` over gloo (world size 2, the oracle injected in place of the
kernels), and the argument checks that need no device."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import ref_predictive as R

NAN = float("nan")
TD = torch.distributions


def close(a, b, rtol=1e-5, atol=1e-6):
    torch.testing.assert_close(a.to(torch.float64), b.to(torch.float64), rtol=rtol, atol=atol, equal_nan=True)


# rows of class probabilities as a network may emit them (float32, as the kernels read them)
CAT_ROWS = [
    [0.2, 0.3, 0.5],              # normalised
    [2.0, 6.0, 2.0],              # unnormalised
    [1.0, 0.0, 0.0],              # one-hot: q = 1 clamps to 1 - eps, the zeros contribute 0 * log(eps) = 0
    [0.0, 0.0, 0.0],              # sums to zero: NaN, as torch's 0 / 0
    [1.0, 1e-9, 1e-12],           # below eps after the renormalisation: clamped
    [0.25, NAN, 0.25],            # a NaN stays NaN through the clamp
    [5e-8, 5e-8, 5e-8],           # tiny but well-conditioned
]


def test_categorical_entropy_and_log_prob_match_torch_distributions():
    p = torch.tensor(CAT_ROWS, dtype=torch.float32)
    d = TD.Categorical(probs=p, validate_args=False)
    close(R.entropy(p, "categorical"), d.entropy())
    y = torch.tensor([2, 0, 1, 0, 2, 0, 1])
    close(R.log_prob(p, y, "categorical"), d.log_prob(y))
    # a label outside [0, C) gives NaN (torch raises)
    assert torch.isnan(R.log_prob(p[:2], torch.tensor([3, -1]), "categorical")).all()


def test_categorical_single_class():
    p = torch.tensor([[0.3], [1.0], [0.0]], dtype=torch.float32)
    d = TD.Categorical(probs=p, validate_args=False)
    close(R.entropy(p, 0), d.entropy())
    close(R.log_prob(p, torch.zeros(3, dtype=torch.int64), 0), d.log_prob(torch.zeros(3)))
    assert torch.isnan(R.entropy(p, 0)[2])


def test_bernoulli_entropy_and_log_prob_match_torch_distributions():
    eps = torch.finfo(torch.float32).eps
    p = torch.tensor([[0.0, 1.0, 0.5, 1e-9],
                      [1 - 1e-9, eps, 1 - eps, 0.3],
                      [0.7, NAN, 0.1, 0.9]], dtype=torch.float32)
    y = torch.tensor([[0., 1., 1., 0.], [1., 0., 1., 1.], [1., 0., 0., 1.]])
    d = TD.Bernoulli(probs=p, validate_args=False)
    close(R.entropy(p, "bernoulli"), d.entropy().sum(-1))
    close(R.log_prob(p, y, "bernoulli"), d.log_prob(y).sum(-1))
    assert torch.isnan(R.entropy(p, 1)[2]) and not torch.isnan(R.entropy(p, 1)[:2]).any()


@pytest.mark.parametrize("kind", ["categorical", "bernoulli"])
def test_finalize_of_a_stack_matches_torch(kind):
    g = torch.Generator().manual_seed(0)
    S, N, C = 6, 9, 5
    probs = torch.rand((S, N, C), generator=g) ** 3
    probs[:, 0] = torch.tensor([1.0, 0, 0, 0, 0])           # every sample agrees: no mutual information
    y = torch.randint(0, C, (N,), generator=g) if kind == "categorical" else (torch.rand((N, C), generator=g) > 0.5).float()
    fam = TD.Categorical if kind == "categorical" else TD.Bernoulli
    red = (lambda t: t) if kind == "categorical" else (lambda t: t.sum(-1))
    mean, pred, expd, mi, ll = R.predictive(probs, kind, y)
    tmean = probs.mean(0)
    close(mean, tmean)
    close(pred, red(fam(probs=tmean, validate_args=False).entropy()))
    close(expd, red(fam(probs=probs, validate_args=False).entropy()).mean(0))
    close(mi, pred - expd, rtol=0, atol=0)
    close(ll, red(fam(probs=tmean, validate_args=False).log_prob(y)))
    assert abs(float(mi[0])) < 1e-12 and (mi[1:] > -1e-6).all()   # mutual information is non-negative


def test_ops_refuse_cpu_tensors():
    from stag_b200 import ops, StagLibraryError
    with pytest.raises(StagLibraryError):
        ops.mc_accumulate(torch.rand(2, 3, 4), torch.zeros(3, 4, dtype=torch.float64), torch.zeros(3, dtype=torch.float64))
    with pytest.raises(StagLibraryError):
        ops.mc_finalize(torch.zeros(3, 4, dtype=torch.float64), torch.zeros(3, dtype=torch.float64), 2)


def _tiny_model(likelihood=None):
    import stag_b200 as sb
    from stag_b200.zoo import GCN
    layers = torch.nn.ModuleList([sb.layers.StagLayer(GCN(4, 3))])
    return sb.models.StagModel(layers, **({} if likelihood is None else {"likelihood": likelihood}))


def test_predictive_refuses_other_likelihoods_and_bad_counts():
    import stag_b200 as sb

    class Poisson(sb.likelihoods.Likelihood):
        def __init__(self):
            super().__init__(TD.Poisson)

        def condition(self, feat):
            return TD.Poisson(feat)

    g = sb.rand_graph(5, 12)
    with pytest.raises(NotImplementedError):
        _tiny_model(Poisson()).predictive(g, torch.rand(5, 4), 4)
    with pytest.raises(ValueError):
        _tiny_model().predictive(g, torch.rand(5, 4), 0)
    with pytest.raises(ValueError):
        _tiny_model().predictive(g, torch.rand(5, 4), 4, chunk_samples=0)


# ---- sample sharding over gloo ----------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, ret):
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from stag_b200 import parallel as P, models
    try:
        S, N, C = 7, 11, 6
        g = torch.Generator().manual_seed(5)
        probs = torch.rand((S, N, C), generator=g)             # the same global samples on every rank
        labels = {"categorical": torch.randint(0, C, (N,), generator=g),
                  "bernoulli": (torch.rand((N, C), generator=g) > 0.5).float()}
        base, n = P.shard_samples(S, rank, world)
        got = [None] * world
        dist.all_gather_object(got, (base, n))
        assert sorted(i for b, m in got for i in range(b, b + m)) == list(range(S))
        calls = []
        real = dist.all_reduce

        def counting_all_reduce(t, *a, **k):
            calls.append((t.dtype, t.numel()))
            return real(t, *a, **k)

        dist.all_reduce = counting_all_reduce
        for kind, y in labels.items():
            seen = []

            def accumulate(out, acc_sum, acc_ent, kind):
                seen.append(out.shape[0])
                return R.accumulate(out, acc_sum, acc_ent, kind)

            calls.clear()
            chunks = (probs[base + s0: base + min(s0 + 2, n)] for s0 in range(0, n, 2))
            res = models.mc_predictive(chunks, S, kind, y=y, group=dist.group.WORLD, accumulate=accumulate,
                                       finalize=R.finalize)
            # one collective over one flat float64 buffer holding both accumulators
            assert calls == [(torch.float64, N * C + N)], calls
            assert sum(seen) == n and max(seen) <= 2
            one = R.predictive(probs, kind, y)                  # one process, all samples
            for a, b in zip(res[:5], one):
                torch.testing.assert_close(a, b, rtol=1e-12, atol=1e-15, equal_nan=True)
            assert res.n_samples == S
        dist.all_reduce = real
        # a model that runs its samples as sequential passes has no sample_base: it cannot shard
        import stag_b200 as sb
        gr = sb.rand_graph(5, 12)
        try:
            _tiny_model().predictive(gr, torch.rand(5, 4), 4, group=dist.group.WORLD)
            raise AssertionError("sharded predictive of a sequential model did not raise")
        except NotImplementedError:
            pass
        ret[rank] = "ok"
    finally:
        dist.destroy_process_group()


def test_sharded_predictive_world_size_2_gloo():
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(2, _free_port(), ret), nprocs=2, join=True)
    assert dict(ret) == {0: "ok", 1: "ok"}
