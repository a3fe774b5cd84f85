"""CPU: the host logic of ``StagModel.loss_backward`` -- the chunk plan and the Philox rewinds of ``_sample_chunks``, the
per-chunk weights of ``models.mc_loss_backward``, chunked gradients against the one-chunk gradient in float64 on a
torch-only stand-in for the model, a gloo world-size-2 run whose summed gradients are the single-process gradient, and the
argument checks that need no device."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

S, N, D = 12, 9, 5
KL = 0.3


def _data(dtype=torch.float64):
    g = torch.Generator().manual_seed(0)
    x = torch.randn((N, D), generator=g, dtype=dtype)
    y = (torch.rand(N, generator=g) > 0.5).to(dtype)
    eps = 1.0 + 0.5 * torch.randn((S, D), generator=g, dtype=dtype)     # the "noise" of sample s
    w = torch.randn(D, generator=g, dtype=dtype).requires_grad_(True)
    b = torch.randn((), generator=g, dtype=dtype).requires_grad_(True)
    return x, y, eps, w, b


def _sample_nll(x, y, e, w, b):
    """[c] NLLs of the samples e [c, D] of a logistic model with multiplicative noise on its weights."""
    p = torch.sigmoid(x @ (w * e).T + b)                                  # [N, c]
    return -(y[:, None] * p.log() + (1 - y[:, None]) * (1 - p).log()).mean(0)


def _reg(w, b, e, sample_based):
    """Analytic: independent of the samples; sample-based: a mean over the chunk's samples, as ops.fused_kl_fallback."""
    if sample_based:
        return (w * e).pow(2).sum(-1).mean() + b * b
    return (w - 1).pow(2).sum() + b * b


def _stand_in_chunks(x, y, eps, w, b, base, n, chunk, sample_based):
    for s0 in range(0, n, chunk):
        e = eps[base + s0: base + min(s0 + chunk, n)]
        yield e.shape[0], _sample_nll(x, y, e, w, b).sum(), _reg(w, b, e, sample_based)


def _full_objective(x, y, eps, w, b, sample_based):
    return _sample_nll(x, y, eps, w, b).mean() + KL * _reg(w, b, eps, sample_based)


def test_chunk_plan_rewinds_the_philox_state_before_every_batched_chunk():
    import stag_b200 as sb
    from stag_b200 import random as R
    model = _tiny_model()
    sb.manual_seed(11)
    R.next_offset()
    entry = R.get_state()
    calls = []

    def run(c, base):
        calls.append((c, base, R.get_state()))
        R.next_offset(), R.next_offset()                                   # a pass of two stochastic layers
        return c

    assert list(model._sample_chunks(3, S, 5, True, run)) == [5, 5, 2]
    assert calls == [(5, 3, entry), (5, 8, entry), (2, 13, entry)]
    assert R.get_state() == (entry[0], entry[1] + 2)                       # where one pass of all samples leaves it
    calls.clear()
    assert list(model._sample_chunks(0, S, 5, False, run)) == [5, 5, 2]
    # sequential passes draw sample index 0 and continue the stream
    assert [(c, base) for c, base, _ in calls] == [(5, 0), (5, 0), (2, 0)]
    assert [st[1] for _, _, st in calls] == [entry[1] + 2, entry[1] + 4, entry[1] + 6]
    assert list(model._sample_chunks(0, 4, 9, True, run)) == [4]


def test_chunk_weights_and_returned_values():
    """Chunk objective nll_c / S + (c / S) kl_scaling reg_c, one backward per chunk; the values returned are the sums."""
    from stag_b200 import models
    p = torch.tensor(2.0, dtype=torch.float64, requires_grad=True)
    nlls, regs, counts = [1.0, 2.5, 4.0], [0.7, 0.9, 1.3], [5, 5, 2]
    seen = []

    def backward(objective):
        seen.append(float(objective.detach()))
        objective.backward()

    chunks = ((c, p * a, p * r) for c, a, r in zip(counts, nlls, regs))
    res = models.mc_loss_backward(chunks, S, KL, backward=backward)
    want = [a / S + c / S * KL * r for c, a, r in zip(counts, nlls, regs)]
    assert seen == pytest.approx([2 * v for v in want], rel=1e-15)
    assert float(p.grad) == pytest.approx(sum(want), rel=1e-15)
    assert isinstance(res, models.LossTerms) and not res.nll.requires_grad and not res.reg.requires_grad
    assert float(res.nll) == pytest.approx(2 * sum(nlls) / S, rel=1e-15)
    assert float(res.reg) == pytest.approx(2 * KL * sum(c / S * r for c, r in zip(counts, regs)), rel=1e-15)
    # a model without vi layers has the Python number 0.0 as its KL
    res = models.mc_loss_backward(iter([(3, p * 1.0, 0.0)]), 3, KL)
    assert float(res.reg) == 0.0 and res.reg.dtype == res.nll.dtype
    with pytest.raises(ValueError):
        models.mc_loss_backward(iter([]), S, KL)


@pytest.mark.parametrize("sample_based", [False, True])
def test_chunked_gradient_equals_the_one_chunk_gradient_in_float64(sample_based):
    from stag_b200 import models
    x, y, eps, w, b = _data()
    # one chunk: the loss_terms expression, bit for bit
    models.mc_loss_backward(_stand_in_chunks(x, y, eps, w, b, 0, S, S, sample_based), S, KL)
    one = (w.grad.clone(), b.grad.clone())
    w.grad = b.grad = None
    nll, reg = _sample_nll(x, y, eps, w, b).sum() / S, _reg(w, b, eps, sample_based) * KL
    (nll + reg).backward()
    assert torch.equal(one[0], w.grad) and torch.equal(one[1], b.grad)
    w.grad = b.grad = None
    _full_objective(x, y, eps, w, b, sample_based).backward()
    torch.testing.assert_close((w.grad, b.grad), one, rtol=1e-12, atol=0)
    for chunk in (1, 5, 7, S + 3):
        w.grad = b.grad = None
        res = models.mc_loss_backward(_stand_in_chunks(x, y, eps, w, b, 0, S, chunk, sample_based), S, KL)
        torch.testing.assert_close((w.grad, b.grad), one, rtol=1e-12, atol=0)
        torch.testing.assert_close(res.nll, nll.detach(), rtol=1e-12, atol=0)
        torch.testing.assert_close(res.reg, reg.detach(), rtol=1e-12, atol=0)


def _tiny_model(cls=None):
    import stag_b200 as sb
    from stag_b200.zoo import GCN
    layers = torch.nn.ModuleList([sb.layers.StagLayer(GCN(4, 3))])
    return (cls or sb.models.StagModel)(layers)


def test_loss_backward_refuses_bad_counts_and_contrastive_models():
    import stag_b200 as sb
    g, x, y = sb.rand_graph(5, 12), torch.rand(5, 4), torch.zeros(5, dtype=torch.int64)
    with pytest.raises(ValueError):
        _tiny_model().loss_backward(g, x, y, n_samples=0)
    with pytest.raises(ValueError):
        _tiny_model().loss_backward(g, x, y, n_samples=4, chunk_samples=0)
    with pytest.raises(NotImplementedError):
        _tiny_model(sb.models.StagModelContrastive).loss_backward(g, x, y, n_samples=4)


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
        calls = []
        real = dist.all_reduce

        def counting_all_reduce(t, *a, **k):
            calls.append(t.numel())
            return real(t, *a, **k)

        for sample_based in (False, True):
            x, y, eps, w, b = _data(torch.float32)                     # the same global samples on every rank
            bucket = P.GradBucket([w, b], group=dist.group.WORLD)
            base, n = P.shard_samples(S, rank, world)
            dist.all_reduce = counting_all_reduce
            calls.clear()
            res = models.mc_loss_backward(_stand_in_chunks(x, y, eps, w, b, base, n, 4, sample_based), S, KL,
                                          group=dist.group.WORLD)
            assert calls == [2], calls                                 # the two values, in one collective
            bucket.allreduce(average=False)
            dist.all_reduce = real
            got = (w.grad.clone(), b.grad.clone())
            w.grad = b.grad = None
            nll, reg = _sample_nll(x, y, eps, w, b).mean(), KL * _reg(w, b, eps, sample_based)
            (nll + reg).backward()                                      # one process, all samples
            torch.testing.assert_close(got, (w.grad, b.grad), rtol=1e-5, atol=1e-7)
            torch.testing.assert_close(res.nll, nll.detach(), rtol=1e-5, atol=0)
            torch.testing.assert_close(res.reg, reg.detach(), rtol=1e-5, atol=0)
        # a model that runs its samples as sequential passes has no sample_base, and fewer samples than ranks cannot
        # be sharded
        import stag_b200 as sb
        g = sb.rand_graph(5, 12)
        try:
            _tiny_model().loss_backward(g, torch.rand(5, 4), torch.zeros(5, dtype=torch.int64), n_samples=4,
                                        group=dist.group.WORLD)
            raise AssertionError("sharded loss_backward of a sequential model did not raise")
        except NotImplementedError:
            pass
        try:
            models._shard("loss_backward", 1, dist.group.WORLD, True)
            raise AssertionError("one sample sharded over two ranks did not raise")
        except ValueError:
            pass
        ret[rank] = "ok"
    finally:
        dist.destroy_process_group()


def test_sharded_loss_backward_world_size_2_gloo():
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(2, _free_port(), ret), nprocs=2, join=True)
    assert dict(ret) == {0: "ok", 1: "ok"}


def test_trainable_uniform_posterior():
    """A vi layer with a Uniform posterior (one of the variants loss_backward is tested on) keeps low / high as trainable
    parameters: Uniform declares its arg_constraints as a property, so they are read from the instance."""
    import stag_b200 as sb
    q = torch.distributions.Uniform(torch.full((4,), 0.5), torch.full((4,), 1.5))
    layer = sb.layers.StagLayer(sb.zoo.GCN(4, 3), q_a=q, vi=True)
    assert sorted(n for n, _ in layer.q_a.named_parameters()) == ["high", "low"]
    assert layer.q_a.fused_parameters()[0] == "uniform"
    layer.kl_divergence().backward()
    assert layer.q_a.low.grad is not None and layer.q_a.high.grad is not None
