"""GPU: Monte-Carlo training in bounded memory (StagModel.loss_backward) against loss(n_samples=S).backward() on the zoo
models and vi variants in train mode (dropout 0): gradients and returned values for every chunk size, bitwise for one
chunk; the Philox state and the device-counter mark; two sample shards summing to the single-call gradient; sequential
passes of an amortised posterior against the explicit per-pass loop; BatchNorm running statistics; and peak memory that
does not grow with the number of samples, up to 256 samples at the ogbn-arxiv shape."""
import gc

import pytest
import torch

from test_gpu_predictive import labels, make_graph, make_model

pytestmark = pytest.mark.gpu

S = 12


def make_vi_model(name, D=16, H=32, C=7):
    """Two GCN layers with trainable posteriors (vi=True) and a softmax head."""
    import stag_b200 as sb
    from stag_b200.layers import StagLayer, FeatOnlyLayer
    td = torch.distributions
    z = sb.zoo
    torch.manual_seed(2)
    normal = lambda k: td.Normal(torch.ones(k), torch.full((k,), 0.5))  # noqa: E731
    relu = torch.relu
    second = StagLayer(z.GCN(H, C), q_a=normal(H), vi=True)
    if name == "vi_normal":                                     # per-channel Normal, analytic KL
        first = StagLayer(z.GCN(D, H, activation=relu), q_a=normal(D), vi=True)
    elif name == "vi_uniform":
        first = StagLayer(z.GCN(D, H, activation=relu), q_a=td.Uniform(torch.full((D,), 0.5), torch.full((D,), 1.5)),
                          vi=True)
    elif name == "vi_mixture":                                  # no analytic KL: the fused sample-based fallback
        mix = td.MixtureSameFamily(td.Categorical(torch.ones(2, device="cuda")),
                                   td.Normal(torch.tensor([0.0, 1.0], device="cuda"), torch.tensor([0.3, 0.3], device="cuda")))
        first = StagLayer(z.GCN(D, H, activation=relu), q_a=normal(D), p_a=mix, vi=True)
    elif name == "vi_relu":
        first = StagLayer(z.GCN(D, H, activation=relu), q_a=normal(D), relu=True, vi=True)
    elif name == "bernoulli_norm":                              # Bernoulli noise with in-norm, next to a vi layer
        first = StagLayer(z.GCN(D, H, activation=relu), q_a=td.Bernoulli(torch.full((D,), 0.8)), norm=True)
    elif name == "vi_norm":                                     # vi with in-norm: sequential passes
        first = StagLayer(z.GCN(D, H, activation=relu), q_a=normal(D), norm=True, vi=True)
    layers = [first, second, FeatOnlyLayer(torch.nn.Softmax(-1))]
    return sb.models.StagModel(torch.nn.ModuleList(layers)).cuda().train()


def grads(model):
    return {k: p.grad.clone() for k, p in model.named_parameters() if p.grad is not None}


def zero(model):
    for p in model.parameters():
        p.grad = None


def rel(a, b):
    a, b = a.detach().double(), b.detach().double()
    scale = float(b.abs().max())
    return float((a - b).abs().max()) / scale if scale > 0 else float((a - b).abs().max())


def loss_reference(model, g, x, y, mask, n, seed, kl_scaling=None):
    """Gradients, values and final Philox state of loss(n_samples=n).backward() from `seed`."""
    import stag_b200 as sb
    zero(model)
    sb.manual_seed(seed)
    nll, reg = model.loss_terms(g, x, y, mask=mask, n_samples=n, kl_scaling=kl_scaling)
    (nll + reg).backward()
    reg = reg.detach() if torch.is_tensor(reg) else reg
    return grads(model), (float(nll.detach()), float(reg)), sb.random.get_state()


def chunked(model, g, x, y, mask, n, chunk, seed, kl_scaling=None):
    import stag_b200 as sb
    zero(model)
    sb.manual_seed(seed)
    res = model.loss_backward(g, x, y, mask=mask, n_samples=n, chunk_samples=chunk, kl_scaling=kl_scaling)
    return grads(model), (float(res.nll), float(res.reg)), sb.random.get_state()


ZOO = ["gcn", "sage_mean", "sage_pool", "gin", "gat", "gated_gcn"]
VI = ["vi_normal", "vi_uniform", "vi_mixture", "vi_relu", "bernoulli_norm", "vi_norm"]


@pytest.mark.parametrize("name", ZOO + VI)
def test_chunks_match_loss_backward(name):
    """Every gradient and both returned values of loss_backward(S, chunk) match loss(S).backward() from the same Philox
    state, bit for bit with one chunk.  The dense transform picks its split-K from the row count chunk x N, so smaller
    chunks agree to rounding."""
    g, N = make_graph(1)
    model = make_model(name)[0].train() if name in ZOO else make_vi_model(name)
    assert model._can_batch() == (name not in ("gated_gcn", "vi_norm"))
    x = torch.randn(N, 16, device="cuda")
    y = labels(N, 7, "categorical", seed=9).clamp_(max=6)
    mask = torch.rand(N, device="cuda") < 0.6
    kl = 0.37
    ref, ref_vals, ref_state = loss_reference(model, g, x, y, mask, S, 31, kl)
    assert ref and all(torch.isfinite(t).all() for t in ref.values())
    if name in VI:
        assert ref_vals[1] != 0.0
    for chunk in (None, 5, 1):
        got, vals, state = chunked(model, g, x, y, mask, S, chunk, 31, kl)
        assert state == ref_state, chunk
        assert got.keys() == ref.keys()
        if chunk is None:
            assert vals == ref_vals
            for k in ref:
                assert torch.equal(got[k], ref[k]), k
            continue
        for k in ref:
            assert rel(got[k], ref[k]) <= 1e-5, (chunk, k, rel(got[k], ref[k]))
        for a, b in zip(vals, ref_vals):
            assert abs(a - b) <= 1e-5 * abs(b), (chunk, vals, ref_vals)


@pytest.mark.parametrize("name", ["gcn", "gated_gcn"])
def test_philox_state_and_device_counter_mark(name):
    """The state after loss_backward is the state after loss(S).backward(), and the offsets it reserved (what
    advance_device_counter adds at the end of a captured step) are the same: the rewinds leave the mark alone."""
    import stag_b200 as sb
    g, N = make_graph(4)
    model = make_model(name)[0].train()
    x = torch.randn(N, 16, device="cuda")
    y = labels(N, 7, "categorical", seed=2).clamp_(max=6)
    sb.random.enable_device_counter("cuda")
    try:
        sb.manual_seed(8)
        model.loss(g, x, y, n_samples=S).backward()
        after = sb.random.get_state()
        n_ref = sb.random.advance_device_counter()
        for chunk in (5, 1):
            sb.manual_seed(8)
            model.loss_backward(g, x, y, n_samples=S, chunk_samples=chunk)
            assert sb.random.get_state() == after
            assert sb.random.advance_device_counter() == n_ref > 0
    finally:
        sb.random.disable_device_counter()


def test_two_sample_shards_sum_to_the_single_call_gradient():
    """Samples [0, 6) and [6, 12) drawn through sample_base (the shares of two ranks under parallel.shard_samples), each
    scaled by the global S, sum to the gradient of loss(S).backward()."""
    import stag_b200 as sb
    from stag_b200 import models, parallel
    g, N = make_graph(2)
    model = make_vi_model("vi_mixture")
    x = torch.randn(N, 16, device="cuda")
    y = labels(N, 7, "categorical", seed=3).clamp_(max=6)
    ref, ref_vals, _ = loss_reference(model, g, x, y, None, S, 5)
    total, vals, shards = {}, [0.0, 0.0], []
    for rank in range(2):
        base, n = parallel.shard_samples(S, rank, 2)
        zero(model)
        sb.manual_seed(5)
        res = models.mc_loss_backward(model._loss_chunks(g, x, y, None, base, n, 4, True), S, model.kl_scaling)
        got = grads(model)
        shards.append(got)
        for k, t in got.items():
            total[k] = t if k not in total else total[k] + t
        vals = [vals[0] + float(res.nll), vals[1] + float(res.reg)]
    assert total.keys() == ref.keys()
    for k in ref:
        assert rel(total[k], ref[k]) <= 1e-5, (k, rel(total[k], ref[k]))
        if "base_layer" in k:                                   # the shards really are different samples
            assert not torch.equal(shards[0][k], shards[1][k]), k
    for a, b in zip(vals, ref_vals):
        assert abs(a - b) <= 1e-5 * abs(b)


def test_sequential_amortised_passes_match_the_per_pass_loop():
    """An amortised `re` posterior in layer 2 conditions on the stochastic features of layer 1: its KL depends on the
    pass.  loss_backward(S, chunk_samples=1) backpropagates one pass at a time with that pass's KL, which is the
    reference's per-pass loop; loss_terms takes the KL of the last pass instead."""
    import stag_b200 as sb
    from stag_b200.layers import StagLayer, FeatOnlyLayer
    D, H, C, n = 16, 32, 7, 6
    torch.manual_seed(2)
    normal = lambda k: torch.distributions.Normal(torch.ones(k), torch.full((k,), 0.5))  # noqa: E731
    layers = [StagLayer(sb.zoo.GCN(D, H, activation=torch.relu), q_a=normal(D)),
              StagLayer(sb.zoo.GCN(H, C), q_a=sb.distributions.AmortizedDistribution(H, 1), vi=True),
              FeatOnlyLayer(torch.nn.Softmax(-1))]
    model = sb.models.StagModel(torch.nn.ModuleList(layers), kl_scaling=0.5).cuda().train()
    assert not model._can_batch()
    g, N = make_graph(6)
    x = torch.randn(N, D, device="cuda")
    y = labels(N, C, "categorical", seed=4).clamp_(max=C - 1)
    zero(model)
    sb.manual_seed(12)
    kls = []
    for _ in range(n):
        out = model._forward(g, x)
        nll = model.likelihood.nll_samples(out.unsqueeze(0), y).sum()
        kl = layers[1].kl_divergence()
        kls.append(float(kl))
        (nll / n + kl * (0.5 / n)).backward()
    ref, ref_state = grads(model), sb.random.get_state()
    assert len(set(kls)) == n                                   # the KL does depend on the pass
    got, vals, state = chunked(model, g, x, y, None, n, 1, 12)
    assert state == ref_state and got.keys() == ref.keys()
    for k in ref:
        assert rel(got[k], ref[k]) <= 1e-6, (k, rel(got[k], ref[k]))
    assert abs(vals[1] - 0.5 * sum(kls) / n) <= 1e-6 * abs(vals[1])


def test_batchnorm_running_statistics_end_where_loss_leaves_them():
    import stag_b200 as sb
    from stag_b200.layers import StagLayer, FeatOnlyLayer
    D, H, C = 16, 32, 7
    torch.manual_seed(2)
    normal = lambda k: torch.distributions.Normal(torch.ones(k), torch.full((k,), 0.5))  # noqa: E731
    bn = torch.nn.BatchNorm1d(H)
    # no bias before the BatchNorm: its gradient is zero up to rounding, which no relative bound can compare
    layers = [StagLayer(sb.zoo.GCN(D, H, bias=False), q_a=normal(D), vi=True), FeatOnlyLayer(bn), FeatOnlyLayer(torch.nn.ReLU()),
              StagLayer(sb.zoo.GCN(H, C), q_a=normal(H), vi=True), FeatOnlyLayer(torch.nn.Softmax(-1))]
    model = sb.models.StagModel(torch.nn.ModuleList(layers)).cuda().train()
    assert model._can_batch()
    g, N = make_graph(7)
    x = torch.randn(N, D, device="cuda")
    y = labels(N, C, "categorical", seed=5).clamp_(max=C - 1)
    start = {k: v.clone() for k, v in model.state_dict().items()}
    ref, _, _ = loss_reference(model, g, x, y, None, S, 9)
    stats = [t.clone() for t in (bn.running_mean, bn.running_var, bn.num_batches_tracked)]
    assert int(stats[2]) == S
    for chunk in (5, 1):
        model.load_state_dict(start)
        got, _, _ = chunked(model, g, x, y, None, S, chunk, 9)
        torch.testing.assert_close(bn.running_mean, stats[0], rtol=1e-5, atol=1e-6)
        torch.testing.assert_close(bn.running_var, stats[1], rtol=1e-5, atol=1e-6)
        assert torch.equal(bn.num_batches_tracked, stats[2])
        for k in ref:
            assert rel(got[k], ref[k]) <= 1e-5, (chunk, k)


def _peak(model, g, x, y, n, c):
    torch.cuda.synchronize()
    gc.collect()
    before = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    r = model.loss_backward(g, x, y, n_samples=n, chunk_samples=c)
    del r
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated() - before


@pytest.mark.parametrize("name", ["gcn", "gated_gcn"])
def test_memory_does_not_grow_with_the_number_of_samples(name):
    """loss_backward(16 c, c) peaks no higher than loss_backward(2 c, c): each chunk's graph is freed before the next
    chunk runs.  The warm-up call allocates the gradients."""
    g, N = make_graph(3, N=20000, E=200000)
    C = 40
    model = make_model(name, D=64, H=64, C=C)[0].train()
    x = torch.randn(N, 64, device="cuda")
    y = labels(N, C, "categorical", seed=1).clamp_(max=C - 1)
    c = 4
    _peak(model, g, x, y, c, c)
    two = _peak(model, g, x, y, 2 * c, c)
    many = _peak(model, g, x, y, 16 * c, c)
    assert many <= two + (1 << 20), (two, many)


def test_arxiv_shape_256_samples_in_chunks_of_16():
    """A training step over 256 samples of a 3-layer vi GCN (hidden 256) at the ogbn-arxiv shape: all samples at once
    would hold [256, N, 256] activations (44.4 GB each) until the backward; in chunks of 16 it needs the memory of 16."""
    import bench
    import stag_b200 as sb
    from stag_b200.layers import StagLayer, FeatOnlyLayer
    src, dst = bench.synth_graph()
    N = bench.N_NODES
    g = sb.Graph(torch.from_numpy(src), torch.from_numpy(dst), N).to("cuda")
    normal = lambda k: torch.distributions.Normal(torch.ones(k), torch.full((k,), 0.5))  # noqa: E731
    torch.manual_seed(0)
    layers = [StagLayer(sb.zoo.GCN(128, 256, activation=torch.relu), q_a=normal(128), vi=True),
              StagLayer(sb.zoo.GCN(256, 256, activation=torch.relu), q_a=normal(256), vi=True),
              StagLayer(sb.zoo.GCN(256, 40), q_a=normal(256), vi=True), FeatOnlyLayer(torch.nn.Softmax(-1))]
    model = sb.models.StagModel(torch.nn.ModuleList(layers)).cuda().train()
    x = torch.randn(N, 128, device="cuda")
    y = torch.randint(0, 40, (N,), device="cuda")
    _peak(model, g, x, y, 16, 16)                                # warm-up: gradients and graph structures
    zero(model)
    sixteen = _peak(model, g, x, y, 16, 16)
    zero(model)
    many = _peak(model, g, x, y, 256, 16)
    assert many <= 1.1 * sixteen, (sixteen, many)
    for k, p in model.named_parameters():
        assert p.grad is not None and torch.isfinite(p.grad).all(), k
