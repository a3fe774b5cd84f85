"""GPU: Monte-Carlo predictive statistics in bounded memory (stag_mc_accumulate / stag_mc_finalize,
StagModel.predictive) against the float64 oracle (oracle/ref_predictive.py): every kernel instantiation with row and
sample strides and NaN rows, bitwise chunk invariance, agreement of every zoo model with forward() from the same Philox
state, sample sharding through sample_base, and memory that does not grow with the number of samples."""
import gc

import numpy as np
import pytest
import torch

from oracle import ref_predictive as R

pytestmark = pytest.mark.gpu

KINDS = ("categorical", "bernoulli")


def close(a, b, rtol=1e-5, atol=1e-6, what=""):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    assert a.shape == b.shape, (what, a.shape, b.shape)
    assert torch.equal(torch.isnan(a), torch.isnan(b)), "%s: NaN pattern" % what
    ok = ~torch.isnan(b)
    err = (a[ok] - b[ok]).abs()
    bound = rtol * b[ok].abs() + atol
    assert bool((err <= bound).all()), "%s: max excess %g" % (what, float((err - bound).max()))


def zeros_acc(N, C):
    return (torch.zeros((N, C), dtype=torch.float64, device="cuda"), torch.zeros(N, dtype=torch.float64, device="cuda"))


def sample_stack(S, N, C, kind, seed, ld=None, ss=None):
    """[S,N,C] view with row stride ld and sample stride ss into a larger buffer; row 1 holds a NaN, row 2 sums to zero
    (Categorical) and row 3 is one-hot (clamp edges)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    ld = ld or C
    ss = ss or N * ld
    buf = torch.rand(S * ss + N * ld + C, device="cuda", generator=g)
    if kind == "categorical":
        buf = buf ** 3                                      # unnormalised, some rows far from uniform
    p = buf.as_strided((S, N, C), (ss, ld, 1))
    if N > 3:
        p[:, 1, C // 2] = float("nan")
        if kind == "categorical":
            p[:, 2] = 0.0
        p[:, 3] = 0.0
        p[:, 3, 0] = 1.0
    return p


def labels(N, C, kind, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    if kind == "categorical":
        y = torch.randint(0, C, (N,), device="cuda", generator=g)
        y[min(4, N - 1)] = C                                  # out of range: NaN
        return y
    return (torch.rand((N, C), device="cuda", generator=g) > 0.5).float()


# every instantiation of mc_accumulate_kernel: C <= 32, 64, 128, 256, 512, 1024
@pytest.mark.parametrize("C", [1, 2, 7, 40, 41, 121, 200, 300, 1024])
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("strided", [False, True])
def test_kernels_match_the_oracle(C, kind, strided):
    from stag_b200 import ops
    S, N = 9, 67
    ld, ss = (C + 5, N * (C + 5) + 13) if strided else (None, None)
    p = sample_stack(S, N, C, kind, seed=C, ld=ld, ss=ss)
    y = labels(N, C, kind, seed=C + 1)
    acc_sum, acc_ent = zeros_acc(N, C)
    ops.mc_accumulate(p, acc_sum, acc_ent, kind)
    r_sum, r_ent = R.accumulate(p.cpu(), *[t.cpu() for t in zeros_acc(N, C)], kind)
    close(acc_sum, r_sum, what="acc_sum")
    close(acc_ent, r_ent, what="acc_ent")
    got = ops.mc_finalize(acc_sum, acc_ent, S, kind, y)
    ref = R.finalize(r_sum, r_ent, S, kind, y.cpu())
    for name, a, b in zip(("mean", "entropy", "expected_entropy", "mutual_information", "log_likelihood"), got, ref):
        close(a, b, what=name)
    assert got[0].dtype == torch.float32 and got[4] is not None
    assert ops.mc_finalize(acc_sum, acc_ent, S, kind)[4] is None


def test_shared_sample_stride_and_unsupported_width():
    """A stride-0 sample dimension (a model whose output does not depend on the noise) reads one row S times; more
    than 1024 classes is refused at the ABI."""
    from stag_b200 import ops, StagError
    N, C, S = 50, 40, 5
    row = torch.rand((N, C), device="cuda")
    acc = zeros_acc(N, C)
    ops.mc_accumulate(row.unsqueeze(0).expand(S, N, C), *acc)
    ref = R.accumulate(row.unsqueeze(0).expand(S, N, C).cpu(), *[t.cpu() for t in zeros_acc(N, C)])
    close(acc[0], ref[0])
    close(acc[1], ref[1])
    mi = ops.mc_finalize(*acc, S)[3]
    assert float(mi.abs().max()) < 1e-6
    with pytest.raises(StagError):
        ops.mc_accumulate(torch.rand((2, 3, 1025), device="cuda"), *zeros_acc(3, 1025))


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("C", [7, 40, 121])
def test_chunked_accumulation_is_bitwise_chunk_invariant(kind, C):
    from stag_b200 import ops
    S, N = 16, 1000
    p = sample_stack(S, N, C, kind, seed=3)
    results = []
    for chunk in (1, 3, 7, S, S):                             # S twice: two runs of the same call
        acc = zeros_acc(N, C)
        for s0 in range(0, S, chunk):
            ops.mc_accumulate(p[s0:s0 + chunk], *acc, kind)
        results.append(acc)
    for acc in results[1:]:
        assert torch.equal(acc[0].nan_to_num(7.0), results[0][0].nan_to_num(7.0))
        assert torch.equal(acc[1].nan_to_num(7.0), results[0][1].nan_to_num(7.0))


# ---- models ---------------------------------------------------------------------------------------------------------
def make_graph(seed, N=300, E=2400):
    import stag_b200 as sb
    rng = np.random.default_rng(seed)
    g = sb.Graph(torch.from_numpy(rng.integers(0, N, E)), torch.from_numpy(rng.integers(0, N, E)), N)
    return sb.add_self_loop(g).to("cuda"), N


def make_model(name, D=16, H=32, C=7):
    import stag_b200 as sb
    from stag_b200.layers import StagLayer, FeatOnlyLayer
    z = sb.zoo
    torch.manual_seed(2)
    normal = lambda k: torch.distributions.Normal(torch.ones(k), torch.full((k,), 0.5))  # noqa: E731
    relu = torch.relu
    lik = sb.likelihoods.CategoricalLikelihood()
    head = FeatOnlyLayer(torch.nn.Softmax(-1))
    if name == "gcn":
        layers = [StagLayer(z.GCN(D, H, activation=relu), q_a=normal(D)), StagLayer(z.GCN(H, C), q_a=normal(H)), head]
    elif name == "gcn_bernoulli":
        layers = [StagLayer(z.GCN(D, H, activation=relu), q_a=normal(D)), StagLayer(z.GCN(H, C), q_a=normal(H)),
                  FeatOnlyLayer(torch.nn.Sigmoid())]
        lik = sb.likelihoods.BernoulliLikelihood()
    elif name in ("sage_mean", "sage_pool"):
        agg = name.split("_")[1]
        layers = [StagLayer(z.GraphSAGE(D, H, activation=relu, aggregator_type=agg), q_a=normal(D)),
                  StagLayer(z.GraphSAGE(H, C, aggregator_type=agg), q_a=normal(H)), head]
    elif name == "gin":
        layers = [StagLayer(z.GIN(D, H), q_a=normal(D)), FeatOnlyLayer(torch.nn.ReLU()),
                  StagLayer(z.GIN(H, C), q_a=normal(H)), head]
    elif name == "gat":
        layers = [StagLayer(z.GAT(D, 8, num_heads=4, activation=torch.nn.functional.elu), q_a=normal(4)),
                  StagLayer(z.GAT(32, C, num_heads=1, last=True, activation=lambda t: torch.softmax(t, -1)),
                            q_a=normal(1))]
    elif name == "gated_gcn":
        # the noise multiplies the D-wide input messages, which are added to A(h): width-preserving, as in the reference
        layers = [StagLayer(z.GatedGCN(D, D), q_a=normal(D)), FeatOnlyLayer(torch.nn.Linear(D, C)), head]
    model = sb.models.StagModel(torch.nn.ModuleList(layers), likelihood=lik).cuda().eval()
    return model, lik.fused_kind


MODELS = ["gcn", "gcn_bernoulli", "sage_mean", "sage_pool", "gin", "gat", "gated_gcn"]


@pytest.mark.parametrize("name", MODELS)
def test_model_predictive_matches_forward_and_the_oracle(name):
    """predictive(S, chunk) draws the samples forward(n_samples=S) draws from the same Philox state and leaves the
    state where that call leaves it.  The dense transform picks its split-K from the row count S_chunk x N, so the
    outputs of a chunk agree with those of the whole batch to rounding, not bit for bit."""
    import stag_b200 as sb
    g, N = make_graph(1)
    model, kind = make_model(name)
    assert model._can_batch() == (name != "gated_gcn")
    x = torch.randn(N, 16, device="cuda")
    C = 7
    y = labels(N, C, kind, seed=9)
    S = 12
    with torch.no_grad():
        sb.manual_seed(31)
        ref_mean = model(g, x, n_samples=S, return_parameters=True)
        after_forward = sb.random.get_state()
        sb.manual_seed(31)
        outs = model._forward_samples(g, x, S)
    ref = R.predictive(outs, kind, y)
    for chunk in (None, 5, 1):
        sb.manual_seed(31)
        pr = model.predictive(g, x, S, chunk_samples=chunk, y=y)
        assert sb.random.get_state() == after_forward
        assert pr.n_samples == S and not pr.mean.requires_grad
        close(pr.mean, ref_mean, rtol=1e-6, atol=1e-7, what="mean chunk=%s" % chunk)
        for field, b in zip(("entropy", "expected_entropy", "mutual_information", "log_likelihood"), ref[1:]):
            close(getattr(pr, field), b, rtol=1e-5, atol=2e-6, what="%s chunk=%s" % (field, chunk))


def test_sharded_accumulators_sum_to_the_single_call():
    """Samples [0, S/2) and [S/2, S) drawn through sample_base (what two ranks of parallel.shard_samples draw) and
    accumulated apart, then summed, equal the accumulators of the same samples in one call."""
    import stag_b200 as sb
    from stag_b200 import ops
    g, N = make_graph(2)
    model, kind = make_model("gcn")
    x = torch.randn(N, 16, device="cuda")
    S = 8
    with torch.no_grad():
        sb.manual_seed(5)
        lo = model._forward_samples(g, x, S // 2, sample_base=0)
        sb.manual_seed(5)
        hi = model._forward_samples(g, x, S // 2, sample_base=S // 2)
    a, b, one = zeros_acc(N, 7), zeros_acc(N, 7), zeros_acc(N, 7)
    ops.mc_accumulate(lo, *a)
    ops.mc_accumulate(hi, *b)
    ops.mc_accumulate(torch.cat([lo, hi]), *one)
    for u, v, w in zip(a, b, one):
        close(u + v, w, rtol=1e-12, atol=0)
    # the halves really are different samples
    assert not torch.equal(lo, hi)


def _peak(model, g, x, n, c):
    torch.cuda.synchronize()
    gc.collect()
    before = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    r = model.predictive(g, x, n, chunk_samples=c)
    del r
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated() - before


@pytest.mark.parametrize("name", ["gcn", "gated_gcn"])
def test_memory_does_not_grow_with_the_number_of_samples(name):
    """predictive(16 c, c) peaks no higher than predictive(2 c, c): every chunk after the first runs beside the same
    accumulators.  predictive(c, c) allocates its accumulators (8 (N C + N) bytes) only once its one chunk has run, so
    against it the bound carries those bytes."""
    g, N = make_graph(3, N=20000, E=200000)
    C = 40
    model, _ = make_model(name, D=64, H=64, C=C)
    x = torch.randn(N, 64, device="cuda")
    c = 4
    _peak(model, g, x, c, c)                                   # warm-up: structures built on first use
    one = _peak(model, g, x, c, c)
    two = _peak(model, g, x, 2 * c, c)
    many = _peak(model, g, x, 16 * c, c)
    assert many <= two + (1 << 20), (two, many)
    assert many <= one + 8 * (N * C + N) + (1 << 20), (one, many)


def test_arxiv_shape_1024_samples_in_chunks_of_32():
    """1024 samples of a 3-layer GCN (hidden 256) at the ogbn-arxiv shape: all samples at once would need [1024, N,
    256] activations (177 GB each); in chunks of 32 the call holds one chunk and the accumulators."""
    import bench
    import stag_b200 as sb
    from stag_b200.layers import StagLayer, FeatOnlyLayer
    src, dst = bench.synth_graph()
    N = bench.N_NODES
    g = sb.Graph(torch.from_numpy(src), torch.from_numpy(dst), N).to("cuda")
    normal = lambda k: torch.distributions.Normal(torch.ones(k), torch.full((k,), 0.5))  # noqa: E731
    torch.manual_seed(0)
    layers = [StagLayer(sb.zoo.GCN(128, 256, activation=torch.relu), q_a=normal(128)),
              StagLayer(sb.zoo.GCN(256, 256, activation=torch.relu), q_a=normal(256)),
              StagLayer(sb.zoo.GCN(256, 40), q_a=normal(256)), FeatOnlyLayer(torch.nn.Softmax(-1))]
    model = sb.models.StagModel(torch.nn.ModuleList(layers)).cuda().eval()
    x = torch.randn(N, 128, device="cuda")
    pr = model.predictive(g, x, 1024, chunk_samples=32)
    torch.cuda.synchronize()
    assert pr.mean.shape == (N, 40) and pr.n_samples == 1024
    assert torch.isfinite(pr.entropy).all() and float(pr.mutual_information.min()) > -1e-5
    close(pr.mean.sum(-1), torch.ones(N), rtol=0, atol=1e-5, what="mean rows sum to one")
