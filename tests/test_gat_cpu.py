"""CPU: host-side decisions of the stochastic GAT path (no device needed): which models batch their Monte-Carlo samples,
which noise specs the attention kernel draws itself and which go through the materialised tensor, and the shape checks
of the attention and per-head aggregation operators."""
import pytest
import torch


def gat_model(amortized=False):
    import stag_b200 as sb
    q = sb.distributions.AmortizedDistribution(16, 4) if amortized else torch.distributions.Normal(torch.ones(4), torch.ones(4))
    layers = torch.nn.ModuleList([
        sb.layers.StagLayer(sb.zoo.GAT(16, 8, num_heads=4), q_a=q),
        sb.layers.StagLayer(sb.zoo.GAT(32, 3, num_heads=1, last=True)),
    ])
    return sb.models.StagModel(layers)


def test_gat_takes_noise_specs_and_sample_batches():
    import stag_b200 as sb
    assert sb.zoo.GAT.accepts_noise_spec and sb.zoo.GAT.accepts_sample_batch
    assert gat_model()._can_batch() is True


def test_amortised_gat_runs_sequential_passes():
    assert gat_model(amortized=True)._can_batch() is False


def test_vi_with_norm_is_not_batched():
    import stag_b200 as sb
    layers = torch.nn.ModuleList([sb.layers.StagLayer(sb.zoo.GAT(8, 4, num_heads=2), norm=True, vi=True)])
    assert sb.models.StagModel(layers)._can_batch() is False


def spec(**kw):
    from stag_b200.ops import NoiseSpec
    args = dict(kind="normal", p0=torch.ones(()), p1=torch.ones(()), K=4, num_edges=10, seed=1, offset=1)
    args.update(kw)
    return NoiseSpec(**args)


def test_routes_of_noise_specs():
    from stag_b200.ops import attention_route
    assert attention_route(spec()) == "fused"
    assert attention_route(spec(kind="uniform", p1=torch.full((), 2.0), relu=True)) == "fused"
    assert attention_route(spec(kind="bernoulli", p0=torch.full((), 0.5), p1=None)) == "fused"
    assert attention_route(spec(p0=torch.ones(10, 4), p1=torch.ones(10, 4))) == "fused"      # amortised [E,H]
    assert attention_route(spec(in_norm=True)) == "materialized"
    # 128 heads: the tensor-core generator's 128-channel groups
    assert attention_route(spec(K=128, generator="hadamard")) == "materialized"
    assert attention_route(spec(K=128, generator="boxmuller")) == "fused"


def test_attention_operator_validates_shapes():
    import stag_b200 as sb
    g = sb.Graph(torch.tensor([0, 1, 2]), torch.tensor([1, 2, 0]), 3)
    el, er = torch.zeros(3, 4), torch.zeros(3, 4)
    with pytest.raises(ValueError, match="el"):
        sb.ops.attention_softmax(g, el[:, :3], er, None)
    with pytest.raises(ValueError, match="rows"):
        sb.ops.attention_softmax(g, torch.zeros(4, 4), er, None)
    with pytest.raises(ValueError, match="K=2"):
        sb.ops.attention_softmax(g, el, er, spec(K=2, num_edges=3))
    with pytest.raises(ValueError, match="edges"):
        sb.ops.attention_softmax(g, el, er, spec(num_edges=5))
    with pytest.raises(ValueError, match="samples"):
        sb.ops.attention_softmax(g, torch.zeros(2, 3, 4), torch.zeros(3, 3, 4), None)
    with pytest.raises(ValueError, match="samples"):
        sb.ops.attention_softmax(g, torch.zeros(2, 3, 4), er, None, n_samples=3)


def test_heads_aggregate_validates_shapes():
    import stag_b200 as sb
    g = sb.Graph(torch.tensor([0, 1, 2]), torch.tensor([1, 2, 0]), 3)
    with pytest.raises(ValueError):
        sb.ops.heads_aggregate(g, torch.zeros(3, 4, 2), torch.zeros(3, 3))          # heads disagree
    with pytest.raises(ValueError):
        sb.ops.heads_aggregate(g, torch.zeros(2, 3, 4, 2), torch.zeros(3, 4))       # per-sample features, one attention
    with pytest.raises(ValueError):
        sb.ops.heads_aggregate(g, torch.zeros(2, 3, 4, 2), torch.zeros(3, 3, 4))    # sample counts disagree
    with pytest.raises(ValueError):
        sb.ops.heads_aggregate(g, torch.zeros(3, 4, 2), torch.zeros(2, 5, 4))       # wrong edge count
