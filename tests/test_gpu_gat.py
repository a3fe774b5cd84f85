"""GPU: stochastic GAT on the fused attention kernel (stag_attention_softmax_s / _s_bwd, csrc/edge_softmax.cu).  The logit
noise drawn inside the kernel equals the materialised noise bit for bit (every kind, parameter shape, relu, head count,
sample count, sample_base and device counter); gradients match float64 autograd; the layer, the sample-batched model,
sample sharding, the materialised routes, determinism, CUDA-graph replays and the full arxiv shape."""
import ctypes

import numpy as np
import pytest
import torch

from test_gpu_spmm import close

pytestmark = pytest.mark.gpu
T = torch.from_numpy
KINDS = ["normal", "uniform", "bernoulli"]
PSHAPES = ["scalar", "channel", "edge", "edge_channel"]


def make_graph(seed, n=300, e=3000):
    """(src, dst, N, Graph on cuda): the last 30 rows have no in-edges, rows 7 and 11 are hubs."""
    import stag_b200 as sb
    rng = np.random.default_rng(seed)
    src, dst = rng.integers(0, n, e), rng.integers(0, n - 30, e)
    dst[:500] = 7
    dst[500:700] = 11
    return src, dst, n, sb.Graph(T(src), T(dst), n).to("cuda")


def make_params(kind, pshape, E, H, rng, grad=False):
    shape = {"scalar": (), "channel": (H,), "edge": (E, 1), "edge_channel": (E, H)}[pshape]

    def t(a):
        return torch.tensor(np.asarray(a, np.float32), device="cuda").requires_grad_(grad)

    if kind == "normal":
        return t(1 + 0.2 * rng.standard_normal(shape)), t(0.3 + 0.2 * rng.random(shape))
    if kind == "uniform":
        return t(0.2 + 0.3 * rng.random(shape)), t(1.2 + 0.5 * rng.random(shape))
    return t(0.3 + 0.6 * rng.random(shape)), None


def raw_variates(spec, S):
    """[S,E,K] raw variates (standard normal / uniform) of a spec, from stag_noise_emit."""
    from stag_b200 import _lib, ops
    lib = _lib.load()
    w = torch.empty((S, spec.num_edges, spec.K), device="cuda")
    raw = torch.empty_like(w)
    nz = ops._fill_noise(spec, spec.lib_kind, spec.K, ops._c(spec.p0), ops._c(spec.p1), None, False, False,
                         spec.sample_base, spec.seed, spec.offset, spec.param_shape)
    _lib.check(lib.stag_noise_emit(ctypes.byref(nz), spec.num_edges, S, w.data_ptr(), raw.data_ptr(),
                                   torch.cuda.current_stream().cuda_stream))
    return raw


def ref_attention(src, dst, N, el, er, w, slope=0.2):
    """float64 restatement of the reference's attention (oracle/ref_layers.py GAT case): per sample s,
    softmax over the in-edges of leaky_relu(el[s,u] + er[s,v]) * w[s]."""
    s_, d_ = T(src).cuda(), T(dst).cuda()
    out = []
    for s in range(w.shape[0]):
        els = el[s] if el.dim() == 3 else el
        ers = er[s] if er.dim() == 3 else er
        e = torch.nn.functional.leaky_relu(els[s_] + ers[d_], slope) * w[s]
        idx = d_.unsqueeze(-1).expand_as(e)
        mx = torch.full((N, e.shape[1]), float("-inf"), dtype=e.dtype, device=e.device).scatter_reduce(
            0, idx, e, reduce="amax", include_self=True)
        ex = torch.exp(e - mx[d_])
        out.append(ex / torch.zeros((N, e.shape[1]), dtype=e.dtype, device=e.device).index_add(0, d_, ex)[d_])
    return torch.stack(out)


def scores(rng, S, N, H, shared):
    shape = (N, H) if shared else (S, N, H)
    return (T(rng.standard_normal(shape).astype(np.float32)).cuda(),
            T(rng.standard_normal(shape).astype(np.float32)).cuda())


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("H", [1, 3, 4, 8, 40])
@pytest.mark.parametrize("S,shared", [(1, True), (3, True), (3, False)])
def test_generated_noise_equals_attention_over_materialised_noise(kind, H, S, shared):
    """Bitwise: the attention with the noise drawn in the kernel equals the attention over spec.materialize(S) -- every
    parameter shape, with and without relu, sample_base != 0 -- and at S = 1 the pre-existing entry point fed that tensor."""
    import stag_b200 as sb
    from stag_b200.ops import NoiseSpec
    src, dst, N, g = make_graph(H + 10 * S)
    E = len(src)
    rng = np.random.default_rng(H * 7 + S)
    el, er = scores(rng, S, N, H, shared)
    for pshape in PSHAPES:
        for relu in (False, True):
            p0, p1 = make_params(kind, pshape, E, H, rng)
            spec = NoiseSpec(kind, p0, p1, H, E, relu=relu, seed=11, offset=5 + H, sample_base=2 * S - 1,
                             n_samples=S, batched=True)
            a = sb.ops.attention_softmax(g, el, er, spec, 0.2, n_samples=S)
            w = spec.materialize(n_samples=S)
            ref = sb.ops.attention_softmax(g, el, er, w, 0.2, n_samples=S)
            assert a.shape == (S, E, H)
            assert torch.equal(a, ref), (pshape, relu)
            if S == 1:
                assert torch.equal(a[0], sb.ops.attention_softmax(g, el, er, w[0], 0.2)), (pshape, relu)
            close(a, ref_attention(src, dst, N, el.double(), er.double(), w.double()), what="a %s %s" % (pshape, relu))


def test_generated_noise_follows_the_device_counter():
    """A non-zero device counter shifts the Philox call counter of the attention kernel exactly as that of
    stag_noise_emit: still bitwise equal to the materialised noise, and different from the counter-free draw."""
    import stag_b200 as sb
    from stag_b200.ops import NoiseSpec
    src, dst, N, g = make_graph(3)
    E, H, S = len(src), 4, 2
    rng = np.random.default_rng(3)
    el, er = scores(rng, S, N, H, False)
    p0, p1 = make_params("normal", "channel", E, H, rng)
    spec = NoiseSpec("normal", p0, p1, H, E, seed=4, offset=9, n_samples=S, batched=True)
    a0 = sb.ops.attention_softmax(g, el, er, spec, 0.2, n_samples=S)
    ctr = sb.random.enable_device_counter(torch.device("cuda"))
    try:
        ctr.fill_(5)
        a5 = sb.ops.attention_softmax(g, el, er, spec, 0.2, n_samples=S)
        assert torch.equal(a5, sb.ops.attention_softmax(g, el, er, spec.materialize(n_samples=S), 0.2, n_samples=S))
        assert not torch.equal(a5, a0)
    finally:
        sb.random.disable_device_counter()


@pytest.mark.parametrize("kind", ["normal", "uniform"])
@pytest.mark.parametrize("pshape", PSHAPES)
@pytest.mark.parametrize("relu", [False, True])
@pytest.mark.parametrize("H,shared", [(4, True), (5, False)])
def test_gradients_match_float64_autograd(kind, pshape, relu, H, shared):
    """d el, d er, d p0, d p1 against float64 autograd of the reference attention fed the same raw variates."""
    import stag_b200 as sb
    from stag_b200.ops import NoiseSpec
    src, dst, N, g = make_graph(H + len(pshape))
    E, S = len(src), 3
    rng = np.random.default_rng(H)
    el0, er0 = scores(rng, S, N, H, shared)
    p0, p1 = make_params(kind, pshape, E, H, rng, grad=True)
    da = T(rng.standard_normal((S, E, H)).astype(np.float32)).cuda()
    el, er = el0.clone().requires_grad_(True), er0.clone().requires_grad_(True)
    spec = NoiseSpec(kind, p0, p1, H, E, relu=relu, seed=7, offset=1, sample_base=1, n_samples=S, batched=True)
    a = sb.ops.attention_softmax(g, el, er, spec, 0.2, n_samples=S)
    a.backward(da)
    raw = raw_variates(spec, S).double()
    eld, erd = el0.double().requires_grad_(True), er0.double().requires_grad_(True)
    q0, q1 = p0.detach().double().requires_grad_(True), p1.detach().double().requires_grad_(True)
    b0, b1 = q0.expand(E, H), q1.expand(E, H)
    w = b0 + b1 * raw if kind == "normal" else b0 + raw * (b1 - b0)
    if relu:
        w = w.relu()
    ref = ref_attention(src, dst, N, eld, erd, w)
    ref.backward(da.double())
    close(a, ref, what="a")
    close(el.grad, eld.grad, what="d el")
    close(er.grad, erd.grad, what="d er")
    close(p0.grad, q0.grad, what="d p0")
    close(p1.grad, q1.grad, what="d p1")


@pytest.mark.parametrize("H", [4, 3])
def test_external_noise_gradient_matches_float64_autograd(H):
    import stag_b200 as sb
    src, dst, N, g = make_graph(40 + H)
    E, S = len(src), 2
    rng = np.random.default_rng(H)
    el0, er0 = scores(rng, S, N, H, False)
    w0 = T((1 + 0.4 * rng.standard_normal((S, E, H))).astype(np.float32)).cuda()
    da = T(rng.standard_normal((S, E, H)).astype(np.float32)).cuda()
    el, er, w = (t.clone().requires_grad_(True) for t in (el0, er0, w0))
    sb.ops.attention_softmax(g, el, er, w, 0.2).backward(da)
    eld, erd, wd = (t.double().requires_grad_(True) for t in (el0, er0, w0))
    ref_attention(src, dst, N, eld, erd, wd).backward(da.double())
    close(el.grad, eld.grad, what="d el")
    close(er.grad, erd.grad, what="d er")
    close(w.grad, wd.grad, what="d w")


def test_fused_path_refuses_hadamard_and_in_norm_at_the_abi():
    from stag_b200 import _lib, ops
    src, dst, N, g = make_graph(5)
    E, H = len(src), 128
    lib = _lib.load()
    st = g._s
    csc, _ = st.csx(True)
    el = torch.zeros(N, H, device="cuda")
    a = torch.empty(E, H, device="cuda")
    one = torch.ones((), device="cuda")
    for kind, in_norm, code in ((_lib.NOISE_NORMAL_HADAMARD, False, _lib.STAG_EUNSUPPORTED),
                                (_lib.NOISE_NORMAL, True, _lib.STAG_EINVAL)):
        nz = ops._fill_noise(None, kind, H, one, one, None, False, in_norm, 0, 1, 1, _lib.PARAM_SCALAR)
        rc = lib.stag_attention_softmax_s(ctypes.byref(csc), el.data_ptr(), 0, el.data_ptr(), 0, H, 1, ctypes.byref(nz),
                                          0.2, a.data_ptr(), 0, 0, torch.cuda.current_stream().cuda_stream)
        assert rc == code


@pytest.mark.parametrize("route", ["in_norm", "edge_channel"])
def test_materialised_and_amortised_routes_equal_the_materialised_computation(route):
    """An in-norm spec (materialised route) and amortised [E,H] parameters (fused, EDGE_CHANNEL) against the attention
    over the materialised tensor, forward bitwise and parameter gradients."""
    import stag_b200 as sb
    from stag_b200.layers import _in_norm
    from stag_b200.ops import NoiseSpec
    src, dst, N, g = make_graph(9)
    E, H, S = len(src), 4, 2
    rng = np.random.default_rng(9)
    el, er = scores(rng, S, N, H, True)
    pshape = "scalar" if route == "in_norm" else "edge_channel"
    p0, p1 = make_params("normal", pshape, E, H, rng, grad=route == "edge_channel")
    spec = NoiseSpec("normal", p0, p1, H, E, relu=True, in_norm=route == "in_norm", seed=2, offset=8, n_samples=S,
                     batched=True)
    if route == "in_norm":
        assert sb.ops.attention_route(spec) == "materialized"
    else:
        assert sb.ops.attention_route(spec) == "fused"
    da = T(rng.standard_normal((S, E, H)).astype(np.float32)).cuda()
    a = sb.ops.attention_softmax(g, el, er, spec, 0.2, n_samples=S)
    w = spec.materialize(n_samples=S)
    if route == "in_norm":
        w = torch.stack([_in_norm(g, w[s]) for s in range(S)])
    ref = sb.ops.attention_softmax(g, el, er, w, 0.2, n_samples=S)
    assert torch.equal(a.detach(), ref.detach())
    if route == "edge_channel":
        g0, g1 = torch.autograd.grad(a, (p0, p1), da)
        r0, r1 = torch.autograd.grad(ref, (p0, p1), da)
        close(g0, r0, what="d loc")
        close(g1, r1, what="d scale")


def test_runs_are_bitwise_identical():
    import stag_b200 as sb
    from stag_b200.ops import NoiseSpec
    src, dst, N, g = make_graph(13)
    E, S = len(src), 3
    res = []
    for H, pshape in ((4, "channel"), (5, "scalar"), (3, "edge")):
        for _ in range(2):
            rng = np.random.default_rng(H)
            el0, er0 = scores(rng, S, N, H, False)
            el, er = el0.requires_grad_(True), er0.requires_grad_(True)
            p0, p1 = make_params("normal", pshape, E, H, rng, grad=True)
            spec = NoiseSpec("normal", p0, p1, H, E, relu=True, seed=3, offset=3, n_samples=S, batched=True)
            a = sb.ops.attention_softmax(g, el, er, spec, 0.2, n_samples=S)
            (a * torch.linspace(-1, 1, a.numel(), device="cuda").view(a.shape)).sum().backward()
            res.append([t.detach().clone() for t in (a, el.grad, er.grad, p0.grad, p1.grad)])
    for i in range(0, len(res), 2):
        for u, v in zip(res[i], res[i + 1]):
            assert torch.equal(u, v)


def gat_layer(D, F, H, vi=False, **kw):
    import stag_b200 as sb
    torch.manual_seed(D + F + H)
    q_a = torch.distributions.Normal(torch.ones(H), torch.full((H,), 0.5))
    return sb.layers.StagLayer(sb.zoo.GAT(D, F, num_heads=H, **kw), q_a=q_a, vi=vi).cuda()


@pytest.mark.parametrize("H,last", [(4, False), (3, True)])
def test_layer_forward_equals_the_base_layer_on_its_own_sample(H, last, monkeypatch):
    """StagLayer(GAT) hands the spec to the fused attention (no stag_noise_emit on that route); the output equals
    base_layer.forward on the materialised _edge_weight_sample bit for bit."""
    import stag_b200 as sb
    src, dst, N, g = make_graph(17)
    layer = gat_layer(16, 8, H, last=last, residual=True)
    x = torch.randn(N, 16, device="cuda")

    def refuse(*a, **k):
        raise AssertionError("stag_noise_emit on the fused GAT route")

    with monkeypatch.context() as m:
        m.setattr(sb.ops._NoiseEmit, "apply", refuse)
        out = layer(g, x)
    assert layer._noise_tensor is None
    assert torch.equal(out, layer.base_layer(g, x, edge_weight=layer._edge_weight_sample))


def test_vi_layer_gradients_match_the_materialised_path():
    import stag_b200 as sb
    src, dst, N, g = make_graph(19)
    H = 4
    layer = gat_layer(12, 6, H, vi=True)
    x = torch.randn(N, 12, device="cuda")
    gout = torch.randn(N, H * 6, device="cuda")
    named = [(n, p) for n, p in layer.named_parameters() if p.requires_grad and not n.startswith("p_a")]
    params = [p for _, p in named]
    assert any(n.startswith("q_a") for n, _ in named)
    out = layer(g, x)
    fused = torch.autograd.grad(out, params, gout, retain_graph=True)   # the spec's loc / scale feed both passes
    w = layer._noise_spec.materialize()
    ref_out = layer.base_layer(g, x, edge_weight=w)
    ref = torch.autograd.grad(ref_out, params, gout)
    assert torch.equal(out, ref_out)
    for (n, _), u, v in zip(named, fused, ref):
        close(u, v, what=n)


def test_mixture_prior_kl_matches_log_prob_on_the_materialised_sample():
    import stag_b200 as sb
    src, dst, N, g = make_graph(23)
    H = 4
    prior = torch.distributions.MixtureSameFamily(torch.distributions.Categorical(torch.tensor([0.3, 0.7])),
                                                  torch.distributions.Normal(torch.tensor([0.0, 1.0]),
                                                                             torch.tensor([0.5, 1.5])))
    q_a = torch.distributions.Normal(torch.ones(H), torch.full((H,), 0.5))
    layer = sb.layers.StagLayer(sb.zoo.GAT(8, 4, num_heads=H), q_a=q_a, p_a=prior, vi=True).cuda()
    layer(g, torch.randn(N, 8, device="cuda"))
    assert layer._noise_tensor is None
    kl = layer.kl_divergence()
    w = layer._edge_weight_sample
    ref = layer.q_a.log_prob(w).sum(dim=-1).mean() - layer.p_a.log_prob(w.cpu()).sum(dim=-1).mean().to(w.device)
    close(kl, ref, what="kl")


@pytest.mark.parametrize("shared", [True, False])
@pytest.mark.parametrize("last,residual", [(False, False), (True, True)])
def test_sample_batched_layer_equals_single_sample_calls(shared, last, residual):
    import stag_b200 as sb
    from stag_b200.ops import NoiseSpec
    src, dst, N, g = make_graph(29)
    E, H, F, S = len(src), 4, 8, 3
    base = sb.zoo.GAT(16, F, num_heads=H, last=last, residual=residual).cuda()
    x = torch.randn(N, 16, device="cuda") if shared else torch.randn(S, N, 16, device="cuda")
    p0, p1 = make_params("normal", "channel", E, H, np.random.default_rng(0))
    spec = NoiseSpec("normal", p0, p1, H, E, seed=5, offset=2, n_samples=S, batched=True)
    out, att = base(g, x, edge_weight=spec, get_attention=True)
    w = spec.materialize(n_samples=S)
    assert out.shape == (S, N, F if last else H * F) and att.shape == (S, E, H, 1)
    for s in range(S):
        o, a = base(g, x if shared else x[s], edge_weight=w[s], get_attention=True)
        if shared:      # same scores: the attention is the same computation
            assert torch.equal(att[s], a)
        else:           # the dense transform of [S,N,D] and of [N,D] may reduce in different orders
            close(att[s], a, what="attention %d" % s)
        close(out[s], o, what="out %d" % s)


def two_layer_model(H=4, vi=True):
    import stag_b200 as sb
    torch.manual_seed(1)
    q = lambda h: torch.distributions.Normal(torch.ones(h), torch.full((h,), 0.4))  # noqa: E731
    layers = torch.nn.ModuleList([
        sb.layers.StagLayer(sb.zoo.GAT(16, 8, num_heads=H, activation=torch.nn.functional.elu), q_a=q(H), vi=vi),
        sb.layers.StagLayer(sb.zoo.GAT(8 * H, 5, num_heads=1, last=True, activation=lambda t: torch.softmax(t, -1)),
                            q_a=q(1), vi=vi),
    ]).cuda()
    return sb.models.StagModel(layers)


def trained_params(model):
    """Parameters a forward pass reaches: the base layers' and the posteriors' (not the priors')."""
    return [p for layer in model.layers for m in (layer.base_layer, layer.q_a) for p in m.parameters() if p.requires_grad]


def test_two_layer_model_batches_and_matches_per_sample_passes():
    src, dst, N, g = make_graph(31)
    S = 4
    model = two_layer_model()
    assert model._can_batch()
    x = torch.randn(N, 16, device="cuda")
    y = torch.randint(0, 5, (N,), device="cuda")
    nll, reg = model.loss_terms(g, x, y, n_samples=S)
    (nll + reg).backward()
    params = trained_params(model)
    assert torch.isfinite(nll) and all(p.grad is not None for p in params)
    model.zero_grad()
    outs = model._forward_samples(g, x, S)
    gout = torch.randn_like(outs)
    got = torch.autograd.grad(outs, params, gout, retain_graph=True)
    ws = [layer._noise_spec.materialize(n_samples=S) for layer in model.layers]
    ref = []
    for s in range(S):
        h = x
        for layer, w in zip(model.layers, ws):
            h = layer.base_layer(g, h, edge_weight=w[s])
        ref.append(h)
    ref = torch.stack(ref)
    close(outs, ref, what="outputs")
    for p, u, v in zip(params, got, torch.autograd.grad(ref, params, gout)):
        close(u, v, what=str(tuple(p.shape)))


def test_gat_model_shards_samples_over_sample_base():
    """forward(n_samples=8) of a GAT model equals n_samples=4 at sample_base 0 and 4 put together (what
    parallel.shard_samples hands two ranks)."""
    import stag_b200 as sb
    src, dst, N, g = make_graph(37)
    model = two_layer_model(vi=False)
    x = torch.randn(N, 16, device="cuda")
    with torch.no_grad():
        noise = []
        outs = []
        for n, base in ((8, 0), (4, 0), (4, 4)):
            sb.manual_seed(21)
            outs.append(model._forward_samples(g, x, n, sample_base=base))
            noise.append([layer._noise_spec.materialize() for layer in model.layers])
        full, lo, hi = outs
        # the same noise, bit for bit, for every sample of every layer ...
        for wf, wl, wh in zip(*noise):
            assert torch.equal(torch.cat([wl, wh]), wf)
        # ... and the same outputs (the dense transform of 4 N and 8 N rows may reduce in different orders)
        close(torch.cat([lo, hi]), full, rtol=1e-6, what="sharded outputs")
        sb.manual_seed(21)
        pred = model(g, x, n_samples=4, sample_base=4, return_parameters=True)
        assert torch.equal(pred, hi.mean(0))


def test_cuda_graph_replays_equal_eager_steps():
    """A captured two-layer stochastic attention step (fused attention + per-head aggregation per layer, forward and the
    gradients w.r.t. the features, scores and noise parameters): replay i equals eager step i bit for bit, and the steps
    draw fresh noise through the device counter."""
    import stag_b200 as sb
    from stag_b200.ops import NoiseSpec
    dev = torch.device("cuda")
    src, dst, N, g = make_graph(41)
    g._s.csx(True), g._s.csx(False)                       # structure is built outside the capture (host syncs)
    E, H, F, S = len(src), 4, 8, 2
    ft = torch.randn(N, H, F, device=dev, requires_grad=True)
    el, er = torch.randn(N, H, device=dev, requires_grad=True), torch.randn(N, H, device=dev, requires_grad=True)
    loc = torch.ones(H, device=dev, requires_grad=True)
    scale = torch.full((H,), 0.4, device=dev, requires_grad=True)
    gout = torch.randn(S, N, H, F, device=dev)
    ctr = sb.random.enable_device_counter(dev)

    def step():
        h = ft
        for _ in range(2):                                # two layers: two Philox offsets per step
            spec = NoiseSpec("normal", loc, scale, H, E, n_samples=S, batched=True)
            a = sb.ops.attention_softmax(g, el, er, spec, 0.2, n_samples=S)
            h = sb.ops.heads_aggregate(g, h, a)
        grads = torch.autograd.grad(h, (ft, el, er, loc, scale), gout)
        assert sb.random.advance_device_counter() == 2
        return (h.detach(),) + tuple(grads)

    try:
        sb.manual_seed(5)
        ctr.zero_()
        eager = [tuple(t.clone() for t in step()) for _ in range(3)]
        assert not torch.equal(eager[0][0], eager[1][0])
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            step()
        torch.cuda.current_stream().wait_stream(side)
        sb.manual_seed(5)
        ctr.zero_()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            res = step()
        for i in range(3):
            graph.replay()
            torch.cuda.synchronize()
            for u, v in zip(res, eager[i]):
                assert torch.equal(u, v), i
    finally:
        sb.random.disable_device_counter()


def test_full_size_against_the_per_sample_tensor_path():
    """arxiv shape, GAT 128 -> 4 x 32, S = 4: the batched fused layer against the tensor path fed materialize(S)[s], on a
    row subset (the 64 largest in-degrees and 2000 random rows) and on the in-edges of those rows."""
    import bench
    import stag_b200 as sb
    from stag_b200.ops import NoiseSpec
    src, dst = bench.synth_graph()
    N, E, H, F, S = bench.N_NODES, bench.N_EDGES, 4, 32, 4
    g = sb.Graph(T(src), T(dst), N).to("cuda")
    torch.manual_seed(0)
    base = sb.zoo.GAT(128, F, num_heads=H).cuda()
    x = torch.randn(N, 128, device="cuda")
    spec = NoiseSpec("normal", torch.ones(H, device="cuda"), torch.full((H,), 0.4, device="cuda"), H, E, seed=13,
                     offset=2, n_samples=S, batched=True)
    with torch.no_grad():
        out, att = base(g, x, edge_weight=spec, get_attention=True)
        w = spec.materialize(n_samples=S)
        deg = np.bincount(dst, minlength=N)
        rows = np.unique(np.concatenate([np.argsort(-deg)[:64], np.random.default_rng(0).integers(0, N, 2000)]))
        sel = T(np.nonzero(np.isin(dst, rows))[0]).cuda()
        r = T(rows).cuda()
        for s in range(S):
            o, a = base(g, x, edge_weight=w[s], get_attention=True)
            assert torch.equal(att[s][sel], a[sel])
            close(out[s][r], o[r], what="out %d" % s)
