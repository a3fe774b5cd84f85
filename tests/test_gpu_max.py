"""GPU: the max aggregation kernels (stag_spmm_max_fwd / _bwd, csrc/spmm_max.cuh) against the CPU oracle
(oracle/ref_max.py): values and winning edges exactly, gradients to 1e-5, the first-winner tie rule, every noise kind
against the materialised noise, parameter gradients, sample batching, determinism, CUDA-graph replays, the layers
that use it and the full arxiv shape."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import ref_max
from test_gpu_spmm import close

pytestmark = pytest.mark.gpu
T = torch.from_numpy


def make_graph(kind, seed, n=300, e=3000):
    """(src, dst, N, NS, Graph on cuda) with zero in-degree rows, hubs, power-law degrees or two node sets."""
    import stag_b200 as sb
    rng = np.random.default_rng(seed)
    NS = n
    if kind == "bipartite":
        NS = n + 77
        src, dst = rng.integers(0, NS, e), rng.integers(0, n, e)
    elif kind == "power":
        src = rng.integers(0, n, e)
        dst = np.minimum((rng.pareto(1.2, e) * 3).astype(np.int64), n - 1)
    else:
        src, dst = rng.integers(0, n, e), rng.integers(0, n - 40, e)   # the last 40 rows have no in-edges
        if kind == "hub":
            dst[:700] = 7                                                # hub rows above the threshold (128)
            dst[700:1000] = 11
            src[:400] = 3                                                # and a source hub for the CSR walk
    g = sb.Graph(T(src), T(dst), n, num_src=NS if NS != n else None).to("cuda")
    return src, dst, n, NS, g


def abi_max(g, x, nz, D, S, shared=True):
    """(out, arg) [S,N,D] straight from stag_spmm_max_fwd (the operator keeps arg to itself)."""
    from stag_b200 import _lib, ops
    lib, st = _lib.load(), g._s
    N, NS = st.num_nodes, st.num_src
    csc, _ = st.csx(True)
    ws = ops._workspace(st, lib, csc, True, D, S)
    out = torch.empty((S, N, D), device="cuda")
    arg = torch.empty((S, N, D), dtype=torch.int32, device="cuda")
    _lib.check(lib.stag_spmm_max_fwd(ctypes.byref(csc), x.data_ptr(), D, 0 if shared else NS * D, D, S,
                                     ctypes.byref(nz), out.data_ptr(), arg.data_ptr(), D, N * D, ws.data_ptr(),
                                     ws.numel(), torch.cuda.current_stream().cuda_stream))
    return out, arg


def ext_noise(w):
    from stag_b200 import _lib, ops
    return ops._fill_noise(None, _lib.NOISE_EXTERNAL, w.shape[-1], None, None, w, False, False, 0, 0, 0,
                           _lib.PARAM_SCALAR)


def spec_nz(spec):
    from stag_b200 import ops
    return ops._fill_noise(spec, spec.lib_kind, spec.K, ops._c(spec.p0), ops._c(spec.p1), None, spec.relu, False,
                           spec.sample_base, spec.seed, spec.offset, spec.param_shape)


def oracle(src, dst, N, x, w):
    return ref_max.u_mul_e_max(T(src), T(dst), N, x, w)


@pytest.mark.parametrize("gkind", ["zero", "hub", "power", "bipartite"])
@pytest.mark.parametrize("D", [1, 9, 16, 50, 100, 128, 256, 1433])
@pytest.mark.parametrize("per_channel", [True, False])
def test_external_noise_matches_oracle(gkind, D, per_channel):
    import stag_b200 as sb
    src, dst, N, NS, g = make_graph(gkind, D)
    E = len(src)
    K = D if per_channel else 1
    rng = np.random.default_rng(D + 7)
    x = T(rng.standard_normal((NS, D)).astype(np.float32))
    w = T(rng.standard_normal((E, K)).astype(np.float32))
    gout = T(rng.standard_normal((N, D)).astype(np.float32))
    xc, wc = x.cuda().requires_grad_(True), w.cuda().requires_grad_(True)
    out = sb.ops.stochastic_aggregate(g, xc, wc, reduce="max")
    out.backward(gout.cuda())
    xo, wo = x.clone().requires_grad_(True), w.clone().requires_grad_(True)
    ro, ra = oracle(src, dst, N, xo, wo)
    ro.backward(gout)
    assert torch.equal(out.detach().cpu(), ro.detach())
    wn = w.cuda()[None].contiguous()   # the noise struct holds a raw pointer: keep the tensor alive
    _, arg = abi_max(g, x.cuda(), ext_noise(wn), D, 1)
    assert torch.equal(arg[0].cpu().long(), ra)
    close(xc.grad, xo.grad, what="dx")
    if per_channel:
        assert torch.equal(wc.grad.cpu(), wo.grad), "dw"
    else:
        close(wc.grad, wo.grad, what="dw")


def test_ties_go_to_the_first_winner():
    import stag_b200 as sb
    src, dst, N, NS, g = make_graph("hub", 5)
    E, D = len(src), 64
    rng = np.random.default_rng(3)
    x = torch.relu(T(rng.standard_normal((N, D)).astype(np.float32)))   # many exact zeros
    x[10:20] = x[30]                                                    # duplicate rows
    w = T((rng.random((E, D)) < 0.5).astype(np.float32))               # Bernoulli-like 0 / 1 noise
    gout = T(rng.standard_normal((N, D)).astype(np.float32))
    xc, wc = x.cuda().requires_grad_(True), w.cuda().requires_grad_(True)
    out = sb.ops.stochastic_aggregate(g, xc, wc, reduce="max")
    out.backward(gout.cuda())
    xo, wo = x.clone().requires_grad_(True), w.clone().requires_grad_(True)
    ro, ra = oracle(src, dst, N, xo, wo)
    ro.backward(gout)
    wn = w.cuda()[None].contiguous()
    _, arg = abi_max(g, x.cuda(), ext_noise(wn), D, 1)
    assert torch.equal(arg[0].cpu().long(), ra)
    assert (ra >= 0).any() and torch.equal(out.detach().cpu(), ro.detach())
    # the winner is the smallest edge id among the edges reaching the maximum
    msg = x[T(src)] * w
    for v in (7, 11, 0):
        for c in range(0, D, 7):
            es = np.nonzero(dst == v)[0]
            if len(es):
                vals = msg[T(es), c]
                assert ra[v, c] == es[int(torch.nonzero(vals == vals.max())[0, 0])]
    assert torch.equal(wc.grad.cpu(), wo.grad)       # gradients only on the winners
    close(xc.grad, xo.grad, what="dx")


SPECS = [  # kind, generator, p0, p1, pshape, relu
    ("normal", "boxmuller", 1.0, 0.4, "scalar", False),
    ("normal", "boxmuller", 0.2, 1.0, "channel", True),
    ("normal", "boxmuller", 1.0, 0.4, "edge", False),
    ("normal", "hadamard", 1.0, 0.4, "scalar", False),
    ("normal", "hadamard", 0.1, 1.0, "edge", False),
    ("uniform", None, 0.3, 1.7, "scalar", False),
    ("uniform", None, -0.5, 1.0, "channel", True),
    ("bernoulli", None, 0.6, None, "scalar", False),
    ("bernoulli", None, 0.6, None, "edge", False),
]


def make_params(p, pshape, E, D, rng):
    if p is None:
        return None
    if pshape == "scalar":
        return torch.tensor(p, device="cuda")
    if pshape == "channel":
        return torch.tensor(p + 0.1 * rng.standard_normal(D), dtype=torch.float32, device="cuda")
    return torch.tensor(p + 0.1 * rng.standard_normal((E, 1)), dtype=torch.float32, device="cuda")


@pytest.mark.parametrize("spec_args", SPECS)
@pytest.mark.parametrize("D,K", [(128, 128), (50, 50), (256, 256), (16, 1)])
def test_generated_noise_equals_max_over_materialised_noise(spec_args, D, K):
    import stag_b200 as sb
    from stag_b200.ops import NoiseSpec
    kind, gen, p0, p1, pshape, relu = spec_args
    if gen == "hadamard" and (K % 128):
        pytest.skip("the Hadamard generator needs K % 128 == 0")
    if pshape == "channel" and K == 1:
        pytest.skip("per-channel parameters need K == D")
    src, dst, N, NS, g = make_graph("hub", D + 1)
    E, S = len(src), 3
    rng = np.random.default_rng(D)
    spec = NoiseSpec(kind, make_params(p0, pshape, E, K, rng), make_params(p1, pshape, E, K, rng), K, E, relu=relu,
                     seed=5, offset=9, n_samples=S, batched=True, generator=gen)
    x = torch.randn(NS, D, device="cuda")
    out = sb.ops.stochastic_aggregate(g, x, spec, reduce="max", n_samples=S)
    w = spec.materialize(n_samples=S).detach().cpu()
    _, arg = abi_max(g, x, spec_nz(spec), D, S)
    for s in range(S):
        ro, ra = oracle(src, dst, N, x.cpu(), w[s])
        assert torch.equal(out[s].cpu(), ro), s
        assert torch.equal(arg[s].cpu().long(), ra), s


@pytest.mark.parametrize("kind", ["normal", "uniform"])
@pytest.mark.parametrize("pshape", ["scalar", "channel", "edge"])
@pytest.mark.parametrize("relu", [False, True])
def test_parameter_gradients_match_float64_autograd(kind, pshape, relu):
    """r1 / rc / re: d loc, d scale (d low, d high) and dx against float64 autograd on the emitted variates, with the
    winners the kernel picked (the argmax rule)."""
    import stag_b200 as sb
    from stag_b200.ops import NoiseSpec
    src, dst, N, NS, g = make_graph("hub", 17)
    E, D, S = len(src), 64, 2
    rng = np.random.default_rng(11)
    a, b = (1.0, 0.5) if kind == "normal" else (0.2, 1.4)
    p0 = make_params(a, pshape, E, D, rng).requires_grad_(True)
    p1 = make_params(b, pshape, E, D, rng).requires_grad_(True)
    x = torch.randn(NS, D, device="cuda", requires_grad=True)
    gout = torch.randn(S, N, D, device="cuda")
    spec = NoiseSpec(kind, p0, p1, D, E, relu=relu, seed=3, offset=4, n_samples=S, batched=True)
    out = sb.ops.stochastic_aggregate(g, x, spec, reduce="max", n_samples=S)
    out.backward(gout)
    _, arg = abi_max(g, x.detach(), spec_nz(spec), D, S)
    # raw variates: the same stream with loc 0 / scale 1 (low 0 / high 1)
    z = NoiseSpec(kind, torch.zeros((), device="cuda"), torch.ones((), device="cuda"), D, E, seed=3, offset=4,
                  n_samples=S).materialize(n_samples=S).double().cpu()
    q0 = p0.detach().double().cpu().requires_grad_(True)
    q1 = p1.detach().double().cpu().requires_grad_(True)
    xo = x.detach().double().cpu().requires_grad_(True)
    w = q0 + z * q1 if kind == "normal" else q0 + z * (q1 - q0)
    if relu:
        w = w.relu()
    total = 0
    for s in range(S):
        msg = xo[T(src)] * w[s]
        am = arg[s].cpu().long()
        o = torch.where(am >= 0, torch.gather(msg, 0, am.clamp(min=0)), torch.zeros(()).double())
        total = total + (o * gout[s].cpu().double()).sum()
    total.backward()
    close(x.grad, xo.grad, what="dx")
    close(p0.grad, q0.grad, what="dp0")
    close(p1.grad, q1.grad, what="dp1")


@pytest.mark.parametrize("route", ["rec", "in_norm"])
def test_materialised_routes_equal_the_materialised_computation(route):
    import stag_b200 as sb
    from stag_b200.layers import _in_norm
    from stag_b200.ops import NoiseSpec
    src, dst, N, NS, g = make_graph("zero", 23)
    E, D, S = len(src), 32, 2
    if route == "rec":
        p0 = (1 + 0.1 * torch.randn(E, D, device="cuda")).requires_grad_(True)
        p1 = torch.full((E, D), 0.3, device="cuda", requires_grad=True)
        spec = NoiseSpec("normal", p0, p1, D, E, seed=1, offset=2, n_samples=S, batched=True)
    else:
        p0, p1 = torch.tensor(0.0, device="cuda"), torch.tensor(1.0, device="cuda")  # signed in-norm scales
        spec = NoiseSpec("normal", p0, p1, D, E, in_norm=True, seed=1, offset=2, n_samples=S, batched=True)
    x = torch.randn(NS, D, device="cuda", requires_grad=True)
    gout = torch.randn(S, N, D, device="cuda")
    out = sb.ops.stochastic_aggregate(g, x, spec, reduce="max", n_samples=S)
    out.backward(gout)
    grads = (x.grad.clone(), None if route != "rec" else p0.grad.clone())
    x.grad = None
    if route == "rec":
        p0.grad = None
    w = spec.materialize(n_samples=S)
    if route == "in_norm":
        w = torch.stack([_in_norm(g, w[s]) for s in range(S)])
    ref = torch.stack([sb.ops.stochastic_aggregate(g, x, w[s], reduce="max") for s in range(S)])
    ref.backward(gout)
    assert torch.equal(out, ref)
    close(grads[0], x.grad, what="dx")
    if route == "rec":
        close(grads[1], p0.grad, what="dp0")
    wo = w.detach().cpu()
    for s in range(S):
        assert torch.equal(out[s].detach().cpu(), oracle(src, dst, N, x.detach().cpu(), wo[s])[0])


@pytest.mark.parametrize("shared", [True, False])
@pytest.mark.parametrize("kind", ["normal", "uniform"])
def test_sample_batching_equals_single_sample_calls(shared, kind):
    import stag_b200 as sb
    from stag_b200.ops import NoiseSpec
    src, dst, N, NS, g = make_graph("hub", 29)
    E, D, S = len(src), 96, 4
    p0 = torch.full((D,), 1.0 if kind == "normal" else 0.1, device="cuda", requires_grad=True)
    p1 = torch.full((D,), 0.5 if kind == "normal" else 1.5, device="cuda", requires_grad=True)
    spec = NoiseSpec(kind, p0, p1, D, E, seed=8, offset=1, n_samples=S, batched=True)
    x = torch.randn(NS, D, device="cuda") if shared else torch.randn(S, NS, D, device="cuda")
    x.requires_grad_(True)
    gout = torch.randn(S, N, D, device="cuda")
    out = sb.ops.stochastic_aggregate(g, x, spec, reduce="max", n_samples=S)
    out.backward(gout)
    gx, g0, g1 = x.grad.clone(), p0.grad.clone(), p1.grad.clone()
    x.grad = p0.grad = p1.grad = None
    for s in range(S):
        one = spec.with_samples(1, s)
        o = sb.ops.stochastic_aggregate(g, x if shared else x[s], one, reduce="max", n_samples=1)
        assert torch.equal(o[0], out[s].detach()), s
        o.backward(gout[s:s + 1])
    close(gx, x.grad, what="dx")
    close(g0, p0.grad, what="dp0")
    close(g1, p1.grad, what="dp1")


def test_runs_are_bitwise_identical():
    import stag_b200 as sb
    from stag_b200.ops import NoiseSpec
    src, dst, N, NS, g = make_graph("hub", 31)
    E, D, S = len(src), 128, 3
    res = []
    for _ in range(2):
        p0 = torch.full((D,), 1.0, device="cuda", requires_grad=True)
        p1 = torch.full((D,), 0.5, device="cuda", requires_grad=True)
        r0 = torch.full((E, 1), 1.0, device="cuda", requires_grad=True)
        r1 = torch.full((E, 1), 0.5, device="cuda", requires_grad=True)
        x = torch.linspace(-1, 1, NS * D, device="cuda").reshape(NS, D).sin().requires_grad_(True)
        gout = torch.linspace(-2, 3, S * N * D, device="cuda").reshape(S, N, D).cos()
        a = sb.ops.stochastic_aggregate(g, x, NoiseSpec("normal", p0, p1, D, E, relu=True, seed=2, offset=3,
                                                        n_samples=S, batched=True), reduce="max", n_samples=S)
        b = sb.ops.stochastic_aggregate(g, x, NoiseSpec("uniform", r0, r1, D, E, seed=2, offset=4, n_samples=S,
                                                        batched=True), reduce="max", n_samples=S)
        (a + b).backward(gout)
        _, arg = abi_max(g, x.detach(), spec_nz(NoiseSpec("normal", p0, p1, D, E, relu=True, seed=2, offset=3,
                                                          n_samples=S)), D, S)
        res.append([t.detach().clone() for t in (a, b, arg, x.grad, p0.grad, p1.grad, r0.grad, r1.grad)])
    for u, v in zip(*res):
        assert torch.equal(u, v)


@pytest.mark.parametrize("generator", ["boxmuller", "hadamard"])
def test_cuda_graph_replays_equal_eager_steps(generator):
    import stag_b200 as sb
    from stag_b200.ops import NoiseSpec
    dev = torch.device("cuda")
    src, dst, N, NS, g = make_graph("hub", 37)
    E, D, S = len(src), 128, 2
    g._s.csx(True), g._s.csx(False)
    x = torch.randn(NS, D, device=dev, requires_grad=True)
    gout = torch.randn(S, N, D, device=dev)
    one, sg = torch.ones((), device=dev), torch.full((), 0.4, device=dev)
    ctr = sb.random.enable_device_counter(dev)

    def step():
        spec = NoiseSpec("normal", one, sg, D, E, n_samples=S, batched=True, generator=generator)
        out = sb.ops.stochastic_aggregate(g, x, spec, reduce="max", n_samples=S)
        dx, = torch.autograd.grad(out, x, gout)
        assert sb.random.advance_device_counter() == 1
        return out.detach(), dx

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
            out, dx = step()
        for i in range(3):
            graph.replay()
            torch.cuda.synchronize()
            assert torch.equal(out, eager[i][0]) and torch.equal(dx, eager[i][1]), i
    finally:
        sb.random.disable_device_counter()


def test_sage_pool_layer_matches_oracle():
    import stag_b200 as sb
    src, dst, N, NS, g = make_graph("zero", 41, n=80, e=500)
    E, D, O = len(src), 16, 8
    torch.manual_seed(0)
    base = sb.zoo.GraphSAGE(D, O, aggregator_type="pool").cuda()
    with torch.no_grad():
        base.bias.normal_()
        base.fc_pool.bias.normal_()
    layer = sb.layers.StagLayer(base)
    feat = torch.randn(N, D, device="cuda", requires_grad=True)
    w = torch.randn(E, D, device="cuda", requires_grad=True)
    layer.rsample_noise = lambda graph, sample_dimension, **kw: w
    gout = torch.randn(N, O, device="cuda")
    out = layer(g, feat)
    out.backward(gout)
    P = {k: v.detach().cpu().requires_grad_(True) for k, v in base.named_parameters()}
    fo, wo = feat.detach().cpu().requires_grad_(True), w.detach().cpu().requires_grad_(True)
    ro = ref_max.sage_pool_forward(T(src), T(dst), N, fo, wo, P["fc_pool.weight"], P["fc_pool.bias"],
                                   P["fc_self.weight"], P["fc_neigh.weight"], P["bias"])
    ro.backward(gout.cpu())
    close(out, ro, what="out")
    close(feat.grad, fo.grad, what="dfeat")
    close(w.grad, wo.grad, what="dw")
    for k, p in base.named_parameters():
        close(p.grad, P[k].grad, what=k)


def test_gin_max_layer_matches_oracle():
    import stag_b200 as sb
    src, dst, N, NS, g = make_graph("hub", 43)
    E, D, O = len(src), 24, 8
    base = sb.zoo.GIN(D, O, aggregator_type="max", init_eps=0.25).cuda()
    layer = sb.layers.StagLayer(base)
    feat = torch.randn(N, D, device="cuda", requires_grad=True)
    w = torch.randn(E, D, device="cuda", requires_grad=True)
    layer.rsample_noise = lambda graph, sample_dimension, **kw: w
    gout = torch.randn(N, O, device="cuda")
    out = layer(g, feat)
    out.backward(gout)
    Wl = base.apply_func.weight.detach().cpu().requires_grad_(True)
    bl = base.apply_func.bias.detach().cpu().requires_grad_(True)
    fo, wo = feat.detach().cpu().requires_grad_(True), w.detach().cpu().requires_grad_(True)
    ro = ref_max.gin_max_forward(T(src), T(dst), N, fo, wo, Wl, bl, eps=0.25)
    ro.backward(gout.cpu())
    close(out, ro, what="out")
    close(feat.grad, fo.grad, what="dfeat")
    close(w.grad, wo.grad, what="dw")
    close(base.apply_func.weight.grad, Wl.grad, what="apply_func.weight")
    close(base.apply_func.bias.grad, bl.grad, what="apply_func.bias")


def test_sample_batched_model_with_a_pool_layer_runs():
    import stag_b200 as sb
    src, dst, N, NS, g = make_graph("hub", 47)
    D, C = 32, 5
    layers = torch.nn.ModuleList([
        sb.layers.StagLayer(sb.zoo.GraphSAGE(D, 16, aggregator_type="pool", activation=torch.relu)),
        sb.layers.StagLayer(sb.zoo.GCN(16, C, activation=lambda t: torch.softmax(t, -1))),
    ]).cuda()
    model = sb.models.StagModel(layers)
    assert model._can_batch()
    feat = torch.randn(N, D, device="cuda")
    y = torch.randint(0, C, (N,), device="cuda")
    nll, reg = model.loss_terms(g, feat, y, n_samples=4)
    (nll + reg).backward()
    assert torch.isfinite(nll) and layers[0].base_layer.fc_pool.weight.grad.abs().sum() > 0


@pytest.mark.parametrize("red", ["max", "min"])
@pytest.mark.parametrize("msg", ["u_mul_e", "copy_u", "copy_e"])
def test_update_all_with_fn_max_and_min(red, msg):
    import stag_b200 as sb
    fn = sb.function
    src, dst, N, NS, g = make_graph("zero", 53)
    E, D = len(src), 12
    x, w = torch.randn(N, D, device="cuda"), torch.randn(E, D, device="cuda")
    g.ndata["h"], g.edata["w"] = x, w
    mfun = {"u_mul_e": fn.u_mul_e("h", "w", "m"), "copy_u": fn.copy_u("h", "m"), "copy_e": fn.copy_e("w", "m")}[msg]
    g.update_all(mfun, getattr(fn, red)("m", "o"))
    xo = x.cpu() if msg != "copy_e" else torch.ones(N, D)
    wo = None if msg == "copy_u" else w.cpu()
    ref = (ref_max.u_mul_e_max if red == "max" else ref_max.u_mul_e_min)(T(src), T(dst), N, xo, wo)[0]
    assert torch.equal(g.ndata["o"].cpu(), ref)


@pytest.fixture(scope="module")
def arxiv():
    import bench
    import stag_b200 as sb
    src, dst = bench.synth_graph()
    g = sb.Graph(torch.from_numpy(src), torch.from_numpy(dst), bench.N_NODES).to("cuda")
    return src, dst, g, bench.N_NODES, bench.N_EDGES, bench.WIDTH


@pytest.mark.parametrize("generator", ["boxmuller", "hadamard"])
def test_full_size_against_oracle_on_a_row_subset(arxiv, generator):
    """One sample at the arxiv shape; a subset of rows (the 64 largest in-degrees -- hub rows included -- and 2000
    random ones) is checked against the oracle fed the materialised noise of their in-edges."""
    import stag_b200 as sb
    from stag_b200.ops import NoiseSpec
    src, dst, g, N, E, D = arxiv
    spec = NoiseSpec("normal", torch.ones((), device="cuda"), torch.full((), 0.4, device="cuda"), D, E, seed=13,
                     offset=2, n_samples=1, batched=True, generator=generator)
    x = torch.randn(N, D, device="cuda")
    out = sb.ops.stochastic_aggregate(g, x, spec, reduce="max", n_samples=1)
    out_abi, arg = abi_max(g, x, spec_nz(spec), D, 1)
    assert torch.equal(out, out_abi)
    deg = np.bincount(dst, minlength=N)
    rng = np.random.default_rng(0)
    rows = np.unique(np.concatenate([np.argsort(-deg)[:64], rng.integers(0, N, 2000)]))
    assert deg[rows].max() > 128
    sel = np.nonzero(np.isin(dst, rows))[0]
    w = spec.materialize(n_samples=1)[0][T(sel).cuda()].cpu()
    ro, ra = oracle(src[sel], dst[sel], N, x.cpu(), w)
    ra = torch.where(ra >= 0, T(sel)[ra.clamp(min=0)], ra)
    r = T(rows)
    assert torch.equal(out[0].cpu()[r], ro[r])
    assert torch.equal(arg[0].cpu().long()[r], ra[r])
