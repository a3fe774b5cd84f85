"""GPU: stag_gemm_tcgen05 (tcgen05.mma kind::tf32, 3xTF32 split, TMEM accumulator) through ops.dense_transform
against a float64 matmul: fp32-level accuracy, fused row scale / bias / relu epilogue, ragged M / K / N, gradients
(also above 256 input channels, and through GCN / SAGE layers of 512 channels) and non-finite inputs.  The route-by-route
ABI tests are in test_gpu_gemm_routes.py."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def rel(a, b):
    return float((a.double().cpu() - b.double().cpu()).abs().max() / b.double().abs().max().clamp(min=1e-30))


@pytest.mark.parametrize("M,K,N", [(1, 8, 16), (127, 16, 7), (128, 32, 16), (129, 50, 40), (1000, 128, 128),
                                   (5000, 128, 40), (300, 1433, 16), (4096, 256, 256), (777, 100, 121),
                                   (64, 9, 16), (2049, 33, 200)])
def test_matches_float64(M, K, N):
    from stag_b200 import ops
    g = torch.Generator().manual_seed(M + K + N)
    a = torch.randn(M, K, generator=g).cuda()
    w = torch.randn(K, N, generator=g).cuda()
    out = ops.dense_transform(a, w)
    ref = a.double() @ w.double()
    assert out.shape == (M, N)
    assert rel(out, ref) < 1e-5, rel(out, ref)


def test_epilogue_and_batched_samples():
    from stag_b200 import ops
    g = torch.Generator().manual_seed(0)
    S, N, K, C = 3, 500, 64, 40
    a = torch.randn(S, N, K, generator=g).cuda()
    w = torch.randn(K, C, generator=g).cuda()
    b = torch.randn(C, generator=g).cuda()
    rs = torch.rand(N, generator=g).cuda() + 0.5
    out = ops.dense_transform(a, w, row_scale=rs, bias=b, relu=True)
    ref = torch.relu((a.double() @ w.double()) * rs.double()[None, :, None] + b.double())
    assert out.shape == (S, N, C)
    assert rel(out, ref) < 1e-5


@pytest.mark.parametrize("M,K,N", [(2708, 1433, 16), (2708, 1433, 7), (500, 999, 33), (1300, 640, 64), (130, 4100, 40)])
def test_split_k_cluster(M, K, N):
    """Few row tiles and a long K (Cora's first layer): K is split over a thread-block cluster and the partial
    accumulators are added in rank 0's shared memory in rank order -- fp32-level accuracy, the fused epilogue
    still applied once, bitwise run-to-run."""
    from stag_b200 import ops
    g = torch.Generator().manual_seed(M + K + N)
    a = torch.randn(M, K, generator=g).cuda()
    w = torch.randn(K, N, generator=g).cuda()
    b = torch.randn(N, generator=g).cuda()
    rs = (torch.rand(M, generator=g) + 0.5).cuda()
    out = ops.dense_transform(a, w, row_scale=rs, bias=b, relu=True)
    ref = torch.relu((a.double() @ w.double()) * rs.double()[:, None] + b.double())
    assert rel(out, ref) < 1e-5, rel(out, ref)
    assert torch.equal(out, ops.dense_transform(a, w, row_scale=rs, bias=b, relu=True))
    plain = ops.dense_transform(a, w)
    assert rel(plain, a.double() @ w.double()) < 1e-5


@pytest.mark.parametrize("M,K,N", [(300001, 128, 128), (300001, 128, 40), (250000, 160, 64), (200003, 100, 121),
                                   (190000, 96, 16), (150000, 32, 256), (400000, 64, 7), (169343 * 4, 128, 128)])
def test_persistent_tma_form_many_tiles_per_cta(M, K, N):
    """Row counts far beyond 148 x 128: every CTA of the persistent TMA form walks many row tiles, so its rings (sizes that
    do not divide the K blocks of a tile), both TMEM accumulators and every mbarrier phase wrap many times.  Ragged M,
    K tails filled by the TMA unit, N from one MMA column block to the 256-column maximum; fused epilogue; elementwise
    tolerance against float64; bitwise run-to-run."""
    from stag_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(M + K + N)
    a = torch.randn(M, K, generator=g, device="cuda")
    w = torch.randn(K, N, generator=g, device="cuda")
    b = torch.randn(N, generator=g, device="cuda")
    rs = torch.rand(M, generator=g, device="cuda") + 0.5
    out = ops.dense_transform(a, w, row_scale=rs, bias=b, relu=True)
    ref = torch.relu((a.double() @ w.double()) * rs.double()[:, None] + b.double())
    scale = float(ref.abs().max())
    assert bool(((out.double() - ref).abs() <= 1e-5 * ref.abs() + 2e-6 * scale).all())
    assert torch.equal(out, ops.dense_transform(a, w, row_scale=rs, bias=b, relu=True))
    del out, ref
    plain = ops.dense_transform(a, w)
    ref = a.double() @ w.double()
    assert bool(((plain.double() - ref).abs() <= 1e-5 * ref.abs() + 2e-6 * float(ref.abs().max())).all())


def test_gradients():
    from stag_b200 import ops
    g = torch.Generator().manual_seed(1)
    a = torch.randn(700, 48, generator=g).cuda().requires_grad_(True)
    w = torch.randn(48, 24, generator=g).cuda().requires_grad_(True)
    b = torch.randn(24, generator=g).cuda().requires_grad_(True)
    rs = (torch.rand(700, generator=g) + 0.5).cuda()
    go = torch.randn(700, 24, generator=g).cuda()
    ops.dense_transform(a, w, row_scale=rs, bias=b, relu=True).backward(go)
    a2, w2, b2 = [t.detach().double().requires_grad_(True) for t in (a, w, b)]
    torch.relu((a2 @ w2) * rs.double()[:, None] + b2).backward(go.double())
    assert rel(a.grad, a2.grad) < 1e-5 and rel(w.grad, w2.grad) < 1e-5 and rel(b.grad, b2.grad) < 1e-5


def test_unsupported_width_falls_to_cublas_in_python_only():
    """Nout > 256 is refused by the C entry point (STAG_EUNSUPPORTED) and routed to torch.matmul above it."""
    import ctypes
    from stag_b200 import _lib, ops
    lib = _lib.load()
    a = torch.randn(10, 8).cuda()
    wt = torch.randn(300, 8).cuda()
    out = torch.empty(10, 300).cuda()
    rc = lib.stag_gemm_tcgen05(a.data_ptr(), 8, wt.data_ptr(), 8, 10, 300, 8, 0, 0, 0, out.data_ptr(), 300, 0, 0, 0)
    assert rc == _lib.STAG_EUNSUPPORTED
    assert ops.dense_transform(a, wt.t().contiguous()).shape == (10, 300)


# ---------------------------------------------------------------------------------------------------------------------
# per-element bounds against float64 (oracle/ref_gemm.py): |got - ref| <= 2^-17 x the same sum over absolute values
def _within(got, ref, scale, what, bound=2.0 ** -17):
    got, ref, scale = (t.detach().double().cpu() for t in (got, ref, scale))
    bad = ~((got - ref).abs() <= bound * scale)
    assert not bool(bad.any()), "%s: %d of %d entries beyond the bound" % (what, int(bad.sum()), bad.numel())


@pytest.mark.parametrize("transposed", [False, True])
@pytest.mark.parametrize("K", [257, 300, 512, 1433])
def test_gradients_above_256_input_channels(K, transposed):
    """dA = g W^T has K output columns: above 256 it runs on 256-row slices of W, each into its columns of dA.
    S-batched [S, N, K] input, [N] row scale shared by the samples, bias, relu; dA, dW and dbias against float64."""
    from stag_b200 import ops
    g = torch.Generator().manual_seed(K + transposed)
    S, N, C = 2, 300, 40
    a = torch.randn(S, N, K, generator=g).cuda().requires_grad_(True)
    w0 = torch.randn(K, C, generator=g) / K ** 0.5
    w = (w0.t().contiguous() if transposed else w0).cuda().requires_grad_(True)
    b = torch.randn(C, generator=g).cuda().requires_grad_(True)
    rs = (torch.rand(N, generator=g) + 0.5).cuda()
    go = torch.randn(S, N, C, generator=g).cuda()
    out = ops.dense_transform(a, w, row_scale=rs, bias=b, relu=True, transposed=transposed)
    out.backward(go)
    ad, wd, rsd = a.detach().double().cpu(), w0.double(), rs.double().cpu()[None, :, None]
    ref = (ad @ wd) * rsd + b.detach().double().cpu()
    _within(out, ref.clamp(min=0), (ad.abs() @ wd.abs()) * rsd + b.detach().double().cpu().abs(), "out")
    # the relu mask of the kernel's own output: the backward is checked, not the sign of entries near 0
    ge = go.double().cpu() * (out.detach().double().cpu() > 0)
    gs = ge * rsd
    _within(a.grad, gs @ wd.t(), gs.abs() @ wd.abs().t(), "dA")
    gw = (ad.reshape(-1, K).t() @ gs.reshape(-1, C))
    gw_scale = ad.reshape(-1, K).abs().t() @ gs.reshape(-1, C).abs()
    _within(w.grad, gw.t() if transposed else gw, gw_scale.t() if transposed else gw_scale, "dW")
    _within(b.grad, ge.sum((0, 1)), ge.abs().sum((0, 1)), "dbias")


def _graph(N, E, seed):
    import stag_b200 as sb
    rng = np.random.default_rng(seed)
    src, dst = rng.integers(0, N, E), rng.integers(0, N, E)
    return sb.Graph(torch.from_numpy(src), torch.from_numpy(dst), N).to("cuda"), src, dst


def _agg(src, dst, N, x, scale_src=None, scale_dst=None):
    """float64 sum over in-edges with optional per-node scales (the aggregation of GCN / SAGE 'mean')."""
    if scale_src is not None:
        x = x * scale_src[:, None]
    out = torch.zeros((N,) + x.shape[1:], dtype=x.dtype).index_add(0, torch.from_numpy(dst), x[torch.from_numpy(src)])
    return out if scale_dst is None else out * scale_dst[:, None]


def _step_check(params, ref_fn, inputs, go, what):
    """Gradients of the model (params, already backpropagated) against float64 autograd of ref_fn, per element within
    2^-15 of the same gradient taken over absolute values (a chain of two GEMMs and two aggregations)."""
    def grads(absolute):
        ts = [p.detach().double().cpu() for p in params]
        xs = [x.detach().double().cpu() for x in inputs]
        gg = go.double().cpu()
        if absolute:
            ts, xs, gg = [t.abs() for t in ts], [x.abs() for x in xs], gg.abs()
        ts = [t.requires_grad_(True) for t in ts]
        (ref_fn(ts, xs) * gg).sum().backward()
        return [t.grad for t in ts]
    for p, r, s in zip(params, grads(False), grads(True)):
        assert p.grad is not None and bool(torch.isfinite(p.grad).all())
        _within(p.grad, r, s, what, bound=2.0 ** -15)


def test_gcn_training_step_through_512_hidden_channels():
    """GCN(300 -> 512) then GCN(512 -> 40): the second layer's input needs a gradient through K = 512."""
    import stag_b200 as sb
    torch.manual_seed(0)
    N, E = 400, 4000
    G, src, dst = _graph(N, E, 1)
    l1, l2 = sb.zoo.GCN(300, 512).cuda(), sb.zoo.GCN(512, 40).cuda()
    for m in (l1, l2):
        torch.nn.init.normal_(m.bias)
    x = torch.randn(N, 300).cuda()
    go = torch.randn(N, 40).cuda()
    params = [l1.weight, l1.bias, l2.weight, l2.bias]
    opt = torch.optim.SGD(params, lr=0.1)
    opt.zero_grad()
    out = l2(G, l1(G, x))
    out.backward(go)
    ss, ds = (G._s.scale(k, "rsqrt").double().cpu() for k in (False, True))

    def ref(ts, xs):
        w1, b1, w2, b2 = ts
        h = _agg(src, dst, N, xs[0], ss, ds) @ w1 + b1
        return _agg(src, dst, N, h, ss, ds) @ w2 + b2
    _step_check(params, ref, [x], go, "GCN 300 -> 512 -> 40")
    before = l2.weight.detach().clone()
    opt.step()
    assert not torch.equal(before, l2.weight.detach())


def test_sage_layer_with_512_input_channels():
    import stag_b200 as sb
    torch.manual_seed(1)
    N, E = 400, 4000
    G, src, dst = _graph(N, E, 2)
    layer = sb.zoo.GraphSAGE(512, 40, aggregator_type="mean").cuda()
    torch.nn.init.normal_(layer.bias)
    x = torch.randn(N, 512).cuda().requires_grad_(True)
    go = torch.randn(N, 40).cuda()
    params = [layer.fc_self.weight, layer.fc_neigh.weight, layer.bias, x]
    layer(G, x).backward(go)
    inv = G._s.scale(True, "inv").double().cpu()

    def ref(ts, xs):
        ws, wn, b, xx = ts
        return xx @ ws.t() + _agg(src, dst, N, xx, None, inv) @ wn.t() + b
    _step_check(params, ref, [], go, "SAGE mean 512 -> 40")


def _nonfinite_inputs(M, K, N, seed):
    g = torch.Generator().manual_seed(seed)
    a = torch.randn(M, K, generator=g)
    w = torch.randn(K, N, generator=g)
    b = torch.randn(N, generator=g)
    a[3, 5], a[7, 0], a[M - 1, K - 1] = float("nan"), float("inf"), float("-inf")
    w[K - 1, 2], w[1, N - 1] = float("nan"), float("inf")
    return a, w, b, [3, 7, M - 1], [2, N - 1]


@pytest.mark.parametrize("form", [1, 2])
@pytest.mark.parametrize("relu", [False, True])
def test_nan_and_inf_rows_and_columns(form, relu):
    """NaN / +-Inf in row i of A -> NaN in all of out row i; in column j of W -> NaN in all of out column j; relu keeps
    NaN (as torch.relu); every other entry within the bound.  Form 1 is reached through an A that is not 16-byte
    aligned, form 2 through an aligned one (the kernel of each layout is asserted in test_gpu_gemm_routes.py)."""
    from oracle import ref_gemm
    from stag_b200 import ops
    M, K, N = 300, 100, 40
    a, w, b, rows, cols = _nonfinite_inputs(M, K, N, form)
    buf = torch.empty(M * K + 4, device="cuda")
    off = 0 if form == 2 else 1
    ac = buf[off:off + M * K].view(M, K)
    ac.copy_(a)
    out = ops.dense_transform(ac, w.cuda(), bias=b.cuda(), relu=relu).cpu().double().numpy()
    assert np.isnan(out[rows]).all() and np.isnan(out[:, cols]).all()
    kr, kc = np.setdiff1d(np.arange(M), rows), np.setdiff1d(np.arange(N), cols)
    a2, w2, b2 = a.numpy()[kr], w.numpy()[:, kc], b.numpy()[kc]
    assert ref_gemm.violations(out[np.ix_(kr, kc)], ref_gemm.reference(a2, w2, None, b2, relu),
                               ref_gemm.bound(a2, w2, None, b2)) == 0


def test_nan_agrees_with_the_wide_output_branch():
    """Nout > 256 runs on torch.matmul; relu of a NaN row is NaN on both sides of the 256 limit."""
    from stag_b200 import ops
    a, w, b, rows, _ = _nonfinite_inputs(200, 64, 300, 5)
    a[:, :], w[:, :] = torch.nan_to_num(a, posinf=1.0, neginf=-1.0), torch.nan_to_num(w, posinf=1.0, neginf=-1.0)
    a[rows] = float("nan")
    a, w, b = a.cuda(), w.cuda(), b.cuda()
    wide = ops.dense_transform(a, w, bias=b, relu=True)
    narrow = ops.dense_transform(a, w[:, :256].contiguous(), bias=b[:256].contiguous(), relu=True)
    for out in (wide, narrow):
        nan_rows = torch.isnan(out).all(1).nonzero().flatten().tolist()
        assert nan_rows == rows and not bool(torch.isnan(out[[i for i in range(200) if i not in rows]]).any())
