"""CPU: the max-aggregation oracle against a brute-force loop, the public surface of GraphSAGE 'pool' / GIN 'max' /
fn.max, and the argument checks of the operator and of the C ABI (no device needed)."""
import ctypes
import os
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT
from oracle import ref_max


def brute_max(src, dst, N, x, w):
    """Python loop over the edges in id order: strict > keeps the first winner; empty rows 0 / -1."""
    D = x.shape[1]
    out = np.zeros((N, D))
    arg = -np.ones((N, D), dtype=np.int64)
    for e in range(len(src)):
        for c in range(D):
            m = float(x[src[e], c]) * float(w[e, c] if w.shape[1] > 1 else w[e, 0])
            v = dst[e]
            if arg[v, c] < 0 or m > out[v, c]:
                out[v, c], arg[v, c] = m, e
    return out, arg


def tie_graph(seed, N=12, E=60, D=5, K=5):
    rng = np.random.default_rng(seed)
    src, dst = rng.integers(0, N, E), rng.integers(0, N - 3, E)   # the last three rows have no in-edges
    x = rng.integers(-2, 3, (N, D)).astype(np.float64)             # small integers: many ties, negative messages
    x[3] = x[5]                                                     # duplicate rows
    w = rng.integers(0, 3, (E, K)).astype(np.float64)               # zeros as Bernoulli noise makes them
    return src, dst, N, x, w


@pytest.mark.parametrize("seed,K", [(0, 5), (1, 1), (2, 5)])
def test_oracle_max_matches_brute_force_with_ties(seed, K):
    src, dst, N, x, w = tie_graph(seed, K=K)
    out, arg = ref_max.u_mul_e_max(torch.from_numpy(src), torch.from_numpy(dst), N, torch.from_numpy(x),
                                   torch.from_numpy(w))
    bo, ba = brute_max(src, dst, N, x, w)
    assert np.array_equal(arg.numpy(), ba)
    assert np.array_equal(out.numpy(), bo)
    assert (arg[N - 3:] == -1).all() and (out[N - 3:] == 0).all()


def test_oracle_max_gradient_lands_on_the_first_winner():
    src, dst, N, x, w = tie_graph(3)
    xt = torch.from_numpy(x).requires_grad_(True)
    wt = torch.from_numpy(w).requires_grad_(True)
    out, arg = ref_max.u_mul_e_max(torch.from_numpy(src), torch.from_numpy(dst), N, xt, wt)
    G = torch.from_numpy(np.random.default_rng(4).standard_normal(out.shape))
    (out * G).sum().backward()
    dx, dw = np.zeros_like(x), np.zeros_like(w)
    a = arg.numpy()
    for v in range(N):
        for c in range(x.shape[1]):
            e = a[v, c]
            if e >= 0:
                dx[src[e], c] += w[e, c] * G[v, c].item()
                dw[e, c] += x[src[e], c] * G[v, c].item()
    assert np.allclose(xt.grad.numpy(), dx) and np.allclose(wt.grad.numpy(), dw)


def test_oracle_max_gradient_by_finite_differences():
    """Away from ties (continuous random data) the gather-at-arg gradient is the derivative."""
    rng = np.random.default_rng(5)
    N, E, D = 9, 40, 4
    src, dst = torch.from_numpy(rng.integers(0, N, E)), torch.from_numpy(rng.integers(0, N - 1, E))
    x = torch.from_numpy(rng.standard_normal((N, D))).requires_grad_(True)
    w = torch.from_numpy(rng.standard_normal((E, D))).requires_grad_(True)
    assert torch.autograd.gradcheck(lambda a, b: ref_max.u_mul_e_max(src, dst, N, a, b)[0], (x, w))
    assert torch.autograd.gradcheck(lambda a, b: ref_max.u_mul_e_min(src, dst, N, a, b)[0], (x, w))


def test_oracle_min_takes_the_first_minimum():
    src, dst, N, x, w = tie_graph(6)
    out, arg = ref_max.u_mul_e_min(torch.from_numpy(src), torch.from_numpy(dst), N, torch.from_numpy(x),
                                   torch.from_numpy(w))
    bo, ba = brute_max(src, dst, N, -x, w)
    assert np.array_equal(arg.numpy(), ba) and np.array_equal(out.numpy(), -bo)


def test_sage_pool_has_the_sageconv_parameters():
    import stag_b200 as sb
    sys.path.insert(0, os.path.join(ROOT, "oracle", "dgl_shim"))
    try:
        import dgl.nn as dglnn
    finally:
        sys.path.pop(0)
    ours, ref = sb.zoo.GraphSAGE(8, 4, aggregator_type="pool"), dglnn.SAGEConv(8, 4, "pool")
    assert {k: tuple(v.shape) for k, v in ours.state_dict().items()} == \
        {k: tuple(v.shape) for k, v in ref.state_dict().items()}
    assert sorted(ours.state_dict()) == ["bias", "fc_neigh.weight", "fc_pool.bias", "fc_pool.weight", "fc_self.weight"]
    ours.load_state_dict(ref.state_dict())
    for k, v in ref.state_dict().items():
        assert torch.equal(ours.state_dict()[k], v)
    # xavier with the relu gain, as SAGEConv.reset_parameters
    bound = torch.nn.init.calculate_gain("relu") * (6.0 / 16) ** 0.5
    assert ours.fc_pool.weight.abs().max() <= bound


def test_gin_max_constructs_and_lstm_still_raises():
    import stag_b200 as sb
    m = sb.zoo.GIN(8, 4, aggregator_type="max")
    assert sorted(m.state_dict()) == ["apply_func.bias", "apply_func.weight", "eps"]
    with pytest.raises(NotImplementedError, match="lstm"):
        sb.zoo.GraphSAGE(8, 4, aggregator_type="lstm")
    with pytest.raises(NotImplementedError):
        sb.zoo.GIN(8, 4, aggregator_type="lstm")


def test_operator_rejects_scales_with_max_and_bad_reduce_names():
    import stag_b200 as sb
    g = sb.rand_graph(5, 20)
    x = torch.randn(5, 8)
    for red in ("max", "min"):
        with pytest.raises(ValueError, match="scale"):
            sb.ops.stochastic_aggregate(g, x, None, reduce=red, src_scale=torch.ones(5))
        with pytest.raises(ValueError, match="scale"):
            sb.ops.stochastic_aggregate(g, x, None, reduce=red, dst_scale=torch.ones(5))
    with pytest.raises(ValueError, match="reduce"):
        sb.ops.stochastic_aggregate(g, x, None, reduce="amax")
    with pytest.raises(NotImplementedError):
        sb.function.run(g, sb.function.copy_u("h", "m"), sb.function.Reduce("lstm", "m", "h"))


def test_abi_rejects_in_norm_and_edge_channel_parameters_with_max(lib):
    from stag_b200 import _lib
    g = _lib.StagGraph()
    g.num_rows, g.num_cols, g.num_edges = 4, 4, 0
    g.indptr = 16  # never dereferenced: the checks come first
    base = dict(kind=_lib.NOISE_NORMAL, K=4, param_shape=_lib.PARAM_SCALAR, p0=16, p1=16)
    for extra in (dict(in_norm=1), dict(param_shape=_lib.PARAM_EDGE_CHANNEL)):
        n = _lib.StagNoise(**{**base, **extra})
        rc = lib.stag_spmm_max_fwd(ctypes.byref(g), 16, 4, 0, 4, 1, ctypes.byref(n), 16, 16, 4, 0, 0, 0, 0)
        assert rc == _lib.STAG_EINVAL, extra
        rc = lib.stag_spmm_max_bwd(ctypes.byref(g), 16, 4, 0, 16, 16, 4, 0, 4, 1, ctypes.byref(n), 16, 4, 0,
                                   0, 0, 0, 0, 0, 0)
        assert rc == _lib.STAG_EINVAL, extra
        assert lib.stag_last_error()
    n = _lib.StagNoise(**base)
    assert lib.stag_spmm_max_fwd(ctypes.byref(g), 16, 4, 0, 4, 1, ctypes.byref(n), 16, 0, 4, 0, 0, 0, 0) == \
        _lib.STAG_EINVAL  # null arg output
