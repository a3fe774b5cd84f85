"""GPU: the calibration table of stag_calibration (csrc/mc_predictive.cu) equals the numpy oracle
(oracle/ref_calibration.py) bit for bit: every kernel instantiation and class-slice layout, padded row strides, masks,
invalid rows, argmax ties and probabilities on bin edges; tables of row chunks add up to the table of one call; two runs
give the same bits; ``StagModel.calibration`` of a predictive mean; the argument errors."""
import math

import numpy as np
import pytest
import torch

from oracle import ref_calibration as R

pytestmark = pytest.mark.gpu

KINDS = ("categorical", "bernoulli")


def make_rows(kind, N, C, seed, ld=None, ldy=None):
    """probs [N,C] (row stride ld) and labels (int64 [N], or [N,C] with row stride ldy) on the GPU, with hand-made rows:
    1 NaN, 2 zero / out of range, 3 one-hot, 4 a tie, 5 values on bin edges, 6 inf, 7 negative; labels out of range at
    rows 8 and 9 (Categorical), 2.0 at row 8 and fractional values at row 10 (Bernoulli)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    ld, ldy = ld or C, ldy or C
    buf = torch.rand(N * ld + C, device="cuda", generator=g)
    if kind == "categorical":
        buf = buf ** 3
    p = buf.as_strided((N, C), (ld, 1))
    if kind == "categorical":
        y = torch.randint(0, C, (N,), device="cuda", generator=g)
    else:
        ybuf = (torch.rand(N * ldy + C, device="cuda", generator=g) > 0.5).float()
        y = ybuf.as_strided((N, C), (ldy, 1))
    if N > 10:
        p[1, C // 2] = float("nan")
        p[2] = 0.0
        if kind == "bernoulli":
            p[2, C // 2] = 1.5
        p[3] = 0.0
        p[3, C - 1] = 1.0
        p[4] = 0.25                                   # every class tied: the first wins
        p[5] = torch.tensor([0.25, 0.5, 0.0, 1.0], device="cuda").repeat(C)[:C] if kind == "bernoulli" else 0.0
        if kind == "categorical":
            p[5, 0] = 1.0                             # q = 1/4, 1/4, 1/2: on the edges of B = 2, 4, 64
            p[5, 1 % C] += 1.0
            p[5, 2 % C] += 2.0
        p[6, 0] = float("inf")
        p[7, C - 1] = -0.5
        if kind == "categorical":
            y[8], y[9] = C, -1
        else:
            y[8, 0] = 2.0
            y[10] = 0.3
    return p, y


def oracle(p, y, kind, B, mask=None):
    return R.table_fn(p.cpu(), y.cpu(), kind, B, None if mask is None else mask.cpu())


@pytest.mark.parametrize("C", [1, 2, 7, 40, 41, 121, 200, 1024])
@pytest.mark.parametrize("B", [1, 2, 15, 64])
@pytest.mark.parametrize("kind", KINDS)
def test_kernel_table_equals_the_oracle(C, B, kind):
    from stag_b200 import ops
    N = 700
    for padded in (False, True):
        ld, ldy = (C + 3, C + 5) if padded else (None, None)
        p, y = make_rows(kind, N, C, seed=C * 100 + B, ld=ld, ldy=ldy)
        mask = None
        if padded:
            mask = torch.rand(N, device="cuda", generator=torch.Generator(device="cuda").manual_seed(B)) < 0.7
            mask[:12] = True                                   # keep the hand-made rows
        got = ops.calibration_table(p, y, kind, B, mask=mask)
        ref = oracle(p, y, kind, B, mask)
        assert torch.equal(got.cpu(), ref), (C, B, kind, padded, (got.cpu() != ref).nonzero()[:5].flatten().tolist())
        assert int(ref[1]) == (6 if kind == "categorical" else 5) and int(ref[0]) > 0


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("C", [7, 40, 121])
def test_many_rows_per_warp_and_two_runs(kind, C):
    """200 000 rows: every warp walks many rows (the prefetch of the next row) and every CTA flushes once."""
    from stag_b200 import ops
    N, B = 200_000, 15
    p, y = make_rows(kind, N, C, seed=5)
    mask = torch.rand(N, device="cuda", generator=torch.Generator(device="cuda").manual_seed(6)) < 0.7
    a = ops.calibration_table(p, y, kind, B, mask=mask)
    b = ops.calibration_table(p, y, kind, B, mask=mask)
    assert torch.equal(a, b)
    assert torch.equal(a.cpu(), oracle(p, y, kind, B, mask))


@pytest.mark.parametrize("kind", KINDS)
def test_row_chunks_add_up_to_one_call(kind):
    from stag_b200 import ops
    N, C, B = 2000, 41, 15
    p, y = make_rows(kind, N, C, seed=11, ld=C + 2)
    mask = torch.rand(N, device="cuda", generator=torch.Generator(device="cuda").manual_seed(12)) < 0.8
    one = ops.calibration_table(p, y, kind, B, mask=mask)
    for chunk in (1, 7, math.ceil(N / 3)):
        t = torch.zeros_like(one)
        for r0 in range(0, N, chunk):
            assert ops.calibration_table(p[r0:r0 + chunk], y[r0:r0 + chunk], kind, B, mask=mask[r0:r0 + chunk],
                                         out=t) is t
        assert torch.equal(t, one), chunk
    assert torch.equal(one.cpu(), oracle(p, y, kind, B, mask))


def test_empty_and_all_masked_calls_leave_the_table():
    from stag_b200 import ops
    p, y = make_rows("categorical", 50, 9, seed=1)
    t = ops.calibration_table(p, y, n_bins=10, mask=torch.zeros(50, dtype=torch.bool, device="cuda"))
    assert not t.any()
    ops.calibration_table(p[:0], y[:0], n_bins=10, out=t)
    assert not t.any()


# ---- models ---------------------------------------------------------------------------------------------------------
def make_model(kind, D=16, H=32, C=7):
    import stag_b200 as sb
    from stag_b200.layers import StagLayer, FeatOnlyLayer
    torch.manual_seed(2)
    normal = lambda k: torch.distributions.Normal(torch.ones(k), torch.full((k,), 0.5))  # noqa: E731
    head = torch.nn.Softmax(-1) if kind == "categorical" else torch.nn.Sigmoid()
    lik = sb.likelihoods.CategoricalLikelihood() if kind == "categorical" else sb.likelihoods.BernoulliLikelihood()
    layers = [StagLayer(sb.zoo.GCN(D, H, activation=torch.relu), q_a=normal(D)), StagLayer(sb.zoo.GCN(H, C),
                                                                                            q_a=normal(H)),
              FeatOnlyLayer(head)]
    return sb.models.StagModel(torch.nn.ModuleList(layers), likelihood=lik).cuda().eval()


@pytest.mark.parametrize("kind", KINDS)
def test_model_calibration_of_the_predictive_mean(kind):
    import stag_b200 as sb
    from stag_b200.calibration import Calibration
    rng = np.random.default_rng(4)
    N, C = 500, 7
    g = sb.add_self_loop(sb.Graph(torch.from_numpy(rng.integers(0, N, 4000)),
                                  torch.from_numpy(rng.integers(0, N, 4000)), N)).to("cuda")
    model = make_model(kind, C=C)
    x = torch.randn(N, 16, device="cuda")
    y = torch.randint(0, C, (N,), device="cuda") if kind == "categorical" else \
        (torch.rand((N, C), device="cuda") > 0.5).float()
    mask = torch.rand(N, device="cuda") < 0.5
    sb.manual_seed(3)
    mean = model.predictive(g, x, 12, chunk_samples=4).mean
    cal = model.calibration(mean, y, mask=mask)
    assert isinstance(cal, Calibration) and (cal.kind, cal.n_classes, cal.n_bins) == (kind, C, 15)
    assert torch.equal(cal.table.cpu(), oracle(mean, y, kind, 15, mask))
    assert cal.n == int(mask.sum()) and cal.n_invalid == 0
    assert 0.0 <= cal.ece <= 1.0 and 0.0 <= cal.brier <= 2.0
    assert model.calibration(mean, y, n_bins=4).n == N


def test_argument_errors():
    from stag_b200 import ops, StagError, StagLibraryError, _lib
    p, y = make_rows("categorical", 20, 5, seed=2)
    with pytest.raises(StagError) as e:
        ops.calibration_table(torch.rand(3, 1025, device="cuda"), torch.zeros(3, dtype=torch.int64, device="cuda"))
    assert e.value.code == _lib.STAG_EUNSUPPORTED
    for bins in (0, 65):
        with pytest.raises(StagError) as e:
            ops.calibration_table(p, y, n_bins=bins)
        assert e.value.code == _lib.STAG_EINVAL
    with pytest.raises(ValueError):
        ops.calibration_table(p, y[:-1])
    with pytest.raises(ValueError):
        ops.calibration_table(p, y.float())
    with pytest.raises(ValueError):
        ops.calibration_table(p, torch.zeros((20, 4), device="cuda"), "bernoulli")
    with pytest.raises(ValueError):
        ops.calibration_table(p.double(), y)
    with pytest.raises(ValueError):
        ops.calibration_table(p, y, out=torch.zeros(7, dtype=torch.int64, device="cuda"))
    with pytest.raises(StagLibraryError):
        ops.calibration_table(p.cpu(), y.cpu())
    lib = _lib.load()
    assert lib.stag_calibration_table_len(5, 15) == 6 + 45 + 225
    assert lib.stag_calibration(p.data_ptr(), 5, 20, 5, 0, 0, 0, 0, 15, 0, 0) == _lib.STAG_EINVAL   # null pointers
    assert lib.stag_calibration(p.data_ptr(), 4, 20, 5, 0, y.data_ptr(), 0, 0, 15, 0, 0) == _lib.STAG_EINVAL  # ld < C
    t = torch.zeros(276, dtype=torch.int64, device="cuda")
    assert lib.stag_calibration(p.data_ptr(), 5, 2 ** 31, 5, 0, y.data_ptr(), 0, 0, 15, t.data_ptr(), 0) == \
        _lib.STAG_EINVAL                                                                        # N C >= 2^31
