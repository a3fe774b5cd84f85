"""CPU: the numpy oracle of the calibration table (oracle/ref_calibration.py) against sklearn and explicit formulas, the
metrics of ``stag_b200.calibration.Calibration`` on hand-made rows, exact addition of tables over row splits, the
reduction of tables over ranks (gloo, world size 2, the oracle in place of the kernel), and the argument checks that
need no device."""
import math
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import ref_calibration as R

NAN = float("nan")


def calib(probs, y, kind, n_bins=15, mask=None):
    from stag_b200.calibration import calibration
    return calibration(torch.as_tensor(probs), torch.as_tensor(y), kind, n_bins, mask, table_fn=R.table_fn)


def random_rows(kind, N, C, seed):
    rng = np.random.default_rng(seed)
    if kind == "categorical":
        probs = (rng.random((N, C)) ** 3).astype(np.float32)      # unnormalised: the table renormalises
        return probs, rng.integers(0, C, N)
    probs = rng.random((N, C)).astype(np.float32)
    return probs, (rng.random((N, C)) < probs).astype(np.float32)


def renormalised(probs):
    m = probs.astype(np.float64)
    return m / R.row_sum(m)[:, None]


METRICS = ("brier", "ece", "mce", "classwise_ece")


def all_nan(cal):
    vals = [getattr(cal, k) for k in METRICS] + [cal.accuracy if cal.kind == "categorical" else cal.micro_f1]
    rel = cal.reliability()
    return all(math.isnan(v) for v in vals) and bool(torch.isnan(rel.confidence).all() and torch.isnan(rel.frequency).all())


# ---- the oracle against sklearn and explicit formulas ---------------------------------------------------------------
@pytest.mark.parametrize("n_bins", [1, 2, 10, 15, 64])
def test_categorical_matches_sklearn(n_bins):
    skm = pytest.importorskip("sklearn.metrics")
    from sklearn.calibration import calibration_curve
    N, C = 700, 7
    probs, y = random_rows("categorical", N, C, seed=n_bins)
    cal = calib(probs, y, "categorical", n_bins)
    q = renormalised(probs)
    k = probs.argmax(1)
    conf, correct = q[np.arange(N), k], (k == y).astype(np.float64)
    assert cal.n == N and cal.n_invalid == 0
    assert cal.accuracy == pytest.approx(skm.accuracy_score(y, k), abs=1e-15)
    prob_true, prob_pred = calibration_curve(correct, conf, n_bins=n_bins, strategy="uniform")
    rel = cal.reliability()
    full = rel.counts > 0
    np.testing.assert_allclose(rel.frequency[full].numpy(), prob_true, rtol=0, atol=1e-9)
    np.testing.assert_allclose(rel.confidence[full].numpy(), prob_pred, rtol=0, atol=1e-9)
    np.testing.assert_array_equal(rel.edges.numpy(), np.linspace(0, 1, n_bins + 1))
    onehot = np.eye(C)[y]
    assert cal.brier == pytest.approx(((q - onehot) ** 2).sum(1).mean(), abs=1e-9)
    b = np.searchsorted(np.linspace(0, 1, n_bins + 1)[1:-1], conf)
    gaps = np.array([abs(correct[b == i].sum() - conf[b == i].sum()) for i in range(n_bins)])
    counts = np.bincount(b, minlength=n_bins)
    assert cal.ece == pytest.approx(gaps.sum() / N, abs=1e-9)
    assert cal.mce == pytest.approx((gaps[counts > 0] / counts[counts > 0]).max(), abs=1e-9)
    bc = np.searchsorted(np.linspace(0, 1, n_bins + 1)[1:-1], q)
    cw = sum(abs(onehot[:, c][bc[:, c] == i].sum() - q[:, c][bc[:, c] == i].sum())
             for c in range(C) for i in range(n_bins))
    assert cal.classwise_ece == pytest.approx(cw / N / C, abs=1e-9)


@pytest.mark.parametrize("n_bins", [1, 3, 15, 64])
def test_bernoulli_matches_sklearn(n_bins):
    skm = pytest.importorskip("sklearn.metrics")
    from sklearn.calibration import calibration_curve
    N, C = 400, 9
    probs, y = random_rows("bernoulli", N, C, seed=100 + n_bins)
    cal = calib(probs, y, "bernoulli", n_bins)
    p, t = probs.astype(np.float64), y.astype(np.float64)
    assert cal.n == N and cal.n_invalid == 0
    assert cal.micro_f1 == pytest.approx(skm.f1_score(y.astype(int), (probs > 0.5).astype(int), average="micro"),
                                         abs=1e-15)
    prob_true, prob_pred = calibration_curve(t.ravel(), p.ravel(), n_bins=n_bins, strategy="uniform")
    rel = cal.reliability()
    full = rel.counts > 0
    np.testing.assert_allclose(rel.frequency[full].numpy(), prob_true, rtol=0, atol=1e-9)
    np.testing.assert_allclose(rel.confidence[full].numpy(), prob_pred, rtol=0, atol=1e-9)
    assert int(rel.counts.sum()) == N * C
    assert cal.brier == pytest.approx(((p - t) ** 2).mean(), abs=1e-9)
    b = np.searchsorted(np.linspace(0, 1, n_bins + 1)[1:-1], p)
    gaps = np.array([abs(t[b == i].sum() - p[b == i].sum()) for i in range(n_bins)])
    assert cal.ece == pytest.approx(gaps.sum() / (N * C), abs=1e-9)
    cw = sum(abs(t[:, c][b[:, c] == i].sum() - p[:, c][b[:, c] == i].sum()) for c in range(C) for i in range(n_bins))
    assert cal.classwise_ece == pytest.approx(cw / N / C, abs=1e-9)


def test_row_sum_follows_the_warp_order():
    """Lane l adds classes l, l+32, ... in order, then the xor butterfly: checked against an explicit lane loop."""
    rng = np.random.default_rng(3)
    m = (rng.random((5, 77)) * 10.0 ** rng.integers(-8, 8, (5, 77))).astype(np.float32).astype(np.float64)
    for r in range(5):
        lanes = [0.0] * 32
        for c in range(77):
            lanes[c % 32] = lanes[c % 32] + m[r, c]
        for o in (16, 8, 4, 2, 1):
            lanes = [lanes[i] + lanes[i ^ o] for i in range(32)]
        assert R.row_sum(m[r:r + 1])[0] == lanes[0]


def test_edges_are_linspace_values_not_i_over_b():
    """An interior edge is i * (1.0 / B), the double np.linspace makes; where it lies below i / B, a probability of
    exactly i / B is above the edge and falls in bin i, as sklearn bins it."""
    found = 0
    for B in range(2, 101):
        for i in range(1, B):
            if i * (1.0 / B) < i / B:
                # class 0 of the row [i, B - i] has q = i / B, the double nearest to it (s = B exactly)
                t = R.table(np.array([[i, B - i]], np.float32), np.array([1]), "categorical", B)
                cls = t[R.HEAD + 3 * B:].reshape(3, 2, B)
                assert cls[0, 0, i] == 1, (B, i)
                assert np.searchsorted(np.linspace(0, 1, B + 1)[1:-1], i / B) == i
                found += 1
    assert found > 0


# ---- hand-made rows ---------------------------------------------------------------------------------------------------
def test_confidence_on_an_edge_and_one_hot_rows():
    cal = calib(np.array([[0.5, 0.5]], np.float32), [0], "categorical", n_bins=2)
    rel = cal.reliability()
    assert rel.counts.tolist() == [1, 0]                       # 0.5 is not above the edge 0.5: bin 0 = [0, 0.5]
    cal = calib(np.array([[0.0, 1.0, 0.0]], np.float32), [1], "categorical", n_bins=10)
    assert cal.reliability().counts.tolist() == [0] * 9 + [1]
    assert cal.accuracy == 1.0 and cal.brier == 0.0 and cal.ece == 0.0
    cls = cal.table[R.HEAD + 30:].view(3, 3, 10)
    assert cls[0, 0].tolist() == [1] + [0] * 9                 # q = 0 falls in bin 0
    assert cls[0, 1].tolist() == [0] * 9 + [1]
    assert cls[1, 1, 9] == 2 ** 32 and cls[2, 1, 9] == 1
    cal = calib(np.array([[0.0, 1.0, 0.5]], np.float32), np.array([[0.0, 1.0, 1.0]], np.float32), "bernoulli", 2)
    cls = cal.table[R.HEAD + 6:].view(3, 3, 2)
    assert cls[0].tolist() == [[1, 0], [0, 1], [1, 0]]
    assert cal.table[:6].tolist() == [1, 0, 1, 0, 1, int(0.25 * 2 ** 32)]   # tp, fp, fn; 0.5 is not > 0.5


def test_argmax_ties_go_to_the_first_class():
    probs = np.array([[0.4, 0.2, 0.4], [0.1, 0.45, 0.45], [0.25, 0.25, 0.25]], np.float32)
    assert calib(probs, [0, 1, 0], "categorical").accuracy == 1.0
    assert calib(probs, [2, 2, 2], "categorical").accuracy == 0.0
    wide = np.zeros((1, 70), np.float32)
    wide[0, [5, 37, 69]] = 0.3                                 # tied classes held by lanes 5, 5 and 5 (slots 0, 1, 2)
    assert calib(wide, [5], "categorical").accuracy == 1.0
    wide[0, 5] = 0.0
    wide[0, 36] = 0.3                                          # lanes 4 and 5: the lower class wins
    assert calib(wide, [36], "categorical").accuracy == 1.0


CAT_INVALID = [([NAN, 0.5, 0.5], 0), ([float("inf"), 0.5, 0.5], 0), ([-0.1, 0.5, 0.6], 1), ([0.0, 0.0, 0.0], 0),
               ([0.2, 0.3, 0.5], -1), ([0.2, 0.3, 0.5], 3)]
BERN_INVALID = [([NAN, 0.5], [0.0, 1.0]), ([1.5, 0.5], [0.0, 1.0]), ([-0.5, 0.5], [0.0, 1.0]),
                ([0.5, 0.5], [NAN, 1.0]), ([0.5, 0.5], [2.0, 1.0]), ([0.5, float("inf")], [0.0, 1.0])]


@pytest.mark.parametrize("case", range(len(CAT_INVALID)))
def test_each_invalid_categorical_row_counts_once(case):
    row, label = CAT_INVALID[case]
    good = np.array([[0.1, 0.7, 0.2], [0.6, 0.3, 0.1]], np.float32)
    probs = np.concatenate([good, np.array([row], np.float32)])
    cal = calib(probs, [1, 0, label], "categorical")
    assert cal.n == 2 and cal.n_invalid == 1 and all_nan(cal)
    # the refused row enters no other entry
    ref = calib(good, [1, 0], "categorical").table
    assert torch.equal(cal.table[2:], ref[2:])


@pytest.mark.parametrize("case", range(len(BERN_INVALID)))
def test_each_invalid_bernoulli_row_counts_once(case):
    row, label = BERN_INVALID[case]
    good_p, good_y = np.array([[0.1, 0.7]], np.float32), np.array([[0.0, 1.0]], np.float32)
    cal = calib(np.concatenate([good_p, np.array([row], np.float32)]),
                np.concatenate([good_y, np.array([label], np.float32)]), "bernoulli")
    assert cal.n == 1 and cal.n_invalid == 1 and all_nan(cal)
    assert torch.equal(cal.table[2:], calib(good_p, good_y, "bernoulli").table[2:])


def test_all_masked_gives_a_zero_table_and_nan_metrics():
    probs, y = random_rows("categorical", 20, 4, seed=1)
    cal = calib(probs, y, "categorical", mask=torch.zeros(20, dtype=torch.bool))
    assert not cal.table.any() and all_nan(cal)
    # a masked-out row is not read: its NaN does not count
    probs[3] = NAN
    mask = torch.ones(20, dtype=torch.bool)
    mask[3] = False
    cal = calib(probs, y, "categorical", mask=mask)
    assert cal.n == 19 and cal.n_invalid == 0


# ---- exact addition ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["categorical", "bernoulli"])
def test_tables_of_row_splits_add_to_the_whole(kind):
    N, C, B = 301, 13, 15
    probs, y = random_rows(kind, N, C, seed=7)
    whole = calib(probs, y, kind, B)
    for cuts in ([0, 1, N], [0, 100, 200, N], list(range(0, N, 7)) + [N]):
        parts = [calib(probs[a:b], y[a:b], kind, B) for a, b in zip(cuts[:-1], cuts[1:])]
        total = parts[0]
        for p in parts[1:]:
            total = total + p
        assert torch.equal(total.table, whole.table)
    assert whole.ece == total.ece
    assert torch.equal(whole.reliability().confidence.nan_to_num(7.0), total.reliability().confidence.nan_to_num(7.0))


def test_add_refuses_mismatched_tables():
    from stag_b200.calibration import Calibration
    a = calib(*random_rows("categorical", 5, 4, 0), "categorical", 15)
    with pytest.raises(ValueError):
        a + calib(*random_rows("categorical", 5, 4, 0), "categorical", 10)
    with pytest.raises(ValueError):
        a + calib(*random_rows("categorical", 5, 3, 0), "categorical", 15)
    with pytest.raises(ValueError):
        a + Calibration("bernoulli", 4, 15, a.table.clone())
    with pytest.raises(ValueError):
        Calibration("categorical", 4, 15, a.table[:-1])
    with pytest.raises(ValueError):
        a.micro_f1
    with pytest.raises(ValueError):
        calib(*random_rows("bernoulli", 5, 4, 0), "bernoulli").accuracy


# ---- no device --------------------------------------------------------------------------------------------------------
def test_ops_and_model_refuse_what_they_cannot_run():
    import stag_b200 as sb
    from stag_b200 import ops, StagLibraryError
    with pytest.raises(StagLibraryError):
        ops.calibration_table(torch.rand(4, 3), torch.zeros(4, dtype=torch.int64))
    with pytest.raises(StagLibraryError):
        sb.calibration.calibration(torch.rand(4, 3), torch.zeros(4, dtype=torch.int64), "categorical")

    class Poisson(sb.likelihoods.Likelihood):
        def __init__(self):
            super().__init__(torch.distributions.Poisson)

        def condition(self, feat):
            return torch.distributions.Poisson(feat)

    layers = torch.nn.ModuleList([sb.layers.StagLayer(sb.zoo.GCN(4, 3))])
    with pytest.raises(NotImplementedError):
        sb.models.StagModel(layers, likelihood=Poisson()).calibration(torch.rand(4, 3), torch.zeros(4))
    with pytest.raises(StagLibraryError):
        sb.models.StagModel(layers).calibration(torch.rand(4, 3), torch.zeros(4, dtype=torch.int64))


# ---- ranks ------------------------------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, ret):
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        for kind in ("categorical", "bernoulli"):
            N, C, B = 157, 11, 15
            probs, y = random_rows(kind, N, C, seed=21)             # the same rows on every rank
            mask = torch.from_numpy(np.random.default_rng(22).random(N) < 0.7)
            half = (N + 1) // 2
            rows = slice(0, half) if rank == 0 else slice(half, N)
            mine = calib(probs[rows], y[rows], kind, B, mask=mask[rows])
            calls = []
            real = dist.all_reduce

            def counting_all_reduce(t, *a, **k):
                calls.append((t.dtype, t.numel()))
                return real(t, *a, **k)

            dist.all_reduce = counting_all_reduce
            try:
                assert mine.all_reduce(dist.group.WORLD) is mine
            finally:
                dist.all_reduce = real
            assert calls == [(torch.int64, R.table_len(C, B))], calls
            one = calib(probs, y, kind, B, mask=mask)
            assert torch.equal(mine.table, one.table), kind
        ret[rank] = "ok"
    finally:
        dist.destroy_process_group()


def test_all_reduce_over_two_ranks_equals_one_process_gloo():
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(2, _free_port(), ret), nprocs=2, join=True)
    assert dict(ret) == {0: "ok", 1: "ok"}
