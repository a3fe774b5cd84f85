"""CPU: the oracle (oracle/ref_*.py) against the golden vectors minted from the reference's
own code (oracle/make_golden.py) and, given a checkout of the reference, against the live reference."""
import os
import sys

import numpy as np
import pytest
import torch

from conftest import golden, LAYER_CASES, ROOT
from oracle import ref_index, ref_layers, ref_philox, ref_spmm

RTOL, ATOL = 1e-5, 1e-6


def close(a, b, rtol=RTOL, atol=ATOL):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    scale = max(np.abs(b).max(), 1e-30) if b.size else 1.0
    np.testing.assert_allclose(a, b, rtol=rtol, atol=atol * max(scale, 1.0))


def test_philox_known_answers():
    for ctr, key, want in ref_philox.KAT:
        got = ref_philox.philox4x32_10(*[np.uint32(c) for c in ctr], key[0], key[1])
        assert tuple(int(np.asarray(g).reshape(-1)[0]) for g in got) == want


def test_philox_variate_ranges():
    u = ref_philox.uniform(1000, 8, 0, 42, 0)
    assert u.min() >= 0.0 and u.max() < 1.0
    z = ref_philox.std_normal(20000, 8, 1, 42, 3)
    assert abs(z.mean()) < 0.02 and abs(z.std() - 1.0) < 0.02 and np.isfinite(z).all()


@pytest.mark.parametrize("by_dst", [True, False])
def test_index_oracle_matches_stable_sort(by_dst):
    rng = np.random.default_rng(0)
    for n, e in ((1, 0), (1, 5), (7, 0), (50, 300), (1000, 20000)):
        src, dst = rng.integers(0, n, e), rng.integers(0, n, e)
        indptr, indices, eid = ref_index.csx_build(src, dst, n, by_dst)
        key = torch.from_numpy(dst if by_dst else src)
        perm = torch.sort(key, stable=True).indices.numpy() if e else np.zeros(0, np.int64)
        assert np.array_equal(eid, perm.astype(np.int32))
        assert np.array_equal(indices, (src if by_dst else dst)[perm].astype(np.int32))
        assert indptr[0] == 0 and indptr[-1] == e and len(indptr) == n + 1
        assert np.array_equal(np.diff(indptr), np.bincount(dst if by_dst else src, minlength=n))


def test_index_order_is_the_reduction_order():
    """Summing messages in CSC order (stable by edge id) is bitwise what index_add in edge-id
    order (the dgl shim's fn.sum) produces -- the order the golden outputs were made with."""
    d = golden("powerlaw_d50")
    src, dst, N = d["src"], d["dst"], int(d["num_nodes"])
    indptr, indices, eid = ref_index.csx_build(src, dst, N, True)
    x, w = d["feat"], d["w"]
    m = x[src] * w
    want = torch.zeros(N, x.shape[1]).index_add(0, torch.from_numpy(dst), torch.from_numpy(m)).numpy()
    got = np.zeros_like(want)
    for v in range(N):
        acc = np.zeros(x.shape[1], np.float32)
        for j in range(indptr[v], indptr[v + 1]):
            acc = acc + m[eid[j]]
        got[v] = acc
    assert np.array_equal(got, want)


@pytest.mark.parametrize("name", LAYER_CASES)
def test_layer_restatement_matches_reference_golden(name):
    d = golden(name)
    r = ref_layers.replay_layer_case(name, d)
    close(r["out"], d["out"])
    close(r["dfeat"], d["dfeat"])
    if "dw" in d:
        close(r["dw"], d["dw"])
    if "w_used" in d:
        close(r["w_used"], d["w_used"])
    for k, g in r["grads"].items():
        close(g, d["g_" + k.replace(".", "__")])


def test_model_restatement_matches_reference_golden():
    d = golden("model_rc_vi")
    nll, reg, grads = ref_layers.replay_model_rc_vi(d)
    close(nll, d["nll"])
    close(reg, d["reg"])
    keys = [k for k in d.files if k.startswith("g_")]
    assert keys
    for k in keys:
        close(grads[k[2:].replace("__", ".")], d[k], rtol=1e-4)


def test_readout_restatement():
    d = golden("readout")
    f, bnn = torch.from_numpy(d["feat"]), torch.from_numpy(d["batch_num_nodes"])
    close(ref_spmm.readout(f, bnn, "sum"), d["sum"])
    close(ref_spmm.readout(f, bnn, "mean"), d["mean"])


def test_aggregate_contract_equals_gcn_pieces():
    d = golden("gcn_both")
    src, dst, N = torch.from_numpy(d["src"]), torch.from_numpy(d["dst"]), int(d["num_nodes"])
    x, w = torch.from_numpy(d["feat"]), torch.from_numpy(d["w"])
    s, t = ref_spmm.gcn_norms(src, dst, N, "both")
    agg = ref_spmm.aggregate(src, dst, N, x, w, src_scale=s, dst_scale=t)
    out = agg @ torch.from_numpy(d["p_weight"]) + torch.from_numpy(d["p_bias"])
    close(out, d["out"])


@pytest.mark.skipif(not (os.environ.get("STAG_REFERENCE") and os.path.isdir(os.path.join(os.environ["STAG_REFERENCE"], "stag"))),
                    reason="needs a checkout of the reference project (yuanqing-wang/stag) named by STAG_REFERENCE")
def test_golden_reproducible_from_live_reference(tmp_path, monkeypatch):
    """Re-run make_golden.py against the reference checkout named by STAG_REFERENCE and compare with the committed
    fixtures."""
    import subprocess
    env = dict(os.environ)
    code = ("import sys; sys.path.insert(0, %r); import oracle.make_golden as m; m.OUT=%r; m.main()"
            % (ROOT, str(tmp_path)))
    subprocess.run([sys.executable, "-W", "ignore", "-c", code], check=True, env=env, stdout=subprocess.DEVNULL)
    for name in ("t_r1_gcn", "gcn_both", "sage_mean", "model_rc_vi", "amortized_rec", "hub_d128"):
        a, b = np.load(os.path.join(str(tmp_path), name + ".npz")), golden(name)
        assert sorted(a.files) == sorted(b.files)
        for k in a.files:
            np.testing.assert_allclose(a[k], b[k], rtol=1e-5, atol=1e-6)


def test_hadamard_generator_restatement_law():
    """The numpy restatement of the tensor-core generator (oracle/ref_philox.py): constants, orthogonality of the
    mixing matrix, exactness of the sums and the law of the output on 1.3e6 draws."""
    from scipy import stats
    from oracle import ref_philox as rp
    H = rp.hadamard_matrix()
    assert np.array_equal(H @ H.T, 128 * np.eye(128))
    v = rp.e4m3_value((np.arange(256) & rp.WH_AND) | rp.WH_OR)
    m2, m4 = (v ** 2).mean(), (v ** 4).mean()
    assert m2 == 105186885 / 524288
    assert abs(m4 / m2 ** 2 - 3.0) < 1e-3                      # input law: excess kurtosis 8e-4
    assert abs(float(rp.WH_INV_SD) - 1 / np.sqrt(128 * m2)) < 1e-9
    assert np.abs(v).max() * 128 < 2 ** 12 and np.all(v * 256 == np.round(v * 256))   # sums exact in fp32
    s = rp.hadamard_sums(5000, 256, 1, 42, 3)
    assert np.array_equal(s.astype(np.float32).astype(np.float64), s)
    z = rp.hadamard_normal(5000, 256, 1, 42, 3).astype(np.float64)
    n = z.size
    assert abs(z.mean()) < 5 / np.sqrt(n) and abs(z.var() - 1) < 5 * np.sqrt(2.0 / n)
    assert abs(stats.kurtosis(z.ravel())) < 5 * np.sqrt(24.0 / n)
    assert stats.kstest(z.ravel(), "norm").pvalue > 1e-3


def test_generators_accept_edge_id_subsets():
    """`num_edges` may be an array of edge ids (row subsets of graphs too large to materialise [E,K] for: the
    products-shape parity test): the variates of exactly those edges, for every distribution kind."""
    from oracle import ref_philox
    ids = np.array([7, 3, 49, 3, 0], dtype=np.int64)
    for kind, K, p0, p1 in [("normal", 40, 1.0, 0.4), ("normal_hadamard", 256, 1.0, 0.4), ("uniform", 24, 0.3, 1.7),
                            ("bernoulli", 16, 0.8, None)]:
        full = ref_philox.noise(kind, 50, K, 2, 11, 3, p0, p1)
        assert np.array_equal(ref_philox.noise(kind, ids, K, 2, 11, 3, p0, p1), full[ids]), kind
