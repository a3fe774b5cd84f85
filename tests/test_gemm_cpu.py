"""CPU: the oracle and tolerance of the dense-transform tests (oracle/ref_gemm.py), the route table of
tests/test_gpu_gemm_routes.py, and the argument checks of ops.dense_transform.

The GPU tests hold stag_gemm_tcgen05 to 2^-17 (|rs| (|A| @ |W|) + |b|) per element.  Here, for every route shape, the
float64 emulation of the kernel's 3xTF32 product (both splits) is inside that bound, while a 1xTF32 product and splits
that drop A_lo W_hi or A_hi W_lo are outside it: the bound is tight enough to see a missing term."""
import os
import sys
import zlib

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from conftest import ROOT  # noqa: E402,F401  (puts the repository root on sys.path)
from oracle import ref_gemm  # noqa: E402
import test_gpu_gemm_routes as routes  # noqa: E402  (the route table; its tests need a GPU, its helpers do not)

MAX_ROWS = 2048


def test_tf32_rounding_and_splits():
    f = lambda v: np.array(v, np.float32)  # noqa: E731
    ulp = 2.0 ** -10
    # round to nearest, ties away from zero
    assert ref_gemm.tf32_rna(f([1 + ulp / 2, -(1 + ulp / 2), 1 + ulp / 2 - 2 ** -23, 1 + 1.5 * ulp])).tolist() == \
        [1 + ulp, -(1 + ulp), 1.0, 1 + 2 * ulp]
    assert ref_gemm.tf32_trunc(f([1 + ulp - 2 ** -23, -(1 + ulp - 2 ** -23)])).tolist() == [1.0, -1.0]
    x = np.random.default_rng(0).standard_normal(10000).astype(np.float32) * np.float32(2.0 ** 20)
    for form in (1, 2):
        for op in ("a", "w"):
            hi, lo = ref_gemm.split(x, form, op)
            for p in (hi, lo):
                assert not (p.view(np.uint32) & 0x1FFF).any(), "a split part is not a tf32 value"
            err = np.abs(hi.astype(np.float64) + lo - x)
            assert (err <= 2.0 ** -21 * np.abs(x)).all()
    assert np.isnan(ref_gemm.tf32_rna(f([np.nan]))).all() and ref_gemm.tf32_rna(f([np.inf]))[0] == np.inf
    # an infinite input splits into (Inf, NaN): a product with it is NaN, not Inf
    hi, lo = ref_gemm.split(f([np.inf, -np.inf]), 2, "a")
    assert np.isinf(hi).all() and np.isnan(lo).all()


def test_route_table_covers_the_dispatcher():
    cases = routes.make_cases(routes.B200_SMS)
    got, runs = routes.coverage(cases, routes.B200_SMS)
    rings = sorted({(r["nlo"], r["nst"]) for _, e, r in runs if r["form"] == 2})
    splits = sorted({r["ksplit"] for _, e, r in runs if r["form"] == 1})
    print("\n%d cases, %d child runs, %d route features; rings %s, ksplit %s"
          % (len(cases), len(runs) - len(cases), len(got), rings, splits))
    assert rings == sorted(routes.RINGS) and splits == list(range(1, 9))


def test_route_rule_at_the_documented_points():
    """(nlo, nst) at npad 16 per nkb range, and the npad limits of the split, from the launcher's arithmetic."""
    c = lambda M, K, N, **kw: routes.case("x", M, K, N, 0, **kw)  # noqa: E731
    want = {(29, 32): (2, 3), (25, 28): (2, 4), (21, 24): (2, 5), (17, 20): (3, 5), (13, 16): (3, 6), (9, 12): (3, 7),
            (1, 4): (3, 8)}
    for (k0, k1), ring in want.items():
        for nkb in (k0, k1):
            r = routes.route(c(1000, 32 * nkb, 16), 148)
            assert r["form"] == 2 and (r["nlo"], r["nst"]) == ring, (nkb, r)
    for N, ks in ((32, 5), (48, 4), (64, 3), (144, 2), (160, 1)):
        r = routes.route(c(128, 640, N, a_off=1), 148)
        assert r["form"] == 1 and r["ksplit"] == ks, (N, r)
    assert routes.route(c(1000, 32 * 33, 16), 148)["form"] == 1        # W_hi + W_lo over 128 KB
    assert routes.route(c(128, 640, 16, a_off=1), 148, ksplit_cap=3)["ksplit"] == 3


def _shapes():
    seen, out = set(), []
    for c in routes.make_cases(routes.B200_SMS):
        key = (min(c["M"], MAX_ROWS), c["K"], c["N"])
        if key not in seen:
            seen.add(key)
            out.append(key)
    return out


@pytest.mark.parametrize("M,K,N", _shapes())
def test_bound_accepts_3xtf32_and_sees_a_dropped_term(M, K, N):
    rng = np.random.default_rng(zlib.crc32(repr([M, K, N]).encode()))
    a, w, rs, b = ref_gemm.scaled_inputs(rng, M, K, N)
    for relu in (False, True):
        ref = ref_gemm.reference(a, w, rs, b, relu)
        tol = ref_gemm.bound(a, w, rs, b)
        for form in (1, 2):
            three = ref_gemm.emulate(a, w, form, ("hh", "lh", "hl"), rs, b, relu)
            assert ref_gemm.violations(three, ref, tol) == 0, (form, relu)
    pre, tol = ref_gemm.reference(a, w, rs), ref_gemm.bound(a, w, rs)
    for form in (1, 2):
        for terms in (("hh",), ("hh", "hl"), ("hh", "lh")):
            n = ref_gemm.violations(ref_gemm.emulate(a, w, form, terms, rs), pre, tol)
            assert n > 0, "form %d, terms %s: inside the bound" % (form, terms)


def test_bound_sees_a_wrong_row_scale_bias_or_row():
    rng = np.random.default_rng(3)
    a, w, rs, b = ref_gemm.scaled_inputs(rng, 300, 64, 40)
    ref, tol = ref_gemm.reference(a, w, rs, b), ref_gemm.bound(a, w, rs, b)
    assert ref_gemm.violations(ref, ref, tol) == 0
    ref0, tol0 = ref_gemm.reference(a, w, rs), ref_gemm.bound(a, w, rs)
    for i in range(300):                     # every row scale off by 2^-13 is seen in its row, whatever its size
        rs2 = rs.copy()
        rs2[i] *= np.float32(1 + 2.0 ** -13)
        assert ref_gemm.violations(ref_gemm.reference(a, w, rs2), ref0, tol0) > 0, i
    for j in range(40):
        b2 = b.copy()
        b2[j] *= np.float32(1 + 2.0 ** -15)
        assert ref_gemm.violations(ref_gemm.reference(a, w, rs, b2), ref, tol) > 0, j
    swapped = ref.copy()
    swapped[[5, 6]] = swapped[[6, 5]]
    assert ref_gemm.violations(swapped, ref, tol) > 0
    nan = ref.copy()
    nan[2, 3] = np.nan
    assert ref_gemm.violations(nan, ref, tol) == 1


# ---------------------------------------------------------------------------------------------------------------------
# argument checks of ops.dense_transform: before any device work, so they hold for CPU tensors too
@pytest.mark.parametrize("transposed", [False, True])
@pytest.mark.parametrize("nout", [40, 300])
def test_dense_transform_rejects_bad_row_scale_and_bias(transposed, nout):
    from stag_b200 import _lib, ops
    K = 24
    a = torch.randn(3, 10, K)
    w = torch.randn(nout, K) if transposed else torch.randn(K, nout)
    for n in (7, 29, 31, 60, 0):             # neither M = 30 nor a divisor of it
        with pytest.raises(ValueError, match="row_scale"):
            ops.dense_transform(a, w, row_scale=torch.rand(n), transposed=transposed)
    with pytest.raises(ValueError, match="gradient"):
        ops.dense_transform(a, w, row_scale=torch.rand(10, requires_grad=True), transposed=transposed)
    for shape in ((nout - 1,), (1,), (nout, 1), (1, nout), (nout + 1,)):
        with pytest.raises(ValueError, match="bias"):
            ops.dense_transform(a, w, bias=torch.randn(shape), transposed=transposed)
    if nout <= 256:
        # well-formed arguments pass the checks and reach the device requirement
        for n in (30, 10, 5, 1):
            with pytest.raises(_lib.StagLibraryError):
                ops.dense_transform(a, w, row_scale=torch.rand(n), bias=torch.randn(nout), transposed=transposed)
