"""GPU: every route of the dense transform stag_gemm_tcgen05, driven through the bare C ABI (ctypes) and checked per
element against the float64 oracle of oracle/ref_gemm.py.

ops.dense_transform always passes compact, aligned buffers, so it reaches only part of the host's dispatcher.  The
header promises more: free leading dimensions, any base alignment, optional row scale / bias / relu.  `route()` below
restates the host's choice (csrc/gemm_tcgen05.cu, stag_gemm_tcgen05):
  - form 2 (gemm_tma_kernel, persistent): lda % 4 == 0, A 16-byte aligned, npad * nkb * 256 <= 128 KB; the A-tile
    rings (nlo, nst) and the TMEM columns per accumulator follow from the shared-memory arithmetic;
  - form 1 (gemm_tcgen05_kernel): everything else; few row tiles and >= 4 K blocks split K over a cluster of ksplit
    CTAs (at most 8, two K blocks each, partial tiles within the shared memory behind the epilogue scratch).
`coverage()` asserts that CASES (plus the child runs with STAG_GEMM_FORM=1 and STAG_GEMM_KSPLIT) reach every ring size,
TMEM width, ksplit value, alignment / vector-path switch and output width the dispatcher distinguishes.  The ring
sizes are reached through shapes only: the launcher's ring knobs are never set.

Each case must
  - launch the predicted kernel, with the predicted grid (ksplit CTAs per row tile on form 1, min(tiles, SMs) on
    form 2) and, on form 2, the shared memory of the predicted ring (torch.profiler trace);
  - match  act(rs * (A @ W) + b)  within 2^-17 (|rs| (|A| @ |W|) + |b|) per element, while the 1xTF32 emulation of
    its own inputs on its own split does not (so the bound can see a dropped term);
  - be bitwise equal on a second run;
  - leave the quiet-NaN canary in the margins around every buffer and in the row padding of `out` (ldo > Nout).
Inputs carry row scales of A and column scales of W from 2^-30 to 2^30, so a wrong row or column fails at its own size.

`python tests/test_gpu_gemm_routes.py child ...` is the child-process mode: the traced checks run in a fresh interpreter
(the profiler of a process that earlier test modules have profiled in may record no kernel), and the knobs are read
once per process.
"""
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import zlib

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import ref_gemm  # noqa: E402  (numpy only)

pytestmark = pytest.mark.gpu

CANARY = 0x7FC0DEAD            # a quiet-NaN bit pattern: never produced from finite inputs
MARGIN = 64                    # canary floats before and after every buffer
B200_SMS = 148                 # SM count the case list is laid out for when no device is visible
GM, GK, G2_TILE, G2_MAXST = 128, 32, 128 * 32 * 4, 8
NOUTS = (1, 7, 15, 16, 17, 33, 40, 100, 121, 128, 129, 200, 255, 256)
RINGS = ((2, 3), (2, 4), (2, 5), (3, 5), (3, 6), (3, 7), (3, 8))
KSPLIT_CAPS = (1, 3)


def sm_count():
    if torch.cuda.is_available():
        return torch.cuda.get_device_properties(0).multi_processor_count
    return B200_SMS


# ---------------------------------------------------------------------------------------------------------------------
# the host's route choice
def route(c, sms, force_form1=False, ksplit_cap=None):
    """-> dict(form, kernel, grid, ...) that stag_gemm_tcgen05 picks for case `c`."""
    M, K, N = c["M"], c["K"], c["N"]
    npad, nkb = (N + 15) // 16 * 16, (K + GK - 1) // GK
    cols = 32
    while cols < npad:
        cols <<= 1
    a_aligned = (4 * c["a_off"]) % 16 == 0
    if (c["lda"] % 4 == 0 and a_aligned and npad * nkb * 256 <= 128 * 1024 and M * c["lda"] < (1 << 40)
            and not force_form1):
        fixed = npad * nkb * 256 + 4 * 32 * 32 * 4 + 1024
        tiles = (227 * 1024 - 1024 - fixed) // G2_TILE
        nlo = 3 if tiles >= 8 else 2
        nst = min(tiles - nlo, G2_MAXST)
        ntiles = (M + GM - 1) // GM
        return dict(form=2, kernel="gemm_tma_kernel", nlo=nlo, nst=nst, ncol=cols, ntiles=ntiles,
                    grid=(min(ntiles, sms), 1, 1), dyn_smem=fixed + (nst + nlo) * G2_TILE)
    grid = (M + GM - 1) // GM
    ksplit, limit = 1, None
    if grid * 2 <= sms and nkb >= 4 and grid < 65536:
        lims = {"grid": 2 * sms // grid, "max": 8, "nkb": nkb // 2, "npad": 158 // npad + 1}
        ksplit = min(lims.values())
        limit = min(lims, key=lambda k: (lims[k], k != "npad"))
        if ksplit_cap is not None and 1 <= ksplit_cap < ksplit:
            ksplit, limit = ksplit_cap, "cap"
    return dict(form=1, kernel="gemm_tcgen05_kernel", ksplit=ksplit, limit=limit, npad=npad, ncol=cols,
                grid=(ksplit, grid, 1) if ksplit > 1 else (grid, 1, 1))


# ---------------------------------------------------------------------------------------------------------------------
# cases
def case(name, M, K, N, form, lda=None, ldw=None, ldo=None, a_off=0, w_off=0, o_off=0, b_off=0, rs=True, bias=True,
         act=0):
    return dict(name=name, M=M, K=K, N=N, form=form, lda=K if lda is None else lda, ldw=K if ldw is None else ldw,
                ldo=N if ldo is None else ldo, a_off=a_off, w_off=w_off, o_off=o_off, b_off=b_off, rs=rs, bias=bias,
                act=act)


def make_cases(sms):
    T = GM
    cs = [
        # ---- form 2: every (nlo, nst) the launcher picks, npad 16 (nkb 29-32, 25-28, 21-24, 17-20, 13-16, 9-12, 1-4)
        case("f2_ring23_K1000_N16", 300, 1000, 16, 2, act=1),
        case("f2_ring24_K800_N7", 129, 800, 7, 2, rs=False),
        case("f2_ring25_K700_N15", 1000, 700, 15, 2, bias=False, act=1),
        case("f2_ring35_K600_N1", 257, 600, 1, 2),
        case("f2_ring36_K500_N16_M64", 64, 500, 16, 2, ldo=20),
        case("f2_ring37_K300_N16", 1, 300, 16, 2, act=1, b_off=1),
        case("f2_ring38_K128_N16", 777, 128, 16, 2, ldw=131),
        case("f2_ring38_K61_lda64_N17", 500, 61, 17, 2, lda=64, act=1),
        # ---- form 2: TMEM widths 32 / 64 / 128 / 256, the output widths, alignment switches of W / out / bias
        case("f2_N33_ldo41", 300, 96, 33, 2, ldo=41, act=1),
        case("f2_N40_wmis_omis", 1000, 128, 40, 2, w_off=1, o_off=1),
        case("f2_N100_lda72_K64", 450, 64, 100, 2, lda=72, act=1, b_off=1),
        case("f2_N121_ldo128", 333, 128, 121, 2, ldo=128, rs=False, bias=False),
        case("f2_N128", 1000, 128, 128, 2, act=1),
        case("f2_N129_K96", 200, 96, 129, 2, ldw=100),
        case("f2_N200_K64_omis", 130, 64, 200, 2, o_off=1, act=1),
        case("f2_N255_K33", 100, 33, 255, 2, lda=36, ldo=260, w_off=3),
        case("f2_N256_K64", 513, 64, 256, 2, act=1, b_off=2),
        case("f2_N7_K5_lda8", 90, 5, 7, 2, lda=8, ldw=5),
        case("f2_N1_M1_K1_lda4", 1, 1, 1, 2, lda=4, act=1),
        case("f2_N16_K32_plain", 256, 32, 16, 2, rs=False, bias=False),
        case("f2_N15_K40_ldo17", 1500, 40, 15, 2, ldo=17, act=1),
        # ---- form 2: row tiles below / equal to / above the SM count, and both accumulators wrapping
        case("f2_tiles_eq_sms", sms * T - 3, 64, 40, 2, act=1),
        case("f2_tiles_above_sms", sms * T + 1000, 128, 128, 2, ldo=132),
        case("f2_acc_wrap", 3 * sms * T + 77, 48, 121, 2, act=1, b_off=1),
        # ---- form 1: misaligned A (pointer + 1 float, lda % 4 != 0), W too large for form 2, npad <= / > 128
        case("f1_amis_N16", 300, 64, 16, 1, a_off=1, act=1),
        case("f1_lda_odd_N40", 500, 61, 40, 1, act=1, ldo=41),
        case("f1_lda65_N128", 400, 64, 128, 1, lda=65, w_off=1, o_off=1),
        case("f1_bigW_N256_K100", 300, 100, 256, 1, act=1, b_off=1),
        case("f1_bigW_N129_K200", 1000, 200, 129, 1, ldw=203, ldo=136),
        case("f1_bigW_N200_K128_ragged", 129, 128, 200, 1, rs=False, act=1),
        case("f1_bigW_N255_K70", 700, 70, 255, 1, o_off=3, bias=False),
        case("f1_amis_N1", 77, 33, 1, 1, a_off=2, act=1),
        case("f1_amis_N7", 1, 7, 7, 1, a_off=1, lda=9),
        case("f1_amis_N15", 260, 128, 15, 1, a_off=3, b_off=1),
        case("f1_amis_N17", 128, 96, 17, 1, a_off=1, ldo=21, act=1),
        case("f1_amis_N33", 100, 64, 33, 1, a_off=1, rs=False),
        case("f1_amis_N100", 640, 64, 100, 1, a_off=1, act=1, w_off=2),
        case("f1_amis_N121", 200, 32, 121, 1, a_off=1, ldo=125),
        case("f1_amis_N256", 150, 64, 256, 1, a_off=1, bias=False, act=1),
        case("f1_many_tiles", 3 * sms * T + 5, 40, 40, 1, a_off=1, act=1),
        # ---- form 1: ksplit 1 .. 8 (one row tile, nkb = 2 k) and the npad limits (npad 32 -> 5, 48 -> 4, 64 -> 3,
        #      144 -> 2, 160 -> 1), one grid-limited split, and ksplit 1 below 4 K blocks / above sms / 2 row tiles
        case("f1_ks1_nkb3", 100, 90, 16, 1, a_off=1),
        case("f1_ks1_grid", (sms // 2 + 1) * T, 300, 16, 1, a_off=1),
        case("f1_ks2_nkb4", 128, 123, 16, 1, a_off=1, act=1),
        case("f1_ks3_nkb6", 100, 187, 16, 1, a_off=1, ldo=19),
        case("f1_ks4_nkb8", 64, 250, 16, 1, lda=251, b_off=1),
        case("f1_ks5_nkb10", 128, 319, 7, 1, a_off=1, act=1),
        case("f1_ks6_nkb12", 30, 380, 16, 1, a_off=1, w_off=1),
        case("f1_ks7_nkb14", 128, 443, 1, 1, a_off=1, rs=False),
        case("f1_ks8_nkb16", 100, 507, 16, 1, a_off=1, act=1, o_off=1),
        case("f1_ks8_K1433", 2 * T + 5, 1433, 16, 1, a_off=1, act=1),
        case("f1_ks_grid_limited", (sms // 2) * T - 7, 512, 16, 1, a_off=1),
        case("f1_ks5_npad32", 200, 640, 17, 1, a_off=1, act=1),
        case("f1_ks4_npad48", 128, 640, 40, 1, a_off=1, ldo=44),
        case("f1_ks3_npad64", 100, 640, 64, 1, a_off=1, b_off=1),
        case("f1_ks2_npad144", 128, 300, 129, 1, act=1),
        case("f1_ks1_npad160", 128, 300, 150, 1),
    ]
    return cs


SMS = sm_count()
CASES = make_cases(SMS)
_ids = [c["name"] for c in CASES]
assert len(set(_ids)) == len(_ids), "duplicate case names"


def child_runs(cases, sms):
    """The (case, env) pairs run in child processes: the form-2 cases on form 1, and every split case under each cap."""
    runs = []
    for c in cases:
        if route(c, sms)["form"] == 2:
            runs.append((c, {"STAG_GEMM_FORM": "1"}))
    for cap in KSPLIT_CAPS:
        for c in cases:
            r = route(c, sms)
            if r["form"] == 1 and r["ksplit"] > cap:
                runs.append((c, {"STAG_GEMM_KSPLIT": str(cap)}))
    return runs


def route_env(c, sms, env):
    cap = env.get("STAG_GEMM_KSPLIT")
    return route(c, sms, force_form1=env.get("STAG_GEMM_FORM") == "1", ksplit_cap=int(cap) if cap else None)


def features(c, r, sms):
    """Route features of one run of case `c` on route `r`."""
    f = r["form"]
    out = {("form", f), ("nout", f, c["N"]), ("ncol", f, r["ncol"]),
           ("rs", f, c["rs"]), ("bias", f, c["bias"]), ("act", f, c["act"])}
    if c["ldw"] > c["K"]:
        out.add(("ldw>K", f))
    if c["w_off"] % 4:
        out.add(("wt misaligned", f))
    if c["ldo"] > c["N"]:
        out.add(("ldo>Nout", f))
    if c["ldo"] % 4:
        out.add(("ldo%4", f))
    if c["o_off"] % 4:
        out.add(("out misaligned", f))
    if c["bias"] and c["b_off"] % 4:
        out.add(("bias misaligned", f))
    if f == 2:
        ntiles = r["ntiles"]
        out.add(("ring", r["nlo"], r["nst"]))
        out.add(("M<128",) if c["M"] < GM else ("M>=128",))
        if c["M"] % GM:
            out.add(("ragged M",))
        if c["K"] % GK:
            out.add(("K%32",))
        if c["K"] % 4 and c["lda"] % 4 == 0:
            out.add(("K%4, lda padded",))
        if c["lda"] > c["K"]:
            out.add(("lda>K",))
        out.add(("tiles vs sms", "below" if ntiles < sms else "equal" if ntiles == sms else "above"))
        if ntiles > 2 * sms:
            out.add(("both accumulators wrap",))
    else:
        out.add(("ksplit", r["ksplit"]))
        if r["limit"] == "npad":
            out.add(("ksplit npad limit", r["npad"], r["ksplit"]))
        out.add(("npad<=128",) if r["npad"] <= 128 else ("npad>128",))
        if c["a_off"] % 4:
            out.add(("f1 via A misaligned",))
        if c["lda"] % 4:
            out.add(("f1 via lda%4",))
        npad, nkb = r["npad"], (c["K"] + GK - 1) // GK
        if npad * nkb * 256 > 128 * 1024:
            out.add(("f1 via W too large",))
    return out


def required():
    req = {("form", 1), ("form", 2)}
    req |= {("ring",) + p for p in RINGS}
    req |= {("ncol", 2, n) for n in (32, 64, 128, 256)}
    req |= {("M<128",), ("M>=128",), ("ragged M",), ("K%32",), ("K%4, lda padded",), ("lda>K",),
            ("tiles vs sms", "below"), ("tiles vs sms", "equal"), ("tiles vs sms", "above"), ("both accumulators wrap",)}
    req |= {("f1 via A misaligned",), ("f1 via lda%4",), ("f1 via W too large",), ("npad<=128",), ("npad>128",)}
    req |= {("ksplit", k) for k in range(1, 9)}
    req |= {("ksplit npad limit", n, k) for n, k in ((32, 5), (48, 4), (64, 3), (144, 2), (160, 1))}
    for f in (1, 2):
        req |= {("nout", f, n) for n in NOUTS}
        req |= {(k, f) for k in ("ldw>K", "wt misaligned", "ldo>Nout", "ldo%4", "out misaligned", "bias misaligned")}
        req |= {(k, f, v) for k in ("rs", "bias") for v in (True, False)}
        req |= {("act", f, v) for v in (0, 1)}
    return req


def coverage(cases=None, sms=None):
    """Assert that the in-process cases and the child runs reach every route feature; -> (features, per-run routes)."""
    cases = CASES if cases is None else cases
    sms = SMS if sms is None else sms
    runs = [(c, {}) for c in cases] + child_runs(cases, sms)
    got, routes = set(), []
    for c, env in runs:
        r = route_env(c, sms, env)
        if not env:
            assert r["form"] == c["form"], "%s: meant for form %d, the dispatcher picks form %d" % (
                c["name"], c["form"], r["form"])
        got |= features(c, r, sms)
        routes.append((c["name"], env, r))
    missing = sorted(required() - got, key=repr)
    assert not missing, "route features no case reaches: %s" % missing
    return got, routes


# ---------------------------------------------------------------------------------------------------------------------
# buffers
class Buf:
    """Flat device buffer filled with CANARY; the logical [rows, cols] view (row stride ld) starts MARGIN + off in."""

    def __init__(self, rows, cols, ld, off=0):
        self.base = MARGIN + off
        span = (rows - 1) * ld + cols if rows > 0 else 0
        self.raw = torch.full((self.base + span + MARGIN,), CANARY, dtype=torch.int32, device="cuda")
        self.rows, self.cols, self.ld = rows, cols, ld

    def view(self):
        return self.raw.view(torch.float32).as_strided((self.rows, self.cols), (self.ld, 1), self.base)

    @property
    def ptr(self):
        return self.raw.data_ptr() + 4 * self.base

    def fill(self, data):
        self.view().copy_(torch.from_numpy(np.ascontiguousarray(data, np.float32)).cuda())
        return self

    def assert_canary(self, what):
        raw = self.raw.cpu().numpy()
        inside = np.zeros(raw.shape, bool)
        if self.rows > 0:
            idx = self.base + np.arange(self.rows)[:, None] * self.ld + np.arange(self.cols)[None, :]
            inside[idx.reshape(-1)] = True
        bad = np.flatnonzero((raw != CANARY) & ~inside)
        assert bad.size == 0, "%s: %d floats outside the logical region were written (first at %d)" % (
            what, bad.size, bad[0] - self.base)


def inputs(c):
    """Data of case `c`: the same for a shape whatever the layout, alignment or process."""
    key = repr([c[k] for k in ("M", "K", "N")])
    rng = np.random.default_rng(zlib.crc32(key.encode()))
    return ref_gemm.scaled_inputs(rng, c["M"], c["K"], c["N"])


def traced(fn):
    """Run fn() under torch.profiler; -> (rc, [(kernel name, grid, shared memory bytes)] of the stag kernels)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        rc = fn()
        torch.cuda.synchronize()
    fd, path = tempfile.mkstemp(suffix=".json")
    os.close(fd)
    try:
        prof.export_chrome_trace(path)
        with open(path) as f:
            ev = json.load(f)
    finally:
        os.unlink(path)
    ev = ev["traceEvents"] if isinstance(ev, dict) else ev
    ks = []
    for e in ev:
        if e.get("cat") == "kernel" and "stag::" in e.get("name", ""):
            a = e.get("args", {})
            assert "grid" in a, "profiler kernel event without a grid: %s" % sorted(a)
            ks.append((e["name"], tuple(a["grid"]), a.get("shared memory")))
    return rc, ks


def run_case(c, env=None, trace=True):
    """Run case `c` through the C ABI and check it.  -> dict(route, kernel, grid, smem) of what was observed."""
    from stag_b200 import _lib
    lib = _lib.load()
    r = route_env(c, SMS, env or {})
    a, w, rs, b = inputs(c)
    M, K, N = c["M"], c["K"], c["N"]
    ab = Buf(M, K, c["lda"], c["a_off"]).fill(a)
    wb = Buf(N, K, c["ldw"], c["w_off"]).fill(w.T)
    rb = Buf(1, M, M).fill(rs[None]) if c["rs"] else None
    bb = Buf(1, N, N, c["b_off"]).fill(b[None]) if c["bias"] else None
    st = torch.cuda.current_stream().cuda_stream

    def call(ob):
        return lib.stag_gemm_tcgen05(ab.ptr, c["lda"], wb.ptr, c["ldw"], M, N, K, rb.ptr if rb else 0,
                                     bb.ptr if bb else 0, c["act"], ob.ptr, c["ldo"], 0, 0, st)
    o1 = Buf(M, N, c["ldo"], c["o_off"])
    if trace:
        rc, ks = traced(lambda: call(o1))
    else:
        rc, ks = call(o1), None
        torch.cuda.synchronize()
    assert rc == 0, "%s: rc %d: %s" % (c["name"], rc, lib.stag_last_error().decode())
    obs = dict(route=r)
    if ks is not None:
        names = [k[0] for k in ks]
        assert len(ks) == 1 and r["kernel"] in names[0], "%s: expected one %s, launched %s" % (
            c["name"], r["kernel"], names)
        obs.update(kernel=r["kernel"], grid=ks[0][1], smem=ks[0][2])
        assert tuple(ks[0][1]) == r["grid"], "%s: grid %s, the dispatcher's rule gives %s" % (
            c["name"], ks[0][1], r["grid"])
        if r["form"] == 2:
            # dynamic shared memory pins the ring: nst + nlo tiles of 16 KB beside W and the scratch (+ static)
            assert ks[0][2] is not None and 0 <= ks[0][2] - r["dyn_smem"] < 4096, (c["name"], ks[0][2], r["dyn_smem"])
    for bf, what in ((ab, "a"), (wb, "wt"), (rb, "row_scale"), (bb, "bias")):
        if bf is not None:
            bf.assert_canary("%s: %s" % (c["name"], what))
    o1.assert_canary(c["name"] + ": out")
    out = o1.view().cpu().numpy().astype(np.float64)

    rsx, bx = (rs if c["rs"] else None), (b if c["bias"] else None)
    ref = ref_gemm.reference(a, w, rsx, bx, relu=bool(c["act"]))
    tol = ref_gemm.bound(a, w, rsx, bx)
    bad = ref_gemm.violations(out, ref, tol)
    if bad:
        err = np.abs(out - ref)
        i, j = np.unravel_index(np.nanargmax(np.where(np.isnan(err), np.inf, err / tol)), err.shape)
        raise AssertionError("%s (%s): %d of %d entries beyond 2^-17 (|rs||A||W| + |b|); worst [%d, %d]: got %r, "
                             "want %r, bound %.3e" % (c["name"], r, bad, out.size, i, j, out[i, j], ref[i, j],
                                                      tol[i, j]))
    # the bound sees a dropped split term: the 1xTF32 product of these inputs on this route's split is outside it
    one = ref_gemm.emulate(a, w, r["form"], ("hh",), rsx)
    assert ref_gemm.violations(one, ref_gemm.reference(a, w, rsx), ref_gemm.bound(a, w, rsx)) > 0, \
        "%s: the 1xTF32 emulation is within the bound" % c["name"]

    o2 = Buf(M, N, c["ldo"], c["o_off"])
    assert call(o2) == 0
    torch.cuda.synchronize()
    assert torch.equal(o1.raw, o2.raw), "%s: two runs differ" % c["name"]
    return obs


# ---------------------------------------------------------------------------------------------------------------------
# 1. routes
# torch.profiler records no kernel events in a process that has been through some other test modules' profiling first,
# so every traced check runs in a fresh child interpreter (one for the whole table) and each test reports its result.
@pytest.fixture(scope="module")
def routed():
    return run_child({}, ["routes"])


@pytest.mark.parametrize("c", CASES, ids=_ids)
def test_route_matches_the_float64_oracle(c, routed):
    res = routed[c["name"]]
    assert res["ok"], res["error"]
    r = route(c, SMS)
    print("\n%s: %s grid %s%s" % (c["name"], res["kernel"], res["grid"], " (nlo, nst) = (%d, %d)" % (r["nlo"], r["nst"])
                                    if r["form"] == 2 else " ksplit %d" % r["ksplit"]))


def test_coverage_of_the_dispatcher():
    """The route rule of this device reaches every feature (the same check runs on CPU for 148 SMs)."""
    got, routes = coverage()
    print("\nroute features reached:", len(got))
    for name, env, r in routes:
        print("  %-28s %-26s %s" % (name, env or "", {k: v for k, v in r.items() if k != "dyn_smem"}))


# ---------------------------------------------------------------------------------------------------------------------
# 2. argument handling
def test_argument_errors_and_empty_input():
    from stag_b200 import _lib
    lib = _lib.load()
    st = torch.cuda.current_stream().cuda_stream
    M, K, N = 10, 8, 16
    a = Buf(M, K, K).fill(np.ones((M, K)))
    wt = Buf(N, K, K).fill(np.ones((N, K)))
    o = Buf(M, N, N)

    def call(M=M, K=K, N=N, lda=K, ldw=K, ldo=N, act=0, pa=None, pw=None, po=None):
        return lib.stag_gemm_tcgen05(a.ptr if pa is None else pa, lda, wt.ptr if pw is None else pw, ldw, M, N, K,
                                     0, 0, act, o.ptr if po is None else po, ldo, 0, 0, st)
    n0 = lib.stag_launch_count()
    assert call(M=0) == _lib.STAG_OK
    assert call(M=0, pa=0, pw=0, po=0) == _lib.STAG_OK
    bad = [dict(M=-1), dict(K=0), dict(K=-3), dict(N=0), dict(lda=K - 1), dict(ldw=K - 1), dict(ldo=N - 1),
           dict(act=2), dict(act=-1), dict(pa=0), dict(pw=0), dict(po=0)]
    for kw in bad:
        assert call(**kw) == _lib.STAG_EINVAL, (kw, lib.stag_last_error())
    assert call(N=257, ldo=257) == _lib.STAG_EUNSUPPORTED
    assert b"257" in lib.stag_last_error()
    torch.cuda.synchronize()
    assert lib.stag_launch_count() == n0, "a refused or empty call launched a kernel"
    o.assert_canary("refused calls: out")
    assert (o.raw.cpu().numpy() == CANARY).all(), "a refused or empty call wrote the output"


# ---------------------------------------------------------------------------------------------------------------------
# 3. non-finite inputs on both forms, through the ABI
NONFINITE = [(n, act) for n in ("f2_N40_wmis_omis", "f1_amis_N100", "f1_ks8_nkb16") for act in (0, 1)]


@pytest.mark.parametrize("form_case,act", NONFINITE, ids=["%s-act%d" % x for x in NONFINITE])
def test_nan_and_inf_rows_and_columns(form_case, act, routed):
    res = routed["nonfinite %s %d" % (form_case, act)]
    assert res["ok"], res["error"]


def check_nonfinite(form_case, act):
    """NaN in row i of A -> out row i NaN; NaN in column j of W -> out column j NaN; +-Inf -> NaN (the split's
    Inf - Inf); relu keeps NaN; every other entry within the bound."""
    from stag_b200 import _lib
    lib = _lib.load()
    c = dict(next(x for x in CASES if x["name"] == form_case), act=act)
    r = route(c, SMS)
    a, w, rs, b = inputs(c)
    M, K, N = c["M"], c["K"], c["N"]
    a[3, 5] = np.nan
    a[7, 0] = np.inf
    a[M - 1, K - 1] = -np.inf
    w[K - 1, 2] = np.nan
    w[1, N - 1] = np.inf
    bad_rows, bad_cols = [3, 7, M - 1], [2, N - 1]
    ab = Buf(M, K, c["lda"], c["a_off"]).fill(a)
    wb = Buf(N, K, c["ldw"], c["w_off"]).fill(w.T)
    rb = Buf(1, M, M).fill(rs[None])
    bb = Buf(1, N, N, c["b_off"]).fill(b[None])
    ob = Buf(M, N, c["ldo"], c["o_off"])
    rc, ks = traced(lambda: lib.stag_gemm_tcgen05(ab.ptr, c["lda"], wb.ptr, c["ldw"], M, N, K, rb.ptr, bb.ptr, act,
                                                  ob.ptr, c["ldo"], 0, 0, torch.cuda.current_stream().cuda_stream))
    assert rc == 0 and len(ks) == 1 and r["kernel"] in ks[0][0], (rc, ks)
    ob.assert_canary("out")
    out = ob.view().cpu().numpy().astype(np.float64)
    assert np.isnan(out[bad_rows]).all(), "rows with NaN / Inf in A must be NaN"
    assert np.isnan(out[:, bad_cols]).all(), "columns with NaN / Inf in W must be NaN"
    keep_r = np.setdiff1d(np.arange(M), bad_rows)
    keep_c = np.setdiff1d(np.arange(N), bad_cols)
    a2, w2 = a[keep_r], w[:, keep_c]
    ref = ref_gemm.reference(a2, w2, rs[keep_r], b[keep_c], relu=bool(act))
    tol = ref_gemm.bound(a2, w2, rs[keep_r], b[keep_c])
    assert ref_gemm.violations(out[np.ix_(keep_r, keep_c)], ref, tol) == 0
    return dict(kernel=r["kernel"], grid=list(ks[0][1]))


# ---------------------------------------------------------------------------------------------------------------------
# 4. the same inputs on form 1, and under a split cap (knobs read once per process: child interpreters)
def run_child(env, args=(), timeout=900):
    e = dict(os.environ)
    e.update(env)
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "child"] + list(args), env=e, capture_output=True,
                       text=True, timeout=timeout, cwd=ROOT)
    assert r.returncode == 0, "child %s failed:\n%s\n%s" % (env, r.stdout[-4000:], r.stderr[-4000:])
    return json.loads(r.stdout.strip().splitlines()[-1])


@pytest.mark.parametrize("env", [{"STAG_GEMM_FORM": "1"}] + [{"STAG_GEMM_KSPLIT": str(k)} for k in KSPLIT_CAPS],
                         ids=["form1"] + ["ksplit_cap%d" % k for k in KSPLIT_CAPS])
def test_same_inputs_under_a_knob(env):
    want = [c["name"] for c, e in child_runs(CASES, SMS) if e == env]
    assert want
    out = run_child(env)
    assert out["ran"] == want, (out["ran"], want)
    seen = sorted({(o["kernel"], tuple(o["grid"])) for o in out["obs"]})
    print("\n%s: %d cases, launches %s" % (env, len(want), seen))


def _child(argv):
    torch.cuda.set_device(0)
    if argv and argv[0] == "routes":
        # every case, each reported on its own: one failing case does not hide the others
        res = {}
        jobs = [(c["name"], lambda c=c: run_case(c)) for c in CASES]
        jobs += [("nonfinite %s %d" % x, lambda x=x: check_nonfinite(*x)) for x in NONFINITE]
        for name, job in jobs:
            try:
                o = job()
                res[name] = dict(ok=True, kernel=o["kernel"], grid=list(o["grid"]))
            except Exception as ex:  # noqa: BLE001  (reported per case)
                res[name] = dict(ok=False, error="%s: %s" % (type(ex).__name__, ex))
        print(json.dumps(res))
        return
    env = {k: os.environ[k] for k in ("STAG_GEMM_FORM", "STAG_GEMM_KSPLIT") if k in os.environ}
    ran, obs = [], []
    for c, e in child_runs(CASES, SMS):
        if e == env:
            o = run_case(c, env)
            ran.append(c["name"])
            obs.append(dict(kernel=o["kernel"], grid=list(o["grid"])))
    print(json.dumps({"ran": ran, "obs": obs}))


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "child":
    _child(sys.argv[2:])
