"""GPU: every kernel instantiation behind the fused aggregation entry points (stag_spmm_fwd / _bwd, stag_spmm_max_fwd /
_bwd), driven through the bare C ABI (ctypes) and checked against a float64 oracle.

The Python layer (stag_b200.ops) always passes compact aligned buffers and graphs with every optional schedule, so
it reaches only part of the dispatcher.  The header promises more: free row and sample strides, shared X, optional
`row_order` / `items` / `erow` / `eidf`, OVERWRITE vs ACCUMULATE parameter gradients, `dx` = NULL, bitwise results.
Each entry of ROUTES is a small case that must launch the named kernel(s) (checked with torch.profiler) and match:
  - sums: the oracle on the noise stag_noise_emit writes (pinned to oracle/ref_philox.py by test_gpu_rng /
    test_gpu_hadamard), elementwise |a - b| <= 1e-5 |b| + 1e-6 max|b|; summed parameter gradients with the slack rule
    of test_gpu_rng.test_fused_parameter_gradients;
  - max: values (bits) and winning edges exactly.
Every output buffer sits between canary margins and must keep the canary outside its logical region.
The graph has rows whose in-degree (CSC) and out-degree (CSR) is exactly 0, 1, 127, 128, 129, 255, 256, 257 and 385:
the hub threshold and segment are 128 edges.

`python tests/test_gpu_abi_routes.py child ...` is the child-process mode used for the knobs read once per process
(STAG_NCB, STAG_WQ_VARIANT).
"""
import ctypes
import json
import os
import re
import shutil
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

from oracle import ref_max, ref_spmm  # noqa: E402  (torch CPU only)

pytestmark = pytest.mark.gpu

CANARY = 0x7FC0DEAD            # a quiet-NaN bit pattern: never produced by the kernels
MARGIN = 64                    # canary floats before and after every output buffer
DEGS = (0, 1, 127, 128, 129, 255, 256, 257, 385)
N_NODES = 720
IN_ROWS = tuple(range(10, 19))    # in-degree DEGS[i] (CSC rows)
OUT_ROWS = tuple(range(20, 29))   # out-degree DEGS[i] (CSR rows)
TIE_U = (2, 3)                    # sources of stored edges 127 and 128 of the in-degree-257 row
FILL0 = 80                        # nodes FILL0.. carry the random filler edges; 0..FILL0-1 are otherwise isolated
KIND = {"none": 0, "ext": 1, "normal": 2, "uniform": 3, "bernoulli": 4, "hadamard": 5}
PSHAPE = {"r1": 0, "rc": 1, "re": 2, "rec": 3}
SCHED = ("row_order", "items", "erow", "eidf")
NO_SCHED = ("items", "erow", "eidf")
FAMILIES = ("agg_kernel", "agg_stream_kernel", "agg_stream_grads_kernel", "agg_wh_quad_kernel", "edge_param_grads",
            "max_row_kernel", "max_wh_kernel", "max_edge_kernel", "hub_finalize", "max_hub_finalize", "param_finalize")


# ---------------------------------------------------------------------------------------------------------------------
# kernel names
def norm_name(name):
    """'void stag::agg_kernel<2, 2, 0, true, false, true>(stag::AggParams)' -> 'agg_kernel<2,2,0,1,0,1>'
    (nm -C and the profiler print bools as true / false, Nsight Compute as 1 / 0)."""
    n = name.strip()
    if n.startswith("void "):
        n = n[5:]
    depth, cut = 0, len(n)
    for i, ch in enumerate(n):   # drop the parameter list: the first '(' outside the template brackets
        if ch == "<":
            depth += 1
        elif ch == ">":
            depth -= 1
        elif ch == "(" and depth == 0:
            cut = i
            break
    n = n[:cut].replace(" ", "").replace("stag::", "")
    return re.sub(r"\btrue\b", "1", re.sub(r"\bfalse\b", "0", n))


def in_family(name):
    return any(name == f or name.startswith(f + "<") or name.startswith(f + "_") for f in FAMILIES)


def traced(fn):
    """Run fn() under torch.profiler (CUDA activity); -> (result, set of normalised stag kernel names)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        r = fn()
        torch.cuda.synchronize()
    if isinstance(r, int) and r != 0:
        return r, set()      # refused before any launch: the caller checks the code
    kernels = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    assert kernels, "torch.profiler recorded no CUDA kernel events: the route of this case cannot be checked"
    return r, {norm_name(k) for k in kernels if "stag::" in k}


# ---------------------------------------------------------------------------------------------------------------------
# graphs
def boundary_coo(seed=0):
    """COO (original edge order shuffled) with the DEGS rows on both sides, isolated rows, and a tie pair."""
    rng = np.random.default_rng(seed)
    fill = np.arange(FILL0, N_NODES)
    src, dst = [], []
    for r, d in zip(IN_ROWS, DEGS):
        dst.append(np.full(d, r))
        src.append(rng.choice(fill, d))
    for r, d in zip(OUT_ROWS, DEGS):
        src.append(np.full(d, r))
        dst.append(rng.choice(fill, d))
    src.append(rng.choice(fill, 2000))
    dst.append(rng.choice(fill, 2000))
    src, dst = np.concatenate(src), np.concatenate(dst)
    perm = rng.permutation(len(src))
    src, dst = src[perm], dst[perm]
    e = np.flatnonzero(dst == IN_ROWS[DEGS.index(257)])   # increasing edge id = stored order of the row
    src[e[127]], src[e[128]] = TIE_U
    return src.astype(np.int64), dst.astype(np.int64)


_COO = {}


def coo(seed=0):
    if seed not in _COO:
        _COO[seed] = boundary_coo(seed)
    return _COO[seed]


def stream():
    return torch.cuda.current_stream().cuda_stream


class DevGraph:
    """stag_csx_build with the optional schedules in `drop` passed as NULL."""

    def __init__(self, src, dst, n, by_dst, drop=()):
        from stag_b200 import _lib
        lib = _lib.load()
        E = len(src)
        thr = lib.stag_hub_threshold()
        dev = "cuda"
        t = {"src": torch.from_numpy(src).to(dev), "dst": torch.from_numpy(dst).to(dev)}
        i32 = lambda k: torch.empty(max(k, 1), dtype=torch.int32, device=dev)  # noqa: E731
        t.update(indptr=i32(n + 1), indices=i32(E), eid=i32(E), hub_rows=i32(E // thr + 1),
                 hub_seg_ptr=i32(E // thr + 2), row_order=i32(n), erow=i32(E), eidf=i32(E),
                 items=torch.empty((lib.stag_csx_items_capacity(E, n), 4), dtype=torch.int32, device=dev))
        ws_bytes = lib.stag_csx_workspace_bytes(E, n)
        ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device=dev)
        counts = (ctypes.c_int32 * 3)(-7, -7, -7)
        p = {k: (0 if k in drop else t[k].data_ptr()) for k in SCHED}
        _lib.check(lib.stag_csx_build(t["src"].data_ptr(), t["dst"].data_ptr(), E, n, 1 if by_dst else 0,
                                      t["indptr"].data_ptr(), t["indices"].data_ptr(), t["eid"].data_ptr(),
                                      t["hub_rows"].data_ptr(), t["hub_seg_ptr"].data_ptr(), p["row_order"],
                                      p["items"], p["erow"], p["eidf"], counts, ws.data_ptr(), ws_bytes, stream()))
        self.counts = tuple(counts)
        self.t, self.drop, self.E, self.N = t, tuple(drop), E, n
        g = _lib.StagGraph()
        g.num_rows, g.num_cols, g.num_edges = n, n, E
        g.indptr, g.indices, g.eid = t["indptr"].data_ptr(), t["indices"].data_ptr(), t["eid"].data_ptr()
        g.num_hubs, g.num_hub_segs = counts[0], counts[1]
        g.hub_rows, g.hub_seg_ptr = t["hub_rows"].data_ptr(), t["hub_seg_ptr"].data_ptr()
        g.row_order, g.items, g.erow, g.eidf = p["row_order"], p["items"], p["erow"], p["eidf"]
        g.num_items = counts[2] if "items" not in drop else 0
        self.g = g

    def host(self, name):
        n = {"indptr": self.N + 1, "indices": self.E, "eid": self.E, "erow": self.E, "eidf": self.E,
             "row_order": self.N, "hub_rows": self.counts[0], "hub_seg_ptr": self.counts[0] + 1,
             "items": self.counts[2]}[name]
        return self.t[name][:n].cpu().numpy().copy()


# ---------------------------------------------------------------------------------------------------------------------
# canary buffers and layouts
class Buf:
    """Flat device buffer filled with CANARY; the logical tensor starts MARGIN (+ off) elements in."""

    def __init__(self, span, off=0, dtype=torch.float32):
        self.base = MARGIN + off
        self.raw = torch.full((self.base + span + MARGIN,), CANARY, dtype=torch.int32, device="cuda")
        self.dtype = dtype
        self.views = []

    def view(self, shape, strides):
        self.views.append((shape, strides))
        t = self.raw if self.dtype == torch.int32 else self.raw.view(torch.float32)
        return t.as_strided(shape, strides, self.base)

    @property
    def ptr(self):
        return self.raw.data_ptr() + 4 * self.base

    def assert_canary(self, what):
        raw = self.raw.cpu().numpy()
        touched = np.zeros(raw.shape, bool)
        for shape, strides in self.views:
            idx = self.base + sum(np.arange(n).reshape((-1,) + (1,) * (len(shape) - 1 - i)) * st
                                  for i, (n, st) in enumerate(zip(shape, strides)))
            touched[np.asarray(idx).reshape(-1)] = True
        bad = np.flatnonzero((raw != CANARY) & ~touched)
        assert bad.size == 0, "%s: %d floats outside the logical region were written (first at %d)" % (
            what, bad.size, bad[0] - self.base)


def geometry(layout, S, R, D):
    """-> (element offset, row stride, sample stride) of an [S,R,D] operand."""
    if layout == "compact":
        return 0, D, R * D
    if layout == "pad":            # ld > D (still a multiple of 4), gaps between the samples
        ld = D + 8
        return 0, ld, R * ld + 40
    if layout == "off4":           # base 4 bytes off 16-byte alignment: the scalar-load instantiations
        return 1, D, R * D
    if layout == "off8":
        return 2, D, R * D
    if layout == "inter":          # samples interleaved: [R,S,D]
        return 0, S * D, D
    raise KeyError(layout)


def place(data, layout, shared=False, dtype=torch.float32):
    """data [S,R,D] numpy -> (Buf, view, ld, sample stride); shared: one [R,D] operand with sample stride 0."""
    S, R, D = data.shape
    off, ld, ss = geometry(layout, S, R, D)
    if shared:
        ss = 0
    span = (S - 1) * ss + (R - 1) * ld + D
    b = Buf(span, off, dtype)
    v = b.view((S, R, D), (ss, ld, 1))
    v[:1].copy_(torch.from_numpy(data[:1]).to(v))
    if not shared:
        v.copy_(torch.from_numpy(data).to(v))
    return b, v, ld, ss


def out_buf(S, R, D, layout, dtype=torch.float32, fill=None):
    off, ld, ss = geometry(layout, S, R, D)
    b = Buf((S - 1) * ss + (R - 1) * ld + D, off, dtype)
    v = b.view((S, R, D), (ss, ld, 1))
    if fill is not None:
        v.fill_(fill)
    return b, v, ld, ss


# ---------------------------------------------------------------------------------------------------------------------
# cases
class Case(dict):
    __getattr__ = dict.get

    @property
    def id(self):
        return self["name"]


def R(expect, entry, D, kind, pshape="r1", K="D", S=3, layout="compact", drop=(), **kw):
    c = Case(expect=tuple(expect), entry=entry, D=D, kind=kind, pshape=pshape, K=K, S=S, layout=layout, drop=drop)
    c.update(kw)
    bits = [entry, kind, pshape if kind in ("normal", "uniform", "bernoulli", "hadamard") else None,
            "K1" if K == 1 else None, "D%d" % D, "S%d" % S, layout, "relu" if kw.get("relu") else None,
            "innorm" if kw.get("in_norm") else None, "shared" if kw.get("shared") else None,
            "mean" if kw.get("mean") else None, "nodx" if kw.get("no_dx") else None,
            "no-" + "-".join(drop) if drop else None, kw.get("tag")]
    c["name"] = "_".join(b for b in bits if b)
    return c


def make_params(kind, pshape, E, K, relu, rng):
    if kind in ("none", "ext"):
        return None, None
    shape = {"r1": (1,), "rc": (K,), "re": (E,), "rec": (E, K)}[pshape]
    if kind in ("normal", "hadamard"):
        a = (0.2 if relu else 1.0) + 0.1 * rng.standard_normal(shape)
        b = (1.0 if relu else 0.3) + 0.2 * rng.uniform(size=shape)
    elif kind == "uniform":
        a = (-0.5 if relu else 0.5) + 0.1 * rng.standard_normal(shape)
        b = a + 1.0 + 0.1 * rng.uniform(size=shape)
    else:
        a, b = 0.6 + 0.2 * rng.uniform(size=shape), None
    T = lambda v: None if v is None else torch.from_numpy(np.asarray(v, np.float32)).cuda()  # noqa: E731
    return T(a), T(b)


def noise_struct(c, K, p0, p1, ext, sample_base, in_norm=None):
    from stag_b200 import _lib
    nz = _lib.StagNoise()
    nz.kind, nz.K, nz.param_shape = KIND[c.kind], K, PSHAPE[c.pshape]
    nz.relu = int(bool(c.relu))
    nz.in_norm = int(bool(c.in_norm if in_norm is None else in_norm))
    nz.sample_base = sample_base
    nz.p0 = 0 if p0 is None else p0.data_ptr()
    nz.p1 = 0 if p1 is None else p1.data_ptr()
    nz.external = 0 if ext is None else ext.data_ptr()
    nz.seed, nz.offset = 1234 + c.get("seed", 0), 77
    nz.counter = 0
    return nz


def emitted(c, K, p0, p1, E, S, sample_base):
    """The materialised noise (w, raw variate) [S,E,K] of the case's spec, float64 on the host."""
    from stag_b200 import _lib
    lib = _lib.load()
    nz = noise_struct(c, K, p0, p1, None, sample_base, in_norm=False)
    w = torch.empty((S, E, K), device="cuda")
    raw = torch.empty((S, E, K), device="cuda")
    _lib.check(lib.stag_noise_emit(ctypes.byref(nz), E, S, w.data_ptr(), raw.data_ptr(), stream()))
    torch.cuda.synchronize()
    return w.cpu().double(), raw.cpu().double()


def close(a, b, what, rtol=1e-5, extra=0.0):
    """test_gpu_spmm.close: |a - b| <= rtol |b| + 1e-6 max|b| (+ extra, elementwise), elementwise."""
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    if not b.size:
        return
    assert np.isfinite(a).all(), "%s: %d non-finite entries (canary left in the logical region?)" % (
        what, int((~np.isfinite(a)).sum()))
    scale = max(np.abs(b).max(), 1e-30)
    bad = np.abs(a - b) > rtol * np.abs(b) + 1e-6 * scale + extra
    assert not bad.any(), "%s: %d entries beyond tolerance (worst |a-b| = %.3e, max|ref| = %.3e)" % (
        what, int(bad.sum()), np.abs(a - b)[bad].max(), scale)


def close_sum(a, b, n_terms, what):
    """Summed parameter gradients: max|a - b| <= 2e-5 max|b| + 1e-6 sqrt(n_terms) (test_fused_parameter_gradients)."""
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    assert np.isfinite(a).all(), "%s: non-finite entries" % what
    err = np.abs(a - b).max()
    lim = 2e-5 * np.abs(b).max() + 1e-6 * np.sqrt(n_terms)
    assert err <= lim, "%s: max err %.3e > %.3e" % (what, err, lim)


def param_reduce(g, pshape, E, K):
    """[S,E,K] per-(sample, edge, channel) terms -> the parameter shape."""
    if pshape == "r1":
        return g.sum().reshape(1)
    if pshape == "rc":
        return g.sum((0, 1)).reshape(K)
    if pshape == "re":
        return g.sum((0, 2)).reshape(E)
    return g.sum(0).reshape(E * K)


# ---------------------------------------------------------------------------------------------------------------------
# one call through the C ABI, its oracle and its canaries
def run_case(c, check=True, trace=True, sample_slice=None):
    """Run case `c`.  -> (dict of logical outputs as numpy, set of launched kernel names or None).
    sample_slice=(s0, n): run samples s0..s0+n-1 of the case's data as one launch with sample_base + s0."""
    call, finish = prepare(c, sample_slice)
    if trace:
        rc, names = traced(call)
    else:
        rc, names = call(), None
        torch.cuda.synchronize()
    return finish(rc, names, check)


def prepare(c, sample_slice=None, st=None):
    """Inputs, canary buffers and the C call of case `c` on stream `st` (default: the current stream).
    -> (call() -> return code, finish(rc, names, check) -> (outputs, names))."""
    from stag_b200 import _lib
    lib = _lib.load()
    # the data depend on the operation, not on the layout or the schedules: those runs must agree bitwise
    key = repr([c.get(k) for k in ("entry", "kind", "pshape", "K", "D", "S", "relu", "in_norm", "shared", "mean")])
    rng = np.random.default_rng(zlib.crc32(key.encode()))
    src, dst = coo(c.get("graph_seed", 0))
    N, E, D = N_NODES, len(src), c.D
    S_all = c.S
    s0, S = (0, S_all) if sample_slice is None else sample_slice
    K = 1 if c.K == 1 else D
    by_dst = c.entry in ("fwd", "max_fwd")
    G = DevGraph(src, dst, N, by_dst, c.drop)
    p0, p1 = make_params(c.kind, c.pshape, E, K, c.relu, rng)
    ext_all = (1 + 0.4 * rng.standard_normal((S_all, E, K))).astype(np.float32) if c.kind == "ext" else None
    Sx = 1 if c.shared else S_all
    x_all = rng.standard_normal((Sx, N, D)).astype(np.float32)
    if c.entry in ("max_fwd", "max_bwd"):
        x_all[:, TIE_U[0]] = x_all[:, TIE_U[1]] = 50.0 + np.abs(x_all[:, TIE_U[0]])   # equal winning products
        if ext_all is not None:
            ei = np.flatnonzero(src == TIE_U[0])[0], np.flatnonzero(src == TIE_U[1])[0]
            ext_all[:, ei[1]] = ext_all[:, ei[0]] = np.abs(ext_all[:, ei[0]]) + 1.0
    dout_all = rng.standard_normal((S_all, N, D)).astype(np.float32)
    ss = rng.uniform(0.5, 1.5, N).astype(np.float32) if not c.no_scales else None
    ds = rng.uniform(0.5, 1.5, N).astype(np.float32) if not c.no_scales else None
    if c.mean:
        ds = (1.0 / np.maximum(np.bincount(dst, minlength=N), 1)).astype(np.float32)
    sb = c.get("sample_base", 5) + s0
    x = x_all if c.shared else x_all[s0:s0 + S]
    ext = None if ext_all is None else torch.from_numpy(np.ascontiguousarray(ext_all[s0:s0 + S])).cuda()
    nz = noise_struct(c, K, p0, p1, ext, sb)
    dev = lambda a: None if a is None else torch.from_numpy(a).cuda()  # noqa: E731
    ssd, dsd = dev(ss), dev(ds)
    ptr = lambda t: 0 if t is None else t.data_ptr()  # noqa: E731
    ws_bytes = lib.stag_spmm_workspace_bytes(ctypes.byref(G.g), D, S)
    ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device="cuda")
    st = stream() if st is None else st
    lay = c.layout
    xb, _, ldx, xss = place(x, lay, shared=c.shared)
    bufs, res = {}, {}
    n_p = {"r1": 1, "rc": K, "re": E, "rec": E * K}[c.pshape]
    accumulate = c.pshape in ("re", "rec")

    if c.entry == "fwd":
        ob, ov, ldo, oss = out_buf(S, N, D, lay)
        bufs["out"] = ob
        nsb = None
        if c.in_norm and not c.no_ns:
            nsb = Buf(S * N * K)
            nsv = nsb.view((S, N, K), (N * K, K, 1))
            bufs["norm_scale_out"] = nsb

        def call():
            return lib.stag_spmm_fwd(ctypes.byref(G.g), xb.ptr, ldx, xss, D, S, ctypes.byref(nz), ptr(ssd), ptr(dsd),
                                     ob.ptr, ldo, oss, 0 if nsb is None else nsb.ptr, ws.data_ptr(), ws_bytes, st)
    elif c.entry == "bwd":
        gb, _, ldg, gss = place(dout_all[s0:s0 + S], lay)
        ob = None
        if not c.no_dx:
            ob, ov, lddx, dxss = out_buf(S, N, D, lay)
            bufs["dx"] = ob
        else:
            lddx, dxss = D, N * D
        pg = c.kind in ("normal", "uniform")
        dpb = []
        if pg:
            for k in ("dparam0", "dparam1"):
                b = Buf(n_p)
                b.view((n_p,), (1,)).fill_(7.0)
                bufs[k] = b
                dpb.append(b)
        dwb = None
        if c.kind == "ext":
            dwb = Buf(S * E * K)
            dwv = dwb.view((S, E, K), (E * K, K, 1))
            bufs["dw_external"] = dwb

        def call():
            return lib.stag_spmm_bwd(ctypes.byref(G.g), xb.ptr, ldx, xss, gb.ptr, ldg, gss, D, S, ctypes.byref(nz),
                                     ptr(ssd), ptr(dsd), 0 if ob is None else ob.ptr, lddx, dxss,
                                     dpb[0].ptr if pg else 0, dpb[1].ptr if pg else 0, 0 if dwb is None else dwb.ptr,
                                     ws.data_ptr(), ws_bytes, st)
    elif c.entry == "max_fwd":
        ob, ov, ldo, oss = out_buf(S, N, D, lay)
        ab, av, _, _ = out_buf(S, N, D, lay, dtype=torch.int32)
        bufs["out"], bufs["arg"] = ob, ab

        def call():
            return lib.stag_spmm_max_fwd(ctypes.byref(G.g), xb.ptr, ldx, xss, D, S, ctypes.byref(nz), ob.ptr, ab.ptr,
                                         ldo, oss, ws.data_ptr(), ws_bytes, st)
    else:  # max_bwd: the winners come from the oracle forward (exact)
        arg_all = np.stack([max_oracle(src, dst, N, x_all[0 if c.shared else s], wf)[1]
                            for s, wf in enumerate(_max_weights(c, K, p0, p1, E, S_all, sb - s0, ext_all))])
        gb, _, ldg, gss = place(dout_all[s0:s0 + S], lay)
        abuf, _, _, _ = place(arg_all[s0:s0 + S].astype(np.int32), lay, dtype=torch.int32)
        ob = None
        if not c.no_dx:
            ob, ov, lddx, dxss = out_buf(S, N, D, lay)
            bufs["dx"] = ob
        else:
            lddx, dxss = D, N * D
        pg = c.kind in ("normal", "uniform") and not c.no_dparam
        dpb = []
        if pg:
            for k in ("dparam0", "dparam1"):
                b = Buf(n_p)
                b.view((n_p,), (1,)).fill_(7.0)
                bufs[k] = b
                dpb.append(b)
        dwb = None
        if c.kind == "ext":
            dwb = Buf(S * E * K)
            dwv = dwb.view((S, E, K), (E * K, K, 1))
            bufs["dw_external"] = dwb

        def call():
            return lib.stag_spmm_max_bwd(ctypes.byref(G.g), xb.ptr, ldx, xss, gb.ptr, abuf.ptr, ldg, gss, D, S,
                                         ctypes.byref(nz), 0 if ob is None else ob.ptr, lddx, dxss,
                                         dpb[0].ptr if pg else 0, dpb[1].ptr if pg else 0,
                                         0 if dwb is None else dwb.ptr, ws.data_ptr(), ws_bytes, st)

    locals_ = dict(locals())
    return call, lambda rc, names, check: _finish(c, rc, names, check, locals_)


def _finish(c, rc, names, check, L):
    from stag_b200 import _lib
    lib = _lib.load()
    bufs, res = L["bufs"], {}
    src, dst, N, E, D, S, K, s0 = (L[k] for k in ("src", "dst", "N", "E", "D", "S", "K", "s0"))
    x, x_all, ext_all, dout_all, ss, ds = (L[k] for k in ("x", "x_all", "ext_all", "dout_all", "ss", "ds"))
    p0, p1, sb, accumulate = L["p0"], L["p1"], L["sb"], L["accumulate"]
    arg_all = L.get("arg_all")
    if c.expect_rc is not None:
        assert rc == c.expect_rc, (rc, lib.stag_last_error())
        return {}, names
    assert rc == 0, lib.stag_last_error().decode()

    # ---- logical outputs --------------------------------------------------------------------------------------------
    for k, b in bufs.items():
        shape, strides = b.views[0]
        res[k] = b.view(shape, strides).cpu().numpy().copy()
        b.views = b.views[:1]
    for k, b in bufs.items():
        b.assert_canary(c.id + ": " + k)
    if not check:
        return res, names

    # ---- oracle ---------------------------------------------------------------------------------------------------
    T = torch.from_numpy
    srcT, dstT = T(src), T(dst)
    if c.kind == "none":
        w = torch.ones((S, E, K), dtype=torch.float64)
        raw = None
    elif c.kind == "ext":
        w = T(ext_all[s0:s0 + S]).double()
        raw = None
    else:
        w, raw = emitted(c, K, p0, p1, E, S, sb)
    xd = T(x).double()
    ssT = None if ss is None else T(ss).double()
    dsT = None if ds is None else T(ds).double()
    # The Uniform streaming kernel folds the weight into w = A' + B' X with X = 2^23 + h and A' = low - 128 (high - low)
    # (one FFMA per channel).  A' carries a rounding error of up to 2^-17 (high - low) -- the same for every edge of
    # scalar parameters -- so a row's error grows with sum |w x|, not with |out|.  Those rows get a bound relative
    # to the sum of the absolute terms.
    fold_u = c.kind == "uniform" and any(n.startswith("agg_stream_kernel<3,") for n in (names or ()))

    def abs_extra(src_, dst_, xs_, ws_, a_, b_):
        if not fold_u:
            return 0.0
        return 1e-5 * ref_spmm.aggregate(src_, dst_, N, xs_.abs(), ws_.abs(), src_scale=a_, dst_scale=b_).numpy()
    if c.entry == "fwd":
        outs, scales, extra = [], [], []
        for s in range(S):
            ws_ = w[s]
            if c.in_norm:
                ws_, sc = ref_spmm.in_norm(dstT, N, ws_)
                scales.append(sc)
            outs.append(ref_spmm.aggregate(srcT, dstT, N, xd[0 if c.shared else s], ws_, src_scale=ssT, dst_scale=dsT))
            extra.append(abs_extra(srcT, dstT, xd[0 if c.shared else s], ws_, ssT, dsT))
        close(res["out"], torch.stack(outs).numpy(), c.id + ": out", extra=np.asarray(extra) if fold_u else 0.0)
        empty = np.bincount(dst, minlength=N) == 0
        assert (res["out"][:, empty] == 0).all(), c.id + ": rows without in-edges must be exact 0"
        if "norm_scale_out" in res:
            close(res["norm_scale_out"], torch.stack(scales).numpy(), c.id + ": norm_scale_out")
    elif c.entry == "bwd":
        gd = T(dout_all[s0:s0 + S]).double()
        if "dx" in res:
            dxr = torch.stack([ref_spmm.aggregate(dstT, srcT, N, gd[s], w[s], src_scale=dsT, dst_scale=ssT)
                               for s in range(S)])
            extra = [abs_extra(dstT, srcT, gd[s], w[s], dsT, ssT) for s in range(S)]
            close(res["dx"], dxr.numpy(), c.id + ": dx", extra=np.asarray(extra) if fold_u else 0.0)
            empty = np.bincount(src, minlength=N) == 0
            assert (res["dx"][:, empty] == 0).all(), c.id + ": rows without out-edges must be exact 0"
        # dw[s,e,c] = (ss[u] x[s,u,c]) (ds[v] dout[s,v,c])
        xs_ = xd[:, src] * (1 if ssT is None else ssT[src][None, :, None])
        gs_ = gd[:, dst] * (1 if dsT is None else dsT[dst][None, :, None])
        dw = (xs_ * gs_)
        if K == 1:
            dw = dw.sum(-1, keepdim=True)
        if "dw_external" in res:
            close(res["dw_external"], dw.numpy(), c.id + ": dw_external")
        if "dparam0" in res:
            check_param_grads(c, res, dw, w, raw, E, K, D, S, accumulate)
    elif c.entry == "max_fwd":
        for s in range(S):
            o, a = max_oracle(src, dst, N, x[0 if c.shared else s], w[s].float().numpy())
            assert np.array_equal(res["out"][s].view(np.int32), o.view(np.int32)), \
                "%s: max values differ (sample %d, %d entries)" % (c.id, s, int((res["out"][s] != o).sum()))
            assert np.array_equal(res["arg"][s], a), "%s: winning edges differ (sample %d, %d entries)" % (
                c.id, s, int((res["arg"][s] != a).sum()))
    else:
        arg = T(arg_all[s0:s0 + S].astype(np.int64))
        gd = T(dout_all[s0:s0 + S]).double()
        win = torch.zeros((S, E, D), dtype=torch.float64)
        eids = torch.arange(E)
        win = (arg[:, dst] == eids[None, :, None]).double()     # [S,E,D]: edge e wins (s, dst[e], c)
        wD = w.expand(S, E, D) if K == 1 else w
        if "dx" in res:
            msg = win * wD * gd[:, dst]
            dxr = torch.zeros((S, N, D), dtype=torch.float64).index_add(1, srcT, msg)
            close(res["dx"], dxr.numpy(), c.id + ": dx")
        dw = win * xd[:, src] * gd[:, dst] if not c.shared else win * xd[0][src][None] * gd[:, dst]
        if K == 1:
            dw = dw.sum(-1, keepdim=True)
        if "dw_external" in res:
            close(res["dw_external"], dw.numpy(), c.id + ": dw_external")
        if "dparam0" in res:
            check_param_grads(c, res, dw, w, raw, E, K, D, S, accumulate)
    return res, names


def check_param_grads(c, res, dw, w, raw, E, K, D, S, accumulate):
    if c.relu:
        dw = dw * (w > 0)
    if c.kind == "normal":
        g0, g1 = dw, dw * raw
    else:
        g1 = dw * raw
        g0 = dw - g1
    n_terms = S * {"r1": E * D, "rc": E * (D // K), "re": D, "rec": 1}[c.pshape]
    for k, g in (("dparam0", g0), ("dparam1", g1)):
        ref = param_reduce(g, c.pshape, E, K).numpy()
        got = res[k].astype(np.float64)
        if accumulate:
            got = got - 7.0        # EDGE shapes accumulate into the caller's buffer
        close_sum(got, ref, n_terms, "%s: %s" % (c.id, k))


def max_oracle(src, dst, N, x, w):
    """fp32 products, first edge in edge-id order wins; -> (out float32 [N,D], arg int32 [N,D])."""
    T = torch.from_numpy
    o, a = ref_max.u_mul_e_max(T(src), T(dst), N, T(np.ascontiguousarray(x, np.float32)),
                               T(np.ascontiguousarray(w, np.float32)))
    return o.numpy(), a.numpy().astype(np.int32)


def _max_weights(c, K, p0, p1, E, S, sample_base, ext_all):
    if c.kind == "none":
        return [np.ones((E, K), np.float32)] * S
    if c.kind == "ext":
        return list(ext_all)
    w, _ = emitted(c, K, p0, p1, E, S, sample_base)
    return [w[s].float().numpy() for s in range(S)]


# ---------------------------------------------------------------------------------------------------------------------
# the route table
# D = 64 / 40 / 128 / 96 give the streaming kernel's (NB, FULL) = (1, 1) / (1, 0) / (2, 1) / (2, 0)
ROUTES = []
_STREAM_D = ((64, "1,1"), (40, "1,0"), (128, "2,1"), (96, "2,0"))
for _D, _nf in _STREAM_D:
    ROUTES.append(R(["agg_stream_kernel<0,%s,0>" % _nf, "hub_finalize_kernel"], "fwd", _D, "none", mean=True))
    ROUTES.append(R(["agg_stream_kernel<2,%s,0>" % _nf], "fwd", _D, "normal", "r1" if _D != 96 else "re"))
    ROUTES.append(R(["agg_stream_kernel<3,%s,0>" % _nf], "fwd", _D, "uniform", "re" if _D == 64 else "r1"))
    ROUTES.append(R(["agg_stream_kernel<4,%s,0>" % _nf], "fwd", _D, "bernoulli", "r1"))
    ROUTES.append(R(["agg_stream_kernel<4,%s,1>" % _nf, "hub_finalize_kernel"], "fwd", _D, "bernoulli", "r1",
                    in_norm=True))
ROUTES += [
    # two-sum / per-edge-weight streaming kernel (forward) and its gradient form (backward)
    R(["agg_stream_grads_kernel<0,1,0,1>"], "fwd", 64, "ext", K=1),
    R(["agg_stream_grads_kernel<0,1,0,2>"], "fwd", 128, "normal", "r1", K=1, shared=True),
    R(["agg_stream_grads_kernel<2,0,0,1>"], "fwd", 64, "normal", "rc"),
    R(["agg_stream_grads_kernel<2,0,0,2>"], "fwd", 128, "normal", "r1", relu=True),
    R(["agg_stream_grads_kernel<3,0,0,1>"], "fwd", 40, "uniform", "rc", mean=True),
    R(["agg_stream_grads_kernel<3,0,0,2>"], "fwd", 128, "uniform", "r1", relu=True),
    R(["agg_stream_grads_kernel<2,0,1,1>", "param_finalize_kernel", "hub_finalize_kernel"], "bwd", 64, "normal", "rc"),
    R(["agg_stream_grads_kernel<2,0,1,2>", "param_finalize_kernel"], "bwd", 128, "normal", "r1", shared=True),
    R(["agg_stream_grads_kernel<3,0,1,1>", "param_finalize_kernel"], "bwd", 96, "uniform", "rc", relu=True),
    R(["agg_stream_grads_kernel<3,0,1,2>", "param_finalize_kernel"], "bwd", 128, "uniform", "r1", no_dx=True),
    # row-per-group family, forward: no schedules (FOLD) / relu / in-norm / per-channel parameters / 4-byte offsets
    R(["agg_kernel<0,0,0,1,0,0>", "hub_finalize_kernel"], "fwd", 64, "none", drop=("items",)),
    R(["agg_kernel<0,0,0,0,0,0>"], "fwd", 64, "none", layout="off4"),
    R(["agg_kernel<0,0,0,1,0,0>"], "fwd", 128, "normal", "re", K=1, relu=True),
    R(["agg_kernel<1,0,0,1,0,0>"], "fwd", 64, "ext", layout="pad"),
    R(["agg_kernel<1,0,0,0,0,0>"], "fwd", 40, "ext", layout="off8"),
    R(["agg_kernel<2,2,0,1,0,1>", "hub_finalize_kernel"], "fwd", 128, "normal", "r1", drop=NO_SCHED),
    R(["agg_kernel<2,2,0,0,0,1>"], "fwd", 64, "normal", "re", layout="off4", drop=SCHED),
    R(["agg_kernel<2,3,0,1,0,1>"], "fwd", 64, "uniform", "r1", drop=("erow",)),
    R(["agg_kernel<2,3,0,0,0,1>"], "fwd", 128, "uniform", "re", layout="off4"),
    R(["agg_kernel<2,4,0,1,0,1>"], "fwd", 96, "bernoulli", "re", drop=("eidf",), mean=True),
    R(["agg_kernel<2,4,0,0,0,1>"], "fwd", 40, "bernoulli", "r1", layout="off4"),
    R(["agg_kernel<2,2,0,1,0,0>"], "fwd", 128, "normal", "r1", in_norm=True),
    R(["agg_kernel<2,2,0,0,0,0>"], "fwd", 64, "normal", "re", relu=True, layout="off4"),
    R(["agg_kernel<2,3,0,1,0,0>"], "fwd", 64, "uniform", "re", relu=True),
    R(["agg_kernel<2,3,0,0,0,0>"], "fwd", 40, "uniform", "r1", in_norm=True, layout="off4"),
    R(["agg_kernel<2,4,0,1,0,0>"], "fwd", 64, "bernoulli", "r1", in_norm=True, drop=NO_SCHED),
    R(["agg_kernel<2,4,0,0,0,0>"], "fwd", 128, "bernoulli", "re", in_norm=True, layout="off4"),
    R(["agg_kernel<2,2,1,1,0,0>"], "fwd", 64, "normal", "rc", in_norm=True),
    R(["agg_kernel<2,2,1,0,0,0>"], "fwd", 40, "normal", "rc", layout="off4"),
    R(["agg_kernel<2,3,1,1,0,0>"], "fwd", 640, "uniform", "rc"),
    R(["agg_kernel<2,3,1,0,0,0>"], "fwd", 64, "uniform", "rc", relu=True, layout="off4"),
    R(["agg_kernel<2,4,1,1,0,0>"], "fwd", 128, "bernoulli", "rc", shared=True),
    R(["agg_kernel<2,4,1,0,0,0>"], "fwd", 64, "bernoulli", "rc", in_norm=True, layout="off4"),
    R(["agg_kernel<2,2,2,1,0,0>"], "fwd", 64, "normal", "rec", in_norm=True),
    R(["agg_kernel<2,2,2,0,0,0>"], "fwd", 40, "normal", "rec", relu=True, layout="off4"),
    R(["agg_kernel<2,3,2,1,0,0>"], "fwd", 128, "uniform", "rec", layout="inter"),
    R(["agg_kernel<2,3,2,0,0,0>"], "fwd", 64, "uniform", "rec", layout="off4"),
    R(["agg_kernel<2,4,2,1,0,0>"], "fwd", 96, "bernoulli", "rec"),
    R(["agg_kernel<2,4,2,0,0,0>"], "fwd", 64, "bernoulli", "rec", layout="off8"),
    # row-per-group family, backward (GRADS)
    R(["agg_kernel<0,0,0,1,1,0>", "hub_finalize_kernel"], "bwd", 64, "none", layout="pad"),
    R(["agg_kernel<0,0,0,0,1,0>"], "bwd", 40, "none", layout="off4"),
    R(["agg_kernel<0,0,0,1,1,0>", "param_finalize_kernel"], "bwd", 64, "normal", "r1", K=1),
    R(["agg_kernel<0,0,0,0,1,0>"], "bwd", 64, "uniform", "re", K=1, S=1, drop=("erow",), layout="off4"),
    R(["agg_kernel<1,0,0,1,1,0>"], "bwd", 64, "ext", layout="inter"),
    R(["agg_kernel<1,0,0,0,1,0>"], "bwd", 40, "ext", layout="off4", shared=True),
    R(["agg_kernel<2,2,0,1,1,0>", "param_finalize_kernel"], "bwd", 640, "normal", "r1"),
    R(["agg_kernel<2,2,0,0,1,0>"], "bwd", 64, "normal", "r1", layout="off4", relu=True),
    R(["agg_kernel<2,2,0,1,1,0>"], "bwd", 128, "normal", "re", S=1, drop=("erow",)),
    R(["agg_kernel<2,2,0,0,1,0>"], "bwd", 64, "normal", "re", S=1, drop=("erow",), layout="off4"),
    R(["agg_kernel<2,3,0,1,1,0>"], "bwd", 64, "uniform", "re", S=1, drop=SCHED, relu=True),
    R(["agg_kernel<2,3,0,0,1,0>", "param_finalize_kernel"], "bwd", 40, "uniform", "r1", layout="off4"),
    R(["agg_kernel<2,2,1,1,1,0>", "param_finalize_kernel"], "bwd", 640, "normal", "rc"),
    R(["agg_kernel<2,2,1,0,1,0>"], "bwd", 64, "normal", "rc", layout="off4", no_dx=True),
    R(["agg_kernel<2,3,1,1,1,0>"], "bwd", 128, "uniform", "rc", drop=("items",)),
    R(["agg_kernel<2,3,1,0,1,0>"], "bwd", 40, "uniform", "rc", layout="off4"),
    R(["agg_kernel<2,2,2,1,1,0>"], "bwd", 64, "normal", "rec", S=1, drop=("erow",)),
    R(["agg_kernel<2,2,2,0,1,0>"], "bwd", 40, "normal", "rec", S=1, drop=("erow",), layout="off4", relu=True),
    R(["agg_kernel<2,3,2,1,1,0>"], "bwd", 128, "uniform", "rec", S=1, drop=("erow", "items")),
    R(["agg_kernel<2,3,2,0,1,0>"], "bwd", 64, "uniform", "rec", S=1, drop=("erow",), layout="off8"),
    R(["agg_kernel<2,4,0,1,1,0>"], "bwd", 64, "bernoulli", "r1"),
    R(["agg_kernel<2,4,0,0,1,0>"], "bwd", 40, "bernoulli", "re", layout="off4"),
    R(["agg_kernel<2,4,1,1,1,0>"], "bwd", 128, "bernoulli", "rc", shared=True),
    R(["agg_kernel<2,4,1,0,1,0>"], "bwd", 64, "bernoulli", "rc", layout="off4"),
    R(["agg_kernel<2,4,2,1,1,0>"], "bwd", 96, "bernoulli", "rec"),
    R(["agg_kernel<2,4,2,0,1,0>"], "bwd", 64, "bernoulli", "rec", layout="off4"),
    # per-edge parameter gradients, edge-parallel (graphs with erow)
    R(["edge_param_grads_fast_kernel", "agg_stream_kernel<2,2,1,0>"], "bwd", 128, "normal", "re"),
    R(["edge_param_grads_fast_kernel"], "bwd", 256, "normal", "re", no_dx=True, shared=True),
    R(["edge_param_grads_kernel<2,1>"], "bwd", 64, "normal", "rec"),
    R(["edge_param_grads_kernel<2,1>"], "bwd", 128, "normal", "re", relu=True),
    R(["edge_param_grads_kernel<2,0>"], "bwd", 64, "normal", "rec", layout="off4"),
    R(["edge_param_grads_kernel<3,1>"], "bwd", 128, "uniform", "re"),
    R(["edge_param_grads_kernel<3,1>"], "bwd", 40, "uniform", "rec", relu=True, no_dx=True),
    R(["edge_param_grads_kernel<3,0>"], "bwd", 64, "uniform", "re", K=1, layout="off4"),
    # tensor-core generator, default form
    R(["agg_wh_quad_kernel<4,4,1,2,1,1>", "hub_finalize_kernel"], "fwd", 128, "hadamard", "r1"),
    R(["agg_wh_quad_kernel<4,4,1,2,1,1>"], "fwd", 256, "hadamard", "re", shared=True),
    # max
    R(["max_row_kernel<0,1,0>", "max_hub_finalize_kernel"], "max_fwd", 64, "none"),
    R(["max_row_kernel<0,0,0>"], "max_fwd", 40, "none", layout="off4"),
    R(["max_row_kernel<1,1,0>"], "max_fwd", 64, "ext", layout="pad"),
    R(["max_row_kernel<1,0,0>"], "max_fwd", 64, "ext", K=1, layout="off4"),
    R(["max_row_kernel<2,1,0>"], "max_fwd", 128, "normal", "rc", drop=SCHED),
    R(["max_row_kernel<2,0,0>"], "max_fwd", 64, "normal", "re", relu=True, layout="off4"),
    R(["max_row_kernel<3,1,0>"], "max_fwd", 64, "uniform", "r1", layout="inter"),
    R(["max_row_kernel<3,0,0>"], "max_fwd", 40, "uniform", "rc", layout="off8"),
    R(["max_row_kernel<4,1,0>"], "max_fwd", 64, "bernoulli", "r1", shared=True),
    R(["max_row_kernel<4,0,0>"], "max_fwd", 64, "bernoulli", "re", layout="off4"),
    R(["max_wh_kernel<0>", "max_hub_finalize_kernel"], "max_fwd", 128, "hadamard", "r1"),
    R(["max_row_kernel<0,1,1>", "hub_finalize_kernel"], "max_bwd", 64, "none"),
    R(["max_row_kernel<0,0,1>"], "max_bwd", 40, "none", layout="off4"),
    R(["max_row_kernel<1,1,1>", "max_edge_kernel<1,1>"], "max_bwd", 64, "ext"),
    R(["max_row_kernel<1,0,1>", "max_edge_kernel<1,0>"], "max_bwd", 64, "ext", K=1, layout="off4"),
    R(["max_row_kernel<2,1,1>", "param_finalize_kernel"], "max_bwd", 64, "normal", "rc"),
    R(["max_row_kernel<2,0,1>", "param_finalize_kernel"], "max_bwd", 64, "normal", "r1", relu=True, layout="off4"),
    R(["max_row_kernel<3,1,1>", "param_finalize_kernel"], "max_bwd", 128, "uniform", "r1", layout="pad"),
    R(["max_row_kernel<3,0,1>"], "max_bwd", 40, "uniform", "rc", layout="off4", shared=True),
    R(["max_row_kernel<4,1,1>"], "max_bwd", 64, "bernoulli", "rc"),
    R(["max_row_kernel<4,0,1>"], "max_bwd", 64, "bernoulli", "r1", layout="off4"),
    R(["max_wh_kernel<1>"], "max_bwd", 128, "hadamard", "r1"),
    R(["max_edge_kernel<2,1>"], "max_bwd", 64, "normal", "re", no_dx=True),
    R(["max_edge_kernel<2,0>", "max_row_kernel<2,0,1>"], "max_bwd", 64, "normal", "re", K=1, layout="off4"),
    R(["max_edge_kernel<3,1>"], "max_bwd", 128, "uniform", "re", relu=True),
    R(["max_edge_kernel<3,0>"], "max_bwd", 40, "uniform", "re", layout="off4"),
]
# the seven other forms of the tensor-core kernel (STAG_WQ_VARIANT, read once per process: child interpreters)
WQ_FORMS = {1: "agg_wh_quad_kernel<4,4,0,2,1,0>", 2: "agg_wh_quad_kernel<4,2,0,3,0,0>",
            3: "agg_wh_quad_kernel<8,2,1,2,0,0>", 4: "agg_wh_quad_kernel<4,4,1,2,0,0>",
            5: "agg_wh_quad_kernel<4,4,1,2,2,0>", 6: "agg_wh_quad_kernel<4,4,1,2,1,0>",
            7: "agg_wh_quad_kernel<4,4,1,2,2,1>"}
WQ_CASE = R([], "fwd", 256, "hadamard", "r1", tag="wq")
EXCLUDED = {}

_ids = [c.id for c in ROUTES]
assert len(set(_ids)) == len(_ids), "duplicate route ids"


def route_names():
    names = {n for c in ROUTES for n in c.expect}
    return names | set(WQ_FORMS.values())


# ---------------------------------------------------------------------------------------------------------------------
# 1. routes
@pytest.mark.parametrize("case", ROUTES, ids=_ids)
def test_route_launches_its_kernel_and_matches_the_oracle(case):
    _, names = run_case(case)
    missing = [n for n in case.expect if n not in names]
    assert not missing, "%s: expected %s, launched %s" % (case.id, missing, sorted(names))


def library_instantiations():
    from stag_b200 import _lib
    path = os.environ.get("STAG_B200_LIB") or _lib.LIB_PATH
    nm = shutil.which("nm")
    assert nm, "nm (binutils) is needed to list the library's kernels"
    out = subprocess.run([nm, "-C", path], capture_output=True, text=True, timeout=120, check=True).stdout
    found = set()
    for line in out.splitlines():
        parts = line.split(None, 2)
        if len(parts) == 3 and "stag::" in parts[2]:
            n = norm_name(parts[2])
            if in_family(n):
                found.add(n)
    return found


def test_every_instantiation_has_a_route():
    found = library_instantiations()
    assert len(found) > 100, sorted(found)
    covered = route_names() | set(EXCLUDED)
    missing = sorted(found - covered)
    assert not missing, "instantiations with no route and no exclusion: %s" % missing
    stale = sorted(n for n in covered if n not in found)
    assert not stale, "routes name kernels the library does not contain: %s" % stale


# ---------------------------------------------------------------------------------------------------------------------
# 2. optional graph schedules
def radix_coo():
    rng = np.random.default_rng(9)
    n, e = 9000, 30000
    src, dst = rng.integers(0, n, e), rng.integers(0, n, e)
    dst[:400] = 17
    dst[400:528] = 18          # exactly 128: not a hub
    src[:300] = 5
    return src.astype(np.int64), dst.astype(np.int64), n


@pytest.mark.parametrize("which", ["single_cta", "radix"])
@pytest.mark.parametrize("by_dst", [1, 0])
def test_null_schedules_leave_the_structure_unchanged(which, by_dst):
    if which == "single_cta":
        (src, dst), n = coo(), N_NODES
    else:
        src, dst, n = radix_coo()
    full = DevGraph(src, dst, n, by_dst)
    ref = {k: full.host(k) for k in ("indptr", "indices", "eid", "hub_rows", "hub_seg_ptr") + SCHED}
    for mask in range(1, 16):
        drop = tuple(k for i, k in enumerate(SCHED) if mask >> i & 1)
        g = DevGraph(src, dst, n, by_dst, drop)
        assert g.counts[:2] == full.counts[:2], (drop, g.counts, full.counts)
        if "items" not in drop:
            assert g.counts[2] == full.counts[2], (drop, g.counts, full.counts)
        for k in ref:
            if k not in drop:
                assert np.array_equal(g.host(k), ref[k]), (which, by_dst, drop, k)


@pytest.mark.parametrize("entry", ["fwd", "max_fwd"])
def test_every_kind_and_parameter_shape_on_a_graph_without_schedules(entry):
    kinds = [("none", "r1"), ("ext", "r1")] + [(k, p) for k in ("normal", "uniform", "bernoulli")
                                               for p in ("r1", "rc", "re", "rec")]
    for kind, pshape in kinds:
        if entry == "max_fwd" and pshape == "rec":
            continue
        for drop in (SCHED, ("row_order", "items")):
            run_case(R([], entry, 64, kind, pshape, drop=drop), trace=False)


def test_row_order_does_not_change_the_result():
    for entry, kind, pshape in (("fwd", "normal", "rc"), ("fwd", "bernoulli", "r1"), ("bwd", "normal", "rc"),
                                ("max_fwd", "uniform", "r1"), ("max_bwd", "normal", "rc")):
        a, _ = run_case(R([], entry, 64, kind, pshape, drop=("items",)), check=False, trace=False)
        b, _ = run_case(R([], entry, 64, kind, pshape, drop=("items", "row_order")), check=False, trace=False)
        for k in a:
            if k.startswith("dparam") and entry == "bwd":
                # the summed scalar / per-channel parameter gradients of the row-per-group kernel collect per-CTA
                # partials in the order the rows are visited: row_order moves their last bits (include/stag_b200.h)
                close_sum(a[k], b[k], 3 * len(coo()[0]), (entry, kind, k))
                continue
            assert np.array_equal(a[k].view(np.int32), b[k].view(np.int32)), (entry, kind, k)


def test_per_edge_gradients_without_erow_need_one_sample():
    from stag_b200 import _lib
    for pshape in ("re", "rec"):
        run_case(R([], "bwd", 64, "normal", pshape, S=2, drop=("erow",), expect_rc=_lib.STAG_EINVAL), trace=False)


# ---------------------------------------------------------------------------------------------------------------------
# 3. strided / offset / interleaved buffers: bitwise equal to the compact call when the kernel is the same
@pytest.mark.parametrize("entry,kind,pshape,D", [("fwd", "normal", "r1", 128), ("fwd", "ext", "r1", 64),
                                                 ("fwd", "bernoulli", "rc", 64), ("bwd", "normal", "rc", 64),
                                                 ("bwd", "uniform", "re", 128), ("max_fwd", "normal", "r1", 64),
                                                 ("max_bwd", "uniform", "rc", 64), ("fwd", "hadamard", "r1", 128)])
def test_strided_layouts_equal_the_compact_call(entry, kind, pshape, D):
    base, base_names = run_case(R([], entry, D, kind, pshape))
    for layout in ("pad", "inter", "off4", "off8"):
        if kind == "hadamard" and layout in ("off4", "off8"):
            continue
        res, names = run_case(R([], entry, D, kind, pshape, layout=layout))
        if names == base_names:
            for k in base:
                assert np.array_equal(res[k].view(np.int32), base[k].view(np.int32)), (layout, k)


def test_strided_hadamard_rows_are_refused():
    from stag_b200 import _lib
    run_case(R([], "fwd", 128, "hadamard", "r1", layout="off4", expect_rc=_lib.STAG_EUNSUPPORTED), trace=False)


# ---------------------------------------------------------------------------------------------------------------------
# 4. boundary degrees: the route cases all run on the boundary graph; here the tie across a segment boundary
@pytest.mark.parametrize("kind", ["none", "ext"])
def test_max_tie_across_a_hub_segment_goes_to_the_first_edge(kind):
    src, dst = coo()
    row = IN_ROWS[DEGS.index(257)]
    e = np.flatnonzero(dst == row)
    res, _ = run_case(R([], "max_fwd", 64, kind))
    assert (res["arg"][:, row] == e[127]).all(), np.unique(res["arg"][:, row])
    run_case(R([], "max_bwd", 64, kind))


def test_boundary_graph_has_the_intended_degrees():
    src, dst = coo()
    indeg, outdeg = np.bincount(dst, minlength=N_NODES), np.bincount(src, minlength=N_NODES)
    assert tuple(indeg[list(IN_ROWS)]) == DEGS
    assert tuple(outdeg[list(OUT_ROWS)]) == DEGS


# ---------------------------------------------------------------------------------------------------------------------
# 5. column blocks and the tensor-core forms (knobs read once per process: child interpreters)
def run_child(env, args, timeout=600):
    e = dict(os.environ)
    e.update(env)
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "child"] + args, env=e, capture_output=True,
                       text=True, timeout=timeout, cwd=ROOT)
    assert r.returncode == 0, "child %s %s failed:\n%s\n%s" % (env, args, r.stdout[-4000:], r.stderr[-4000:])
    return json.loads(r.stdout.strip().splitlines()[-1])


def ncb_cases():
    cases = []
    for D in (64, 128, 192, 256, 640):
        for S in (1, 3):
            for shared in (True, False):
                for kind, pshape in (("none", "r1"), ("ext", "r1"), ("normal", "r1"), ("uniform", "rc"),
                                     ("bernoulli", "re"), ("normal", "rec")):
                    cases.append(R([], "fwd", D, kind, pshape, S=S, shared=shared, tag="ncb"))
    return cases


def big_graph(N, E, seed, hub_rows=(7, 11)):
    rng = np.random.default_rng(seed)
    src = rng.integers(0, N, E).astype(np.int64)
    dst = rng.integers(0, N, E).astype(np.int64)
    dst[:600] = hub_rows[0]
    dst[600:728] = hub_rows[1]   # exactly 128
    return src, dst


def subset_check(src, dst, rows, got, x_rows_fn, w_of_edges, ss=None, ds=None, what=""):
    """float64 sum over the in-edges of `rows` only."""
    sel = np.isin(dst, rows)
    e = np.flatnonzero(sel)
    xs = torch.from_numpy(x_rows_fn(src[e])).double()
    if ss is not None:
        xs = xs * torch.from_numpy(ss[src[e]]).double()[:, None]
    m = xs * w_of_edges(e)
    pos = {r: i for i, r in enumerate(rows)}
    idx = torch.tensor([pos[v] for v in dst[e]], dtype=torch.int64)
    ref = torch.zeros((len(rows), xs.shape[1]), dtype=torch.float64).index_add(0, idx, m)
    if ds is not None:
        ref = ref * torch.from_numpy(ds[rows]).double()[:, None]
    close(got, ref.numpy(), what)


def test_natural_column_blocks_box_muller():
    """A gathered operand just above 96 MB splits into column blocks without any knob."""
    from stag_b200 import _lib
    lib = _lib.load()
    N, E, D, S = 200_000, 600_000, 128, 3
    src, dst = big_graph(N, E, 3)
    c = R([], "fwd", D, "normal", "r1", S=S)
    G = DevGraph(src, dst, N, True)
    rng = np.random.default_rng(4)
    x = torch.randn((N, D), device="cuda")
    p0, p1 = make_params("normal", "r1", E, D, False, rng)
    ds = rng.uniform(0.5, 1.5, N).astype(np.float32)
    dsd = torch.from_numpy(ds).cuda()
    nz = noise_struct(c, D, p0, p1, None, 5)
    out = torch.empty((S, N, D), device="cuda")
    wsb = lib.stag_spmm_workspace_bytes(ctypes.byref(G.g), D, S)
    ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
    rc, names = traced(lambda: lib.stag_spmm_fwd(ctypes.byref(G.g), x.data_ptr(), D, 0, D, S, ctypes.byref(nz), 0,
                                                 dsd.data_ptr(), out.data_ptr(), D, N * D, 0, ws.data_ptr(), wsb,
                                                 stream()))
    assert rc == 0, lib.stag_last_error()
    assert "agg_stream_kernel<2,1,0,0>" in names, sorted(names)   # 64-channel column blocks
    rows = np.concatenate([[7, 11], np.random.default_rng(5).choice(N, 300, replace=False)])
    w, _ = emitted(c, D, p0, p1, E, S, 5)
    xh = x.cpu().numpy()
    for s in range(S):
        subset_check(src, dst, rows, out[s, rows].cpu().numpy(), lambda u: xh[u], lambda e: w[s, e], ds=ds,
                     what="natural ncb sample %d" % s)


# ---------------------------------------------------------------------------------------------------------------------
# 6. gathered operands beyond 2^31 floats: 64-bit row offsets in the row-per-group kernels
def test_operand_beyond_2g_floats():
    from stag_b200 import _lib
    lib = _lib.load()
    N, E, D, LDX = 70_000, 300_000, 128, 32_768
    src, dst = big_graph(N, E, 6)
    G = DevGraph(src, dst, N, True)
    rng = np.random.default_rng(7)
    xbuf = torch.empty((N - 1) * LDX + D, device="cuda")          # 9.2 GB; only the first D columns are written
    xv = xbuf.as_strided((N, D), (LDX, 1))
    xv.copy_(torch.randn((N, D), device="cuda"))
    xh = xv.cpu().numpy()
    rows = np.concatenate([[7, 11], rng.choice(N, 200, replace=False), [N - 1]])
    wsb = lib.stag_spmm_workspace_bytes(ctypes.byref(G.g), D, 2)
    ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
    try:
        for kind, expect in (("normal", "agg_kernel<2,2,0,1,0,1>"), ("ext", "agg_kernel<1,0,0,1,0,0>"),
                             ("max", "max_row_kernel<2,1,0>")):
            S = 2
            c = R([], "fwd", D, "normal" if kind == "max" else kind, "rc" if kind == "max" else "r1", S=S)
            p0, p1 = make_params(c.kind, c.pshape, E, D, False, rng)
            ext = (1 + 0.3 * torch.randn((S, E, D), device="cuda")) if kind == "ext" else None
            nz = noise_struct(c, D, p0, p1, ext, 0)
            out = torch.empty((S, N, D), device="cuda")
            arg = torch.empty((S, N, D), dtype=torch.int32, device="cuda")
            if kind == "max":
                call = lambda: lib.stag_spmm_max_fwd(ctypes.byref(G.g), xbuf.data_ptr(), LDX, 0, D, S,  # noqa: E731
                                                     ctypes.byref(nz), out.data_ptr(), arg.data_ptr(), D, N * D,
                                                     ws.data_ptr(), wsb, stream())
            else:
                call = lambda: lib.stag_spmm_fwd(ctypes.byref(G.g), xbuf.data_ptr(), LDX, 0, D, S,  # noqa: E731
                                                 ctypes.byref(nz), 0, 0, out.data_ptr(), D, N * D, 0, ws.data_ptr(),
                                                 wsb, stream())
            rc, names = traced(call)
            assert rc == 0, lib.stag_last_error()
            assert expect in names, (kind, sorted(names))
            w = ext.cpu().double() if ext is not None else emitted(c, D, p0, p1, E, S, 0)[0]
            for s in range(S):
                if kind == "max":
                    sel = np.flatnonzero(np.isin(dst, rows))
                    sub_src, sub_dst = src[sel], dst[sel]
                    remap = {r: i for i, r in enumerate(rows)}
                    o, a = ref_max.u_mul_e_max(torch.from_numpy(sub_src), torch.tensor([remap[v] for v in sub_dst]),
                                               len(rows), torch.from_numpy(xh), w[s][sel].float())
                    a = torch.where(a >= 0, torch.from_numpy(sel)[a.clamp(min=0)], a)
                    assert np.array_equal(out[s, rows].cpu().numpy(), o.numpy()), "max values (sample %d)" % s
                    assert np.array_equal(arg[s, rows].cpu().numpy(), a.numpy().astype(np.int32)), "arg %d" % s
                else:
                    subset_check(src, dst, rows, out[s, rows].cpu().numpy(), lambda u: xh[u], lambda e: w[s, e],
                                 what="%s beyond 2^31 sample %d" % (kind, s))
        # the tensor-core generator gathers with 32-bit byte offsets: refused before any launch
        c = R([], "fwd", D, "hadamard", "r1", S=1)
        p0, p1 = make_params("hadamard", "r1", E, D, False, rng)
        nz = noise_struct(c, D, p0, p1, None, 0)
        n0 = lib.stag_launch_count()
        rc = lib.stag_spmm_fwd(ctypes.byref(G.g), xbuf.data_ptr(), LDX, 0, D, 1, ctypes.byref(nz), 0, 0,
                               out.data_ptr(), D, N * D, 0, ws.data_ptr(), wsb, stream())
        assert rc == _lib.STAG_EUNSUPPORTED, (rc, lib.stag_last_error())
        assert lib.stag_launch_count() == n0
    finally:
        del xbuf, xv
        torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------------------------------
# 7. the remaining header contracts (OVERWRITE / ACCUMULATE, dx = NULL, Bernoulli in stag_spmm_bwd and norm_scale_out
#    are asserted by the route cases above)
def test_two_streams_with_their_own_workspaces_equal_serial_calls():
    cases = [R([], "fwd", 128, "normal", "r1"), R([], "bwd", 64, "normal", "rc"), R([], "max_fwd", 64, "uniform"),
             R([], "fwd", 64, "bernoulli", "rc", drop=NO_SCHED)]
    serial = [run_case(c, check=False, trace=False)[0] for c in cases]
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    for a, b in ((0, 1), (2, 3), (0, 3)):
        with torch.cuda.stream(s1):
            ca, fa = prepare(cases[a], st=s1.cuda_stream)
        with torch.cuda.stream(s2):
            cb, fb = prepare(cases[b], st=s2.cuda_stream)
        torch.cuda.synchronize()
        ra, rb = ca(), cb()        # both enqueued before either is waited for, each with its own workspace
        torch.cuda.synchronize()
        for got, want in ((fa(ra, None, False)[0], serial[a]), (fb(rb, None, False)[0], serial[b])):
            for k in want:
                assert np.array_equal(got[k].view(np.int32), want[k].view(np.int32)), k


_SPLIT = [c for c in ROUTES if c.S > 1]


@pytest.mark.parametrize("case", _SPLIT, ids=[c.id for c in _SPLIT])
def test_sample_s_equals_a_single_sample_launch(case):
    full, _ = run_case(case, check=False, trace=False)
    for s in range(case.S):
        one, _ = run_case(case, check=False, trace=False, sample_slice=(s, 1))
        for k in ("out", "dx", "arg", "dw_external", "norm_scale_out"):
            if k in full:
                assert np.array_equal(one[k][0].view(np.int32), full[k][s].view(np.int32)), (s, k)


# The child-process cases (section 5) run last: placed before the two large in-process cases above, torch.profiler in
# this process recorded no kernel events for those.
@pytest.mark.parametrize("ncb", [2, 3])
def test_forced_column_blocks(ncb):
    out = run_child({"STAG_NCB": str(ncb)}, ["ncb"])
    assert out["ok"] == len(ncb_cases())


def test_tensor_core_forms():
    tmp = tempfile.mkdtemp()
    try:
        base, _ = run_case(WQ_CASE)
        report = {}
        for v, name in WQ_FORMS.items():
            path = os.path.join(tmp, "wq%d.npy" % v)
            out = run_child({"STAG_WQ_VARIANT": str(v)}, ["wq", path])
            assert name in out["names"], (v, out["names"])
            report[v] = bool(np.array_equal(np.load(path).view(np.int32), base["out"].view(np.int32)))
        print("STAG_WQ_VARIANT bitwise equal to the default form:", report)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


# ---------------------------------------------------------------------------------------------------------------------
# child-process mode
def _child(argv):
    torch.cuda.set_device(0)
    if argv[0] == "ncb":
        n = 0
        for c in ncb_cases():
            run_case(c)
            n += 1
        print(json.dumps({"ok": n}))
    elif argv[0] == "wq":
        res, names = run_case(WQ_CASE)
        np.save(argv[1], res["out"])
        print(json.dumps({"names": sorted(names)}))


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "child":
    _child(sys.argv[2:])
