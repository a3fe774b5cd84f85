"""Host-side operators over the C ABI (include/stag_b200.h).

``stochastic_aggregate`` is the operator the zoo layers call where the reference
calls ``graph.update_all(fn.u_mul_e('h','_edge_weight','m'), fn.sum('m','h'))``
(stag/zoo/gcn.py:63,95; stag/zoo/graph_sage.py:57,72,86).  The ``edge_weight=`` slot
of the reference's operator interface (stag/layers.py:109-113) carries either

* a tensor ``[E,K]`` / ``[E,1]`` / ``[E]`` -> EXTERNAL noise (the shared-noise parity seam),
* a :class:`NoiseSpec`                      -> noise generated inside the kernel, never stored,
* ``None``                                  -> plain copy_u / sum.

PyTorch is used for device memory, streams and autograd plumbing only; all compute
happens in libstag_b200.so.  There is no CPU fallback.
"""
import ctypes
import os

import torch

from . import _lib, random as _random
from .graph import as_graph

# 'auto' = the tensor-core generator wherever the fused kernel takes it (K % 128 == 0 or padded to it: NoiseSpec.hadamard_width; scalar / per-edge parameters
# without gradients, no relu / in-norm: 1.35 ms per arxiv launch against 1.56), else Box-Muller
_DEFAULT_NORMAL_GENERATOR = "auto"
_KIND = {"normal": _lib.NOISE_NORMAL, "uniform": _lib.NOISE_UNIFORM, "bernoulli": _lib.NOISE_BERNOULLI}


def _stream(dev):
    return torch.cuda.current_stream(dev).cuda_stream


def _ptr(t):
    return 0 if t is None else t.data_ptr()


def _require_cuda(t, what):
    if t.device.type != "cuda":
        raise _lib.StagLibraryError(
            "stag_b200: %s is on %s; the stochastic aggregation runs on CUDA only (no CPU fallback)"
            % (what, t.device))


class NoiseSpec:
    """Lazy description of the multiplicative edge noise of one StagLayer forward.

    kind         'normal' | 'uniform' | 'bernoulli'
    p0, p1       parameters in natural units (loc/scale, low/high, probs/None); tensors on
                 the graph's device; may require grad (vi=True)
    K            noise width (feat.shape[-1], 1, or base_layer.sample_dimension)
    param_shape  'scalar' | 'channel' | 'edge' | 'edge_channel'   (before expand([E,K]))
    relu, in_norm    stag/layers.py:98-105
    seed, offset     Philox key / call counter (reserved at construction)
    sample_base      global index of the first Monte-Carlo sample of this call
    generator        how standard normals are drawn: 'boxmuller' (16-bit Box-Muller in the CUDA cores),
                     'hadamard' (Walsh-Hadamard mix of random FP8 bytes on the tensor cores,
                     csrc/spmm_tc.cuh, spmm_wq.cuh) or None = hadamard wherever the fused kernel takes it (K a
                     multiple of 128 -- or within a third of one on graphs of >= 2^18 edges, run zero-padded:
                     ``hadamard_width`` -- scalar or per-edge parameters without gradients, no relu / in-norm),
                     else boxmuller; env STAG_NORMAL_GENERATOR (boxmuller | hadamard | auto) overrides the None case.  The forward, the transposed pass and
                     ``materialize`` of one spec always use the same generator.  (The tensor-core kernel addresses the
                     gathered operand with 32-bit byte offsets: beyond 4 GB per sample -- 8.4 M nodes at 128 channels --
                     it is refused with STAG_EUNSUPPORTED; pass generator='boxmuller' there.)
    """

    def __init__(self, kind, p0, p1, K, num_edges, relu=False, in_norm=False, seed=None, offset=None,
                 sample_base=0, n_samples=1, batched=False, generator=None):
        if kind not in _KIND:
            raise ValueError("unsupported noise kind %r" % (kind,))
        if generator not in (None, "boxmuller", "hadamard"):
            raise ValueError("generator must be None, 'boxmuller' or 'hadamard'; got %r" % (generator,))
        self.kind = kind
        self.generator = generator
        self.K = int(K)
        self.num_edges = int(num_edges)
        self.relu = bool(relu)
        self.in_norm = bool(in_norm)
        self.sample_base = int(sample_base)
        self.n_samples = int(n_samples)
        self.batched = bool(batched)  # caller wants [S,N,D] back even when S == 1
        if seed is None or offset is None:
            seed, offset = _random.next_offset()
        self.seed, self.offset = int(seed), int(offset)
        self.p0, self.p1, self.param_shape = self._normalise(p0, p1)

    def _normalise(self, p0, p1):
        E, K = self.num_edges, self.K

        def classify(p):
            n = p.numel()
            if n == 1:
                return _lib.PARAM_SCALAR
            if p.dim() >= 1 and p.shape[-1] == K and n == K and K != 1:
                return _lib.PARAM_CHANNEL
            if n == E and (p.dim() == 1 or p.shape[-1] == 1):
                return _lib.PARAM_EDGE
            if n == E * K and p.shape[-1] == K:
                return _lib.PARAM_EDGE_CHANNEL
            raise ValueError("noise parameter of shape %s does not expand to [E=%d, K=%d]"
                             % (tuple(p.shape), E, K))

        shapes = [classify(p) for p in (p0, p1) if p is not None]
        shape = max(shapes)

        def widen(p):
            if p is None:
                return None
            if classify(p) == shape:
                return p
            # mixed shapes (e.g. scalar loc with per-channel scale): expand to the wider one
            target = {_lib.PARAM_CHANNEL: (K,), _lib.PARAM_EDGE: (E, 1), _lib.PARAM_EDGE_CHANNEL: (E, K)}[shape]
            return p.expand(target)

        return widen(p0), widen(p1), shape

    @property
    def requires_grad(self):
        return any(p is not None and p.requires_grad for p in (self.p0, self.p1))

    @property
    def hadamard_ok(self):
        """The tensor-core generator can serve every pass of this spec at its own width."""
        return (self.kind == "normal" and self.K % 128 == 0 and not self.relu and not self.in_norm
                and self.param_shape in (_lib.PARAM_SCALAR, _lib.PARAM_EDGE) and not self.requires_grad)

    @property
    def hadamard_width(self):
        """Width the tensor-core generator runs this spec at: K itself when it is made of 128-channel groups, K rounded
        up to the next group when that costs at most a third more channels and the graph has >= 2^18 edges (products'
        100 -> 128: 49.4 -> 41.4 ms per step), else 0.  The variates of channel c depend on (edge, sample, c)
        only, so the first K channels of the padded problem ARE the problem."""
        ok = (self.kind == "normal" and not self.relu and not self.in_norm
              and self.param_shape in (_lib.PARAM_SCALAR, _lib.PARAM_EDGE) and not self.requires_grad)
        if not ok or self.K < 96:
            return 0
        Kp = (self.K + 127) // 128 * 128
        if Kp == self.K:
            return Kp
        # padding costs a pad and a slice launch: only where the pass is long enough to pay for them (a function of the
        # edge count alone, so that every view of this spec -- other sample counts, the emitted tensor -- agrees)
        return Kp if 3 * Kp <= 4 * self.K and self.num_edges >= (1 << 18) else 0

    @property
    def lib_kind(self):
        """STAG_NOISE_* of this spec (one generator for forward, backward and materialize)."""
        if self.kind != "normal":
            return _KIND[self.kind]
        gen = self.generator or os.environ.get("STAG_NORMAL_GENERATOR") or _DEFAULT_NORMAL_GENERATOR
        if gen == "hadamard":
            if not self.hadamard_width:
                raise ValueError("generator='hadamard' needs K >= 96 within a third of a multiple of 128, scalar or per-edge "
                                 "parameters without gradients and no relu / in-norm")
            return _lib.NOISE_NORMAL_HADAMARD
        if gen == "auto" and self.hadamard_width:
            return _lib.NOISE_NORMAL_HADAMARD
        return _lib.NOISE_NORMAL

    def with_samples(self, n_samples, sample_base=0):
        out = NoiseSpec.__new__(NoiseSpec)
        out.__dict__.update(self.__dict__)
        out.n_samples, out.sample_base = int(n_samples), int(sample_base)
        return out

    def materialize(self, n_samples=None, return_raw=False):
        """The noise tensor w [E,K] (or [S,E,K]) from the same Philox stream the fused
        kernels consume -- differentiable w.r.t. the parameters (compat path)."""
        S = self.n_samples if n_samples is None else int(n_samples)
        w = _NoiseEmit.apply(self, S, self.p0, self.p1)
        if self.relu:
            w = w.relu()
        return w if (S > 1 or n_samples is not None) else w[0]


def spec_samples(edge_weight, feat):
    """``n_samples`` argument for :func:`stochastic_aggregate` implied by the edge_weight slot:
    S for a sample-batched NoiseSpec, else None (plain [N,D] -> [N,D])."""
    if isinstance(edge_weight, NoiseSpec) and (edge_weight.batched or feat.dim() == 3):
        return edge_weight.n_samples
    return None


def _fill_noise(spec, kind, K, p0, p1, ext, relu, in_norm, sample_base, seed, offset, param_shape):
    n = _lib.StagNoise()
    n.kind, n.K, n.param_shape = kind, K, param_shape
    n.relu, n.in_norm, n.sample_base = int(relu), int(in_norm), int(sample_base)
    n.p0, n.p1, n.external = _ptr(p0), _ptr(p1), _ptr(ext)
    n.seed, n.offset = seed, offset
    # device-side addend to the call counter (stag_b200.random.enable_device_counter): a step captured in a CUDA graph
    # draws fresh noise on every replay
    ctr = _random.device_counter(p0.device if p0 is not None else (ext.device if ext is not None else None))
    n.counter = 0 if ctr is None else ctr.data_ptr()
    return n


def _c(t):
    if t is None:
        return None
    if t.dtype == torch.float32 and t.is_contiguous():
        return t.detach()
    return t.detach().to(torch.float32).contiguous()


class _on_device:
    """`with torch.cuda.device(dev)` only when dev is not already the current device (the context manager costs
    several microseconds per call, which is what a small-graph launch is made of)."""

    def __init__(self, dev):
        self.ctx = None if torch.cuda.current_device() == (dev.index or 0) else torch.cuda.device(dev)

    def __enter__(self):
        if self.ctx is not None:
            self.ctx.__enter__()

    def __exit__(self, *a):
        if self.ctx is not None:
            return self.ctx.__exit__(*a)


def _workspace(st, lib, gstruct, by_dst, D, S):
    """Scratch buffer of the graph, sized once per (orientation, D, S)."""
    key = (by_dst, D, S)
    cache = st.__dict__.setdefault("_ws_bytes", {})
    if key not in cache:
        cache[key] = lib.stag_spmm_workspace_bytes(ctypes.byref(gstruct), D, S)
    return st.workspace(cache[key])


class _NoiseEmit(torch.autograd.Function):
    """stag_noise_emit with reparameterisation gradients (torch reductions; compat path)."""

    @staticmethod
    def forward(ctx, spec, S, p0, p1):
        dev = p0.device
        _require_cuda(p0, "noise parameter")
        lib = _lib.load()
        E, K = spec.num_edges, spec.K
        kind = spec.lib_kind
        Kl = spec.hadamard_width if kind == _lib.NOISE_NORMAL_HADAMARD else K   # the tensor-core stream comes in groups of 128
        p0c, p1c = _c(p0), _c(p1)
        w = torch.empty((S, E, Kl), dtype=torch.float32, device=dev)
        need_raw = spec.kind != "bernoulli" and any(
            p is not None and p.requires_grad for p in (p0, p1))
        raw = torch.empty_like(w) if need_raw else None
        nz = _fill_noise(spec, kind, Kl, p0c, p1c, None, False, False, spec.sample_base,
                         spec.seed, spec.offset, spec.param_shape)
        with torch.cuda.device(dev):
            _lib.check(lib.stag_noise_emit(ctypes.byref(nz), E, S, w.data_ptr(), _ptr(raw), _stream(dev)))
        if Kl != K:
            w = w[..., :K].contiguous()
            raw = None if raw is None else raw[..., :K].contiguous()
        ctx.kind = spec.kind
        ctx.shapes = (p0.shape, None if p1 is None else p1.shape)
        ctx.save_for_backward(raw)
        return w

    @staticmethod
    def backward(ctx, gw):
        (raw,) = ctx.saved_tensors
        s0, s1 = ctx.shapes
        g0 = g1 = None
        if raw is not None:
            if ctx.kind == "normal":
                a, b = gw, gw * raw
            else:  # uniform: w = low + u (high - low)
                b = gw * raw
                a = gw - b
            if ctx.needs_input_grad[2]:
                g0 = a.sum(0).sum_to_size(s0) if len(s0) else a.sum()
            if ctx.needs_input_grad[3] and s1 is not None:
                g1 = b.sum(0).sum_to_size(s1) if len(s1) else b.sum()
        return None, None, g0, g1


class _StochasticSpMM(torch.autograd.Function):
    @staticmethod
    def forward(ctx, feat, p0, p1, ext, cfg):
        g = cfg["graph"]
        st = g._s
        dev = feat.device
        _require_cuda(feat, "feat")
        lib = _lib.load()
        S, shared = cfg["S"], cfg["shared"]
        N, NS, D = st.num_nodes, st.num_src, feat.shape[-1]  # destination rows, rows of the gathered operand
        x = _c(feat)
        p0c, p1c, extc = _c(p0), _c(p1), _c(ext)
        out = torch.empty((S, N, D), dtype=torch.float32, device=dev)
        ns = None
        if cfg["in_norm"]:
            ns = torch.empty((S, N, cfg["K"]), dtype=torch.float32, device=dev)
        with _on_device(dev):
            csc, _ = st.csx(True)
            ws = _workspace(st, lib, csc, True, D, S)
            nz = _fill_noise(None, cfg["kind"], cfg["K"], p0c, p1c, extc, cfg["relu"], cfg["in_norm"],
                             cfg["sample_base"], cfg["seed"], cfg["offset"], cfg["param_shape"])
            _lib.check(lib.stag_spmm_fwd(
                ctypes.byref(csc), x.data_ptr(), D, 0 if shared else NS * D, D, S, ctypes.byref(nz),
                _ptr(cfg["src_scale"]), _ptr(cfg["dst_scale"]), out.data_ptr(), D, N * D,
                _ptr(ns), ws.data_ptr(), ws.numel(), _stream(dev)))
        ctx.cfg = cfg
        ctx.feat_shape = feat.shape
        ctx.param_shapes = (None if p0 is None else p0.shape, None if p1 is None else p1.shape)
        ctx.ext_shape = None if ext is None else ext.shape
        need_x = any(ctx.needs_input_grad[1:4])
        ctx.save_for_backward(x if need_x else None, p0c, p1c, extc, ns)
        return out

    @staticmethod
    def backward(ctx, gout):
        cfg = ctx.cfg
        g = cfg["graph"]
        st = g._s
        x, p0c, p1c, extc, ns = ctx.saved_tensors
        lib = _lib.load()
        dev = gout.device
        S, shared = cfg["S"], cfg["shared"]
        N, NS, D, K = st.num_nodes, st.num_src, gout.shape[-1], cfg["K"]
        need_dx = ctx.needs_input_grad[0]
        need_dp = (ctx.needs_input_grad[1] or ctx.needs_input_grad[2]) and cfg["kind"] in (
            _lib.NOISE_NORMAL, _lib.NOISE_UNIFORM)
        need_dext = ctx.needs_input_grad[3] and cfg["kind"] == _lib.NOISE_EXTERNAL
        gout = gout.to(torch.float32).contiguous()
        if cfg["in_norm"]:
            if need_dp or need_dext:
                raise NotImplementedError(
                    "fused gradients w.r.t. the noise through in-norm are not available; "
                    "StagLayer routes vi=True + norm=True through the emitted-noise path")
            gout = gout * ns  # d/d(sum) of s[v,c] * sum  (s constant w.r.t. x)
        dx = dp0 = dp1 = dext = None
        with _on_device(dev):
            csr, _ = st.csx(False)
            ws = _workspace(st, lib, csr, False, D, S)
            if need_dx:
                dx = torch.empty((S, NS, D), dtype=torch.float32, device=dev)

            def noise(sample_base, ext_slice=None):
                return _fill_noise(None, cfg["kind"], K, p0c, p1c, extc if ext_slice is None else ext_slice,
                                   cfg["relu"], False, sample_base, cfg["seed"], cfg["offset"],
                                   cfg["param_shape"])

            if not (need_dp or need_dext):
                if need_dx:
                    # transposed aggregation only: the forward kernel on the CSR with the scales swapped
                    nz = noise(cfg["sample_base"])
                    _lib.check(lib.stag_spmm_fwd(
                        ctypes.byref(csr), gout.data_ptr(), D, N * D, D, S, ctypes.byref(nz),
                        _ptr(cfg["dst_scale"]), _ptr(cfg["src_scale"]), dx.data_ptr(), D, NS * D,
                        0, ws.data_ptr(), ws.numel(), _stream(dev)))
            else:
                edge_params = need_dp and cfg["param_shape"] >= _lib.PARAM_EDGE
                if need_dext:
                    dext = torch.empty((S, st.num_edges, K), dtype=torch.float32, device=dev)
                if need_dp:
                    pshape = cfg["param_shape"]
                    n = {_lib.PARAM_SCALAR: 1, _lib.PARAM_CHANNEL: K, _lib.PARAM_EDGE: st.num_edges,
                         _lib.PARAM_EDGE_CHANNEL: st.num_edges * K}[pshape]
                    dp0 = torch.zeros(n, dtype=torch.float32, device=dev)
                    dp1 = torch.zeros(n, dtype=torch.float32, device=dev)
                # per-edge parameter gradients: all samples in one launch (edge-parallel kernel) when the graph
                # carries the row of every stored edge, else one sample per launch
                groups = [(s, 1) for s in range(S)] if (edge_params and not csr.erow) else [(0, S)]
                for s0, ns_ in groups:
                    nz = noise(cfg["sample_base"] + s0,
                               None if extc is None else extc[s0:s0 + ns_])
                    xs = x if shared else x[s0:s0 + ns_]
                    _lib.check(lib.stag_spmm_bwd(
                        ctypes.byref(csr), xs.data_ptr(), D, 0 if shared else NS * D,
                        gout[s0:s0 + ns_].data_ptr(), D, N * D, D, ns_, ctypes.byref(nz),
                        _ptr(cfg["src_scale"]), _ptr(cfg["dst_scale"]),
                        0 if dx is None else dx[s0:s0 + ns_].data_ptr(), D, NS * D,
                        _ptr(dp0), _ptr(dp1), 0 if dext is None else dext[s0:s0 + ns_].data_ptr(),
                        ws.data_ptr(), ws.numel(), _stream(dev)))
        gfeat = gp0 = gp1 = gext = None
        if need_dx:
            gfeat = (dx.sum(0) if shared else dx).reshape(ctx.feat_shape)
        if need_dp:
            s0, s1 = ctx.param_shapes
            if ctx.needs_input_grad[1]:
                gp0 = dp0.reshape(s0) if dp0.numel() == max(1, _numel(s0)) else dp0.reshape(-1).sum_to_size(s0)
            if ctx.needs_input_grad[2] and s1 is not None:
                gp1 = dp1.reshape(s1) if dp1.numel() == max(1, _numel(s1)) else dp1.reshape(-1).sum_to_size(s1)
        if need_dext:
            gext = dext.reshape(ctx.ext_shape) if dext.numel() == _numel(ctx.ext_shape) else dext
        return gfeat, gp0, gp1, gext, None


def _numel(shape):
    n = 1
    for d in shape:
        n *= int(d)
    return n


def stochastic_aggregate(graph, feat, edge_weight=None, reduce="sum", src_scale=None, dst_scale=None,
                         n_samples=None):
    """out[(s,) v, c] = dst_scale[v] * sum_{e:(u->v)} w[(s,) e, c] * (src_scale[u] * feat[(s,) u, c]).

    feat ``[N,D]`` -> out ``[N,D]`` (or ``[S,N,D]`` when ``n_samples=S`` shares feat over S
    Monte-Carlo samples); feat ``[S,N,D]`` -> out ``[S,N,D]``.  ``reduce='mean'`` divides
    by clamp(in_degree, 1) (dgl fn.mean).  ``reduce='max'`` / ``'min'`` take the max / min of the
    messages w * feat[u] instead (dgl fn.max / fn.min): ties go to the first edge in edge-id order,
    which alone receives the gradient; rows without in-edges are 0.  No scales with max / min.
    """
    if reduce not in ("sum", "mean", "max", "min"):
        raise ValueError("reduce must be 'sum', 'mean', 'max' or 'min'; got %r" % (reduce,))
    if reduce in ("max", "min") and (src_scale is not None or dst_scale is not None):
        raise ValueError("reduce=%r takes no src_scale / dst_scale" % (reduce,))
    g = as_graph(graph)
    st = g._s
    N, E = st.num_nodes, st.num_edges
    _require_cuda(feat, "feat")
    if feat.dim() == 2:
        shared, S = True, (1 if n_samples is None else int(n_samples))
        squeeze = n_samples is None
    elif feat.dim() == 3:
        shared, S, squeeze = False, feat.shape[0], False
        if n_samples is not None and int(n_samples) != S:
            raise ValueError("feat has %d samples but n_samples=%s" % (S, n_samples))
    else:
        raise ValueError("feat must be [N,D] or [S,N,D]; got %s" % (tuple(feat.shape),))
    if feat.shape[-2] != st.num_src:
        raise ValueError("feat has %d rows, graph has %d source nodes" % (feat.shape[-2], st.num_src))
    D = feat.shape[-1]
    if reduce in ("max", "min"):
        if reduce == "min":  # min_e w x = -max_e w (-x): ties go to the first minimum
            out = -_aggregate_max(g, -feat, edge_weight, S, shared)
        else:
            out = _aggregate_max(g, feat, edge_weight, S, shared)
        return out[0] if squeeze else out
    if reduce == "mean":
        m = st.scale(True, "inv")
        dst_scale = m if dst_scale is None else dst_scale * m
    cfg = {"graph": g, "S": S, "shared": shared, "relu": False, "in_norm": False, "sample_base": 0,
           "seed": 0, "offset": 0, "param_shape": _lib.PARAM_SCALAR, "K": D,
           "src_scale": _c(src_scale), "dst_scale": _c(dst_scale)}
    p0 = p1 = ext = None
    if edge_weight is None:
        cfg["kind"] = _lib.NOISE_NONE
    elif isinstance(edge_weight, NoiseSpec):
        spec = edge_weight
        if spec.num_edges != E:
            raise ValueError("noise spec was made for %d edges, graph has %d" % (spec.num_edges, E))
        if spec.K not in (1, D):
            raise ValueError("noise width K=%d must be 1 or feat width %d" % (spec.K, D))
        cfg.update(kind=spec.lib_kind, K=spec.K, relu=spec.relu, in_norm=spec.in_norm,
                   sample_base=spec.sample_base, seed=spec.seed, offset=spec.offset,
                   param_shape=spec.param_shape)
        p0, p1 = spec.p0, spec.p1
        if cfg["kind"] == _lib.NOISE_NORMAL_HADAMARD and D % 128:
            # the tensor-core generator works on 128-channel groups: zero-padded operand, sliced result (both differentiable
            # torch); hadamard_width said that the extra channels cost less than the generator saves
            Dp = spec.hadamard_width
            cfg["K"] = Dp
            out = _StochasticSpMM.apply(torch.nn.functional.pad(feat, (0, Dp - D)), p0, p1, None, cfg)[..., :D]
            return out[0] if squeeze else out
        pad = (-D) % 4
        if pad and D > 128 and not spec.in_norm and spec.param_shape != _lib.PARAM_EDGE_CHANNEL:
            # A width that is not a multiple of 4 (Cora's 1433) has rows that are not 16-byte aligned, which leaves only
            # the scalar-guarded kernels.  Zero-padded channels contribute nothing and the variate of a channel depends
            # on (edge, channel, sample) only, so the padded problem has the same first D outputs and gradients; the
            # pad / slice pair is differentiable torch.  (Narrow rows -- PPI's 50, molhiv's 9 -- are launch-bound: the
            # two extra launches cost more than the vector loads save, measured.)
            Dp = D + pad
            featp = torch.nn.functional.pad(feat, (0, pad))
            if spec.K == D:
                cfg["K"] = Dp
                if spec.param_shape == _lib.PARAM_CHANNEL:
                    p0 = torch.nn.functional.pad(p0, (0, pad))
                    p1 = None if p1 is None else torch.nn.functional.pad(p1, (0, pad), value=1.0)
            out = _StochasticSpMM.apply(featp, p0, p1, None, cfg)[..., :D]
            return out[0] if squeeze else out
    else:
        w = edge_weight
        _require_cuda(w, "edge_weight")
        if w.dim() == 1:
            w = w.unsqueeze(-1)
        K = w.shape[-1]
        if K not in (1, D):
            raise ValueError("edge_weight width %d must be 1 or feat width %d" % (K, D))
        if w.dim() == 2:
            if w.shape[0] != E:
                raise AssertionError("edge_weight has %d rows, graph has %d edges" % (w.shape[0], E))
            w = w.unsqueeze(0).expand(S, E, K)
        elif w.dim() != 3 or w.shape[0] != S or w.shape[1] != E:
            raise ValueError("edge_weight must be [E,K] or [S,E,K]; got %s" % (tuple(edge_weight.shape),))
        cfg.update(kind=_lib.NOISE_EXTERNAL, K=K)
        ext = w
    out = _StochasticSpMM.apply(feat, p0, p1, ext, cfg)
    return out[0] if squeeze else out


class _StochasticMax(torch.autograd.Function):
    """stag_spmm_max_fwd / stag_spmm_max_bwd: out[s,v,c] = max over the in-edges of w * feat[u], with the winning edge
    id kept for the backward (only the winner receives the gradient)."""

    @staticmethod
    def forward(ctx, feat, p0, p1, ext, cfg):
        g = cfg["graph"]
        st = g._s
        dev = feat.device
        lib = _lib.load()
        S, shared = cfg["S"], cfg["shared"]
        N, NS, D = st.num_nodes, st.num_src, feat.shape[-1]
        x = _c(feat)
        p0c, p1c, extc = _c(p0), _c(p1), _c(ext)
        out = torch.empty((S, N, D), dtype=torch.float32, device=dev)
        arg = torch.empty((S, N, D), dtype=torch.int32, device=dev)
        with _on_device(dev):
            csc, _ = st.csx(True)
            ws = _workspace(st, lib, csc, True, D, S)
            nz = _fill_noise(None, cfg["kind"], cfg["K"], p0c, p1c, extc, cfg["relu"], False, cfg["sample_base"],
                             cfg["seed"], cfg["offset"], cfg["param_shape"])
            _lib.check(lib.stag_spmm_max_fwd(
                ctypes.byref(csc), x.data_ptr(), D, 0 if shared else NS * D, D, S, ctypes.byref(nz),
                out.data_ptr(), arg.data_ptr(), D, N * D, ws.data_ptr(), ws.numel(), _stream(dev)))
        ctx.cfg = cfg
        ctx.feat_shape = feat.shape
        ctx.param_shapes = (None if p0 is None else p0.shape, None if p1 is None else p1.shape)
        ctx.ext_shape = None if ext is None else ext.shape
        need_x = any(ctx.needs_input_grad[1:4])
        ctx.save_for_backward(x if need_x else None, p0c, p1c, extc, arg)
        return out

    @staticmethod
    def backward(ctx, gout):
        cfg = ctx.cfg
        st = cfg["graph"]._s
        x, p0c, p1c, extc, arg = ctx.saved_tensors
        lib = _lib.load()
        dev = gout.device
        S, shared = cfg["S"], cfg["shared"]
        N, NS, D, K = st.num_nodes, st.num_src, gout.shape[-1], cfg["K"]
        need_dx = ctx.needs_input_grad[0]
        need_dp = (ctx.needs_input_grad[1] or ctx.needs_input_grad[2]) and cfg["kind"] in (
            _lib.NOISE_NORMAL, _lib.NOISE_UNIFORM)
        need_dext = ctx.needs_input_grad[3] and cfg["kind"] == _lib.NOISE_EXTERNAL
        gout = gout.to(torch.float32).contiguous()
        dx = torch.empty((S, NS, D), dtype=torch.float32, device=dev) if need_dx else None
        dext = torch.empty((S, st.num_edges, K), dtype=torch.float32, device=dev) if need_dext else None
        dp0 = dp1 = None
        if need_dp:
            n = {_lib.PARAM_SCALAR: 1, _lib.PARAM_CHANNEL: K, _lib.PARAM_EDGE: st.num_edges}[cfg["param_shape"]]
            dp0 = torch.zeros(n, dtype=torch.float32, device=dev)
            dp1 = torch.zeros(n, dtype=torch.float32, device=dev)
        if need_dx or need_dp or need_dext:
            with _on_device(dev):
                csr, _ = st.csx(False)
                ws = _workspace(st, lib, csr, False, D, S)
                nz = _fill_noise(None, cfg["kind"], K, p0c, p1c, extc, cfg["relu"], False, cfg["sample_base"],
                                 cfg["seed"], cfg["offset"], cfg["param_shape"])
                _lib.check(lib.stag_spmm_max_bwd(
                    ctypes.byref(csr), _ptr(x), D, 0 if shared else NS * D, gout.data_ptr(), arg.data_ptr(), D, N * D,
                    D, S, ctypes.byref(nz), _ptr(dx), D, NS * D, _ptr(dp0), _ptr(dp1), _ptr(dext),
                    ws.data_ptr(), ws.numel(), _stream(dev)))
        gfeat = gp0 = gp1 = gext = None
        if need_dx:
            gfeat = (dx.sum(0) if shared else dx).reshape(ctx.feat_shape)
        if need_dp:
            s0, s1 = ctx.param_shapes
            if ctx.needs_input_grad[1]:
                gp0 = dp0.reshape(s0) if dp0.numel() == max(1, _numel(s0)) else dp0.reshape(-1).sum_to_size(s0)
            if ctx.needs_input_grad[2] and s1 is not None:
                gp1 = dp1.reshape(s1) if dp1.numel() == max(1, _numel(s1)) else dp1.reshape(-1).sum_to_size(s1)
        if need_dext:
            gext = dext.reshape(ctx.ext_shape) if dext.numel() == _numel(ctx.ext_shape) else dext
        return gfeat, gp0, gp1, gext, None


def _aggregate_max(g, feat, edge_weight, S, shared):
    """[S,N,D] max over the in-edges of w * feat[u] (see :func:`stochastic_aggregate`).  In-norm specs and [E,K]
    parameters go through the materialised noise tensor (differentiable through _NoiseEmit): the in-norm scale of
    Normal noise can be negative and flip the max, and the fused kernels take neither."""
    st = g._s
    E, D = st.num_edges, feat.shape[-1]
    cfg = {"graph": g, "S": S, "shared": shared, "relu": False, "sample_base": 0, "seed": 0, "offset": 0,
           "param_shape": _lib.PARAM_SCALAR, "K": D, "kind": _lib.NOISE_NONE}
    if isinstance(edge_weight, NoiseSpec):
        spec = edge_weight
        if spec.num_edges != E:
            raise ValueError("noise spec was made for %d edges, graph has %d" % (spec.num_edges, E))
        if spec.K not in (1, D):
            raise ValueError("noise width K=%d must be 1 or feat width %d" % (spec.K, D))
        if spec.in_norm or spec.param_shape == _lib.PARAM_EDGE_CHANNEL:
            w = spec.materialize(n_samples=S)                                   # [S,E,K], relu applied
            if spec.in_norm:
                from .layers import _in_norm
                w = torch.stack([_in_norm(g, w[s]) for s in range(S)])
            return _aggregate_max(g, feat, w, S, shared)
        cfg.update(kind=spec.lib_kind, K=spec.K, relu=spec.relu, sample_base=spec.sample_base, seed=spec.seed,
                   offset=spec.offset, param_shape=spec.param_shape)
        p0, p1 = spec.p0, spec.p1
        Dp = D
        if cfg["kind"] == _lib.NOISE_NORMAL_HADAMARD and D % 128:
            Dp = spec.hadamard_width                        # the tensor-core stream comes in groups of 128 channels
        elif D % 4 and D > 128 and spec.K == D:
            Dp = D + (-D) % 4                               # 16-byte rows for the vector loads (as the sum path)
        if Dp != D:
            if spec.K == D:
                cfg["K"] = Dp
                if spec.param_shape == _lib.PARAM_CHANNEL:
                    p0 = torch.nn.functional.pad(p0, (0, Dp - D))
                    p1 = None if p1 is None else torch.nn.functional.pad(p1, (0, Dp - D), value=1.0)
            featp = torch.nn.functional.pad(feat, (0, Dp - D))
            return _StochasticMax.apply(featp, p0, p1, None, cfg)[..., :D]
        return _StochasticMax.apply(feat, p0, p1, None, cfg)
    if edge_weight is None:
        return _StochasticMax.apply(feat, None, None, None, cfg)
    w = edge_weight
    _require_cuda(w, "edge_weight")
    if w.dim() == 1:
        w = w.unsqueeze(-1)
    K = w.shape[-1]
    if K not in (1, D):
        raise ValueError("edge_weight width %d must be 1 or feat width %d" % (K, D))
    if w.dim() == 2:
        if w.shape[0] != E:
            raise AssertionError("edge_weight has %d rows, graph has %d edges" % (w.shape[0], E))
        w = w.unsqueeze(0).expand(S, E, K)
    elif w.dim() != 3 or w.shape[0] != S or w.shape[1] != E:
        raise ValueError("edge_weight must be [E,K] or [S,E,K]; got %s" % (tuple(edge_weight.shape),))
    cfg.update(kind=_lib.NOISE_EXTERNAL, K=K)
    return _StochasticMax.apply(feat, None, None, w, cfg)


class _HeadsAggregate(torch.autograd.Function):
    """out[(s,) v, k, :] = sum over the in-edges e = (u, v) of a[(s,) e, k] * ft[(s,) u, k, :]  -- the weighted aggregation
    of a multi-head attention layer (GATConv's ``u_mul_e('ft', 'a') -> sum``).  One launch per head on the per-edge-weight
    kernel, covering every Monte-Carlo sample, each reading its F columns of ``ft`` IN PLACE (row stride H F; sample
    stride 0 when ``ft`` is shared) and writing its F columns of ``out`` in place: no ``[E, H*F]`` expansion of the
    attention, no per-head copies.  The attention is permuted to ``[H, S, E]`` so that the weights of head k are one
    ``[S, E, 1]`` external tensor.  Backward: per head the transposed pass (d ft) and the SDDMM (d a) in one
    ``stag_spmm_bwd`` call."""

    @staticmethod
    def forward(ctx, ft, a, graph):
        st = graph._s
        dev = ft.device
        _require_cuda(ft, "feat")
        lib = _lib.load()
        N, NS, E = st.num_nodes, st.num_src, st.num_edges
        H, F = ft.shape[-2], ft.shape[-1]
        batched = a.dim() == 3
        S = a.shape[0] if batched else 1
        shared = ft.dim() == 3
        x = _c(ft.to(torch.float32)).reshape(-1, NS, H * F)
        at = a.detach().to(torch.float32).reshape(S, E, H).permute(2, 0, 1).contiguous()   # [H, S, E]: a head's weights
        xs = 0 if shared else NS * H * F
        out = torch.empty((S, N, H * F), dtype=torch.float32, device=dev)
        with _on_device(dev):
            csc, _ = st.csx(True)
            ws = _workspace(st, lib, csc, True, F, S)
            for k in range(H):
                nz = _fill_noise(None, _lib.NOISE_EXTERNAL, 1, None, None, at[k], False, False, 0, 0, 0, _lib.PARAM_SCALAR)
                _lib.check(lib.stag_spmm_fwd(
                    ctypes.byref(csc), x.data_ptr() + 4 * k * F, H * F, xs, F, S, ctypes.byref(nz), 0, 0,
                    out.data_ptr() + 4 * k * F, H * F, N * H * F, 0, ws.data_ptr(), ws.numel(), _stream(dev)))
        ctx.graph, ctx.dims, ctx.flags = graph, (N, NS, E, H, F, S), (batched, shared)
        ctx.save_for_backward(x, at)
        return out.reshape(S, N, H, F) if batched else out.reshape(N, H, F)

    @staticmethod
    def backward(ctx, gout):
        x, at = ctx.saved_tensors
        N, NS, E, H, F, S = ctx.dims
        batched, shared = ctx.flags
        st = ctx.graph._s
        lib = _lib.load()
        dev = gout.device
        g2 = gout.to(torch.float32).contiguous().reshape(S, N, H * F)
        xs = 0 if shared else NS * H * F
        need_dx, need_da = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        dx = torch.empty((S, NS, H * F), dtype=torch.float32, device=dev) if need_dx else None
        dat = torch.empty((H, S, E), dtype=torch.float32, device=dev) if need_da else None
        with _on_device(dev):
            csr, _ = st.csx(False)
            ws = _workspace(st, lib, csr, False, F, S)
            for k in range(H):
                nz = _fill_noise(None, _lib.NOISE_EXTERNAL, 1, None, None, at[k], False, False, 0, 0, 0, _lib.PARAM_SCALAR)
                if need_da:
                    _lib.check(lib.stag_spmm_bwd(
                        ctypes.byref(csr), x.data_ptr() + 4 * k * F, H * F, xs, g2.data_ptr() + 4 * k * F, H * F,
                        N * H * F, F, S, ctypes.byref(nz), 0, 0, 0 if dx is None else dx.data_ptr() + 4 * k * F, H * F,
                        NS * H * F, 0, 0, dat[k].data_ptr(), ws.data_ptr(), ws.numel(), _stream(dev)))
                elif need_dx:
                    _lib.check(lib.stag_spmm_fwd(
                        ctypes.byref(csr), g2.data_ptr() + 4 * k * F, H * F, N * H * F, F, S, ctypes.byref(nz), 0, 0,
                        dx.data_ptr() + 4 * k * F, H * F, NS * H * F, 0, ws.data_ptr(), ws.numel(), _stream(dev)))
        gft = gat = None
        if dx is not None:
            gft = (dx.sum(0) if shared and batched else dx).reshape((NS, H, F) if shared else (S, NS, H, F))
        if dat is not None:
            gat = dat.permute(1, 2, 0) if batched else dat[:, 0].t()
        return gft, gat, None


def heads_aggregate(graph, ft, a):
    """Per-head weighted aggregation ``[N_src, H, F], [E, H] -> [N, H, F]``, or over S Monte-Carlo samples
    ``[S, N_src, H, F]`` (or a shared ``[N_src, H, F]``), ``[S, E, H] -> [S, N, H, F]`` (see :class:`_HeadsAggregate`)."""
    g = as_graph(graph)
    ok = ft.dim() in (3, 4) and a.dim() in (2, 3) and a.shape[-1] == ft.shape[-2] and a.shape[-2] == g.number_of_edges()
    if ok and a.dim() == 2:
        ok = ft.dim() == 3
    elif ok:
        ok = ft.dim() == 3 or ft.shape[0] == a.shape[0]
    if not ok:
        raise ValueError("heads_aggregate: feat [N,H,F] or [S,N,H,F] and attention [E,H] or [S,E,H] expected, got %s and %s"
                         % (tuple(ft.shape), tuple(a.shape)))
    return _HeadsAggregate.apply(ft, a, g)


def segment_reduce(graph, feat, mean=False):
    """SumNodes / MeanNodes readout (stag/layers.py:156-178): [N,D] -> [B,D] by batch_num_nodes."""
    return _SegmentReduce.apply(feat, as_graph(graph), bool(mean))


class _SegmentReduce(torch.autograd.Function):
    @staticmethod
    def forward(ctx, feat, g, mean):
        _require_cuda(feat, "feat")
        lib = _lib.load()
        dev = feat.device
        x = _c(feat).reshape(feat.shape[0], -1)
        ptr = g._s.node_ptr()
        B, D = ptr.numel() - 1, x.shape[1]
        out = torch.empty((B, D), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            _lib.check(lib.stag_segment_reduce(x.data_ptr(), D, ptr.data_ptr(), B, D, int(mean),
                                               out.data_ptr(), D, _stream(dev)))
        ctx.g, ctx.mean, ctx.shape = g, mean, feat.shape
        return out.reshape((B,) + tuple(feat.shape[1:]))

    @staticmethod
    def backward(ctx, gout):
        bnn = ctx.g.batch_num_nodes()
        go = gout.reshape(gout.shape[0], -1)
        if ctx.mean:
            go = go / bnn.to(go).clamp(min=1).unsqueeze(-1)
        return torch.repeat_interleave(go, bnn, dim=0).reshape(ctx.shape), None, None


class _EdgeSoftmax(torch.autograd.Function):
    """stag_edge_softmax: softmax of ``logits [E,H]`` over the in-edges of every destination node
    (dgl.nn.edge_softmax, stag/zoo/gat.py:122), one fused pass per direction."""

    @staticmethod
    def forward(ctx, logits, g):
        _require_cuda(logits, "logits")
        lib = _lib.load()
        dev = logits.device
        lg = logits.detach().to(torch.float32).contiguous()
        E, H = lg.shape
        out = torch.empty_like(lg)
        with torch.cuda.device(dev):
            csc, _ = g._s.csx(True)
            _lib.check(lib.stag_edge_softmax(ctypes.byref(csc), lg.data_ptr(), H, out.data_ptr(), _stream(dev)))
        ctx.g = g
        ctx.save_for_backward(out)
        return out

    @staticmethod
    def backward(ctx, da):
        (a,) = ctx.saved_tensors
        lib = _lib.load()
        dev = a.device
        da = da.to(torch.float32).contiguous()
        dl = torch.empty_like(a)
        with torch.cuda.device(dev):
            csc, _ = ctx.g._s.csx(True)
            _lib.check(lib.stag_edge_softmax_bwd(ctypes.byref(csc), a.data_ptr(), da.data_ptr(), a.shape[1],
                                                 dl.data_ptr(), _stream(dev)))
        return dl, None


class _AttentionSoftmax(torch.autograd.Function):
    """a[(s,) e, h] = softmax over the in-edges of v_e of  w[(s,) e, h] * leaky_relu(el[(s,) u_e, h] + er[(s,) v_e, h])  --
    GAT's attention (stag/zoo/gat.py:113-122) without the [E,H] logits and their autograd graph.  The noise w is none, an
    external tensor, or drawn inside the kernel from a NoiseSpec (S samples per launch, stag_attention_softmax_s);
    unbatched calls without a spec take the S = 1 entry points (stag_attention_softmax).  Backward: one pass over the CSC
    rows gives d er, the per-edge d(el + er), d w (external) or the parameter gradients (generated); d el is the sum per
    SOURCE node of the per-edge values, taken by the aggregation kernel on the CSR (edge values as external weights of a
    ones operand).  No atomics: deterministic."""

    @staticmethod
    def forward(ctx, el, er, p0, p1, ext, cfg):
        _require_cuda(el, "el")
        lib = _lib.load()
        dev = el.device
        st = cfg["graph"]._s
        E, H, S = st.num_edges, el.shape[-1], cfg["S"]
        elc, erc = _c(el), _c(er)
        p0c, p1c, extc = _c(p0), _c(p1), _c(ext)
        a = torch.empty((S, E, H), dtype=torch.float32, device=dev)
        with _on_device(dev):
            csc, _ = st.csx(True)
            if cfg["legacy"]:
                _lib.check(lib.stag_attention_softmax(ctypes.byref(csc), elc.data_ptr(), erc.data_ptr(), _ptr(extc),
                                                      cfg["slope"], H, a.data_ptr(), _stream(dev)))
            else:
                nz = _attention_noise(cfg, p0c, p1c, extc)
                _lib.check(lib.stag_attention_softmax_s(
                    ctypes.byref(csc), elc.data_ptr(), 0 if cfg["el_shared"] else st.num_src * H, erc.data_ptr(),
                    0 if cfg["er_shared"] else st.num_nodes * H, H, S, ctypes.byref(nz), cfg["slope"], a.data_ptr(),
                    0, 0, _stream(dev)))
        ctx.cfg = cfg
        ctx.param_shapes = (None if p0 is None else p0.shape, None if p1 is None else p1.shape)
        ctx.ext_shape = None if ext is None else ext.shape
        ctx.save_for_backward(elc, erc, p0c, p1c, extc, a)
        return a

    @staticmethod
    def backward(ctx, da):
        elc, erc, p0c, p1c, extc, a = ctx.saved_tensors
        cfg = ctx.cfg
        lib = _lib.load()
        dev = a.device
        st = cfg["graph"]._s
        S, E, H = a.shape
        N, NS = st.num_nodes, st.num_src
        need_dp = (ctx.needs_input_grad[2] or ctx.needs_input_grad[3]) and cfg["kind"] in (
            _lib.NOISE_NORMAL, _lib.NOISE_UNIFORM)
        need_dext = ctx.needs_input_grad[4] and cfg["kind"] == _lib.NOISE_EXTERNAL
        d_er = torch.zeros((S, N, H), dtype=torch.float32, device=dev)
        d_el = torch.zeros((S, NS, H), dtype=torch.float32, device=dev)
        dext = torch.zeros_like(a) if need_dext else None
        dp0 = dp1 = None
        if need_dp:
            n = {_lib.PARAM_SCALAR: 1, _lib.PARAM_CHANNEL: H, _lib.PARAM_EDGE: E,
                 _lib.PARAM_EDGE_CHANNEL: E * H}[cfg["param_shape"]]
            dp0 = torch.zeros(n, dtype=torch.float32, device=dev)
            dp1 = torch.zeros(n, dtype=torch.float32, device=dev)
        if E:
            da = da.to(torch.float32).contiguous()
            dpre = torch.empty_like(a)
            with _on_device(dev):
                csc, _ = st.csx(True)
                if cfg["legacy"]:
                    _lib.check(lib.stag_attention_softmax_bwd(
                        ctypes.byref(csc), elc.data_ptr(), erc.data_ptr(), _ptr(extc), cfg["slope"], H, a.data_ptr(),
                        da.data_ptr(), _ptr(dext), dpre.data_ptr(), d_er.data_ptr(), _stream(dev)))
                else:
                    ws = _attention_workspace(st, lib, csc, H, S)
                    nz = _attention_noise(cfg, p0c, p1c, extc)
                    _lib.check(lib.stag_attention_softmax_s_bwd(
                        ctypes.byref(csc), elc.data_ptr(), 0 if cfg["el_shared"] else NS * H, erc.data_ptr(),
                        0 if cfg["er_shared"] else N * H, H, S, ctypes.byref(nz), cfg["slope"], a.data_ptr(),
                        da.data_ptr(), dpre.data_ptr(), d_er.data_ptr(), _ptr(dp0), _ptr(dp1), _ptr(dext),
                        ws.data_ptr(), ws.numel(), _stream(dev)))
                if ctx.needs_input_grad[0]:
                    # d el[s,u,h] = sum over the out-edges of u of dpre[s,e,h]: the aggregation kernel on the CSR, a ones
                    # operand gathered per destination (shared by the samples), the edge values as external weights
                    csr, _ = st.csx(False)
                    ws = _workspace(st, lib, csr, False, H, S)
                    ones = torch.ones((N, H), dtype=torch.float32, device=dev)
                    nz = _fill_noise(None, _lib.NOISE_EXTERNAL, H, None, None, dpre, False, False, 0, 0, 0, _lib.PARAM_SCALAR)
                    _lib.check(lib.stag_spmm_fwd(
                        ctypes.byref(csr), ones.data_ptr(), H, 0, H, S, ctypes.byref(nz), 0, 0, d_el.data_ptr(), H,
                        NS * H, 0, ws.data_ptr(), ws.numel(), _stream(dev)))
        gel = d_el.sum(0) if cfg["el_shared"] else d_el
        ger = d_er.sum(0) if cfg["er_shared"] else d_er
        gp0 = gp1 = gext = None
        if need_dp:
            s0, s1 = ctx.param_shapes
            if ctx.needs_input_grad[2]:
                gp0 = dp0.reshape(s0) if dp0.numel() == max(1, _numel(s0)) else dp0.reshape(-1).sum_to_size(s0)
            if ctx.needs_input_grad[3] and s1 is not None:
                gp1 = dp1.reshape(s1) if dp1.numel() == max(1, _numel(s1)) else dp1.reshape(-1).sum_to_size(s1)
        if need_dext:
            gext = dext.reshape(ctx.ext_shape)
        return gel.reshape(elc.shape), ger.reshape(erc.shape), gp0, gp1, gext, None


def _attention_noise(cfg, p0c, p1c, extc):
    return _fill_noise(None, cfg["kind"], cfg["K"], p0c, p1c, extc, cfg["relu"], False, cfg["sample_base"], cfg["seed"],
                       cfg["offset"], cfg["param_shape"])


def _attention_workspace(st, lib, csc, H, S):
    key = ("attention", H, S)
    cache = st.__dict__.setdefault("_ws_bytes", {})
    if key not in cache:
        cache[key] = lib.stag_attention_workspace_bytes(ctypes.byref(csc), H, S)
    return st.workspace(cache[key])


def attention_route(spec):
    """'fused' when the attention kernel draws the noise of `spec` itself, 'materialized' when the spec goes through its
    noise tensor (in-norm rescales by a per-row sum the kernel does not take; the tensor-core generator works on
    128-channel groups, not one channel per head)."""
    if spec.in_norm or spec.lib_kind == _lib.NOISE_NORMAL_HADAMARD:
        return "materialized"
    return "fused"


def attention_softmax(graph, el, er, edge_weight=None, negative_slope=0.2, n_samples=None):
    """GAT attention from the per-node scores ``el [N_src,H]``, ``er [N,H]`` and the logit noise ``edge_weight``: ``None``,
    a tensor ``[E,H]`` / ``[E,1]`` / ``[E]`` (or ``[S,E,H]``), or a :class:`NoiseSpec` with ``K == H`` drawn inside the
    kernel.  Returns ``[E,H]``, or ``[S,E,H]`` over S Monte-Carlo samples: with ``n_samples=S``, per-sample scores
    ``[S,N,H]``, ``[S,E,H]`` weights or a sample-batched spec; ``[N,H]`` scores are then shared by the samples (see
    :class:`_AttentionSoftmax`)."""
    g = as_graph(graph)
    st = g._s
    E = st.num_edges
    if el.dim() not in (2, 3) or er.dim() not in (2, 3) or el.shape[-1] != er.shape[-1]:
        raise ValueError("attention_softmax: el [(S,)N_src,H] and er [(S,)N,H] expected, got %s and %s"
                         % (tuple(el.shape), tuple(er.shape)))
    H = el.shape[-1]
    if el.shape[-2] != st.num_src or er.shape[-2] != st.num_nodes:
        raise ValueError("attention_softmax: el has %d rows and er %d, graph has %d source and %d destination nodes"
                         % (el.shape[-2], er.shape[-2], st.num_src, st.num_nodes))
    spec = edge_weight if isinstance(edge_weight, NoiseSpec) else None
    S = None if n_samples is None else int(n_samples)
    for t in (el, er) + ((edge_weight,) if (edge_weight is not None and spec is None and edge_weight.dim() == 3) else ()):
        if t.dim() == 3:
            if S is not None and t.shape[0] != S:
                raise ValueError("attention_softmax: inputs disagree on the number of samples (%d and %d)" % (S, t.shape[0]))
            S = t.shape[0]
    if S is None and spec is not None and spec.batched:
        S = spec.n_samples
    batched = S is not None
    S = 1 if S is None else S
    if spec is not None:
        if spec.num_edges != E:
            raise ValueError("noise spec was made for %d edges, graph has %d" % (spec.num_edges, E))
        if spec.K != H:
            raise ValueError("attention noise width K=%d must equal the number of heads H=%d" % (spec.K, H))
        if attention_route(spec) == "materialized":
            w = spec.materialize(n_samples=S)                                       # [S,E,H], relu applied
            if spec.in_norm:
                from .layers import _in_norm
                w = torch.stack([_in_norm(g, w[s]) for s in range(S)])
            a = attention_softmax(g, el, er, w, negative_slope, n_samples=S)
            return a if batched else a[0]
    cfg = {"graph": g, "S": S, "el_shared": el.dim() == 2, "er_shared": er.dim() == 2, "slope": float(negative_slope),
           "kind": _lib.NOISE_NONE, "K": H, "relu": False, "sample_base": 0, "seed": 0, "offset": 0,
           "param_shape": _lib.PARAM_SCALAR, "legacy": False}
    p0 = p1 = ext = None
    if spec is not None:
        cfg.update(kind=spec.lib_kind, relu=spec.relu, sample_base=spec.sample_base, seed=spec.seed, offset=spec.offset,
                   param_shape=spec.param_shape)
        p0, p1 = spec.p0, spec.p1
    elif edge_weight is not None:
        w = edge_weight
        _require_cuda(w, "edge_weight")
        if w.dim() == 3:
            if w.shape[1] != E or w.shape[2] not in (1, H):
                raise ValueError("attention_softmax: edge_weight must be [E,H], [E,1] or [S,E,H], got %s"
                                 % (tuple(edge_weight.shape),))
        else:
            w = w.unsqueeze(-1) if w.dim() == 1 else w.flatten(1)
            if w.shape[0] != E or w.shape[1] not in (1, H):
                raise ValueError("attention_softmax: edge_weight must be [E,H] or [E,1], got %s" % (tuple(edge_weight.shape),))
            w = w.unsqueeze(0)
        ext = w.expand(S, E, H)
        cfg["kind"] = _lib.NOISE_EXTERNAL
    cfg["legacy"] = not batched and spec is None
    a = _AttentionSoftmax.apply(el, er, p0, p1, ext, cfg)
    return a if batched else a[0]


def edge_softmax(graph, logits):
    """Softmax of ``logits [E,H]`` (or ``[E]``) over the in-edges of each destination node."""
    g = as_graph(graph)
    if logits.shape[0] != g._s.num_edges:
        raise ValueError("logits has %d rows, graph has %d edges" % (logits.shape[0], g._s.num_edges))
    flat = logits.reshape(logits.shape[0], -1)
    return _EdgeSoftmax.apply(flat, g).reshape(logits.shape)


class _FusedNLL(torch.autograd.Function):
    """stag_nll: masked mean negative log-likelihood of S sample outputs [S,N,C] -> [S], gradient emitted by the
    same kernel pass (stag/models.py:69-72 over torch.distributions' Categorical / Bernoulli)."""

    @staticmethod
    def forward(ctx, probs, y, mask, kind):
        _require_cuda(probs, "likelihood input")
        lib = _lib.load()
        dev = probs.device
        S, N, C = probs.shape
        pr = probs.detach().to(torch.float32).contiguous()
        yy = y.to(torch.int64).contiguous() if kind == 0 else y.to(torch.float32).contiguous()
        mk = None if mask is None else mask.to(torch.uint8).contiguous()
        nll = torch.empty(S, dtype=torch.float32, device=dev)
        count = torch.empty(1, dtype=torch.float32, device=dev)
        need = ctx.needs_input_grad[0]
        dpr = torch.empty_like(pr) if need else None
        with torch.cuda.device(dev):
            wsb = lib.stag_nll_workspace_bytes(N, S)
            ws = torch.empty(max(wsb, 256), dtype=torch.uint8, device=dev)
            _lib.check(lib.stag_nll(pr.data_ptr(), C, N * C, N, C, S, kind, yy.data_ptr(), C if kind == 1 else 0,
                                    _ptr(mk), nll.data_ptr(), count.data_ptr(), _ptr(dpr), ws.data_ptr(),
                                    ws.numel(), _stream(dev)))
        ctx.save_for_backward(dpr, count)
        return nll

    @staticmethod
    def backward(ctx, g):
        dpr, count = ctx.saved_tensors
        if dpr is None:
            return None, None, None, None
        return dpr * (g.to(torch.float32) / count).reshape(-1, 1, 1), None, None, None


def describe_prior(p_a):
    """(weights, locs, scales) python lists when `p_a` is a Normal with one scalar parameter pair or a
    MixtureSameFamily(Categorical, Normal) over up to 8 scalar components without trainable parameters -- the priors
    ``stag_noise_kl`` evaluates in the kernel -- else None."""
    d = getattr(p_a, "base_distribution", p_a)
    td = torch.distributions
    try:
        if isinstance(d, td.MixtureSameFamily):
            comp, mix = d.component_distribution, d.mixture_distribution
            if not isinstance(comp, td.Normal) or comp.loc.dim() != 1 or comp.loc.numel() > _lib.PRIOR_MAX_COMPONENTS:
                return None
            ts = (mix.probs, comp.loc, comp.scale)
        elif isinstance(d, td.Normal) and d.loc.numel() == 1 and d.scale.numel() == 1:
            ts = (torch.ones(1), d.loc.reshape(1), d.scale.reshape(1))
        else:
            return None
        if any(t.requires_grad for t in ts):
            return None
        return tuple([float(v) for v in t.detach().cpu().reshape(-1)] for t in ts)
    except Exception:
        return None


class _NoiseKL(torch.autograd.Function):
    """(sum log q(w), sum log p(w)) over the regenerated sample of a NoiseSpec (stag_noise_kl): no [E,K] tensor."""

    @staticmethod
    def forward(ctx, spec, prior, p0, p1):
        dev = p0.device
        _require_cuda(p0, "noise parameter")
        lib = _lib.load()
        E, K, S = spec.num_edges, spec.K, spec.n_samples
        p0c, p1c = _c(p0), _c(p1)
        pr = _lib.StagPrior()
        pr.kind, pr.M = _lib.PRIOR_NORMAL_MIXTURE, len(prior[0])
        for m in range(pr.M):
            pr.weight[m], pr.loc[m], pr.scale[m] = prior[0][m], prior[1][m], prior[2][m]
        need = ctx.needs_input_grad[2] or ctx.needs_input_grad[3]
        n = {_lib.PARAM_SCALAR: 1, _lib.PARAM_CHANNEL: K, _lib.PARAM_EDGE: E, _lib.PARAM_EDGE_CHANNEL: E * K}[spec.param_shape]
        d0 = torch.zeros(n, dtype=torch.float32, device=dev) if need else None
        d1 = torch.zeros(n, dtype=torch.float32, device=dev) if need else None
        sums = torch.empty(2, dtype=torch.float64, device=dev)
        ws = torch.empty(max(lib.stag_noise_kl_workspace_bytes(K), 256), dtype=torch.uint8, device=dev)
        nz = _fill_noise(spec, spec.lib_kind, K, p0c, p1c, None, spec.relu, False, spec.sample_base,
                         spec.seed, spec.offset, spec.param_shape)
        with _on_device(dev):
            _lib.check(lib.stag_noise_kl(ctypes.byref(nz), E, S, ctypes.byref(pr), sums.data_ptr(), _ptr(d0), _ptr(d1),
                                         ws.data_ptr(), ws.numel(), _stream(dev)))
        ctx.save_for_backward(d0, d1)
        ctx.shapes = (p0.shape, p1.shape)
        return sums.to(torch.float32)

    @staticmethod
    def backward(ctx, gsums):
        d0, d1 = ctx.saved_tensors
        g0 = g1 = None
        if d0 is not None:
            # d(sum log q - sum log p) came out of the kernel as one tensor: the layer only ever differentiates
            # c * (sums[0] - sums[1]), so gsums = (c, -c)
            c = gsums[0]
            s0, s1 = ctx.shapes
            if ctx.needs_input_grad[2]:
                g0 = (c * d0).reshape(s0) if d0.numel() == max(1, _numel(s0)) else (c * d0).sum_to_size(s0)
            if ctx.needs_input_grad[3]:
                g1 = (c * d1).reshape(s1) if d1.numel() == max(1, _numel(s1)) else (c * d1).sum_to_size(s1)
        return None, None, g0, g1


def fused_kl_fallback(spec, prior):
    """``q.log_prob(w).sum(-1).mean() - p.log_prob(w).sum(-1).mean()`` of the reference's KL fallback
    (stag/layers.py:139-141) over the sample(s) `spec` describes, evaluated by ``stag_noise_kl`` from the regenerated
    variates: no ``[E,K]`` allocation.  `prior` = ``describe_prior(p_a)``.  Differentiable w.r.t. the parameters of q."""
    if spec.kind not in ("normal", "uniform") or spec.in_norm or spec.lib_kind == _lib.NOISE_NORMAL_HADAMARD:
        raise ValueError("fused KL fallback: reparameterised Normal / Uniform posteriors without in-norm only")
    sums = _NoiseKL.apply(spec, prior, spec.p0, spec.p1)
    return (sums[0] - sums[1]) / float(max(spec.n_samples, 1) * max(spec.num_edges, 1))


def fused_nll(probs, y, mask=None, kind="categorical"):
    """``[S]`` masked mean NLLs of ``probs [S,N,C]`` (or ``[N,C]`` -> scalar) under Categorical(probs=.) with labels
    ``y [N]`` or Bernoulli(probs=.) with labels ``y [N,C]``: one kernel pass for all samples, forward and gradient."""
    squeeze = probs.dim() == 2
    if squeeze:
        probs = probs.unsqueeze(0)
    out = _FusedNLL.apply(probs, y, mask, {"categorical": 0, "bernoulli": 1}[kind])
    return out[0] if squeeze else out


class _DenseTransform(torch.autograd.Function):
    """out = act(row_scale * (a @ weight) + bias) on stag_gemm_tcgen05 (3xTF32, fp32 accuracy).
    Backward: dA = g @ W^T through the same kernel, dW / dbias by torch reductions."""

    @staticmethod
    def forward(ctx, a, weight, row_scale, bias, relu, transposed):
        _require_cuda(a, "feat")
        lib = _lib.load()
        dev = a.device
        if transposed:      # weight given as [Nout, K] (torch.nn.Linear layout): already W^T
            Nout, K = weight.shape
            wt = weight.detach().to(torch.float32).contiguous()
        else:               # weight [K, Nout] (GraphConv layout)
            K, Nout = weight.shape
            wt = weight.detach().to(torch.float32).t().contiguous()      # [Nout, K]
        a2 = _c(a).reshape(-1, K)
        M = a2.shape[0]
        out = torch.empty((M, Nout), dtype=torch.float32, device=dev)
        rs = None
        if row_scale is not None:
            rs = _c(row_scale).reshape(-1)
            if rs.numel() != M:                                          # [N] scale shared by the S samples
                rs = rs.repeat(M // rs.numel())
        b = _c(bias)
        with torch.cuda.device(dev):
            _lib.check(lib.stag_gemm_tcgen05(a2.data_ptr(), K, wt.data_ptr(), K, M, Nout, K, _ptr(rs), _ptr(b),
                                             1 if relu else 0, out.data_ptr(), Nout, 0, 0, _stream(dev)))
        ctx.save_for_backward(a2, weight, rs, out if relu else None)
        ctx.relu, ctx.a_shape, ctx.has_bias, ctx.transposed = relu, a.shape, bias is not None, transposed
        return out.reshape(tuple(a.shape[:-1]) + (Nout,))

    @staticmethod
    def backward(ctx, g):
        a2, weight, rs, out = ctx.saved_tensors
        lib = _lib.load()
        dev = g.device
        Nout, K = weight.shape if ctx.transposed else weight.shape[::-1]
        g2 = g.to(torch.float32).reshape(-1, Nout)
        if ctx.relu:
            g2 = g2 * (out > 0)
        gbias = g2.sum(0) if (ctx.has_bias and ctx.needs_input_grad[3]) else None
        if rs is not None:
            g2 = g2 * rs.unsqueeze(-1)
        g2 = g2.contiguous()
        ga = gw = None
        if ctx.needs_input_grad[0]:
            ga = torch.empty((g2.shape[0], K), dtype=torch.float32, device=dev)
            # the "W^T" operand of the transposed product dA = g @ W^T is W [K, Nout] itself
            w = weight.detach().to(torch.float32)
            w = (w.t() if ctx.transposed else w).contiguous()
            with torch.cuda.device(dev):
                _lib.check(lib.stag_gemm_tcgen05(g2.data_ptr(), Nout, w.data_ptr(), Nout, g2.shape[0], K, Nout,
                                                 0, 0, 0, ga.data_ptr(), K, 0, 0, _stream(dev)))
            ga = ga.reshape(ctx.a_shape)
        if ctx.needs_input_grad[1]:
            gw = (g2.t() @ a2) if ctx.transposed else (a2.t() @ g2)
        return ga, gw, None, gbias, None, None


def dense_transform(a, weight, row_scale=None, bias=None, relu=False, transposed=False):
    """``act(row_scale[:,None] * (a @ W) + bias)`` on the tcgen05 tensor-core kernel (3xTF32, fp32-level
    accuracy).  ``weight`` is W [K, Nout] (GraphConv layout) or, with ``transposed=True``, W^T [Nout, K]
    (torch.nn.Linear layout).  Nout > 256 uses torch.matmul (cuBLAS)."""
    nout = weight.shape[0] if transposed else weight.shape[1]
    if nout > 256:
        out = torch.matmul(a, weight.t() if transposed else weight)
        if row_scale is not None:
            out = out * row_scale.reshape((-1,) + (1,) * 1) if out.dim() == 2 else out * row_scale.unsqueeze(-1)
        if bias is not None:
            out = out + bias
        return out.relu() if relu else out
    return _DenseTransform.apply(a, weight, row_scale, bias, relu, transposed)
