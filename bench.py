#!/usr/bin/env python
"""bench.py -- GEdge-samples/s of the fused stochastic SpMM (forward + backward) on the
ogbn-arxiv-shaped synthetic graph of BASELINE.json configs[1]:

    N 169 343 nodes, E 1 166 243 edges, 128 features, 3-layer stag GCN (aggregation widths
    128/128/128), 16 Monte-Carlo samples, Normal(1, sigma) edge noise, vi=False ("arxiv_mle").

One STEP = the stochastic-aggregation work of one training step of that model: for each of
the 3 layers one fused forward launch over the 16 samples (Philox noise generated in the
kernel, GCN degree scalings fused; layer 1 reads one shared X, layers 2-3 read per-sample
[S,N,D] activations) and one fused backward launch (transposed aggregation dX over the
regenerated noise).  edge-samples per step = E * S * 3.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--mode mle|vi] [--dump-outputs DIR]

N > 1: launched by torchrun, one rank per GPU; the MC samples are the sharded unit (rank r
draws Philox sample indices [r*S, (r+1)*S)), no data-path collective, weak scaling.
Prints ONE JSON line on rank 0.

--dump-outputs DIR writes what the last timed step computed as DIR/<name>.npy (float32), on
rank 0: the outputs of the three layers (out1..out3) and the input gradient dx, each [S, R, D]
over a fixed node sample R (see dump_rows), plus dparams [3, 2] (d loc, d scale per layer) in vi
mode; for --impl reference, out and dx [R, D] of its one layer pass.  The inputs depend only on
the arguments, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_NODES, N_EDGES, WIDTH, N_LAYERS, N_SAMPLES = 169343, 1166243, 128, 3, 16
SIGMA = 0.4
METRIC = "GEdge-samples/s fused stochastic SpMM fwd+bwd"
UNIT = "GEdge-samples/s"
WORKLOAD = ("ogbn-arxiv-shaped synthetic graph (N=169343, E=1166243, D=128), arxiv_mle 3-layer stag GCN "
            "aggregation, 16 MC samples, Normal(1,0.4) edge noise")


def synth_graph(seed=0x57A6 + 2):
    """Power-law in/out degrees (alpha ~ 2.1, clipped), random edge order, duplicates and self
    loops allowed (SURVEY.md 8(d))."""
    rng = np.random.default_rng(seed)

    def endpoints():
        ranks = np.arange(1, N_NODES + 1, dtype=np.float64)
        p = ranks ** (-1.0 / 1.1)      # Zipf weights -> degree tail exponent ~ 2.1
        p /= p.sum()
        p = np.minimum(p, 13155.0 / N_EDGES)
        p /= p.sum()
        ids = rng.choice(N_NODES, size=N_EDGES, p=p)
        return rng.permutation(N_NODES)[ids]
    return endpoints().astype(np.int64), endpoints().astype(np.int64)


def dump_rows(src, dst, n_random=1024, n_hubs=32):
    """Node rows kept by --dump-outputs (the full [S, N, D] outputs are 1.39 GB each): a seeded uniform
    sample plus the highest in- and out-degree nodes, whose rows take the hub code paths of the kernels."""
    rng = np.random.default_rng(0xD0)
    hubs = [np.argsort(np.bincount(e, minlength=N_NODES), kind="stable")[-n_hubs:] for e in (dst, src)]
    return np.unique(np.concatenate([rng.choice(N_NODES, n_random, replace=False)] + hubs))


def dump_outputs(out_dir, arrays):
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float32))


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# algorithmic (compulsory, perfect-cache) bytes per launch -- SURVEY.md 8(d) / DESIGN.md
def bytes_fwd(S, shared_x):
    nd = 4 * N_NODES * WIDTH
    per = 4 * N_EDGES + 4 * (N_NODES + 1) + 8 * N_NODES
    return (nd * (1 + S) if shared_x else 2 * nd * S) + per * S


def bytes_bwd(S, vi, shared_x):
    nd = 4 * N_NODES * WIDTH
    per = 8 * N_EDGES + 4 * (N_NODES + 1) + 8 * N_NODES
    x_read = (nd if shared_x else nd * S) if vi else 0
    return 2 * nd * S + x_read + per * S


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower() == "active" for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ---------------------------------------------------------------------------------------------
def run_reference(args, rank):
    """The reference's CPU path: un-fused (noise tensor materialised), restated in C + OpenMP
    (oracle/csrc/stag_ref.c; the reference itself is Python over DGL and cannot travel to the
    box).  Each step = ONE layer x ONE MC sample forward+backward at the arxiv shape."""
    if rank != 0:
        return
    from oracle import cbuild, ref_c
    cbuild.build()
    ref_c.use_all_cores()
    src, dst = synth_graph()
    rng = np.random.default_rng(1)
    x = rng.standard_normal((N_NODES, WIDTH)).astype(np.float32)
    g = rng.standard_normal((N_NODES, WIDTH)).astype(np.float32)
    lp = ref_c.LayerPass(src, dst, N_NODES, x, g, "normal", 1.0, SIGMA, vi=(args.mode == "vi"))
    for w in range(args.warmup):
        lp.run(w)
    t0 = time.perf_counter()
    for k in range(args.steps):
        lp.run(args.warmup + k)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        rows = dump_rows(src, dst)
        dump_outputs(args.dump_outputs, {"out": lp.out[rows], "dx": lp.dx[rows]})
    val = N_EDGES * args.steps / dt / 1e9
    sample = "1 layer x 1 MC sample fwd+bwd per step at the full arxiv shape (noise tensor materialised, as the reference does)"
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "mode": args.mode, "sample": sample},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": ref_c.num_threads(), "kind": "port",
                             "sample": sample},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------
class Path:
    """The hot path at the C ABI: pre-built CSC/CSR, resident buffers, direct ctypes calls."""

    def __init__(self, dev, src, dst, S, sample_base, vi, normal="hadamard"):
        import torch
        import stag_b200 as sb
        from stag_b200 import _lib
        self.torch, self._lib, self.lib = torch, _lib, _lib.load()
        self.dev, self.S, self.vi, self.sample_base = dev, S, vi, sample_base
        # vi = True needs d loc / d scale: the two-sum kernel, Box-Muller normals
        self.normal_kind = _lib.NOISE_NORMAL_HADAMARD if (normal == "hadamard" and not vi) else _lib.NOISE_NORMAL
        self.g = sb.Graph(torch.from_numpy(src), torch.from_numpy(dst), N_NODES).to(dev)
        st = self.g._s
        self.csc, self.csc_keep = st.csx(True)
        self.csr, self.csr_keep = st.csx(False)
        self.ss, self.ds = st.scale(False, "rsqrt"), st.scale(True, "rsqrt")
        gen = torch.Generator(device=dev).manual_seed(1234)
        nd = (N_NODES, WIDTH)
        self.x0 = torch.randn(nd, device=dev, generator=gen)
        self.act = [torch.empty((S,) + nd, device=dev) for _ in range(N_LAYERS)]       # layer outputs
        self.gout = torch.randn((S,) + nd, device=dev, generator=gen)                   # dL/d(out of layer 3)
        self.gbuf = [torch.empty((S,) + nd, device=dev) for _ in range(2)]              # ping-pong dX
        self.dx0 = torch.empty((S,) + nd, device=dev)
        # q_a = Normal(1.0, std): scalar parameters expanded to [E,D] (scripts/arxiv_mle/gcn/run.py:61-62)
        self.loc = torch.ones(1, device=dev)
        self.scale = torch.full((1,), SIGMA, device=dev)
        self.dp = torch.zeros((N_LAYERS, 2, 1), device=dev)
        wsb = max(self.lib.stag_spmm_workspace_bytes(ctypes.byref(self.csc), WIDTH, S),
                  self.lib.stag_spmm_workspace_bytes(ctypes.byref(self.csr), WIDTH, S))
        self.ws = torch.empty(max(wsb, 256), dtype=torch.uint8, device=dev)
        self.stream = torch.cuda.current_stream(dev).cuda_stream
        self.launches = 0
        self.offset = 0

    def noise(self, layer):
        n = self._lib.StagNoise()
        n.kind, n.K, n.param_shape = self.normal_kind, WIDTH, self._lib.PARAM_SCALAR
        n.relu = n.in_norm = 0
        n.sample_base = self.sample_base
        n.p0, n.p1, n.external = self.loc.data_ptr(), self.scale.data_ptr(), 0
        n.seed, n.offset = 42, self.offset + layer
        return n

    def fwd(self, layer, x=None):
        x = self.x0 if layer == 0 and x is None else (x if x is not None else self.act[layer - 1])
        shared = x.dim() == 2
        nd = N_NODES * WIDTH
        nz = self.noise(layer)
        self._lib.check(self.lib.stag_spmm_fwd(
            ctypes.byref(self.csc), x.data_ptr(), WIDTH, 0 if shared else nd, WIDTH, self.S, ctypes.byref(nz),
            self.ss.data_ptr(), self.ds.data_ptr(), self.act[layer].data_ptr(), WIDTH, nd, 0,
            self.ws.data_ptr(), self.ws.numel(), self.stream))

    def bwd(self, layer, gin, gout_buf, x=None):
        nd = N_NODES * WIDTH
        nz = self.noise(layer)
        if not self.vi:
            self._lib.check(self.lib.stag_spmm_fwd(
                ctypes.byref(self.csr), gin.data_ptr(), WIDTH, nd, WIDTH, self.S, ctypes.byref(nz),
                self.ds.data_ptr(), self.ss.data_ptr(), gout_buf.data_ptr(), WIDTH, nd, 0,
                self.ws.data_ptr(), self.ws.numel(), self.stream))
        else:
            x = self.x0 if layer == 0 else self.act[layer - 1]
            shared = x.dim() == 2
            self._lib.check(self.lib.stag_spmm_bwd(
                ctypes.byref(self.csr), x.data_ptr(), WIDTH, 0 if shared else nd, gin.data_ptr(), WIDTH, nd,
                WIDTH, self.S, ctypes.byref(nz), self.ss.data_ptr(), self.ds.data_ptr(),
                gout_buf.data_ptr(), WIDTH, nd, self.dp[layer, 0].data_ptr(), self.dp[layer, 1].data_ptr(), 0,
                self.ws.data_ptr(), self.ws.numel(), self.stream))

    def step(self, events=None):
        """3 x forward, 3 x backward.  `events`: list to which (tag, start, end) CUDA events are appended."""
        torch = self.torch

        def timed(tag, fn):
            if events is None:
                return fn()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            events.append((tag, a, b))
        for layer in range(N_LAYERS):
            timed("fwd_shared" if layer == 0 else "fwd", lambda layer=layer: self.fwd(layer))
        gin = self.gout
        for layer in reversed(range(N_LAYERS)):
            out = self.dx0 if layer == 0 else self.gbuf[layer % 2]
            timed("bwd", lambda layer=layer, gin=gin, out=out: self.bwd(layer, gin, out))
            gin = out
        self.offset += N_LAYERS


def e2e_leg(dev, src, dst, S, sample_base, steps, warmup, dist, normal="hadamard"):
    """Same metric through the public Python API (stag_b200.ops.stochastic_aggregate + autograd)
    with HOST buffers: every step copies X [N,D] from pinned host memory, runs the 3-layer
    forward and backward, and reads dX [N,D] and the scalar objective back to the host."""
    import torch
    import stag_b200 as sb
    g = sb.Graph(torch.from_numpy(src), torch.from_numpy(dst), N_NODES).to(dev)
    st = g._s
    st.csx(True), st.csx(False)
    ss, ds = st.scale(False, "rsqrt"), st.scale(True, "rsqrt")
    loc = torch.ones((), device=dev)
    scale = torch.full((), SIGMA, device=dev)
    x_host = torch.randn(N_NODES, WIDTH).pin_memory()
    # Double buffering, the way a training loop with a prefetching loader runs: the host->device copy of step
    # i + 1 and the device->host copy of step i - 1 travel on their own streams (two copy engines) while step i
    # computes.  Every step still copies its own X in and its own dX + objective out inside the timed region.
    compute = torch.cuda.current_stream(dev)
    h2d_s, d2h_s = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    x_dev = [torch.empty(N_NODES, WIDTH, device=dev) for _ in range(2)]
    dx_host = [torch.empty(N_NODES, WIDTH).pin_memory() for _ in range(2)]
    obj_host = [torch.empty(1).pin_memory() for _ in range(2)]
    in_ready = [torch.cuda.Event() for _ in range(2)]    # X of the step has arrived
    in_free = [torch.cuda.Event() for _ in range(2)]     # the step that read this X buffer has finished
    out_done = [torch.cuda.Event() for _ in range(2)]    # dX + objective of the step are on the host
    keep = [None, None]                                  # device results referenced until their copy is done
    state = {"i": 0}

    def prefetch(i):
        k = i % 2
        with torch.cuda.stream(h2d_s):
            if i >= 2:
                h2d_s.wait_event(in_free[k])
            x_dev[k].copy_(x_host, non_blocking=True)
            in_ready[k].record(h2d_s)

    def one():
        i = state["i"]
        k = i % 2
        if i == 0:
            prefetch(0)
        prefetch(i + 1)
        compute.wait_event(in_ready[k])
        x = x_dev[k].detach().requires_grad_(True)
        h = x
        for layer in range(N_LAYERS):
            spec = sb.ops.NoiseSpec("normal", loc, scale, WIDTH, N_EDGES, n_samples=S, sample_base=sample_base,
                                    batched=True, generator=normal)
            h = sb.ops.stochastic_aggregate(g, h, spec, src_scale=ss, dst_scale=ds, n_samples=S)
        obj = h.mean()
        obj.backward()
        in_free[k].record(compute)
        if i >= 2:
            out_done[k].synchronize()   # the host buffers of step i - 2 have been read
        keep[k] = (x.grad, obj.detach().reshape(1))
        with torch.cuda.stream(d2h_s):
            d2h_s.wait_event(in_free[k])
            dx_host[k].copy_(keep[k][0], non_blocking=True)
            obj_host[k].copy_(keep[k][1], non_blocking=True)
            out_done[k].record(d2h_s)
        state["i"] = i + 1

    for _ in range(warmup):
        one()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        one()
    torch.cuda.synchronize()   # every step's dX and objective are on the host
    dt = time.perf_counter() - t0
    if dist is not None:
        t = torch.tensor([dt], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
    return dt / steps, N_NODES * WIDTH * 4, N_NODES * WIDTH * 4 + 4


def cpu_baseline(mode):
    from oracle import cbuild, ref_c
    cbuild.build()
    ref_c.use_all_cores()
    src, dst = synth_graph()
    rng = np.random.default_rng(1)
    x = rng.standard_normal((N_NODES, WIDTH)).astype(np.float32)
    g = rng.standard_normal((N_NODES, WIDTH)).astype(np.float32)
    lp = ref_c.LayerPass(src, dst, N_NODES, x, g, "normal", 1.0, SIGMA, vi=(mode == "vi"))
    lp.run(0)
    n, t0 = 0, time.perf_counter()
    while n < 3 or (time.perf_counter() - t0 < 10.0 and n < 64):
        lp.run(1 + n)
        n += 1
    dt = time.perf_counter() - t0
    return {"value": N_EDGES * n / dt / 1e9, "unit": UNIT, "cores": ref_c.num_threads(), "kind": "port",
            "sample": "%d x (1 layer x 1 MC sample fwd+bwd) at the full arxiv shape, un-fused C/OpenMP restatement "
                      "of the reference algorithm (oracle/csrc/stag_ref.c), %.1f s" % (n, dt)}


def run_ours(args, rank, world):
    import torch
    local = int(os.environ.get("LOCAL_RANK", 0))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist_.init_process_group("nccl", device_id=dev)
        dist = dist_
    S = N_SAMPLES
    vi = args.mode == "vi"
    src, dst = synth_graph()
    path = Path(dev, src, dst, S, sample_base=rank * S, vi=vi, normal=args.normal)
    for _ in range(max(args.warmup, 3)):
        path.step()
    torch.cuda.synchronize()
    sampler = ClockSampler(local) if rank == 0 else None
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    if sampler:
        sampler.start()
    launches0 = path.lib.stag_launch_count()
    events = []
    t_start, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_start.record()
    for _ in range(args.steps):
        path.step(events)
    t_end.record()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    clocks = sampler.stop() if sampler else None
    ms = t_start.elapsed_time(t_end)
    if dist is not None:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    launches = int(path.lib.stag_launch_count() - launches0)   # counted inside libstag_b200.so
    if args.dump_outputs and rank == 0:
        rows = torch.from_numpy(dump_rows(src, dst)).to(dev)
        arrays = {"out%d" % (i + 1): a.index_select(1, rows).cpu().numpy() for i, a in enumerate(path.act)}
        arrays["dx"] = path.dx0.index_select(1, rows).cpu().numpy()
        if vi:
            arrays["dparams"] = path.dp.reshape(N_LAYERS, 2).cpu().numpy()
        dump_outputs(args.dump_outputs, arrays)
    ms_per_step = ms / args.steps
    edge_samples = N_EDGES * S * N_LAYERS * world
    value = edge_samples / (ms_per_step * 1e-3) / 1e9

    # per-launch-class device times -> roofline of the dominant kernel
    per = {}
    for tag, a, b in events:
        per.setdefault(tag, []).append(a.elapsed_time(b))
    tot = {k: sum(v) for k, v in per.items()}
    dom = max(tot, key=tot.get)
    avg_ms = float(np.mean(per[dom]))
    alg = {"fwd_shared": bytes_fwd(S, True), "fwd": bytes_fwd(S, False),
           "bwd": (2 * bytes_bwd(S, vi, False) + bytes_bwd(S, vi, True)) / 3.0}[dom]
    peak, peak_src = peaks()
    achieved = alg / (avg_ms * 1e-3) / 1e9
    step_bytes = bytes_fwd(S, True) + 2 * bytes_fwd(S, False) + 2 * bytes_bwd(S, vi, False) + bytes_bwd(S, vi, True)
    roof = {"bound": "hbm", "kernel": ("stag::agg_wh_quad_kernel (tensor-core normal generator, %s launches)" if path.normal_kind == path._lib.NOISE_NORMAL_HADAMARD
                       else "stag::agg_stream_kernel<NORMAL, 2 blocks per lane> (%s launches)") % dom, "achieved": achieved, "peak": peak,
            "unit": "GB/s", "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
            "algorithmic_bytes_per_launch": alg, "avg_launch_ms": avg_ms,
            "share_of_step": tot[dom] / sum(tot.values()),
            "per_class_ms": {k: float(np.mean(v)) for k, v in per.items()},
            "whole_step_frac": step_bytes / (ms_per_step * 1e-3) / 1e9 / peak}
    if path.normal_kind == path._lib.NOISE_NORMAL:
        # Secondary ceiling (SURVEY 8(d)): the launch draws E*S*D normals; Box-Muller needs 2 MUFU per normal and the
        # XU pipe runs 16 lanes / clk / SM (measured, profiles/r01_microbench.txt), at the SM clock sampled during the run.
        prop = torch.cuda.get_device_properties(dev)
        mhz = (clocks or {}).get("sm_mhz") or getattr(prop, "clock_rate", 0) / 1e3
        normals = float(N_EDGES) * S * WIDTH
        if mhz:
            xu_peak = prop.multi_processor_count * 16.0 * mhz * 1e6 / 2.0
            roof["rng_ceiling"] = {"normals_per_launch": normals, "achieved_normals_per_s": normals / (avg_ms * 1e-3),
                                   "xu_peak_normals_per_s": xu_peak, "frac": normals / (avg_ms * 1e-3) / xu_peak,
                                   "note": "Box-Muller, 2 MUFU per normal, 16 MUFU lanes/clk/SM measured"}
    prof = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if os.path.exists(prof):
        with open(prof) as f:
            roof["traffic"] = json.load(f).get(dom)

    e2e_s, h2d, d2h = e2e_leg(dev, src, dst, S, rank * S, max(3, min(args.steps, 8)), 5, dist, args.normal)
    e2e = {"value": edge_samples / e2e_s / 1e9, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
           "api": "stag_b200.ops.stochastic_aggregate + autograd, pinned host X in / dX + objective out every step, copies double-buffered on two copy streams"}
    multi = None
    if world > 1 and not args.no_multi:
        # every number in here has a collective inside its timed region (bench_multi.py): strong scaling over the MC
        # samples with the gradient / MC-mean all-reduces, PPI minibatch data parallel, row-partitioned products graph
        import bench_multi
        path.act = path.gbuf = path.gout = path.dx0 = None   # the headline's buffers (7 GB) make room for the legs
        torch.cuda.empty_cache()
        multi = bench_multi.run_all(dev, dist, rank, world, args.steps, args.warmup, args.normal)
    configs = unfused = None
    if world == 1 and not args.no_configs:
        # the other BASELINE.json configurations (C1, C3, C4, C5, vi mode) with the same timing method, and the
        # reference's un-fused algorithm in plain torch ops on this GPU (ADVICE r1: a same-hardware baseline)
        import bench_multi
        path.act = path.gbuf = path.gout = path.dx0 = None
        torch.cuda.empty_cache()
        unfused = bench_multi.unfused_gpu_baseline(dev, src, dst, N_NODES, WIDTH, SIGMA)
        configs = bench_multi.configs_single_gpu(dev, peak)
    if rank != 0:
        return
    cpu = cpu_baseline(args.mode) if (world == 1 and not args.no_cpu_baseline) else None
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "mode": args.mode, "layers": N_LAYERS, "mc_samples_per_gpu": S,
                       "normal_generator": ("hadamard (tensor cores)" if path.normal_kind == path._lib.NOISE_NORMAL_HADAMARD
                                            else "boxmuller (16-bit halves)"),
                       "sharded_unit": "MC samples (Philox sample index), no data-path collective",
                       "l2": "per-launch inputs (1.39 GB activations per layer) exceed the 126 MB L2: nothing is L2-resident "
                             "from one timed launch to the next (ncu: DRAM traffic 1.5x the algorithmic bytes on the per-sample "
                             "launches, 1.7x on the layer-1 launch, whose shared X is re-fetched by most of the 16 samples)"},
            "roofline": roof, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches, "clocks": clocks}
    if multi is not None:
        line["multi_gpu"] = multi
    if configs is not None:
        line["configs"] = configs
        line["unfused_gpu_baseline"] = unfused
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default="mle", choices=["mle", "vi"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="N = 1: skip the `configs` dict (C1, C3, C4, C5, vi)")
    ap.add_argument("--no-multi", action="store_true", help="N > 1: skip the multi_gpu legs (collectives inside the timed region)")
    ap.add_argument("--normal", default="hadamard", choices=["hadamard", "boxmuller"],
                    help="standard-normal generator of the fused kernels: tensor-core Walsh-Hadamard mix "
                         "(agg_wh_quad_kernel) or 16-bit Box-Muller (agg_stream_kernel)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (float32, a fixed node sample)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    run_ours(args, rank, world)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
