"""Stochastic GAT: ms per training step (loss_terms + backward, CUDA events, after warm-up) of two-layer GAT models, the
sequential passes with emitted noise against the fused, sample-batched path, and the attention kernel alone (one S-sample
launch against S one-sample launches).  Also checks the batched outputs against the tensor path fed the same
materialised noise.

    python tools/bench_gat.py [--iters 10] [--out FILE]

Shapes: arxiv (N 169 343, E 1 166 243): 128 -> 4 x 32 -> 40 (one head, last=True), S = 16; Cora-shaped (N 2 708,
E 10 556 random edges plus self-loops, 1 433 features): 1433 -> 8 x 8 -> 7, S = 4.  vi=True, Normal posteriors with
per-head parameters.  Arms:
  emitted    batch_samples=False and the base layers refuse NoiseSpecs: S sequential passes, each materialising its
             [E,H] noise with stag_noise_emit (the path every GAT model took before the attention kernel drew its noise)
  sequential batch_samples=False: S sequential passes on the fused attention (noise drawn in the kernel)
  batched    the default: one pass over [S,N,D] tensors, one attention launch per layer for all S samples"""
import argparse
import ctypes
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def timed(fn, iters, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def make_model(sizes, dev):
    """Two StagLayer(GAT) layers: sizes = (D, F1, H1, C)."""
    import stag_b200 as sb
    D, F1, H1, C = sizes
    torch.manual_seed(0)

    def q(h):
        return torch.distributions.Normal(torch.ones(h), torch.full((h,), 0.5))

    layers = torch.nn.ModuleList([
        sb.layers.StagLayer(sb.zoo.GAT(D, F1, num_heads=H1, activation=torch.nn.functional.elu), q_a=q(H1), vi=True),
        sb.layers.StagLayer(sb.zoo.GAT(F1 * H1, C, num_heads=1, last=True, activation=lambda t: torch.softmax(t, -1)),
                            q_a=q(1), vi=True),
    ]).to(dev)
    return sb.models.StagModel(layers)


def set_arm(model, arm):
    model.batch_samples = arm == "batched"
    for layer in model.layers:
        if arm == "emitted":
            layer.base_layer.accepts_noise_spec = False       # instance attribute: StagLayer materialises the noise
        elif "accepts_noise_spec" in layer.base_layer.__dict__:
            del layer.base_layer.accepts_noise_spec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_gat.py needs a CUDA device")
    import bench
    import stag_b200 as sb
    from stag_b200 import _lib, ops
    from stag_b200.ops import NoiseSpec

    lines = []

    def say(s=""):
        print(s, flush=True)
        lines.append(s)

    dev = torch.device("cuda")
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                             str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:  # noqa: BLE001
        pl = "unknown"
    say("device: %s, power limit %s" % (torch.cuda.get_device_name(dev), pl or "unknown"))
    src, dst = bench.synth_graph()
    arxiv = sb.Graph(torch.from_numpy(src), torch.from_numpy(dst), bench.N_NODES).to(dev)
    rng = np.random.default_rng(0)
    nc, ec = 2708, 10556
    cora = sb.add_self_loop(sb.Graph(torch.from_numpy(rng.integers(0, nc, ec)), torch.from_numpy(rng.integers(0, nc, ec)),
                                     nc)).to(dev)
    cases = [("arxiv 128 -> 4x32 -> 40, S=16", arxiv, (128, 32, 4, 40), 16),
             ("cora 1433 -> 8x8 -> 7, S=4", cora, (1433, 8, 8, 7), 4)]

    say()
    say("training step: loss_terms + backward, ms (%d timed steps after 3 warm-up steps)" % args.iters)
    say("%-34s %10s %12s %10s %10s" % ("model", "emitted", "sequential", "batched", "speed-up"))
    for name, g, sizes, S in cases:
        N = g.number_of_nodes()
        torch.manual_seed(1)
        x = torch.randn(N, sizes[0], device=dev)
        y = torch.randint(0, sizes[3], (N,), device=dev)
        model = make_model(sizes, dev)
        res = {}
        for arm in ("emitted", "sequential", "batched"):
            set_arm(model, arm)
            assert model._can_batch() == (arm == "batched")

            def step():
                model.zero_grad(set_to_none=True)
                nll, reg = model.loss_terms(g, x, y, n_samples=S)
                (nll + reg).backward()

            res[arm] = timed(step, args.iters)
        set_arm(model, "batched")
        say("%-34s %10.3f %12.3f %10.3f %9.2fx" % (name, res["emitted"], res["sequential"], res["batched"],
                                                   res["emitted"] / res["batched"]))

    # attention kernel alone, arxiv, H = 4, shared scores (the first layer), per-head Normal parameters with gradients
    st = arxiv._s
    lib = _lib.load()
    csc, _ = st.csx(True)
    N, E, H, S = bench.N_NODES, bench.N_EDGES, 4, 16
    stream = torch.cuda.current_stream().cuda_stream
    el, er = torch.randn(N, H, device=dev), torch.randn(N, H, device=dev)
    loc, sc = torch.ones(H, device=dev), torch.full((H,), 0.5, device=dev)
    a = torch.empty(S, E, H, device=dev)
    da = torch.randn(S, E, H, device=dev)
    dpre = torch.empty(S, E, H, device=dev)
    d_er = torch.empty(S, N, H, device=dev)
    d0, d1 = torch.empty(H, device=dev), torch.empty(H, device=dev)
    ws = ops._attention_workspace(st, lib, csc, H, S)

    def nz(base):
        return ops._fill_noise(None, _lib.NOISE_NORMAL, H, loc, sc, None, False, False, base, 1, 2, _lib.PARAM_CHANNEL)

    nzs = [nz(s) for s in range(S)]
    R = _lib.check

    def fwd(s0, n):
        R(lib.stag_attention_softmax_s(ctypes.byref(csc), el.data_ptr(), 0, er.data_ptr(), 0, H, n, ctypes.byref(nzs[s0]),
                                       0.2, a[s0].data_ptr(), ws.data_ptr(), ws.numel(), stream))

    def bwd(s0, n):
        R(lib.stag_attention_softmax_s_bwd(ctypes.byref(csc), el.data_ptr(), 0, er.data_ptr(), 0, H, n,
                                           ctypes.byref(nzs[s0]), 0.2, a[s0].data_ptr(), da[s0].data_ptr(),
                                           dpre[s0].data_ptr(), d_er[s0].data_ptr(), d0.data_ptr(), d1.data_ptr(), 0,
                                           ws.data_ptr(), ws.numel(), stream))

    say()
    say("attention kernel alone, arxiv, H=4, generated Normal noise with per-head parameters, ms for %d samples" % S)
    t1f = timed(lambda: fwd(0, S), args.iters * 2)
    tsf = timed(lambda: [fwd(s, 1) for s in range(S)], args.iters * 2)
    t1b = timed(lambda: bwd(0, S), args.iters * 2)
    tsb = timed(lambda: [bwd(s, 1) for s in range(S)], args.iters * 2)
    say("%-46s %10s %12s" % ("", "1 x S=16", "16 x S=1"))
    say("%-46s %10.3f %12.3f" % ("forward (stag_attention_softmax_s)", t1f, tsf))
    say("%-46s %10.3f %12.3f" % ("backward + d loc / d scale (_s_bwd + finalize)", t1b, tsb))

    # batched outputs against the tensor path fed the same materialised noise
    say()
    torch.manual_seed(2)
    base = sb.zoo.GAT(128, 32, num_heads=4).to(dev)
    x = torch.randn(N, 128, device=dev)
    spec = NoiseSpec("normal", loc, sc, H, E, seed=3, offset=4, n_samples=S, batched=True)
    worst_a = worst_o = 0.0
    with torch.no_grad():
        out, att = base(arxiv, x, edge_weight=spec, get_attention=True)
        w = spec.materialize(n_samples=S)
        for s in range(S):
            o, at = base(arxiv, x, edge_weight=w[s], get_attention=True)
            worst_a = max(worst_a, float((att[s] - at).abs().max() / at.abs().max()))
            worst_o = max(worst_o, float((out[s] - o).abs().max() / o.abs().max()))
    say("check, arxiv GAT 128 -> 4x32, S=16 against 16 tensor-path passes on materialize(16): attention max rel err %.3g, "
        "output max rel err %.3g" % (worst_a, worst_o))
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
