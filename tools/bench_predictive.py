"""Monte-Carlo predictive in bounded memory: ms per sample and peak allocated memory of ``forward(n_samples=S)`` against
``StagModel.predictive(S, chunk)``, 1024 samples in chunks of 32 next to what the all-at-once forward would need
(computed from shapes: it does not fit on the card, so it is not run), and ``stag_mc_accumulate`` against the
equivalent torch ops on the same [S,N,C] outputs.

    python tools/bench_predictive.py [--iters 5] [--out FILE]

Shape: ogbn-arxiv (N 169 343, E 1 166 243, bench.synth_graph), 3-layer StagLayer(GCN) 128 -> 256 -> 256 -> 40 with a
softmax head, Normal posteriors with per-channel parameters, eval mode.  Times are CUDA events around whole calls
after one warm-up call; the [32, N, 40] operand of the accumulator comparison (867 MB) is larger than the L2."""
import argparse
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HIDDEN, C = 256, 40


def timed(fn, iters, warmup=1):
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


def peak_bytes(fn):
    """Peak allocated bytes above what was allocated before the call (the result is dropped inside)."""
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    fn()
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated() - before


def make_model(dev):
    import stag_b200 as sb
    from stag_b200.layers import StagLayer, FeatOnlyLayer
    torch.manual_seed(0)

    def normal(k):
        return torch.distributions.Normal(torch.ones(k), torch.full((k,), 0.5))

    layers = [StagLayer(sb.zoo.GCN(128, HIDDEN, activation=torch.relu), q_a=normal(128)),
              StagLayer(sb.zoo.GCN(HIDDEN, HIDDEN, activation=torch.relu), q_a=normal(HIDDEN)),
              StagLayer(sb.zoo.GCN(HIDDEN, C), q_a=normal(HIDDEN)), FeatOnlyLayer(torch.nn.Softmax(-1))]
    return sb.models.StagModel(torch.nn.ModuleList(layers)).to(dev).eval()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_predictive.py needs a CUDA device")
    import bench
    import stag_b200 as sb
    from stag_b200 import ops

    lines = []

    def say(s=""):
        print(s, flush=True)
        lines.append(s)

    dev = torch.device("cuda")
    try:
        card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                               str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:  # noqa: BLE001
        card = "unknown"
    say("device: %s (nvidia-smi name, power limit: %s)" % (torch.cuda.get_device_name(dev), card or "unknown"))
    src, dst = bench.synth_graph()
    N = bench.N_NODES
    g = sb.Graph(torch.from_numpy(src), torch.from_numpy(dst), N).to(dev)
    model = make_model(dev)
    x = torch.randn(N, 128, device=dev)
    GB = 1e9

    say()
    say("arxiv shape, 3-layer GCN 128 -> %d -> %d -> %d, Normal per-channel noise, eval; %d timed calls after 1 warm-up"
        % (HIDDEN, HIDDEN, C, args.iters))
    say("%-28s %12s %14s %16s" % ("call", "ms / call", "ms / sample", "peak alloc GB"))
    S = 64
    with torch.no_grad():
        fwd = lambda: model(g, x, n_samples=S, return_parameters=True)  # noqa: E731
        ms = timed(fwd, args.iters)
        pk = peak_bytes(fwd)
        say("%-28s %12.2f %14.3f %16.2f" % ("forward(n_samples=%d)" % S, ms, ms / S, pk / GB))
    for chunk in (8, 16, 32, 64):
        call = lambda: model.predictive(g, x, S, chunk_samples=chunk)  # noqa: E731
        ms = timed(call, args.iters)
        pk = peak_bytes(call)
        say("%-28s %12.2f %14.3f %16.2f" % ("predictive(%d, chunk=%d)" % (S, chunk), ms, ms / S, pk / GB))
    sb.manual_seed(3)
    with torch.no_grad():
        ref = model(g, x, n_samples=S, return_parameters=True)
    sb.manual_seed(3)
    got = model.predictive(g, x, S, chunk_samples=16).mean
    say("max |predictive(64, 16).mean - forward(64)| / max |forward(64)| = %.2e"
        % float((got - ref).abs().max() / ref.abs().max()))
    del ref, got

    say()
    S, chunk = 1024, 32
    call = lambda: model.predictive(g, x, S, chunk_samples=chunk)  # noqa: E731
    ms = timed(call, 1, warmup=0)
    pk = peak_bytes(call)
    act = S * N * HIDDEN * 4
    say("predictive(%d, chunk=%d): %.1f ms (%.3f ms / sample), peak allocated %.2f GB"
        % (S, chunk, ms, ms / S, pk / GB))
    say("forward(n_samples=%d), from shapes (not run): one [S,N,%d] fp32 activation %.1f GB, a layer's input and output "
        "%.1f GB, output stack [S,N,%d] %.1f GB; the card has %.0f GB"
        % (S, HIDDEN, act / GB, 2 * act / GB, C, S * N * C * 4 / GB, torch.cuda.get_device_properties(dev).total_memory / GB))

    say()
    S = 32
    gen = torch.Generator(device=dev).manual_seed(1)
    probs = torch.softmax(torch.randn((S, N, C), device=dev, generator=gen), -1)
    acc_sum = torch.zeros((N, C), dtype=torch.float64, device=dev)
    acc_ent = torch.zeros(N, dtype=torch.float64, device=dev)
    eps = torch.finfo(torch.float32).eps

    def kernel():
        ops.mc_accumulate(probs, acc_sum, acc_ent)

    def torch_ops():
        # what a user computes with torch today: Categorical(probs=p).entropy() per sample, float64 sums
        q = probs / probs.sum(-1, keepdim=True)
        acc_ent.add_(-(q * q.clamp(eps, 1 - eps).log()).sum(-1).sum(0, dtype=torch.float64))
        acc_sum.add_(probs.sum(0, dtype=torch.float64))

    iters = max(args.iters, 20)
    tk = timed(kernel, iters)
    tt = timed(torch_ops, iters)
    nbytes = S * N * C * 4 + 2 * (N * C * 8 + N * 8)
    say("accumulate [%d, N, %d] fp32 (%.0f MB read) into float64 accumulators, mean of %d calls after 1 warm-up:"
        % (S, C, S * N * C * 4 / 1e6, iters))
    say("  stag_mc_accumulate  %8.3f ms  (%.2f TB/s of probs + accumulator traffic)" % (tk, nbytes / tk / 1e9))
    say("  torch ops           %8.3f ms  (%.1fx)" % (tt, tt / tk))
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
