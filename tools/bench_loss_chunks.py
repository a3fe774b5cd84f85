"""Monte-Carlo training in bounded memory: ms per sample and peak allocated memory of ``loss(n_samples=S).backward()``
against ``StagModel.loss_backward(S, chunk)``, and one 32-sample training step on the products-shaped graph in chunks of
4 samples on one GPU.

    python tools/bench_loss_chunks.py [--iters 3] [--out FILE]

arxiv: ogbn-arxiv shape (N 169 343, E 1 166 243, bench.synth_graph), 3-layer StagLayer(GCN) 128 -> 256 -> 256 -> 40 with
a softmax head, trainable per-channel Normal posteriors (vi=True), train mode, Categorical labels.  ``loss(64).backward()``
runs only when the footprint extrapolated linearly from the 16- and 32-sample peaks fits in 80 % of the free memory.
products: N 2 449 029, E 61 859 140 (the power-law construction of bench_multi.py's C5 legs), 2-layer GCN 100 -> 100 -> 47,
scalar Normal(1, 0.4) noise without gradients (the tensor-core generator, zero-padded to 128), 47 classes.
Times are CUDA events around whole calls after one warm-up call; peaks are taken in separate calls."""
import argparse
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HIDDEN, C = 256, 40
GB = 1e9


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
    """Peak allocated bytes above what was allocated before the call (gradients already allocated)."""
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    fn()
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated() - before


def arxiv_model(dev):
    import stag_b200 as sb
    from stag_b200.layers import StagLayer, FeatOnlyLayer
    torch.manual_seed(0)

    def normal(k):
        return torch.distributions.Normal(torch.ones(k), torch.full((k,), 0.5))

    layers = [StagLayer(sb.zoo.GCN(128, HIDDEN, activation=torch.relu), q_a=normal(128), vi=True),
              StagLayer(sb.zoo.GCN(HIDDEN, HIDDEN, activation=torch.relu), q_a=normal(HIDDEN), vi=True),
              StagLayer(sb.zoo.GCN(HIDDEN, C), q_a=normal(HIDDEN), vi=True), FeatOnlyLayer(torch.nn.Softmax(-1))]
    return sb.models.StagModel(torch.nn.ModuleList(layers)).to(dev).train()


def products_model(dev, width=100, classes=47):
    import stag_b200 as sb
    from stag_b200.layers import StagLayer, FeatOnlyLayer
    torch.manual_seed(0)
    q = torch.distributions.Normal(1.0, 0.4)
    layers = [StagLayer(sb.zoo.GCN(width, width, activation=torch.relu), q_a=q),
              StagLayer(sb.zoo.GCN(width, classes), q_a=q), FeatOnlyLayer(torch.nn.Softmax(-1))]
    return sb.models.StagModel(torch.nn.ModuleList(layers)).to(dev).train()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_loss_chunks.py needs a CUDA device")
    import bench
    import bench_multi
    import stag_b200 as sb

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
    model = arxiv_model(dev)
    x = torch.randn(N, 128, device=dev)
    y = torch.randint(0, C, (N,), device=dev)

    def loss_step(S):
        return lambda: model.loss(g, x, y, n_samples=S).backward()

    def chunked_step(S, c):
        return lambda: model.loss_backward(g, x, y, n_samples=S, chunk_samples=c)

    say()
    say("arxiv shape, 3-layer vi GCN 128 -> %d -> %d -> %d, per-channel Normal posteriors, train mode; %d timed calls "
        "after 1 warm-up" % (HIDDEN, HIDDEN, C, args.iters))
    say("%-30s %12s %14s %16s" % ("call", "ms / call", "ms / sample", "peak alloc GB"))
    peaks = {}
    rows = [("loss(%d).backward()" % S, S, loss_step(S)) for S in (16, 32)]
    rows += [("loss_backward(%d, %d)" % (S, c), S, chunked_step(S, c)) for S in (64, 256) for c in (8, 16, 32)]
    for i, (name, S, fn) in enumerate(rows):
        ms = timed(fn, args.iters)
        pk = peak_bytes(fn)
        peaks[name] = pk
        say("%-30s %12.2f %14.3f %16.2f" % (name, ms, ms / S, pk / GB))
        if i == 1:
            est = peaks["loss(32).backward()"] + 2 * (peaks["loss(32).backward()"] - peaks["loss(16).backward()"])
            free = torch.cuda.mem_get_info(dev)[0]
            if est <= 0.8 * free:
                fn = loss_step(64)
                ms = timed(fn, args.iters)
                pk = peak_bytes(fn)
                say("%-30s %12.2f %14.3f %16.2f" % ("loss(64).backward()", ms, ms / 64, pk / GB))
            else:
                say("loss(64).backward() not run: extrapolated peak %.1f GB, free %.1f GB" % (est / GB, free / GB))
    model.zero_grad(set_to_none=True)
    sb.manual_seed(3)
    nll, reg = model.loss_terms(g, x, y, n_samples=32)
    (nll + reg).backward()
    ref = {k: p.grad.clone() for k, p in model.named_parameters()}
    model.zero_grad(set_to_none=True)
    sb.manual_seed(3)
    res = model.loss_backward(g, x, y, n_samples=32, chunk_samples=8)
    worst = max(float((p.grad - ref[k]).abs().max() / ref[k].abs().max()) for k, p in model.named_parameters())
    say("max over parameters of max |grad(loss_backward(32, 8)) - grad(loss(32))| / max |grad(loss(32))| = %.2e; "
        "nll %.6f vs %.6f" % (worst, float(res.nll), float(nll.detach())))
    say("from shapes: one [S,N,%d] fp32 activation is %.1f GB at S = 64 and %.1f GB at S = 256"
        % (HIDDEN, 64 * N * HIDDEN * 4 / GB, 256 * N * HIDDEN * 4 / GB))
    del model, ref, x, y, g, nll, reg, res
    torch.cuda.empty_cache()

    say()
    Np, Ep, D, K, S, c = 2449029, 61859140, 100, 47, 32, 4
    s5, d5 = bench_multi.powerlaw_graph_device(Np, Ep, 0x57A6 + 5, 17000, dev)
    gp = sb.Graph(s5, d5, Np)
    del s5, d5
    model = products_model(dev, D, K)
    xp = torch.randn(Np, D, device=dev)
    yp = torch.randint(0, K, (Np,), device=dev)
    step = lambda: model.loss_backward(gp, xp, yp, n_samples=S, chunk_samples=c)  # noqa: E731
    ms = timed(step, max(1, args.iters - 1))
    pk = peak_bytes(step)
    say("products shape (N %d, E %d), 2-layer GCN %d -> %d -> %d, scalar Normal(1, 0.4) noise, one GPU:" % (Np, Ep, D, D, K))
    say("  loss_backward(%d, %d): %.1f ms per step (%.2f ms / sample), peak allocated %.2f GB" % (S, c, ms, ms / S, pk / GB))
    say("  from shapes: one [%d,N,%d] fp32 activation is %.1f GB; the card has %.0f GB"
        % (S, D, S * Np * D * 4 / GB, torch.cuda.get_device_properties(dev).total_memory / GB))
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
