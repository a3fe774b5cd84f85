"""Calibration tables on the GPU: ``stag_calibration`` at the arxiv, PPI and 1024-class shapes, against
``stag_mc_accumulate`` on a [32, N, 40] chunk (the yardstick: the calibration pass of a 32-sample predictive must cost
at most a tenth of one accumulate call) and against the equivalent torch ops (argmax, bucketize, float64 scatter_add).

    python tools/bench_calibration.py [--iters 50] [--out FILE]

Times are CUDA events around ``iters`` back-to-back calls after warm-up calls, of the C ABI entry point called through
ctypes with prepared arguments ("abi") and of ``ops.calibration_table`` ("python": argument checks, dtype casts and the
ctypes call, on the host).  Kernel times are device durations from torch.profiler, taken after the event timings.  The
calibration inputs of one call are smaller than the 126 MB L2, so each timed call reads the next of several copies
whose total exceeds 512 MB: every call reads its probabilities from HBM.  GB/s counts the probability bytes of the rows
read (masked-out rows are not read), over the ABI call time."""
import argparse
import math
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

N_ARXIV, C_ARXIV = 169_343, 40
N_PPI, C_PPI = 56_944, 121


def timed(fns, iters, warmup=2):
    """Mean ms per call of ``fns[i % len(fns)]()`` over ``iters`` calls."""
    for i in range(warmup * len(fns)):
        fns[i % len(fns)]()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(iters):
        fns[i % len(fns)]()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def kernel_us(fns, name, calls=20):
    """Mean device duration (us) of the kernels whose name contains ``name`` over ``calls`` calls."""
    from torch.profiler import profile, ProfilerActivity
    for f in fns:
        f()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(calls):
            fns[i % len(fns)]()
        torch.cuda.synchronize()
    total = count = 0
    for e in prof.key_averages():
        if name in e.key:
            total += getattr(e, "self_device_time_total", None) or e.self_cuda_time_total
            count += e.count
    return total / max(count, 1)


def inputs(kind, N, C, copies, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    out = []
    for _ in range(copies):
        logits = torch.randn((N, C), device="cuda", generator=g) * 2.0
        if kind == "categorical":
            p = torch.softmax(logits, -1)
            y = torch.randint(0, C, (N,), device="cuda", generator=g)
        else:
            p = torch.sigmoid(logits)
            y = (torch.rand((N, C), device="cuda", generator=g) < p).float()
        out.append((p, y))
    return out


def torch_table(p, y, B, edges):
    """The Categorical table with torch ops: top-label and per-class counts / sums in float64 (what a user writes
    without the kernel)."""
    N, C = p.shape
    q = p.double() / p.double().sum(-1, keepdim=True)
    conf, k = q.max(-1)
    b = torch.bucketize(conf, edges)
    top = torch.zeros(3 * B, dtype=torch.float64, device=p.device)
    top.scatter_add_(0, b, torch.ones_like(conf))
    top.scatter_add_(0, b + B, conf)
    top.scatter_add_(0, b + 2 * B, (k == y).double())
    onehot = torch.nn.functional.one_hot(y, C).double()
    brier = ((q - onehot) ** 2).sum()
    idx = (torch.bucketize(q, edges) + B * torch.arange(C, device=p.device)).reshape(-1)
    cls = torch.zeros(3 * C * B, dtype=torch.float64, device=p.device)
    cls.scatter_add_(0, idx, torch.ones_like(idx, dtype=torch.float64))
    cls.scatter_add_(0, idx + C * B, q.reshape(-1))
    cls.scatter_add_(0, idx + 2 * C * B, onehot.reshape(-1))
    return top, cls, brier


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_calibration.py needs a CUDA device")
    from stag_b200 import ops, _lib

    lines = []

    def say(s=""):
        print(s, flush=True)
        lines.append(s)

    dev = torch.device("cuda")
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True,
                          text=True, timeout=60).stdout.strip().splitlines()
    say("nvidia-smi: %s" % " | ".join(card))
    say("torch device %d: %s" % (torch.cuda.current_device(), torch.cuda.get_device_name(dev)))
    say("%d timed calls after warm-up, CUDA events; every call reads its probabilities from HBM (rotating copies > L2)"
        % args.iters)
    say()
    say("%-46s %9s %9s %9s %9s %9s" % ("call", "abi ms", "python ms", "kernel ms", "GB/s", "probs MB"))

    def row(name, ms, py_ms, k_us, nbytes):
        say("%-46s %9.4f %9s %9.4f %9.1f %9.1f" % (name, ms, "%.4f" % py_ms if py_ms else "-", k_us / 1e3,
                                                   nbytes / ms / 1e6, nbytes / 1e6))

    def copies_for(nbytes):
        return max(1, math.ceil(512e6 / nbytes))

    # yardstick: stag_mc_accumulate on a [32, N, 40] chunk (867 MB, larger than the L2)
    S = 32
    gen = torch.Generator(device=dev).manual_seed(1)
    probs = torch.softmax(torch.randn((S, N_ARXIV, C_ARXIV), device=dev, generator=gen), -1)
    acc_sum = torch.zeros((N_ARXIV, C_ARXIV), dtype=torch.float64, device=dev)
    acc_ent = torch.zeros(N_ARXIV, dtype=torch.float64, device=dev)
    acc = [lambda: ops.mc_accumulate(probs, acc_sum, acc_ent)]
    t_acc = timed(acc, max(args.iters // 2, 10))
    k_acc = kernel_us(acc, "mc_accumulate_kernel")
    row("stag_mc_accumulate [32, N, 40] (arxiv)", t_acc, None, k_acc, probs.numel() * 4)
    del probs, acc_sum, acc_ent

    results = {}

    def bench(name, kind, N, C, B, mask_frac=None):
        nbytes = N * C * 4
        data = inputs(kind, N, C, copies_for(nbytes), seed=N + C + B)
        mask = None
        if mask_frac is not None:
            mask = torch.rand(N, device=dev, generator=torch.Generator(device=dev).manual_seed(7)) < mask_frac
        table = torch.zeros(ops.calibration_table_len(C, B), dtype=torch.int64, device=dev)
        py = [lambda p=p, y=y: ops.calibration_table(p, y, kind, B, mask=mask, out=table) for p, y in data]
        lib, stream = _lib.load(), torch.cuda.current_stream(dev).cuda_stream
        mk8 = None if mask is None else mask.to(torch.uint8)     # kept alive while the lambdas use its pointer
        mk = 0 if mk8 is None else mk8.data_ptr()
        k = 0 if kind == "categorical" else 1
        abi = [lambda a=(p.data_ptr(), y.data_ptr()): lib.stag_calibration(a[0], C, N, C, k, a[1], C, mk, B,
                                                                           table.data_ptr(), stream) for p, y in data]
        ms = timed(abi, args.iters)
        py_ms = timed(py, args.iters)
        k_us = kernel_us(abi, "calib_kernel")
        read = (int(mask.sum()) if mask is not None else N) * C * 4
        row(name, ms, py_ms, k_us, read)
        results[name] = (ms, k_us)
        return data, mask

    say()
    data, _ = bench("calibration arxiv N 169343 C 40 B 15", "categorical", N_ARXIV, C_ARXIV, 15)
    bench("calibration arxiv, 30 % mask", "categorical", N_ARXIV, C_ARXIV, 15, mask_frac=0.3)
    bench("calibration PPI N 56944 C 121 B 15 Bernoulli", "bernoulli", N_PPI, C_PPI, 15)
    bench("calibration N 169343 C 1024 B 15", "categorical", N_ARXIV, 1024, 15)
    bench("calibration N 169343 C 1024 B 64", "categorical", N_ARXIV, 1024, 64)
    bench("calibration N 169343 C 1024 B 15 Bernoulli", "bernoulli", N_ARXIV, 1024, 15)

    # the same table with torch ops, arxiv shape
    B = 15
    edges = torch.arange(1, B, dtype=torch.float64, device=dev) * (1.0 / B)
    fns = [lambda p=p, y=y: torch_table(p, y, B, edges) for p, y in data]
    t_torch = timed(fns, max(args.iters // 5, 10))
    row("torch ops arxiv (argmax, bucketize, f64 scatter_add)", t_torch, None, float("nan"), N_ARXIV * C_ARXIV * 4)
    p, y = data[0]
    top, cls, brier = torch_table(p, y, B, edges)
    t = ops.calibration_table(p, y, "categorical", B).cpu()
    same = torch.equal(t[6:6 + B], top[:B].long().cpu()) and torch.equal(t[6 + 3 * B:6 + 3 * B + C_ARXIV * B],
                                                                        cls[:C_ARXIV * B].long().cpu())
    say("torch ops and kernel bin counts agree: %s" % same)

    say()
    t_cal, k_cal = results["calibration arxiv N 169343 C 40 B 15"]
    ratio = t_cal / t_acc
    say("arxiv: one stag_calibration call = %.2f %% of one stag_mc_accumulate [32, N, 40] call (limit 10 %%): %s"
        % (100 * ratio, "PASS" if ratio <= 0.10 else "FAIL"))
    say("arxiv: kernel device time %.2f %% of the mc_accumulate kernel's" % (100 * k_cal / k_acc))
    say("arxiv: torch ops take %.1fx the kernel's time" % (t_torch / t_cal))
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
