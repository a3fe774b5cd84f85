"""Quick device timing of stag_gemm_tcgen05 against torch.matmul (cuBLAS fp32) at the arxiv layer shapes.

`--compare OTHER_LIB` instead times the C entry point of this tree's library and of another build of it (e.g. the parent
commit's) in one process, alternating rounds between the two, and prints the card name and power limit beside the
medians: a change to the kernels shows against the run-to-run spread of the same call."""
import argparse
import ctypes
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from stag_b200 import _lib, ops

SHAPES = [(16 * 169343, 128, 128), (16 * 169343, 128, 40), (169343, 128, 128), (2708, 1433, 16)]


def t(fn, n=10):
    for _ in range(3): fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n): fn()
    b.record(); torch.cuda.synchronize()
    return a.elapsed_time(b) / n

def tg(fn, n=20):
    """the same call replayed from a CUDA graph: device time without the host-side call overhead"""
    fn(); torch.cuda.synchronize()
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        fn()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=st):
            for _ in range(n): fn()
    torch.cuda.synchronize()
    return t(g.replay, 5) / n


def versus_cublas():
    for M, K, N in SHAPES:
        a = torch.randn(M, K, device="cuda"); w = torch.randn(K, N, device="cuda"); bias = torch.randn(N, device="cuda")
        ms_ours = t(lambda: ops.dense_transform(a, w, bias=bias, relu=True))
        ms_cublas = t(lambda: torch.relu(a @ w + bias))
        ms_mm = t(lambda: a @ w)
        if M < 200000:
            print("   graph replay: ours %.4f ms, cuBLAS matmul %.4f ms, +bias+relu %.4f ms"
                  % (tg(lambda: ops.dense_transform(a, w, bias=bias, relu=True)), tg(lambda: a @ w), tg(lambda: torch.relu(a @ w + bias))))
        gb = (M * K + M * N) * 4 / 1e9
        print("M=%d K=%d N=%d  tcgen05 3xTF32 %.3f ms (%.0f GB/s, %.1f TFLOP/s eff)   cuBLAS fp32 matmul %.3f ms, +bias+relu %.3f ms"
              % (M, K, N, ms_ours, gb / ms_ours * 1e3, 2.0 * M * K * N / ms_ours / 1e9, ms_mm, ms_cublas))


def compare(other, rounds):
    res, args = _lib.SIGNATURES["stag_gemm_tcgen05"]
    libs = {"this": _lib.load(), "other": ctypes.CDLL(os.path.abspath(other))}
    libs["other"].stag_gemm_tcgen05.restype, libs["other"].stag_gemm_tcgen05.argtypes = res, args
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    print("card %s, power limit %s; %d alternating rounds; graph replay of 20 calls, ms per call" %
          (torch.cuda.get_device_name(0), pl, rounds))
    cur = lambda: torch.cuda.current_stream().cuda_stream  # noqa: E731  (the capture stream inside tg)
    # offset 1: A one float off 16-byte alignment, the first-form kernel at a layer shape
    for M, K, N, off in [s + (0,) for s in SHAPES] + [(169343, 128, 128, 1)]:
        a = torch.randn(M * K + 4, device="cuda")[off:]; wt = torch.randn(N, K, device="cuda")
        bias = torch.randn(N, device="cuda"); out = torch.empty(M, N, device="cuda")
        outs, times = {}, {k: [] for k in libs}
        for name, lib in libs.items():
            call = lambda lib=lib: lib.stag_gemm_tcgen05(a.data_ptr(), K, wt.data_ptr(), K, M, N, K, 0,  # noqa: E731
                                                         bias.data_ptr(), 1, out.data_ptr(), N, 0, 0, cur())
            assert call() == 0
            torch.cuda.synchronize()
            outs[name] = out.clone()
        same = torch.equal(outs["this"], outs["other"])
        for _ in range(rounds):
            for name, lib in libs.items():
                times[name].append(tg(lambda lib=lib: lib.stag_gemm_tcgen05(
                    a.data_ptr(), K, wt.data_ptr(), K, M, N, K, 0, bias.data_ptr(), 1, out.data_ptr(), N, 0, 0, cur())))
        med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
        spread = {k: (min(v), max(v)) for k, v in times.items()}
        print("M=%d K=%d N=%d A+%d bias+relu: this %.4f ms [%.4f, %.4f], other %.4f ms [%.4f, %.4f], ratio %.3f, outputs %s"
              % (M, K, N, off, med["this"], *spread["this"], med["other"], *spread["other"], med["this"] / med["other"],
                 "bitwise equal" if same else "DIFFER"))


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--compare", metavar="OTHER_LIB", help="time this tree's library against another build")
    ap.add_argument("--rounds", type=int, default=7)
    o = ap.parse_args()
    if o.compare:
        compare(o.compare, o.rounds)
    else:
        versus_cublas()
