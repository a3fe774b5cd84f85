"""Max aggregation at the arxiv shape (N 169 343, E 1 166 243, D 128, S 16): time per launch (CUDA events, after
warm-up) of the fused max kernels next to the sum kernels of the same spec, and of the unfused torch equivalent
(materialised [E,D] noise per sample, gather, multiply, scatter_reduce amax, autograd backward).

    python tools/bench_max.py [--iters 20] [--out FILE]

Kernel rows call the C ABI directly on preallocated buffers (no Python operator overhead).  The working set of one
pass (gathered operand 87 MB, outputs 16 x 87 MB) exceeds the 126 MB L2 except the operand itself, which stays
resident by design."""
import argparse
import ctypes
import os
import subprocess
import sys

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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--samples", type=int, default=16)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_max.py needs a CUDA device")
    import bench
    import stag_b200 as sb
    from stag_b200 import _lib, ops
    from stag_b200.ops import NoiseSpec

    lines = []

    def say(s):
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
    N, E, D, S = bench.N_NODES, bench.N_EDGES, bench.WIDTH, args.samples
    say("shape: N %d, E %d, D %d, S %d; %d timed launches after 3 warm-up launches" % (N, E, D, S, args.iters))
    g = sb.Graph(torch.from_numpy(src), torch.from_numpy(dst), N).to(dev)
    st = g._s
    lib = _lib.load()
    csc, _ = st.csx(True)
    csr, _ = st.csx(False)
    ws_c = ops._workspace(st, lib, csc, True, D, S)
    ws_r = ops._workspace(st, lib, csr, False, D, S)
    stream = torch.cuda.current_stream().cuda_stream
    torch.manual_seed(0)
    x = torch.randn(N, D, device=dev)
    gout = torch.randn(S, N, D, device=dev)
    out = torch.empty(S, N, D, device=dev)
    arg = torch.empty(S, N, D, dtype=torch.int32, device=dev)
    dx = torch.empty(S, N, D, device=dev)
    one, sg = torch.ones((), device=dev), torch.full((), 0.4, device=dev)
    loc_e, sc_e = torch.ones(E, 1, device=dev), torch.full((E, 1), 0.4, device=dev)
    d0, d1 = torch.zeros(E, device=dev), torch.zeros(E, device=dev)

    def nz(gen, p0=one, p1=sg, pshape=_lib.PARAM_SCALAR):
        spec = NoiseSpec("normal", p0, p1, D, E, seed=1, offset=2, n_samples=S, generator=gen)
        kind = spec.lib_kind
        return ops._fill_noise(spec, kind, D, p0, p1, None, False, False, 0, 1, 2, pshape)

    nbm, nwh, nre = nz("boxmuller"), nz("hadamard"), nz("boxmuller", loc_e, sc_e, _lib.PARAM_EDGE)
    R = lambda rc: _lib.check(rc)  # noqa: E731

    def max_fwd(n):
        return lambda: R(lib.stag_spmm_max_fwd(ctypes.byref(csc), x.data_ptr(), D, 0, D, S, ctypes.byref(n),
                                                out.data_ptr(), arg.data_ptr(), D, N * D, ws_c.data_ptr(), ws_c.numel(),
                                                stream))

    def sum_fwd(n):
        return lambda: R(lib.stag_spmm_fwd(ctypes.byref(csc), x.data_ptr(), D, 0, D, S, ctypes.byref(n), 0, 0,
                                            out.data_ptr(), D, N * D, 0, ws_c.data_ptr(), ws_c.numel(), stream))

    def max_bwd(n, dp=False):
        return lambda: R(lib.stag_spmm_max_bwd(ctypes.byref(csr), x.data_ptr(), D, 0, gout.data_ptr(), arg.data_ptr(),
                                                D, N * D, D, S, ctypes.byref(n), dx.data_ptr(), D, N * D,
                                                d0.data_ptr() if dp else 0, d1.data_ptr() if dp else 0, 0,
                                                ws_r.data_ptr(), ws_r.numel(), stream))

    def sum_dx(n):
        return lambda: R(lib.stag_spmm_fwd(ctypes.byref(csr), gout.data_ptr(), D, N * D, D, S, ctypes.byref(n), 0, 0,
                                            dx.data_ptr(), D, N * D, 0, ws_r.data_ptr(), ws_r.numel(), stream))

    def sum_bwd(n):
        return lambda: R(lib.stag_spmm_bwd(ctypes.byref(csr), x.data_ptr(), D, 0, gout.data_ptr(), D, N * D, D, S,
                                            ctypes.byref(n), 0, 0, dx.data_ptr(), D, N * D, d0.data_ptr(), d1.data_ptr(),
                                            0, ws_r.data_ptr(), ws_r.numel(), stream))

    it = args.iters
    rows = []
    say("")
    say("%-58s %10s %12s" % ("launch (all %d samples)" % S, "ms", "ms / sample"))

    def row(name, ms):
        rows.append((name, ms))
        say("%-58s %10.3f %12.4f" % (name, ms, ms / S))
        return ms

    t_fwd_bm = row("max forward, Box-Muller, scalar Normal(1, 0.4)", timed(max_fwd(nbm), it))
    row("sum forward, same spec (stag_spmm_fwd)", timed(sum_fwd(nbm), it))
    row("max forward, Hadamard, scalar Normal(1, 0.4)", timed(max_fwd(nwh), it))
    row("sum forward, same spec (stag_spmm_fwd)", timed(sum_fwd(nwh), it))
    max_fwd(nbm)()
    t_dx = row("max dX pass (stag_spmm_max_bwd, dx only), Box-Muller", timed(max_bwd(nbm), it))
    row("sum transposed pass (stag_spmm_fwd on the CSR)", timed(sum_dx(nbm), it))
    t_r1 = row("max backward, dx + r1 parameter gradients", timed(max_bwd(nbm, True), it))
    row("sum backward, dx + r1 (stag_spmm_bwd)", timed(sum_bwd(nbm), it))
    max_fwd(nre)()
    t_re = row("max backward, dx + re ([E,1]) parameter gradients", timed(max_bwd(nre, True), it))
    row("sum backward, dx + re (stag_spmm_bwd)", timed(sum_bwd(nre), it))

    # unfused torch: per Monte-Carlo sample, materialised noise, gather, multiply, scatter_reduce amax, autograd
    srcd, dstd = torch.from_numpy(src).to(dev), torch.from_numpy(dst).to(dev)
    idx = dstd.unsqueeze(-1).expand(E, D)
    xg = x.clone().requires_grad_(True)
    locp, scp = one.clone().requires_grad_(True), sg.clone().requires_grad_(True)
    g1 = gout[0]

    def unfused():
        w = locp + scp * torch.randn(E, D, device=dev)
        m = xg[srcd] * w
        o = torch.zeros(N, D, device=dev).scatter_reduce(0, idx, m, reduce="amax", include_self=False)
        o.backward(g1)

    t_unf = timed(unfused, max(it // 4, 3))
    say("")
    say("%-58s %10.3f %12.4f" % ("unfused torch, one sample: noise + gather + mul + amax + autograd", t_unf, t_unf))
    fused_r1 = (t_fwd_bm + t_r1) / S
    fused_re = (t_fwd_bm + t_re) / S
    fused_dx = (t_fwd_bm + t_dx) / S
    say("")
    say("fused max forward + backward per sample: dx only %.4f ms, dx + r1 %.4f ms, dx + re %.4f ms" % (fused_dx, fused_r1, fused_re))
    say("speed-up over the unfused torch equivalent (dx + r1): %.1fx" % (t_unf / fused_r1))
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
