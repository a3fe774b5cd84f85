"""Build the CUDA library in-tree: stag_b200/_C/libstag_b200.so (sm_100a only).

The library is plain C ABI (include/stag_b200.h) compiled with nvcc; it does not link
against torch.  `python -m stag_b200.build` or `__graft_entry__.build()` runs this.
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT_DIR = os.path.join(HERE, "_C")
LIB_PATH = os.path.join(OUT_DIR, "libstag_b200.so")
SOURCES = ["runtime.cu", "csx_build.cu", "spmm.cu", "gemm_tcgen05.cu", "nll.cu", "mc_predictive.cu", "edge_softmax.cu", "host_api.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden",
]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; the stag_b200 CUDA library cannot be built")


def _stale():
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    deps.append(os.path.join(HERE, "..", "include", "stag_b200.h"))
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False, extra_flags=(), lib_path=None):
    """Compile every .cu under csrc/ for sm_100a and link libstag_b200.so."""
    lib_path = lib_path or LIB_PATH
    if not force and not _stale():
        return lib_path
    os.makedirs(OUT_DIR, exist_ok=True)
    nvcc = _nvcc()
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(OUT_DIR, src.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + list(extra_flags) + (["-Xptxas", "-v"] if verbose else []) + \
              ["-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for src, p in procs:
        out, _ = p.communicate()
        if verbose and out:
            print(out)
        if p.returncode != 0:
            raise RuntimeError("nvcc failed on %s:\n%s" % (src, out))
    cmd = [nvcc, "-shared", "-o", lib_path] + objs + ["-lcudart"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n%s" % r.stdout)
    return lib_path


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
