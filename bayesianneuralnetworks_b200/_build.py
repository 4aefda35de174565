"""Builds libbnn_b200.so (sm_100a) in-tree with nvcc.

The shared library is the whole product data path; it links only libcudart and exports the
C ABI declared in include/bnn_b200.h.  `python -m bayesianneuralnetworks_b200._build` rebuilds it.
"""
import os
import subprocess
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB_PATH = os.path.join(_HERE, "libbnn_b200.so")
SOURCES = ["api.cu", "adam.cu", "ce.cu", "conv.cu", "elementwise.cu", "flipout.cu", "kl.cu", "prune.cu", "sampled_gemm.cu", "sampled_gemm_tma.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC",
    "-diag-suppress", "177",
]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def _stale():
    if not os.path.exists(LIB_PATH):
        return True
    built = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    deps.append(os.path.join(_HERE, "..", "include", "bnn_b200.h"))
    return any(os.path.getmtime(d) > built for d in deps)


def build(force=False, verbose=False):
    """Compile every .cu under csrc/ into libbnn_b200.so; no-op when up to date."""
    if not force and not _stale():
        return LIB_PATH
    nvcc = _nvcc()
    objs = []
    procs = []
    os.makedirs(os.path.join(_HERE, "build"), exist_ok=True)
    for src in SOURCES:
        obj = os.path.join(_HERE, "build", src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, *os.environ.get("BNN_EXTRA_NVCC_FLAGS", "").split(), "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd += ["-Xptxas", "-v"]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for src, proc in procs:
        out, _ = proc.communicate()
        if verbose or proc.returncode != 0:
            sys.stderr.write(out)
        if proc.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}")
    link = [nvcc, "-shared", "-o", LIB_PATH, *objs]
    res = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout)
        raise RuntimeError("link of libbnn_b200.so failed")
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
