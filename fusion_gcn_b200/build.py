"""Builds libagcn_b200.so in-tree with nvcc for sm_100a:  python -m fusion_gcn_b200.build [--force]"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libagcn_b200.so")
SOURCES = ["common.cu", "conv_simt.cu", "wgrad_tc.cu", "conv_tc2.cu", "joint.cu", "joint_big.cu", "gram_tc.cu", "mix_tc.cu", "bn.cu", "optim.cu", "head.cu"]
FLAGS = ["-std=c++17", "-O3", "-lineinfo", "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-Xcompiler", "-fPIC",
         "-Xcompiler", "-fvisibility=hidden"]


def _stale():
    if not os.path.isfile(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "agcn_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def _nvcc():
    """$NVCC, else nvcc on PATH, else the toolkit's own (CUDA_HOME, CUDA_PATH, the default install prefix): a login shell
    need not have the toolkit's bin directory on PATH."""
    if os.environ.get("NVCC"):
        return os.environ["NVCC"]
    found = shutil.which("nvcc")
    if found:
        return found
    for root in (os.environ.get("CUDA_HOME"), os.environ.get("CUDA_PATH"), "/usr/local/cuda"):
        if root and os.path.isfile(os.path.join(root, "bin", "nvcc")):
            return os.path.join(root, "bin", "nvcc")
    raise RuntimeError("nvcc not found: put it on PATH, or set NVCC or CUDA_HOME")


def build(force=False, verbose=False, probes=False):
    """``probes=True`` compiles the A/B switches and limiter probes in (-DAGCN_PROBES); the default library has none."""
    if not force and not probes and not _stale():
        return OUT
    nvcc = _nvcc()
    out = OUT.replace(".so", "_probes.so") if probes else OUT        # the probe build never replaces the product library
    cmd = [nvcc] + FLAGS + (["-DAGCN_PROBES"] if probes else []) + (["-Xptxas", "-v"] if verbose else []) + ["-o", out] + [os.path.join(CSRC, s) for s in SOURCES] + ["-lcuda"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError("nvcc failed building libagcn_b200.so")
    if verbose:
        sys.stderr.write(res.stderr)
    return out


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, probes="--probes" in sys.argv))
