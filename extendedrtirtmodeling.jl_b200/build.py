"""Build the CUDA shared library in-tree with nvcc for sm_100a (no JIT cache, the .so travels with the repo)."""
import glob
import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "liberirt_b200.so")
SOURCES = ["erirt_b200.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC",
              "-shared"]


def find_nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; the CUDA extension cannot be built")


def is_stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    # every file of csrc/ (the sources and every header they include) and the ABI header
    deps = glob.glob(os.path.join(CSRC, "*")) + [os.path.join(HERE, "..", "include", "erirt_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force=False, verbose=False):
    """Compile csrc/*.cu -> liberirt_b200.so.  Returns the library path."""
    if not force and not is_stale():
        return LIB
    extra = os.environ.get("ERIRT_NVCC_EXTRA", "").split()
    cmd = [find_nvcc()] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB] + \
          [os.path.join(CSRC, s) for s in SOURCES] + ["-ldl"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stderr)
    return LIB


if __name__ == "__main__":
    print(build(force=True, verbose=True))
