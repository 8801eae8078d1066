"""In-tree build of libsimstep.so (nvcc, sm_100a only).

`python -m amp_extensions_b200.build` compiles every translation unit under amp_extensions_b200/csrc
(api.cu: the C ABI and most kernels; chain.cu: the column-fused ensemble forward kernel's instantiations) in
parallel and links them into amp_extensions_b200/csrc/libsimstep.so.  nvcc cross-compiles without a GPU.
"""
import hashlib
import os
import shutil
import subprocess
import sys
import tempfile
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(CSRC, "libsimstep.so")
STAMP = os.path.join(CSRC, ".libsimstep.stamp")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC",
]
UNITS = ("api.cu", "chain.cu")


def _sources():
    out = []
    for root in (CSRC, os.path.join(HERE, "..", "include")):
        for name in sorted(os.listdir(root)):
            if name.endswith((".cu", ".cuh", ".h", ".inc")):
                out.append(os.path.join(root, name))
    return out


def _digest():
    h = hashlib.sha256()
    for p in _sources():
        with open(p, "rb") as f:
            h.update(os.path.basename(p).encode())
            h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def have_nvcc():
    return bool(shutil.which("nvcc")) or os.path.exists("/usr/local/cuda/bin/nvcc")


def needs_build():
    if not os.path.exists(LIB) or not os.path.exists(STAMP):
        return True
    with open(STAMP) as f:
        return f.read().strip() != _digest()


def build(force=False, verbose=False):
    """Compile libsimstep.so if sources changed. Returns the library path."""
    if not force and not needs_build():
        return LIB
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found; libsimstep.so cannot be built")
    log = []

    def compile_unit(args):
        name, obj = args
        cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", obj, os.path.join(CSRC, name)]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError(f"nvcc failed on {name}:\n" + res.stdout + res.stderr)
        log.append(res.stderr)

    with tempfile.TemporaryDirectory(prefix="simstep_build_") as tmp:
        objs = [os.path.join(tmp, os.path.splitext(u)[0] + ".o") for u in UNITS]
        with ThreadPoolExecutor(max_workers=len(UNITS)) as pool:
            list(pool.map(compile_unit, zip(UNITS, objs)))
        res = subprocess.run([nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB] + objs,
                             capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError("nvcc link failed:\n" + res.stdout + res.stderr)
    if verbose:
        sys.stderr.write("".join(log))
    with open(STAMP, "w") as f:
        f.write(_digest())
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
