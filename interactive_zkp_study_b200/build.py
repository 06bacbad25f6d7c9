"""Builds libzkp_b200.so (hand-written CUDA for sm_100a behind the C ABI in include/zkp_b200.h).

In-tree, explicit nvcc (no JIT cache): the resulting .so travels with the repository snapshot to
the GPU box.  Translation units are compiled in parallel and cached by content hash.

    python -m interactive_zkp_study_b200.build [--force] [--verbose]
"""
import concurrent.futures
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "_build")
LIB = os.path.join(HERE, "libzkp_b200.so")
ROOT = os.path.dirname(HERE)

UNITS = ["capi_core.cu", "comm.cu", "diag.cu", "msm_g1.cu", "msm_g2.cu", "ntt.cu", "pairing.cu", "poly.cu"]

NVCC_FLAGS = [
    "-std=c++17", "-O3", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
    "-Xcompiler", "-fPIC", "-diag-suppress", "128,550",
    "-I", os.path.join(ROOT, "include"),
] + os.environ.get("ZKP_B200_NVCC_EXTRA", "").split()


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def _digest(unit):
    h = hashlib.sha256()
    h.update(" ".join(NVCC_FLAGS).encode())
    # every header participates in every unit's hash: simple and safe
    names = sorted(f for f in os.listdir(CSRC) if f.endswith((".cuh", ".h")))
    for f in names + [unit]:
        with open(os.path.join(CSRC, f), "rb") as fh:
            h.update(f.encode())
            h.update(fh.read())
    for f in ("zkp_b200.h", "zkp_b200_diag.h"):
        with open(os.path.join(ROOT, "include", f), "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()


def _compile(unit, force, verbose):
    src = os.path.join(CSRC, unit)
    obj = os.path.join(OBJ, unit.replace(".cu", ".o"))
    stamp = obj + ".sha"
    dig = _digest(unit)
    if not force and os.path.exists(obj) and os.path.exists(stamp) and open(stamp).read() == dig:
        return unit, "cached", ""
    cmd = [_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
    p = subprocess.run(cmd, capture_output=True, text=True)
    if p.returncode != 0:
        raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (unit, p.stdout, p.stderr))
    with open(stamp, "w") as fh:
        fh.write(dig)
    return unit, "compiled", p.stderr


def build(force=False, verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    units = [u for u in UNITS if os.path.exists(os.path.join(CSRC, u))]
    with concurrent.futures.ThreadPoolExecutor(max_workers=min(8, len(units))) as ex:
        results = list(ex.map(lambda u: _compile(u, force, verbose), units))
    relink = not os.path.exists(LIB) or any(r[1] == "compiled" for r in results)
    for unit, status, log in results:
        print("[build] %-14s %s" % (unit, status))
        if verbose and log:
            print(log)
    if relink:
        objs = [os.path.join(OBJ, u.replace(".cu", ".o")) for u in units]
        # shared CUDA runtime (libcudart.so.12 is on the loader path of this image and of the GPU box; the rpath
        # covers a bare toolkit install): the .so then carries no copy of the runtime.  libdl for the NCCL binding.
        link = ["-cudart", "static"] if os.environ.get("ZKP_B200_STATIC_CUDART") else \
            ["-cudart", "shared", "-Xlinker", "-rpath=/usr/local/cuda/lib64"]
        cmd = [_nvcc(), "-shared", "-o", LIB] + objs + link + ["-ldl"]
        p = subprocess.run(cmd, capture_output=True, text=True)
        if p.returncode != 0:
            raise RuntimeError("link failed:\n%s\n%s" % (p.stdout, p.stderr))
        print("[build] linked", LIB)
    return LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
