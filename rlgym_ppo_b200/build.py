"""Builds librlppo_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m rlgym_ppo_b200.build [--force] [--verbose]

The library is a plain C-ABI shared object (include/rlppo.h); Python binds it with ctypes (_lib.py)."""
import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "librlppo_b200.so")
STAMP = os.path.join(HERE, "csrc", ".build_stamp")
SOURCES = ["common.cu", "gae_scan.cu", "stats_ring.cu", "optim.cu", "mlp_tcgen05.cu", "mlp_fused.cu", "value_head.cu", "heads.cu", "host_rng.cpp"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr", "-Xptxas", "-v"]
NVCC_FLAGS += os.environ.get("RLPPO_NVCC_EXTRA", "").split()     # e.g. -DRLPPO_DEBUG_BAR (print the barrier a wait timed out on)


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def _digest():
    h = hashlib.sha256()
    files = sorted(f for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".cpp", ".h", ".inc")))
    files = [os.path.join(CSRC, f) for f in files] + [os.path.join(HERE, "..", "include", "rlppo.h")]
    for f in files:
        with open(f, "rb") as fh:
            h.update(fh.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force=False, verbose=False):
    digest = _digest()
    if not force and os.path.exists(OUT) and os.path.exists(STAMP) and open(STAMP).read().strip() == digest:
        return OUT
    nvcc = _nvcc()
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(objdir, src.rsplit(".", 1)[0] + ".o")
        cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    log = []
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        log.append(f"==== {src} ====\n{out}")
        failed |= p.returncode != 0
    with open(os.path.join(objdir, "ptxas.log"), "w") as f:
        f.write("\n".join(log))
    if failed or verbose:
        print("\n".join(log))
    if failed:
        raise RuntimeError("nvcc failed (see output above)")
    subprocess.check_call([nvcc, "-shared", "-o", OUT, *objs, "-gencode", "arch=compute_100a,code=sm_100a"])
    with open(STAMP, "w") as f:
        f.write(digest)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
