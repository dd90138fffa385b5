"""In-tree build of libpllb200.so with nvcc for sm_100a (no GPU needed to compile)."""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libpllb200.so")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-Xcompiler", "-Wall",
          "--expt-relaxed-constexpr", "-Xptxas", "-v"]
# translation unit -> extra flags
UNITS = {
    "api.cu": [],
    "gemm_tcgen05.cu": [],
    "gemm_ln_tcgen05.cu": [],
    "encoder_kernels.cu": [],
    "train_kernels.cu": [],
    "train_api.cu": [],
    "bertscore_kernels.cu": [],
    "seq2seq_kernels.cu": [],
    "seq2seq_api.cu": [],
    # fp64 combiner must round like numpy: no FMA contraction, IEEE division
    "rescore_kernels.cu": ["-fmad=false", "-prec-div=true", "-prec-sqrt=true"],
}


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def _stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "pllb.h"), __file__]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile and link; safe when every rank of a torchrun job calls it at once: an exclusive
    file lock serialises the builders, the late ones find a fresh library and return, and the
    library appears atomically (linked to a temporary name, then os.replace)."""
    if not force and not _stale():
        return LIB
    import fcntl
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    with open(os.path.join(objdir, ".lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and not _stale():      # another process built it while we waited
                return LIB
            return _build_locked(objdir, verbose)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def _build_locked(objdir: str, verbose: bool) -> str:
    nvcc = _nvcc()
    objs = []
    procs = []
    defs = [f"-D{d}" for d in os.environ.get("PLLB_DEFINES", "").split()]     # e.g. PLLB_SPIN_LIMIT=0
    for src, extra in UNITS.items():
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        cmd = [nvcc, *ARCH, *COMMON, *defs, *extra, "-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    log = []
    for src, cmd, p in procs:
        out, _ = p.communicate()
        log.append(f"$ {' '.join(cmd)}\n{out}")
        if p.returncode != 0:
            sys.stderr.write(log[-1])
            raise RuntimeError(f"nvcc failed on {src}")
    tmp = LIB + f".tmp{os.getpid()}"
    cmd = [nvcc, *ARCH, "-shared", "-o", tmp, *objs, "-Xcompiler", "-fPIC", "-ldl"]
    out = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    log.append(f"$ {' '.join(cmd)}\n{out.stdout}")
    if out.returncode != 0:
        sys.stderr.write(log[-1])
        raise RuntimeError("link failed")
    os.replace(tmp, LIB)
    with open(os.path.join(objdir, "build.log"), "w") as f:
        f.write("\n".join(log))
    if verbose:
        print("\n".join(log))
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
