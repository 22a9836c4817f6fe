"""Builds libMFAFFI.so (sm_100a only) in-tree with nvcc; no JIT cache, no torch extension machinery.

    python universal-metal-flash-attention_b200/build.py [--force] [--verbose]

The library links the static CUDA runtime and resolves the few driver-API entry points it needs
(cuTensorMapEncodeTiled) through cudaGetDriverEntryPoint at run time, so it loads on a machine without a GPU
driver too (needed by the CPU-only symbol/ABI tests).
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT_DIR = os.path.join(HERE, "lib")
LIB = os.path.join(OUT_DIR, "libMFAFFI.so")
SOURCES = ["ffi.cu", "attn_simt.cu", "attn_fwd_tc.cu", "attn_bwd_tc.cu", "attn_fwd_tcq.cu", "attn_fwd_split.cu", "quant.cu", "ring.cu", "kvcache_append.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo", "--cudart", "static",
         "-Xcompiler", "-fPIC,-O3", "--expt-relaxed-constexpr", "-ccbin", "/usr/bin/g++"]


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def _extra_flags(stamp):
    """MFA_WATCHDOG=1 in the environment of the BUILD compiles the mbarrier wall-clock watchdog in (sm100_ptx.cuh: a
    protocol bug traps instead of hanging the GPU); MFA_WATCHDOG=0 builds the release library, which spins without a
    limit.  With the variable unset an existing library keeps the mode it was built in (no surprise rebuilds on the GPU
    box); a fresh tree builds release."""
    want = os.environ.get("MFA_WATCHDOG")
    if want is None:
        try:
            return ["-DMFA_MBAR_WATCHDOG"] if "-DMFA_MBAR_WATCHDOG" in open(stamp).read() else []
        except OSError:
            return []
    return ["-DMFA_MBAR_WATCHDOG"] if want not in ("", "0") else []


def build(force=False, verbose=False):
    os.makedirs(OUT_DIR, exist_ok=True)
    stamp = os.path.join(OUT_DIR, "build_flags.txt")
    extra = _extra_flags(stamp)
    want = " ".join(FLAGS + extra)
    have = open(stamp).read() if os.path.exists(stamp) else None
    if have is None and os.path.exists(LIB) and not extra:
        have = want                      # a library built before the stamp existed: release flags
    if have != want:
        force = True
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh"))]
    headers += [os.path.join(HERE, "..", "include", f) for f in ("mfa_ffi.h", "mfa_ffi_ext.h")]
    objs = []
    procs = []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(OUT_DIR, src.replace(".cu", ".o"))
        objs.append(o)
        if force or _stale(o, [s] + headers):
            cmd = [NVCC] + FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o]
            procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write(f"--- {src}\n{out}\n")
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    if force or procs or _stale(LIB, objs + [os.path.join(CSRC, "exports.map")]):
        cmd = [NVCC, "-shared", "--cudart", "static", "-ccbin", "/usr/bin/g++", "-o", LIB] + objs + ["-ldl", "-lpthread", "-lrt", "-Xlinker", "--version-script=" + os.path.join(CSRC, "exports.map")]
        subprocess.run(cmd, check=True)
    with open(stamp, "w") as f:
        f.write(want)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
