"""Build libvasr.so (sm_100a only) in-tree with nvcc.  No torch dependency: the library is a
plain C-ABI shared object (include/vasr.h) with the CUDA runtime linked statically."""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "velocity_asr", "libvasr.so")
SOURCES = ["engine.cu", "gemm.cu", "gemm_tc.cu", "norm_conv.cu", "scan.cu", "mel.cu", "context.cu", "ctc.cu", "beam.cu", "lm.cu", "align.cu"]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
FLAGS = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC,-O3,-Wall", "--expt-relaxed-constexpr"]


def _nvcc():
    for c in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("nvcc not found")


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False, debug=False):
    """debug=True: libvasr_dbg.so with -DVASR_DEBUG (the tuning switches of common.cuh's debug_env_int read the
    environment); load it with VASR_LIB=<path> for A/B runs on one GPU box.  The shipped library has none of them."""
    nvcc = _nvcc()
    objdir = os.path.join(HERE, "build_dbg" if debug else "build")
    target = OUT.replace("libvasr.so", "libvasr_dbg.so") if debug else OUT
    flags = FLAGS + (["-DVASR_DEBUG"] if debug else [])
    os.makedirs(objdir, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(os.path.dirname(HERE), "include", "vasr.h"))
    objs, procs = [], []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(objdir, src.replace(".cu", ".o"))
        objs.append(o)
        if force or _stale(o, [s] + headers):
            cmd = [nvcc] + ARCH + flags + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o]
            procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write(f"--- {src}\n{out}\n")
        failed = failed or p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    if force or procs or _stale(target, objs):
        cmd = [nvcc] + ARCH + ["-shared", "-o", target] + objs + ["-cudart", "static"]
        subprocess.check_call(cmd)
    return target


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, debug="--debug" in sys.argv))
