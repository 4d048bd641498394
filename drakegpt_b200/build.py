"""In-tree nvcc build of the sm_100a kernel library (no JIT cache, no fallback)."""
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(CSRC, "libdrakegpt_b200.so")
SOURCES = ["runtime.cu", "elementwise.cu", "gemm_simt.cu", "attn_simt.cu", "gemm_tc.cu", "attn_tc.cu", "lmhead_ce.cu", "gemm_ln.cu", "dp_adamw.cu", "decode.cu", "api.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
         "-Xcompiler", "-fPIC", "--use_fast_math", "-Xcompiler", "-fvisibility=default"]
# --use_fast_math would change expf/logf/div accuracy in the exact-mode kernels: keep IEEE there
EXACT = {"elementwise.cu", "gemm_simt.cu", "attn_simt.cu"}


def _digest():
    h = hashlib.sha256()
    for f in sorted(os.listdir(CSRC)) + ["../../include/drakegpt_b200.h"]:
        p = os.path.join(CSRC, f)
        if f.endswith((".cu", ".cuh", ".h")) and os.path.isfile(p):
            with open(p, "rb") as fh:
                h.update(f.encode())
                h.update(fh.read())
    h.update(" ".join(FLAGS).encode())
    return h.hexdigest()


def build(force=False, verbose=False, extra_flags=(), suffix=""):
    """Build csrc/libdrakegpt_b200<suffix>.so.  ``extra_flags`` / ``suffix`` make diagnostic variants (e.g.
    ``-DDGPT_ATTN_TS``, the attention backward's phase stamps) that are selected at run time with the DGPT_LIB
    environment variable."""
    lib = LIB.replace(".so", suffix + ".so")
    stamp = lib + ".stamp"
    dig = _digest() + " ".join(extra_flags)
    if not force and os.path.exists(lib) and os.path.exists(stamp) and open(stamp).read() == dig:
        return lib
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(CSRC, src.replace(".cu", suffix + ".o"))
        flags = [f for f in FLAGS if not (src in EXACT and f == "--use_fast_math")] + list(extra_flags)
        cmd = [NVCC, *flags, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write(f"--- nvcc {src} ---\n{out}\n")
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed building drakegpt_b200 kernels")
    subprocess.check_call([NVCC, "-shared", "-o", lib, *objs, "-lcudart"])
    with open(stamp, "w") as fh:
        fh.write(dig)
    return lib


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
