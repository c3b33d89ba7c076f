"""In-tree build of libb200pir.so (sm_100a only).  Run as `python -m sdk_b200.build` or via
__graft_entry__.build(); nvcc cross-compiles without a GPU."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
SO = os.path.join(HERE, "libb200pir.so")
SOURCES = ["api.cu", "poly_kernels.cu", "mul_kernels.cu", "imma_kernels.cu", "wire_kernels.cu", "tc5_kernels.cu", "dpir_gemm.cu"]
HEADERS = ["common.cuh", "kernels.h", "item_write.cuh", "ntt_core.cuh", "tc5_layout.cuh", "tc5_ptx.cuh", "ntt_core4096.cuh", "ntt_tables.hpp", os.path.join("..", "..", "include", "b200pir.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "--extended-lambda",
              "-Xcompiler", "-fPIC", "-ccbin", "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"]


def _stale():
    if not os.path.exists(SO):
        return True
    t = os.path.getmtime(SO)
    return any(os.path.getmtime(os.path.join(CSRC, f)) > t for f in SOURCES + HEADERS)


def build(force=False, verbose=False):
    if not force and not _stale():
        return SO
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(CSRC, src.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for src, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode:
            sys.stderr.write(out)
        if p.returncode:
            raise RuntimeError("nvcc failed on " + src)
    subprocess.check_call([nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", SO] + objs + ["-ccbin", NVCC_FLAGS[-1]])
    return SO


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
