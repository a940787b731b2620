"""Build the sm_100a CUDA library in-tree with nvcc (no JIT cache: the .so must travel with the repo)."""
import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIBNAME = "libturboprune_b200.so"
SOURCES = ["tp_core.cu", "tp_prune.cu", "tp_optim.cu", "tp_igemm.cu", "tp_reduce.cu", "tp_bn.cu", "tp_pool.cu", "tp_data.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr", "-cudart", "static",
]


def lib_path() -> str:
    # TURBOPRUNE_B200_LIB: load another build of the same C ABI instead (e.g. to compare two builds in one GPU run)
    return os.environ.get("TURBOPRUNE_B200_LIB") or os.path.join(LIBDIR, LIBNAME)


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.isfile(cand):
            return cand
    raise RuntimeError("nvcc not found (needed to build turboprune_b200 for sm_100a)")


def _digest() -> str:
    h = hashlib.sha256()
    for root in (CSRC, os.path.join(os.path.dirname(HERE), "include")):
        for name in sorted(os.listdir(root)):
            if name.endswith((".cu", ".cuh", ".h")):
                with open(os.path.join(root, name), "rb") as f:
                    h.update(name.encode()); h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = True) -> str:
    """Compile every .cu for sm_100a and link lib/libturboprune_b200.so. Returns its path."""
    os.makedirs(LIBDIR, exist_ok=True)
    stamp = os.path.join(LIBDIR, "build.sha256")
    dig = _digest()
    default = os.path.join(LIBDIR, LIBNAME)
    if not force and os.path.isfile(default) and os.path.isfile(stamp) and open(stamp).read().strip() == dig:
        return default
    nvcc = _nvcc()
    objs, procs = [], []
    for src in SOURCES:
        obj = os.path.join(LIBDIR, src.replace(".cu", ".o"))
        objs.append(obj)
        cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{out}")
        if verbose and out.strip():
            print(out, file=sys.stderr)
    link = [nvcc, "-shared", "-cudart", "static", "-o", default, *objs]
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}")
    with open(stamp, "w") as f:
        f.write(dig)
    return default


if __name__ == "__main__":
    print(build(force="--force" in sys.argv))
