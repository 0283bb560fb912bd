"""Compile the sm_100a CUDA sources of this package into one C-ABI shared library (in-tree).

    python -m sg2b200.build            # -> <package>/libsg2b200.so          (the product library)
    python -m sg2b200.build --probes   # -> tools/libsg2b200_probes.so       (product sources + diagnostics, tools only)

Plain nvcc, no torch headers: the library's ABI is include/sg2b200.h (raw pointers + sizes).
nvcc cross-compiles for sm_100a on a machine without a GPU.
"""
import os
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_PATH = os.path.join(PKG_DIR, "libsg2b200.so")
SOURCES = ["conv.cu", "elementwise.cu", "small_ops.cu", "precise.cu", "inception.cu"]
PROBE_SOURCES = ["probe.cu"]          # hardware probes / debug readers: never linked into the product library
PROBE_LIB_PATH = os.path.join(PKG_DIR, "..", "tools", "libsg2b200_probes.so")
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "--use_fast_math", "-Xcompiler", "-fPIC", "-Xcompiler", "-O3",
]


def _stale(lib=None):
    lib = lib or LIB_PATH
    if not os.path.exists(lib):
        return True
    t = os.path.getmtime(lib)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    deps.append(os.path.join(PKG_DIR, "..", "include", "sg2b200.h"))
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force=False, verbose=False, probes=False):
    lib = PROBE_LIB_PATH if probes else LIB_PATH
    if not force and not _stale(lib):
        return lib
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    objs = []
    procs = []
    for src in SOURCES + (PROBE_SOURCES if probes else []):
        path = os.path.join(CSRC, src)
        if not os.path.exists(path):
            continue
        obj = os.path.join(CSRC, src.replace(".cu", ".probes.o" if probes else ".o"))
        cmd = [nvcc, *NVCC_FLAGS, *(["-DSG2_BUILD_PROBES"] if probes else []), "-c", path, "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{out}")
        if verbose and out:
            print(out)
    cmd = [nvcc, "-shared", "-o", lib, *objs]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}")
    return lib


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, probes="--probes" in sys.argv))
