"""Builds the engine's shared library in-tree with nvcc for sm_100a.

Output: pdn-jpegxl_b200/libJpegXLFileTypeIO_X64.so (the Linux counterpart of the reference's
JpegXLFileTypeIO_X64.dll, N/JxlFileTypeIO.vcxproj:27,75-85). The .so is git-ignored but travels
to the GPU box with the gpurun snapshot. nvcc cross-compiles without a GPU.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libJpegXLFileTypeIO_X64.so")
SOURCES = ["abi.cu", "decode_engine.cu", "encode_engine.cu", "dev/entropy_kernels.cu", "dev/recon_kernels.cu", "dev/encode_kernels.cu", "dev/layer_kernels.cu", "dev/composite_kernels.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "--expt-relaxed-constexpr",
              "-Xcompiler", "-fPIC,-fvisibility=hidden,-Wall,-Wno-sign-compare,-Wno-unused-function,-Wno-misleading-indentation",
              "-diag-suppress", "177,550"]


def _newer(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def all_deps():
    deps = []
    for root, _, files in os.walk(CSRC):
        for f in files:
            if f.endswith((".cu", ".cuh", ".h", ".cc", ".inc")):   # .inc: generated tables (dev/idct_tables.inc)
                deps.append(os.path.join(root, f))
    deps.append(os.path.join(os.path.dirname(HERE), "include", "JxlFileTypeIO.h"))
    return deps


def build(force=False, verbose=False):
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    deps = all_deps()
    srcs = [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    objs = []
    procs = []
    for s in srcs:
        obj = os.path.join(objdir, s.replace("/", "_") + ".o")
        objs.append(obj)
        if force or _newer(obj, deps):
            cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, s), "-o", obj]
            procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for s, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write("== %s ==\n%s\n" % (s, out))
        failed = failed or p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    if force or procs or _newer(OUT, objs):
        cmd = [nvcc, "-shared", "-o", OUT] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-ldl", "-Xcompiler", "-fPIC"]
        subprocess.run(cmd, check=True)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
