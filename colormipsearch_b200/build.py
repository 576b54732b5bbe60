"""Builds libcdsgpu.so (CUDA kernels + C ABI) in-tree for sm_100a with nvcc.

    python -m colormipsearch_b200.build [--force]

The shared library lands in colormipsearch_b200/lib/libcdsgpu.so; it is git-ignored but travels to the GPU box.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
SO = os.path.join(LIBDIR, "libcdsgpu.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")

CU_SOURCES = ["cds_api.cu", "cds_stream.cu", "cds_kernels.cu", "cds_band.cu", "cds_cand.cu", "cds_topk.cu", "cds_synth.cu", "cds_shape.cu", "cds_ingest.cu", "cds_pairq.cu", "cds_shape_pairq.cu", "cds_inflate.cu", "cds_bestsel.cu"]
CPP_SOURCES = ["cds_tables.cpp", "cds_select.cpp", "cds_tiff.cpp", "cds_formats.cpp"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "--expt-relaxed-constexpr", "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden",
    # the interval tables must come from unfused IEEE double arithmetic, like the JVM's
    "-Xcompiler", "-ffp-contract=off", "--fmad=false",
    "-ccbin", "/usr/bin/g++",
]


def _sources():
    out = [os.path.join(CSRC, f) for f in CU_SOURCES + CPP_SOURCES]
    hdrs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh"))]
    hdrs.append(os.path.join(os.path.dirname(HERE), "include", "cdsgpu.h"))
    return out, hdrs


def needs_build():
    if not os.path.exists(SO):
        return True
    t = os.path.getmtime(SO)
    srcs, hdrs = _sources()
    return any(os.path.getmtime(f) > t for f in srcs + hdrs)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return SO
    os.makedirs(LIBDIR, exist_ok=True)
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    srcs, _ = _sources()
    objs = []
    procs = []
    for src in srcs:
        obj = os.path.join(objdir, os.path.basename(src) + ".o")
        objs.append(obj)
        cmd = [NVCC] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-x", "cu", "-c", src, "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            failed = True
            sys.stderr.write("nvcc failed for %s:\n%s\n" % (src, out))
        elif verbose or out.strip():
            sys.stderr.write(out)
    if failed:
        raise RuntimeError("libcdsgpu build failed")
    cmd = [NVCC, "-shared", "-o", SO] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-ccbin", "/usr/bin/g++",
                                              "-Xcompiler", "-fPIC", "-cudart", "shared", "-lz"]
    subprocess.run(cmd, check=True)
    return SO


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
