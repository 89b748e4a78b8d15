"""Builds the in-tree native libraries of the package (sm_100a only, no JIT cache):

  3dscan_b200/lib/libscan3d.so       CUDA kernels + the C ABI of include/scan3d.h
  3dscan_b200/lib/libscan3d_host.so  C++ host side (image / calibration / PLY I/O, synthetic
                                     pattern generator, reference-named stage functions)

nvcc cross-compiles without a GPU, so this also runs in the CPU-only build container.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
HOST = os.path.join(HERE, "host")
LIB = os.environ.get("SCAN3D_LIBDIR") or os.path.join(HERE, "lib")

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-DSCAN3D_BUILD",
    "-Xcompiler", "-fPIC,-ffp-contract=off,-O2,-Wall", "-Xptxas", "-v",
    "-cudart", "static", "-ccbin", "/usr/bin/g++",
]
# SCAN3D_BUILD_TRACE=1 compiles the pipeline-timeline hooks of the fused kernels in (tools/trace_fused.py);
# they cost ~2 % of the kernel's instructions, so the default build leaves them out.
if os.environ.get("SCAN3D_BUILD_TRACE") == "1":
    NVCC_FLAGS.append("-DS3D_TRACE=1")
CU_SOURCES = ["scan3d_api.cu", "scan3d_stage_kernels.cu", "scan3d_worklist.cu", "scan3d_fused_kernel7.cu",
              "scan3d_aux_kernels.cu", "scan3d_aux_api.cu", "scan3d_shard.cu", "scan3d_mesh_kernels.cu",
              "scan3d_voxel_kernels.cu", "scan3d_align_kernels.cu", "scan3d_surface_kernels.cu",
              "scan3d_components_kernels.cu", "scan3d_decimate_kernels.cu", "scan3d_smooth_kernels.cu",
              "scan3d_fill_kernels.cu", "scan3d_repair_kernels.cu", "scan3d_orient_kernels.cu"]
HOST_SOURCES = ["scan3d_io.cpp", "scan3d_synth.cpp"]
COMPAT_SOURCES = ["scan3d_stages.cpp"]


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def _deps(folder, extra=()):
    out = [os.path.join(d, f) for d in (folder, os.path.join(HERE, "common")) for f in os.listdir(d)
           if f.endswith((".cu", ".cuh", ".h", ".cpp", ".hpp"))]
    out += list(extra)
    out.append(os.path.abspath(__file__))
    return out


def build_cuda(force=False, verbose=False):
    os.makedirs(LIB, exist_ok=True)
    so = os.path.join(LIB, "libscan3d.so")
    hdr = os.path.join(HERE, "..", "include", "scan3d.h")
    if not (force or _stale(so, _deps(CSRC, [hdr, os.path.join(HERE, "..", "include", "scan3d_shard.h")]))):
        return so
    from concurrent.futures import ThreadPoolExecutor

    def compile_one(src):
        obj = os.path.join(LIB, src.replace(".cu", ".o"))
        cmd = [NVCC] + NVCC_FLAGS + ["-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        # registers / spills of every kernel, without ptxas' timing lines (the log is diffable between builds)
        with open(os.path.join(LIB, src + ".ptxas.log"), "w") as f:
            f.write("".join(l + "\n" for l in r.stderr.splitlines() if "Compile time" not in l))
        if verbose or r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed on " + src)
        return obj

    with ThreadPoolExecutor(max_workers=min(len(CU_SOURCES), os.cpu_count() or 1)) as ex:
        objs = list(ex.map(compile_one, CU_SOURCES))
    cmd = [NVCC, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "static",
           "-ccbin", "/usr/bin/g++", "-o", so] + objs + ["-lrt"]
    subprocess.check_call(cmd)
    return so


def build_host(force=False):
    os.makedirs(LIB, exist_ok=True)
    so = os.path.join(LIB, "libscan3d_host.so")
    srcs = [os.path.join(HOST, s) for s in HOST_SOURCES if os.path.exists(os.path.join(HOST, s))]
    if not srcs:
        return None
    hdr = os.path.join(HERE, "..", "include", "scan3d.h")
    if not (force or _stale(so, _deps(HOST, [hdr]))):
        return so
    cmd = ["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-ffp-contract=off",
           "-fopenmp", "-I", os.path.join(HERE, "..", "include"), "-o", so] + srcs + ["-ldl"]
    subprocess.check_call(cmd)
    return so


def build_compat(force=False):
    """libscan3d_compat.so: the reference-named stage functions; links libscan3d.so + libscan3d_host.so."""
    so = os.path.join(LIB, "libscan3d_compat.so")
    srcs = [os.path.join(HOST, s) for s in COMPAT_SOURCES]
    deps = _deps(HOST, [os.path.join(HERE, "..", "include", h) for h in ("scan3d.h", "scan3d_host.h", "scan3d_compat.h")])
    if not (force or _stale(so, deps + [os.path.join(LIB, "libscan3d.so"), os.path.join(LIB, "libscan3d_host.so")])):
        return so
    cmd = ["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-ffp-contract=off",
           "-I", os.path.join(HERE, "..", "include"), "-o", so] + srcs + [
           "-L", LIB, "-lscan3d", "-lscan3d_host", "-Wl,-rpath,$ORIGIN"]
    subprocess.check_call(cmd)
    return so


def build_all(force=False, verbose=False):
    return build_cuda(force, verbose), build_host(force), build_compat(force)


if __name__ == "__main__":
    print(build_all(force="--force" in sys.argv, verbose=True))
