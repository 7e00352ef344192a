"""In-tree build of libictrack.so (nvcc, sm_100a only) and of the host-side C++ drivers.

    python -m invcompcamtrack_b200.build          # library + drivers
nvcc cross-compiles without a GPU; the resulting .so is git-ignored but travels with the repo snapshot.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libictrack.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
# -fmad=false: the reference is built without FMA (CMakeLists.txt:4), contraction would change its fp32 results
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-fmad=false", "-std=c++17",
              "-Xcompiler", "-fPIC", "-ccbin", "g++"] + os.environ.get("ICT_EXTRA_NVCC", "").split()
LIB_SOURCES = ["ict_kernels.cu", "ict_kernel_v2.cu", "ict_kernel_v8.cu", "ict_kernel_x.cu", "ict_kernel_x8.cu", "ict_kernel_r.cu", "ict_kernels_big.cu", "ict_patches.cu", "ict_hypotheses.cu", "ict_evaluate.cu", "ict_capi.cu"]
LIB_DEPS = LIB_SOURCES + ["ict_kernels.cuh", "ict_device.cuh", "ict_kernel_v2.cuh", "ict_kernel_v8.cuh", "ict_kernel_x.cuh", os.path.join("..", "..", "include", "ictrack.h")]


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build_library(force=False, verbose=False):
    """One object per translation unit (compiled in parallel, only the stale ones), then one link.  There is no
    relocatable device code: no kernel calls a device function of another unit."""
    deps = [os.path.join(CSRC, d) for d in LIB_DEPS]
    if not force and not _stale(LIB, deps):
        return LIB
    headers = [d for d in deps if not d.endswith(".cu")]
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    jobs = []
    for src in LIB_SOURCES:
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        if force or _stale(obj, [os.path.join(CSRC, src)] + headers):
            cmd = [NVCC] + NVCC_FLAGS + (["-Xptxas=-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
            jobs.append(cmd)
    if jobs:
        from concurrent.futures import ThreadPoolExecutor
        with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 1)) as ex:
            for r in ex.map(lambda c: subprocess.run(c, capture_output=not verbose, text=True), jobs):
                if r.returncode:
                    raise RuntimeError("nvcc failed:\n%s\n%s" % (" ".join(r.args), (r.stderr or "")[-4000:]))
    objs = [os.path.join(objdir, src.replace(".cu", ".o")) for src in LIB_SOURCES]
    subprocess.run([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", LIB] + objs, check=True)
    return LIB


def build_drivers(force=False):
    """run_track / run_track_nposes: host C++ (reference class interface) linked against libictrack.so."""
    host = os.path.join(CSRC, "host")
    out = []
    for name in ("run_track", "run_track_nposes"):
        src = os.path.join(host, name + ".cpp")
        if not os.path.exists(src):
            continue
        exe = os.path.join(HERE, "bin", name)
        deps = [src] + [os.path.join(host, f) for f in os.listdir(host)] + [LIB]
        if force or _stale(exe, deps):
            os.makedirs(os.path.dirname(exe), exist_ok=True)
            srcs = [src] + [os.path.join(host, f) for f in ("camera.cpp", "pose.cpp", "odometer.cpp", "utilities.cpp")]
            subprocess.run(["g++", "-O2", "-std=c++14", "-I", host, "-I", os.path.join(HERE, "..", "include"), "-o", exe]
                           + srcs + ["-L", HERE, "-lictrack", "-Wl,-rpath," + HERE, "-Wl,-rpath,$ORIGIN/.."], check=True)
        out.append(exe)
    return out


if __name__ == "__main__":
    force = "--force" in sys.argv
    print(build_library(force=force, verbose="-v" in sys.argv))
    for e in build_drivers(force=force):
        print(e)
