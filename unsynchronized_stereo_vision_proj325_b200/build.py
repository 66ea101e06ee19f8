"""In-tree nvcc build of the sm_100a shared library (no JIT cache: the built
.so travels with the repo snapshot to the GPU box)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libusv_b200.so")
OBJ = os.path.join(HERE, "_obj")
MICROBENCH = os.path.join(HERE, "usv_microbench")
HOST_TEST = os.path.join(HERE, "usv_host_test")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["--threads", "0", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr", "-ccbin", "/usr/bin/g++"]

LIB_SOURCES = ["usv_capi.cu", "usv_direct.cu", "usv_dense.cu", "usv_dense_g8.cu", "usv_dense_colour.cu", "usv_dense_census.cu", "usv_dense_census_colour.cu", "usv_census.cu", "usv_distance.cu", "usv_probe.cu", "usv_contours.cu", "usv_resolve.cu", "usv_resolve_rows.cu", "usv_preprocess.cu", "usv_dense_corr.cu", "usv_dense_mma.cu", "usv_dense_umma.cu", "usv_subpixel.cu"]
HOST_SOURCES = ["host/Match.cpp", "host/SearchAlgorithms.cpp", "host/DistanceCalculator.cpp"]


def _newer(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def _run(cmd, verbose):
    if verbose:
        print(" ".join(cmd), flush=True)
    out = subprocess.run(cmd, capture_output=True, text=True)
    if out.returncode != 0:
        raise RuntimeError("build failed: %s\n%s\n%s" % (" ".join(cmd), out.stdout, out.stderr))
    if verbose and (out.stdout or out.stderr):
        print(out.stdout + out.stderr)
    return out.stdout + out.stderr


def build(force=False, verbose=False, ptxas_info=False):
    """Compile every CUDA source for sm_100a into libusv_b200.so (+ tools)."""
    logs = []
    hdrs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h", ".hpp"))]
    inc = os.path.join(HERE, "..", "include")
    hdrs += [os.path.join(inc, f) for f in os.listdir(inc)]
    srcs = [os.path.join(CSRC, s) for s in LIB_SOURCES]
    hosts = [os.path.join(CSRC, s) for s in HOST_SOURCES if os.path.exists(os.path.join(CSRC, s))]
    extra = ["-Xptxas", "-v"] if ptxas_info else []
    # one object per source (only the changed ones are recompiled, in parallel), then one link: no relocatable device
    # code crosses a file boundary
    os.makedirs(OBJ, exist_ok=True)
    todo = []
    objs = []
    for src in srcs + hosts:
        obj = os.path.join(OBJ, os.path.relpath(src, CSRC).replace(os.sep, "_") + ".o")
        objs.append(obj)
        if force or _newer(obj, [src] + hdrs):
            todo.append((src, obj))
    if todo:
        from concurrent.futures import ThreadPoolExecutor
        with ThreadPoolExecutor(max_workers=min(len(todo), os.cpu_count() or 4)) as ex:
            logs.extend(ex.map(lambda so: _run([NVCC] + ARCH + COMMON + extra + ["-c", "-I", inc, "-o", so[1], so[0]], verbose), todo))
    if todo or force or _newer(LIB, objs):
        logs.append(_run([NVCC] + ARCH + ["-shared", "-Xcompiler", "-fPIC", "-ccbin", "/usr/bin/g++", "-o", LIB] + objs, verbose))
    mb = os.path.join(CSRC, "usv_microbench.cu")
    if os.path.exists(mb) and (force or _newer(MICROBENCH, [mb])):
        logs.append(_run([NVCC] + ARCH + COMMON + ["-o", MICROBENCH, mb], verbose))
    ht = os.path.join(CSRC, "host", "usv_host_test.cpp")
    if os.path.exists(ht) and (force or _newer(HOST_TEST, [ht, LIB] + hdrs)):
        logs.append(_run([NVCC] + ARCH + COMMON + ["-I", inc, "-o", HOST_TEST, ht, "-L", HERE, "-lusv_b200",
                                                   "-Xlinker", "-rpath", "-Xlinker", "$ORIGIN"], verbose))
    return "\n".join(logs)


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True, ptxas_info="--ptxas" in sys.argv))
