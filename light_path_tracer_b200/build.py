"""In-tree build of the native code (explicit nvcc / g++ commands, no JIT cache).

    python -m light_path_tracer_b200.build [--force]

Produces, next to this file:
    _C/liblightpath.so     the C-ABI library (include/lightpath.h): CUDA kernels for sm_100a
    _C/_lp_torch.so        thin PyTorch C++ extension: tensors in, C-ABI calls out

Both are git-ignored but travel to the GPU box with the repo snapshot.
nvcc cross-compiles sm_100a without a GPU, so this runs in the build container.
"""
import os
import shutil
import subprocess
import sys
import sysconfig

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "_C")
INCLUDE = os.path.join(ROOT, "include")

LIB = os.path.join(OUT, "liblightpath.so")
EXT = os.path.join(OUT, "_lp_torch.so")

CU_SOURCES = ["lp_host.cu", "lp_trace.cu", "lp_repack.cu", "lp_peer.cu", "lp_remap.cu", "lp_shadow.cu", "lp_rk45.cu", "lp_kerr.cu"]
HEADERS = ["lp_internal.cuh", "lp_rk45_rhs.cuh", "lp_trace.cuh", "lp_remap.cuh", "lp_sincr.cuh", "lp_sintab.h", os.path.join(INCLUDE, "lightpath.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    # the reference's arithmetic has no fused multiply-add (SURVEY.md §2a): never let the
    # compiler contract; the kernels call fma() explicitly where a fused op is exact or opted in
    "-fmad=false",
    "-Xcompiler", "-fPIC,-O2,-ffp-contract=off",
    "-I" + INCLUDE,
]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def _run(cmd, verbose):
    if verbose:
        print(" ".join(cmd), flush=True)
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError("build command failed: " + " ".join(cmd))
    return res.stdout + res.stderr


def build_lib(force=False, verbose=False, ptxas_info=False):
    os.makedirs(OUT, exist_ok=True)
    srcs = [os.path.join(CSRC, s) for s in CU_SOURCES]
    deps = srcs + [h if os.path.isabs(h) else os.path.join(CSRC, h) for h in HEADERS] + [__file__]
    from concurrent.futures import ThreadPoolExecutor
    objs = [os.path.join(OUT, os.path.basename(s)[:-3] + ".o") for s in srcs]
    jobs = [[_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if ptxas_info else []) + ["-c", s, "-o", o]
            for s, o in zip(srcs, objs) if force or _stale(o, deps)]
    with ThreadPoolExecutor(max_workers=max(1, min(len(jobs), os.cpu_count() or 1))) as pool:
        log = "".join(pool.map(lambda cmd: _run(cmd, verbose), jobs))
    if force or _stale(LIB, objs):
        _run([_nvcc(), "-shared", "-o", LIB] + objs, verbose)
    return log


def build_ext(force=False, verbose=False):
    """g++ only: the extension holds no device code, it forwards tensors to the C ABI."""
    import torch
    from torch.utils import cpp_extension as ce
    src = os.path.join(CSRC, "lp_torch.cpp")
    if not (force or _stale(EXT, [src, os.path.join(INCLUDE, "lightpath.h"), LIB, __file__])):
        return
    inc = ce.include_paths() + [sysconfig.get_paths()["include"], INCLUDE]
    cuda_inc = os.path.join(os.path.dirname(os.path.dirname(_nvcc())), "include")
    torch_lib = os.path.join(os.path.dirname(torch.__file__), "lib")
    cmd = ["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-DTORCH_EXTENSION_NAME=_lp_torch",
           "-DTORCH_API_INCLUDE_EXTENSION_H", "-D_GLIBCXX_USE_CXX11_ABI=%d" % int(torch._C._GLIBCXX_USE_CXX11_ABI)]
    cmd += ["-I" + p for p in inc] + ["-I" + cuda_inc]
    cmd += [src, "-o", EXT, "-L" + OUT, "-llightpath", "-Wl,-rpath,$ORIGIN",
            "-L" + torch_lib, "-ltorch", "-ltorch_cpu", "-lc10", "-ltorch_python",
            "-Wl,-rpath," + torch_lib]
    if os.path.exists(os.path.join(torch_lib, "libc10_cuda.so")):
        cmd += ["-lc10_cuda", "-ltorch_cuda"]
    _run(cmd, verbose)


def build(force=False, verbose=False, ptxas_info=False):
    log = build_lib(force=force, verbose=verbose, ptxas_info=ptxas_info)
    build_ext(force=force, verbose=verbose)
    return log


if __name__ == "__main__":
    out = build(force="--force" in sys.argv, verbose=True, ptxas_info="--ptxas" in sys.argv)
    if "--ptxas" in sys.argv:
        print(out)
    print("built", LIB)
    print("built", EXT)
