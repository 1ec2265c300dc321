"""In-tree build of the CUDA extension (libabstract_gym_b200.so) for sm_100a.

nvcc cross-compiles without a GPU; the .so is git-ignored but travels with the gpurun snapshot.
Every translation unit is compiled to an object file in parallel, then linked.
Usage:  python -m abstract_gym_b200.build [--force] [--verbose] [--out PATH] [--debug]
--debug builds libabstract_gym_b200_debug.so with -DAG_DEBUG_BOUNDS (device-side index assertions; load it with
AG_LIB_PATH=<that file>); the release library is untouched.
"""
import concurrent.futures
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
INCLUDE = os.path.join(HERE, "..", "include")
LIB = os.environ.get("AG_LIB_PATH") or os.path.join(HERE, "libabstract_gym_b200.so")   # AG_LIB_PATH: A/B builds
SOURCES = ["ag_kernels.cu", "ag_rollout_lut.cu", "ag_cmap.cu", "ag_motion.cu", "ag_cspace.cu", "ag_host.cu"]
HEADERS = ["ag_device.cuh", "ag_fast.cuh", "ag_rollout.cuh", "ag_cmap.cuh", os.path.join(INCLUDE, "abstract_gym_b200.h")]
OBJDIR = os.path.join(HERE, "build")
DEBUG_LIB = os.path.join(HERE, "libabstract_gym_b200_debug.so")
# the compiled torch custom-op library (torch.ops.abstract_gym_b200.*): a C++ shim over the C ABI, linked against
# libabstract_gym_b200.so (rpath $ORIGIN) and the torch libraries of the running interpreter
OPS_LIB = os.path.join(HERE, "libabstract_gym_b200_ops.so")
OPS_SRC = os.path.join(CSRC, "ag_torch_ops.cpp")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC,-ffp-contract=off,-fvisibility=hidden",
    "-Xptxas", "-v",
]


def find_nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the CUDA extension cannot be built (there is no CPU fallback)")


def sources():
    return [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def _stale(lib) -> bool:
    t = os.path.getmtime(lib)
    deps = [os.path.join(CSRC, s) for s in sources()] + [h if os.path.isabs(h) else os.path.join(CSRC, h) for h in HEADERS]
    deps.append(os.path.abspath(__file__))
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def needs_build() -> bool:
    if os.environ.get("AG_LIB_PATH"):
        return False
    return not os.path.exists(LIB) or _stale(LIB)


def build_debug(force: bool = False, verbose: bool = False) -> str:
    """the -DAG_DEBUG_BOUNDS library (csrc/ag_device.cuh AG_CHECK_INDEX); tests/test_gpu_parity.py runs a subset on it"""
    if not force and os.path.exists(DEBUG_LIB) and not _stale(DEBUG_LIB):
        return DEBUG_LIB
    # -split-compile: the debug library's speed does not matter, its build time does (the release library is built
    # without it: split compilation changes the generated code slightly, and the measured numbers are the normal build's)
    return build(verbose=verbose, out=DEBUG_LIB, defines=["-DAG_DEBUG_BOUNDS", "-split-compile", "0"])


def build(force: bool = False, verbose: bool = False, out: str = None, defines=()) -> str:
    if out is None and not force and not needs_build():
        return LIB
    nvcc = find_nvcc()
    extra = os.environ.get("AG_NVCC_EXTRA", "").split() + list(defines)      # A/B builds, e.g. -DAG_LUT_B1=10
    env = {k: v for k, v in os.environ.items() if k not in ("CC", "CXX")}
    target = out or LIB
    objdir = OBJDIR if out is None else target + ".obj"
    os.makedirs(objdir, exist_ok=True)
    logs = {}

    def compile_one(src):
        obj = os.path.join(objdir, os.path.splitext(src)[0] + ".o")
        cmd = [nvcc] + NVCC_FLAGS + extra + ["-I", INCLUDE, "-c", "-o", obj, os.path.join(CSRC, src)]
        r = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        logs[src] = " ".join(cmd) + "\n" + r.stdout
        return r.returncode, obj

    with concurrent.futures.ThreadPoolExecutor(max_workers=len(sources())) as ex:
        results = list(ex.map(compile_one, sources()))
    rc = max(r for r, _ in results)
    link_out = ""
    if rc == 0:
        cmd = [nvcc, "--shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", target] + [o for _, o in results]
        r = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        rc, link_out = r.returncode, " ".join(cmd) + "\n" + r.stdout
    log = (out + ".log") if out else os.path.join(HERE, "build.log")
    text = "".join(logs[s] for s in sources()) + link_out
    with open(log, "w") as f:
        f.write(text)
    if verbose or rc != 0:
        sys.stderr.write(text)
    if rc != 0:
        raise RuntimeError("nvcc failed (%d); see %s" % (rc, log))
    return target


def ops_needs_build() -> bool:
    if not os.path.exists(OPS_LIB):
        return True
    t = os.path.getmtime(OPS_LIB)
    deps = [OPS_SRC, os.path.join(INCLUDE, "abstract_gym_b200.h"), os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build_ops(force: bool = False, verbose: bool = False) -> str:
    """g++ -shared csrc/ag_torch_ops.cpp -> libabstract_gym_b200_ops.so (needs libabstract_gym_b200.so: build() first)"""
    if not force and not ops_needs_build():
        return OPS_LIB
    build()
    import torch
    from torch.utils import cpp_extension as ce
    cxx = shutil.which("g++") or "g++"
    abi = int(getattr(torch._C, "_GLIBCXX_USE_CXX11_ABI", 1))
    cuda_home = os.environ.get("CUDA_HOME") or "/usr/local/cuda"
    cmd = [cxx, "-O2", "-std=c++17", "-fPIC", "-shared", "-fvisibility=hidden", "-D_GLIBCXX_USE_CXX11_ABI=%d" % abi,
           "-DTORCH_API_INCLUDE_EXTENSION_H"]
    for inc in ce.include_paths() + [os.path.join(cuda_home, "include"), INCLUDE]:
        cmd += ["-I", inc]
    cmd += [OPS_SRC, "-o", OPS_LIB]
    for d in ce.library_paths():
        cmd += ["-L", d]
    cmd += ["-L", HERE, "-L", os.path.join(cuda_home, "lib64"), "-lc10", "-lc10_cuda", "-ltorch_cpu", "-ltorch_cuda", "-ltorch",
            "-labstract_gym_b200", "-lcudart", "-Wl,-rpath,$ORIGIN"]
    env = {k: v for k, v in os.environ.items() if k not in ("CC", "CXX")}
    r = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    with open(os.path.join(HERE, "build_ops.log"), "w") as f:
        f.write(" ".join(cmd) + "\n" + r.stdout)
    if verbose or r.returncode != 0:
        sys.stderr.write(r.stdout)
    if r.returncode != 0:
        raise RuntimeError("g++ failed (%d) building the torch op library; see build_ops.log" % r.returncode)
    return OPS_LIB


if __name__ == "__main__":
    if "--debug" in sys.argv:
        print(build_debug(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
        sys.exit(0)
    out = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else None
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv, out=out))
    if out is None:
        print(build_ops(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
