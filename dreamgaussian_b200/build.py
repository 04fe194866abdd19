"""Build recipe of libdgr_b200.so: one nvcc invocation, sm_100a only, in-tree output (dreamgaussian_b200/lib/).

No torch headers are involved: the library is a plain C-ABI CUDA shared object (include/dgr_b200.h).
nvcc cross-compiles on a machine without a GPU, so this runs in CI and in __graft_entry__.build().
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_DIR = os.path.join(HERE, "lib")
LIB_PATH = os.path.join(LIB_DIR, "libdgr_b200.so")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17", "-shared", "-Xcompiler", "-fPIC",
    "--expt-relaxed-constexpr", "-Xptxas", "-v", "-ldl",
]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (needed to build libdgr_b200.so)")


def sources():
    return sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh"))) + [
        os.path.join(HERE, "..", "include", "dgr_b200.h"), os.path.join(HERE, "..", "include", "dgr_constants.h")]


HASH_PATH = os.path.join(LIB_DIR, "libdgr_b200.srchash")


def source_hash():
    import hashlib
    h = hashlib.sha256(" ".join(NVCC_FLAGS).encode())
    for s in sources():
        with open(s, "rb") as f:
            h.update(os.path.basename(s).encode() + b"\0" + f.read())
    return h.hexdigest()


STEP_SOURCES = ("dgr_common.cuh", "dgr_preprocess.cuh", "dgr_binning.cuh", "dgr_render.cuh", "dgr_backward.cuh", "dgr_api.cu")


def step_kernel_hash():
    """Hash of what determines the kernels of ONE forward+backward step (their sources, the launcher, the constants, the compiler
    flags) — the stamp profiles/r2_ncu_kernels.json carries.  The collective, k-NN, field, optimiser and densification kernels are
    not in that capture and do not invalidate it."""
    import hashlib
    h = hashlib.sha256(" ".join(NVCC_FLAGS).encode())
    for name in STEP_SOURCES + ("dgr_constants.h",):
        path = os.path.join(CSRC, name) if not name.endswith(".h") else os.path.join(HERE, "..", "include", name)
        with open(path, "rb") as f:
            h.update(name.encode() + b"\0" + f.read())
    return h.hexdigest()


def is_stale():
    """Content-hash based (mtimes do not survive a repo snapshot to another machine)."""
    if not os.path.exists(LIB_PATH) or not os.path.exists(HASH_PATH):
        return True
    with open(HASH_PATH) as f:
        return f.read().strip() != source_hash()


def build(force=False, verbose=False):
    """Compile dreamgaussian_b200/csrc/dgr_lib.cu (dgr_api.cu + the batched multi-view entry points) ->
    dreamgaussian_b200/lib/libdgr_b200.so. Returns the path."""
    if not force and not is_stale():
        return LIB_PATH
    os.makedirs(LIB_DIR, exist_ok=True)
    cmd = [_nvcc()] + NVCC_FLAGS + ["-o", LIB_PATH, os.path.join(CSRC, "dgr_lib.cu")]
    # the image's CC may point at a gcc without a usable spec dir; the system compiler is the host compiler
    if os.path.exists("/usr/bin/g++"):
        cmd += ["-ccbin", "/usr/bin/g++"]
    proc = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    log = proc.stdout
    with open(os.path.join(LIB_DIR, "build.log"), "w") as f:
        f.write(" ".join(cmd) + "\n" + log)
    if proc.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + log[-8000:])
    with open(HASH_PATH, "w") as f:
        f.write(source_hash())
    if verbose:
        print(log)
    return LIB_PATH


# ---- the compiled PyTorch host layer over the C ABI (csrc/dgr_torch.cpp): g++ only, links libdgr_b200.so
HOST_PATH = os.path.join(LIB_DIR, "dgr_torch_host.so")
HOST_HASH = os.path.join(LIB_DIR, "dgr_torch_host.srchash")


def _host_hash():
    import hashlib
    import torch
    h = hashlib.sha256(torch.__version__.encode())
    for s in (os.path.join(CSRC, "dgr_torch.cpp"), os.path.join(HERE, "..", "include", "dgr_b200.h")):
        with open(s, "rb") as f:
            h.update(f.read())
    return h.hexdigest()


def build_host(force=False):
    """g++ csrc/dgr_torch.cpp -> lib/dgr_torch_host.so (pybind11 module `dgr_torch_host`).  Returns the path."""
    build()
    if not force and os.path.exists(HOST_PATH) and os.path.exists(HOST_HASH) and open(HOST_HASH).read().strip() == _host_hash():
        return HOST_PATH
    import sysconfig
    import torch
    from torch.utils import cpp_extension as ce
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    inc = ce.include_paths() + [sysconfig.get_paths()["include"], "/usr/local/cuda/include"]
    libdirs = ce.library_paths()
    cmd = [cxx, "-O2", "-std=c++17", "-fPIC", "-shared", "-DTORCH_EXTENSION_NAME=dgr_torch_host", "-DTORCH_API_INCLUDE_EXTENSION_H",
           "-D_GLIBCXX_USE_CXX11_ABI=%d" % int(torch._C._GLIBCXX_USE_CXX11_ABI), "-w",
           os.path.join(CSRC, "dgr_torch.cpp"), "-o", HOST_PATH]
    cmd += ["-I" + i for i in inc] + ["-L" + d for d in libdirs] + ["-L" + LIB_DIR]
    cmd += ["-ltorch", "-ltorch_cpu", "-lc10", "-ltorch_python", "-lc10_cuda", "-ltorch_cuda", "-ldgr_b200", "-Wl,-rpath,$ORIGIN"]
    cmd += ["-Wl,-rpath," + d for d in libdirs]
    proc = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    with open(os.path.join(LIB_DIR, "build_host.log"), "w") as f:
        f.write(" ".join(cmd) + "\n" + proc.stdout)
    if proc.returncode != 0:
        raise RuntimeError("g++ failed on dgr_torch.cpp:\n" + proc.stdout[-6000:])
    with open(HOST_HASH, "w") as f:
        f.write(_host_hash())
    return HOST_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
    print(build_host(force="--force" in sys.argv))
