"""In-tree native build for openembedding_b200.

Two shared libraries with a C ABI (the "narrow waist", like the reference's
``exb_*`` C API in openembedding/entry/c_api.h:32-145), loaded with ctypes:

* ``lib/libexb_core.so``  -- C++17 CPU engine + checkpoint IO (g++)
* ``lib/libexb_cuda.so``  -- sm_100a kernels + CUDA runtime glue (nvcc)

The libraries are built *in tree*, so a copy of the built tree carries them to
another machine; a content hash of sources+flags is stored next to each ``.so`` so an
up-to-date library is loaded without invoking the compiler and without writing to
the tree (which may be read-only after the build).
"""
import concurrent.futures
import hashlib
import os
import shutil
import subprocess
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(_HERE, "csrc")
_LIB = os.path.join(_HERE, "lib")
_OBJ = os.path.join(_HERE, "lib", "obj")

NVCC = os.environ.get("EXB_NVCC", "/usr/local/cuda/bin/nvcc")
CXX = os.environ.get("CXX", "g++")

CUDA_ARCH_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a"]
NVCC_FLAGS = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr",
              "-Xptxas", "-v"] + CUDA_ARCH_FLAGS
CXX_FLAGS = ["-O2", "-std=c++17", "-fPIC", "-Wall", "-Wextra", "-pthread"]


def _sources(sub, exts):
    d = os.path.join(_CSRC, sub)
    out = []
    for root, _, files in os.walk(d):
        for f in sorted(files):
            if f.endswith(exts):
                out.append(os.path.join(root, f))
    return sorted(out)


def _hash(files, flags):
    h = hashlib.sha256()
    h.update(" ".join(flags).encode())
    for f in files:
        h.update(os.path.relpath(f, _HERE).encode())   # location independent: the tree is copied to the GPU box
        with open(f, "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()


def _stamp_ok(lib, digest):
    st = lib + ".stamp"
    return os.path.exists(lib) and os.path.exists(st) and open(st).read().strip() == digest


def _run(cmd, log=None):
    p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if log is not None:
        with open(log, "w") as fh:
            fh.write(" ".join(cmd) + "\n" + p.stdout)
    if p.returncode != 0:
        sys.stderr.write(p.stdout)
        raise RuntimeError("native build failed: " + " ".join(cmd))
    return p.stdout


def core_lib_path():
    return os.path.join(_LIB, "libexb_core.so")


def cuda_lib_path():
    return os.path.join(_LIB, "libexb_cuda.so")


class _BuildLock:
    """inter-process lock: torchrun ranks must not compile the same library concurrently"""

    def __enter__(self):
        import fcntl
        os.makedirs(_LIB, exist_ok=True)
        self.fh = open(os.path.join(_LIB, ".build.lock"), "w")
        fcntl.flock(self.fh, fcntl.LOCK_EX)
        return self

    def __exit__(self, *a):
        import fcntl
        fcntl.flock(self.fh, fcntl.LOCK_UN)
        self.fh.close()


def _core_deps():
    return _sources("core", (".cpp",)) + _sources("core", (".h",))


def _cuda_deps():
    return _sources("cuda", (".cu",)) + _sources("cuda", (".cuh", ".h")) + _sources("core", (".h",))


# An up-to-date library is returned before the lock is taken: the lock file is opened for writing.
def build_core(force=False, verbose=False):
    if not force and _stamp_ok(core_lib_path(), _hash(_core_deps(), CXX_FLAGS)):
        return core_lib_path()
    with _BuildLock():
        return _build_core(force, verbose)


def build_cuda(force=False, verbose=False):
    if not force and _stamp_ok(cuda_lib_path(), _hash(_cuda_deps(), NVCC_FLAGS)):
        return cuda_lib_path()
    with _BuildLock():
        return _build_cuda(force, verbose)


def _build_core(force=False, verbose=False):
    os.makedirs(_LIB, exist_ok=True)
    srcs = _sources("core", (".cpp",))
    deps = _core_deps()
    digest = _hash(deps, CXX_FLAGS)
    lib = core_lib_path()
    if not force and _stamp_ok(lib, digest):
        return lib
    if shutil.which(CXX) is None:
        raise RuntimeError("no C++ compiler to build " + lib)
    tmp = lib + ".tmp%d" % os.getpid()
    _run([CXX] + CXX_FLAGS + ["-shared", "-o", tmp] + srcs, log=os.path.join(_LIB, "core_build.log"))
    os.replace(tmp, lib)
    with open(lib + ".stamp", "w") as fh:
        fh.write(digest)
    if verbose:
        print("built", lib)
    return lib


def _build_cuda(force=False, verbose=False):
    os.makedirs(_OBJ, exist_ok=True)
    srcs = _sources("cuda", (".cu",))
    deps = _cuda_deps()
    digest = _hash(deps, NVCC_FLAGS)
    lib = cuda_lib_path()
    if not force and _stamp_ok(lib, digest):
        return lib
    if not os.path.exists(NVCC):
        raise RuntimeError("nvcc not found and %s is stale/missing" % lib)
    inc = ["-I", os.path.join(_CSRC, "core"), "-I", os.path.join(_CSRC, "cuda")]

    def compile_one(src):
        obj = os.path.join(_OBJ, os.path.basename(src) + ".o")
        hd = _hash([src] + [d for d in deps if d.endswith((".cuh", ".h"))], NVCC_FLAGS)
        st = obj + ".stamp"
        if not force and os.path.exists(obj) and os.path.exists(st) and open(st).read() == hd:
            return obj
        _run([NVCC] + NVCC_FLAGS + inc + ["-c", src, "-o", obj], log=obj + ".log")
        with open(st, "w") as fh:
            fh.write(hd)
        return obj

    with concurrent.futures.ThreadPoolExecutor(max_workers=min(8, len(srcs) or 1)) as ex:
        objs = list(ex.map(compile_one, srcs))
    tmp = lib + ".tmp%d" % os.getpid()
    _run([NVCC, "-shared", "-o", tmp] + CUDA_ARCH_FLAGS + objs + ["-lcudart", "-lcuda"],
         log=os.path.join(_LIB, "cuda_link.log"))
    os.replace(tmp, lib)
    with open(lib + ".stamp", "w") as fh:
        fh.write(digest)
    if verbose:
        print("built", lib)
    return lib


def build_all(force=False, verbose=True):
    a = build_core(force=force, verbose=verbose)
    b = build_cuda(force=force, verbose=verbose)
    return a, b


def ptxas_report():
    """Concatenated ptxas -v output (registers / spills / smem) of the last build."""
    out = []
    if os.path.isdir(_OBJ):
        for f in sorted(os.listdir(_OBJ)):
            if f.endswith(".log"):
                out.append(open(os.path.join(_OBJ, f)).read())
    return "\n".join(out)


if __name__ == "__main__":
    build_all(force="--force" in sys.argv)
